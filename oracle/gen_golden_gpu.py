#!/usr/bin/env python
"""Generate the golden fixture that needs the REAL LightX2V reference on a GPU (oracle tooling, not product code).

One Wan-14B-width DiT block (D = 5120, 40 heads, F = 13824) over a 21x6x10 grid = 1260 tokens, run by the reference's own
WanTransformerWeights + WanTransformerInfer with their stock GPU ops (torch.addmm, torch layer_norm, the bf16 RMSNorm fallback,
fp64 RoPE, flash_attn_varlen_func) on the seeded weights / inputs of oracle/wan_oracle.py.  The full output (1260 x 5120 bf16,
13 MB) is too large to commit, so a fixed seeded sample of 16 rows is stored with the row indices;
tests/test_gpu_reference_dropin.py compares the CUDA path and the oracle restatement with it.

    LIGHTX2V_REFERENCE=<LightX2V checkout> python oracle/gen_golden_gpu.py [OUT_DIR]     # default OUT_DIR: tests/golden
"""
import os
import sys

import torch
from safetensors.torch import save_file

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import ref_loader as R  # noqa: E402
from oracle import wan_oracle as O  # noqa: E402

NAME = "wan14b_block_reference_gpu"
DIM, HEADS, FFN, GRID = 5120, 40, 13824, (21, 6, 10)
ROWS, ROW_SEED, WEIGHTS_SEED, INPUTS_SEED = 16, 0, 1, 2


def main(out_dir):
    assert torch.cuda.is_available(), "the reference's GPU path needs a GPU"
    assert R.import_reference(), f"LightX2V reference not importable: {R._state}"
    from lightx2v.models.networks.wan.infer.transformer_infer import WanTransformerInfer as RefInfer
    from lightx2v.models.networks.wan.weights.transformer_weights import WanTransformerWeights as RefWeights

    S = GRID[0] * GRID[1] * GRID[2]
    W = O.synth_block_weights(1, DIM, FFN, seed=WEIGHTS_SEED, device="cuda")
    x, embed0, context = O.synth_block_inputs(S, DIM, seed=INPUTS_SEED, device="cuda")
    freqs = O.wan_freqs_table(DIM // HEADS).cuda()
    rcfg = R.ref_config(DIM, HEADS, FFN, 1, "t2v", mm_type=None, attn_type="flash_attn2")
    rw = RefWeights(rcfg)
    rw.load(W)
    want = RefInfer(rcfg).infer(rw, torch.tensor([GRID]), None, x.clone(), embed0, torch.tensor([S], device="cuda"), freqs, context)
    rest = O.infer_blocks(W, 1, x.clone(), embed0, GRID, freqs, context, HEADS, attn="flash_attn2")
    torch.cuda.synchronize()
    assert torch.equal(rest, want), "oracle restatement differs from the real reference classes on the GPU"
    rows = torch.randperm(S, generator=torch.Generator().manual_seed(ROW_SEED))[:ROWS].sort().values
    meta = {"dim": str(DIM), "heads": str(HEADS), "ffn": str(FFN), "grid": ",".join(map(str, GRID)), "weights_seed": str(WEIGHTS_SEED),
            "inputs_seed": str(INPUTS_SEED), "device": torch.cuda.get_device_name(0), "torch": torch.__version__,
            "source": "LightX2V WanTransformerInfer, stock GPU ops (mm Default, flash_attn2)"}
    os.makedirs(out_dir, exist_ok=True)
    path = os.path.join(out_dir, NAME + ".safetensors")
    save_file({"rows": rows, "x_out_rows": want[rows.to(want.device)].cpu().contiguous()}, path, metadata=meta)
    print(NAME, tuple(want.shape), want.dtype, "absmax", float(want.float().abs().max()), "bytes", os.path.getsize(path))


if __name__ == "__main__":
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(ROOT, "tests", "golden"))
