"""The drop-in claim exercised against the REAL LightX2V classes (the package found by oracle/ref_loader.py: the build under
oracle/_ref made by oracle/build_ref.py, or the checkout named by LIGHTX2V_REFERENCE; (a) and (b) skip when it is absent):
  (a) `install_into_lightx2v()` registers the B200 ops into the reference's own registries; the reference's OWN WanTransformerWeights
      + WanTransformerInfer, configured with mm_type "B200-bf16" and attention type "b200_fmha", run over libb200dit.so and must
      reproduce the committed fixture (which the same reference classes produced on CPU with torch ops);
  (b) the reference's stock weight tree (mm "Default", flash_attn2) is fed to the B200 infer class;
  (c) the reference's stock GPU path (torch.addmm + flash_attn2, its own classes end to end) vs the B200 infer class on identical
      inputs at 14B width: rtol = atol = 1e-2 (north_star), admitted one-ulp fraction stated and recorded.  The reference's output is
      the committed fixture tests/golden/wan14b_block_reference_gpu.safetensors (oracle/gen_golden_gpu.py), so (c) needs no reference."""
import os

import pytest
import torch
from safetensors import safe_open

from oracle import ref_loader as R
from oracle import wan_oracle as O

pytestmark = pytest.mark.gpu
needs_reference = pytest.mark.skipif(not R.available(), reason="LightX2V reference package not present (LIGHTX2V_REFERENCE unset)")


def _load(path):
    with safe_open(path, framework="pt") as f:
        return {k: f.get_tensor(k) for k in f.keys()}, f.metadata()


def _bad_frac(got, ref, rtol=1e-2, atol=1e-2):
    got, ref = got.float().cpu(), ref.float().cpu()
    return ((got - ref).abs() > atol + rtol * ref.abs()).float().mean().item(), (got - ref).abs().max().item()


@pytest.fixture(scope="module")
def ref():
    assert R.import_reference(), R._state
    return R


@pytest.fixture
def installed(ref):
    """The plugin installed into the reference's registries for the duration of one test (the hard-coded norm keys are restored after)."""
    from lightx2v_b200.host import registry

    assert registry.install_into_lightx2v() is True
    yield ref
    registry.uninstall_from_lightx2v()


@needs_reference
@pytest.mark.parametrize("name", ["wan13b_t2v_2blocks", "wan13b_i2v_1block"])
def test_reference_infer_and_weight_classes_over_b200_ops(installed, golden_dir, name, record):
    from lightx2v.models.networks.wan.infer.transformer_infer import WanTransformerInfer as RefInfer
    from lightx2v.models.networks.wan.weights.transformer_weights import WanTransformerWeights as RefWeights
    from lightx2v.utils.registry_factory import ATTN_WEIGHT_REGISTER, MM_WEIGHT_REGISTER, RMS_WEIGHT_REGISTER

    from lightx2v_b200.host import ops

    assert MM_WEIGHT_REGISTER["B200-bf16"] is ops.MMWeightB200 and ATTN_WEIGHT_REGISTER["b200_fmha"] is ops.FmhaWeightB200
    assert RMS_WEIGHT_REGISTER["sgl-kernel"] is ops.RMSWeightB200
    T, meta = _load(os.path.join(golden_dir, name + ".safetensors"))
    dim, heads, ffn, L, task = int(meta["dim"]), int(meta["heads"]), int(meta["ffn"]), int(meta["layers"]), meta["task"]
    cfg = R.ref_config(dim, heads, ffn, L, task, mm_type="B200-bf16", attn_type="b200_fmha")
    W = {k: v.cuda() for k, v in O.synth_block_weights(L, dim, ffn, task=task, seed=int(meta["weights_seed"])).items()}
    weights = RefWeights(cfg)
    weights.load(W)
    blk = weights.blocks[0].compute_phases
    assert type(blk[1].self_attn_q) is ops.MMWeightB200 and type(blk[1].self_attn_1) is ops.FmhaWeightB200 and type(blk[1].norm1) is ops.LNWeightB200
    infer = RefInfer(cfg)
    x = T["x_in"].cuda().clone()
    out = infer.infer(weights, T["grid"].view(1, 3), None, x, T["embed0"].cuda(), torch.tensor([x.shape[0]]), O.wan_freqs_table(dim // heads).cuda(), T["context"].cuda())
    torch.cuda.synchronize()
    frac, mx = _bad_frac(out, T["x_out"])
    print(f"reference classes over B200 ops, {name}: bad_frac={frac:.3e} max_abs_err={mx:.4f}")
    record(bad_frac=frac, max_abs_err=mx)
    assert frac < 1e-3 and mx < 0.07, (frac, mx)


@needs_reference
def test_reference_weight_tree_feeds_the_b200_infer_class(ref, golden_dir, record):
    from lightx2v.models.networks.wan.weights.transformer_weights import WanTransformerWeights as RefWeights

    from lightx2v_b200.host.wan_infer import WanTransformerInfer

    T, meta = _load(os.path.join(golden_dir, "wan13b_t2v_2blocks.safetensors"))
    dim, heads, ffn, L = int(meta["dim"]), int(meta["heads"]), int(meta["ffn"]), int(meta["layers"])
    cfg = R.ref_config(dim, heads, ffn, L, "t2v", mm_type=None, attn_type="flash_attn2")            # the reference's stock op classes
    W = {k: v.cuda() for k, v in O.synth_block_weights(L, dim, ffn, seed=int(meta["weights_seed"])).items()}
    weights = RefWeights(cfg)
    weights.load(W)
    sa = weights.blocks[0].compute_phases[1]
    assert type(sa.self_attn_q).__module__.startswith("lightx2v.") and type(sa.self_attn_norm_q).__module__.startswith("lightx2v.") and type(sa.norm1).__module__.startswith("lightx2v.")
    infer = WanTransformerInfer(dict(task="t2v", num_layers=L, num_heads=heads, dim=dim, ffn_dim=ffn, mm_config={}))
    x = T["x_in"].cuda().clone()
    out = infer.infer(weights, T["grid"].view(1, 3), None, x, T["embed0"].cuda(), torch.tensor([x.shape[0]]), O.wan_freqs_table(dim // heads), T["context"].cuda())
    torch.cuda.synchronize()
    frac, mx = _bad_frac(out, T["x_out"])
    record(bad_frac=frac, max_abs_err=mx)
    assert frac < 5e-4 and mx < 0.07, (frac, mx)


def test_b200_infer_vs_the_references_own_gpu_path(golden_dir, record):
    """One 14B-width block, 21x6x10 = 1260 tokens: the reference's classes with their stock GPU ops (torch.addmm, torch layer_norm,
    the bf16 RMSNorm fallback, fp64 RoPE, flash_attn_varlen_func; stored as a seeded sample of 16 output rows) against the B200 infer
    class on the same weights and inputs."""
    from lightx2v_b200.host.wan_infer import WanTransformerInfer
    from lightx2v_b200.host.wan_weights import WanTransformerWeights

    T, meta = _load(os.path.join(golden_dir, "wan14b_block_reference_gpu.safetensors"))
    dim, heads, ffn = int(meta["dim"]), int(meta["heads"]), int(meta["ffn"])
    grid = tuple(int(v) for v in meta["grid"].split(","))
    S = grid[0] * grid[1] * grid[2]
    rows, want = T["rows"].cuda(), T["x_out_rows"]
    W = O.synth_block_weights(1, dim, ffn, seed=int(meta["weights_seed"]), device="cuda")
    x, embed0, context = O.synth_block_inputs(S, dim, seed=int(meta["inputs_seed"]), device="cuda")
    freqs = O.wan_freqs_table(dim // heads)
    cfg = dict(task="t2v", num_layers=1, num_heads=heads, dim=dim, ffn_dim=ffn, mm_config={})
    weights = WanTransformerWeights(cfg)
    weights.load(W)
    got = WanTransformerInfer(cfg).infer(weights, torch.tensor([grid]), None, x.clone(), embed0, None, freqs, context)
    torch.cuda.synchronize()
    # the oracle restatement must be the reference's GPU path bit for bit (same ops in the same order)
    rest = O.infer_blocks(W, 1, x.clone(), embed0, grid, freqs.cuda(), context, heads, attn="flash_attn2")
    assert torch.equal(rest[rows].cpu(), want), "oracle restatement differs from the real reference classes on the GPU"
    frac, mx = _bad_frac(got[rows], want)
    print(f"B200 infer vs the reference's own GPU path (14B width): bad_frac={frac:.3e} max_abs_err={mx:.4f}")
    record(bad_frac=frac, max_abs_err=mx)
    assert frac < 1e-3 and mx < 0.07, (frac, mx)
