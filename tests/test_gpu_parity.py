"""GPU (-m gpu): the CUDA path, called through the C ABI (ctypes), against the CPU oracle on the same
seeded inputs and against the committed golden fixtures.  Tolerances: bf16 tensor-core operands ->
rel-L2 <= 1e-2 per op / 2e-2 per DiT forward; fp32 kernels <= 1e-5; rendered pixels <= 1e-3
(north_star); integer bookkeeping bit-exact where the float inputs are identical."""
import os

import numpy as np
import pytest
import torch
import torch.nn.functional as F

pytestmark = pytest.mark.gpu


def _rel(a, b):
    a, b = torch.as_tensor(a).double().cpu(), torch.as_tensor(b).double().cpu()
    return ((a - b).norm() / b.norm()).item()


@pytest.fixture(scope="module")
def dev():
    assert torch.cuda.is_available(), "-m gpu tests need a GPU"
    from ln3diff_b200 import _lib
    _lib.lib()  # fail loudly if the CUDA extension is missing
    return torch.device("cuda", 0)


# ------------------------------------------------------------------ GEMM
@pytest.mark.parametrize("M,N,K", [(128, 128, 64), (256, 512, 1024), (1232, 1024, 768), (16, 6144, 1024),
                                   (77, 256, 128), (3000, 3072, 1024)])
def test_gemm_bf16(dev, M, N, K):
    from ln3diff_b200 import ops
    g = torch.Generator().manual_seed(M + N + K)
    a = (torch.randn(M, K, generator=g) * 0.5).bfloat16()
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16()
    b = torch.randn(N, generator=g)
    ref = a.float() @ w.float().t() + b
    out = ops.gemm(a.to(dev), w.to(dev), b.to(dev))
    assert _rel(out, ref) < 4e-3                       # bf16 output rounding only
    out32 = ops.gemm(a.to(dev), w.to(dev), b.to(dev), out_kind=ops.OUT_F32)
    assert _rel(out32, ref) < 1e-5                     # fp32 accumulate in TMEM


@pytest.mark.parametrize("M,N,K", [(12288, 1024, 4096), (6144, 1024, 1024), (616, 768, 768), (2000, 1024, 64),
                                   (12288, 1024, 1024), (300, 512, 128)])
def test_gemm_bf16_narrow_tile_shapes(dev, M, N, K):
    """Shapes around the host cost model's choice between 256- and 192-column tiles of the CTA-pair GEMM (6 column tiles
    per 1024 columns, the last one 64 wide; ragged M): compared element-wise -- a column-addressing slip would not show
    in a norm."""
    from ln3diff_b200 import ops
    g = torch.Generator().manual_seed(M + 3 * N + K)
    a = (torch.randn(M, K, generator=g) * 0.5).bfloat16()
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16()
    b = torch.randn(N, generator=g)
    ref = a.float() @ w.float().t() + b
    out = ops.gemm(a.to(dev), w.to(dev), b.to(dev)).float().cpu()
    assert _rel(out, ref) < 4e-3
    err = (out - ref).abs() / (ref.abs() + 1.0)
    assert float(err.max()) < 2e-2, (float(err.max()), torch.nonzero(err > 2e-2)[:5])
    nob = ops.gemm(a.to(dev), w.to(dev)).float().cpu()           # no bias
    assert _rel(nob, ref - b) < 4e-3


def test_gemm_epilogues(dev):
    from ln3diff_b200 import ops
    g = torch.Generator().manual_seed(5)
    M, N, K = 1536, 1024, 512
    a = (torch.randn(M, K, generator=g) * 0.5).bfloat16()
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16()
    b = torch.randn(N, generator=g)
    lin = a.float() @ w.float().t() + b
    for act, fn in ((ops.ACT_GELU_ERF, F.gelu), (ops.ACT_GELU_TANH, lambda v: F.gelu(v, approximate="tanh")),
                    (ops.ACT_SILU, F.silu)):
        out = ops.gemm(a.to(dev), w.to(dev), b.to(dev), act=act, out_kind=ops.OUT_F32)
        assert _rel(out, fn(lin)) < 1e-5
    x0 = torch.randn(M, N, generator=g)
    gate = torch.randn(2, N, generator=g)
    x = x0.clone().to(dev)
    xb = torch.empty(M, N, dtype=torch.bfloat16, device=dev)
    ops.gemm(a.to(dev), w.to(dev), b.to(dev), out_kind=ops.OUT_RESID_F32, out=x, gate=gate.to(dev),
             gate_rows=768, out2=xb)
    ref = x0 + gate.repeat_interleave(768, 0) * lin
    assert _rel(x, ref) < 1e-5 and _rel(xb, ref) < 4e-3


def test_gemm_rejects_bad_shapes(dev):
    from ln3diff_b200 import ops
    a = torch.zeros(128, 96, dtype=torch.bfloat16, device=dev)
    w = torch.zeros(128, 96, dtype=torch.bfloat16, device=dev)
    with pytest.raises(RuntimeError, match="multiple of 64"):
        ops.gemm(a, w)


# ------------------------------------------------------------------ attention
# (1,1,384,96) / (1,1,385,97): exactly one 384-row work item and one 96-row KV block, and one row / key past
# them; (5,3,129,191): ragged everywhere; (16,16,768,768), (24,16,256,256), (8,16,768,768): the DiT self-attention
# and decoder in-plane / global shapes -- on 148 SMs the first ends in a round of 68 items, which runs on the
# (2 tiles | 1 tile) tail schedule, and the in-plane shape has a ragged last KV block and an empty third tile
@pytest.mark.parametrize("B,H,Lq,Lkv", [(2, 12, 768, 768), (2, 16, 768, 77), (1, 4, 200, 333),
                                        (2, 16, 768, 1024), (3, 16, 256, 256), (1, 2, 1, 1),
                                        (13, 16, 768, 768), (16, 16, 700, 77), (9, 16, 300, 130),
                                        (1, 1, 384, 96), (1, 1, 385, 97), (5, 3, 129, 191),
                                        (16, 16, 768, 768), (24, 16, 256, 256), (8, 16, 768, 768)])
def test_fmha(dev, B, H, Lq, Lkv):
    from ln3diff_b200 import ops
    g = torch.Generator().manual_seed(Lq * 7 + Lkv)
    D = H * 64
    qkv = torch.randn(B, max(Lq, Lkv), 3 * D, generator=g).bfloat16()
    q, k, v = qkv[:, :Lq, :D], qkv[:, :Lkv, D:2 * D], qkv[:, :Lkv, 2 * D:]
    dq = qkv.to(dev)
    out = ops.fmha(dq[:, :Lq, :D], dq[:, :Lkv, D:2 * D], dq[:, :Lkv, 2 * D:], H)
    qf, kf, vf = (t.float().reshape(B, -1, H, 64).transpose(1, 2) for t in (q, k, v))
    ref = F.scaled_dot_product_attention(qf, kf, vf).transpose(1, 2).reshape(B, Lq, D)
    assert _rel(out, ref) < 6e-3


def test_fmha_peaked_scores(dev):
    """Inputs 3x the unit scale make later KV blocks exceed the running row maximum by more than the lazy-rescale
    threshold (2^8), so blocks are redone against the new maximum and O is rescaled in tensor memory."""
    from ln3diff_b200 import ops
    g = torch.Generator().manual_seed(5)
    B, H, L = 2, 4, 768
    D = H * 64
    qkv = (torch.randn(B, L, 3 * D, generator=g) * 3.0).bfloat16()
    dq = qkv.to(dev)
    out = ops.fmha(dq[:, :, :D], dq[:, :, D:2 * D], dq[:, :, 2 * D:], H)
    qf, kf, vf = (t.float().reshape(B, -1, H, 64).transpose(1, 2) for t in (qkv[:, :, :D], qkv[:, :, D:2 * D],
                                                                            qkv[:, :, 2 * D:]))
    ref = F.scaled_dot_product_attention(qf, kf, vf).transpose(1, 2).reshape(B, L, D)
    assert _rel(out, ref) < 8e-3


# second K/V source appended after the first: a ragged first source (its last block is masked like a final
# one) and the I23D shape (768 latent + 256 DINO tokens)
@pytest.mark.parametrize("B,H,Lq,L1,L2", [(2, 4, 200, 256, 77), (1, 2, 100, 100, 50), (2, 16, 768, 768, 256)])
def test_fmha_second_kv(dev, B, H, Lq, L1, L2):
    from ln3diff_b200 import ops
    g = torch.Generator().manual_seed(17 + L1)
    D = H * 64
    q = torch.randn(B, Lq, D, generator=g).bfloat16()
    k1, v1 = torch.randn(B, L1, D, generator=g).bfloat16(), torch.randn(B, L1, D, generator=g).bfloat16()
    k2, v2 = torch.randn(B, L2, D, generator=g).bfloat16(), torch.randn(B, L2, D, generator=g).bfloat16()
    out = ops.fmha(q.to(dev), k1.to(dev), v1.to(dev), H, k2=k2.to(dev), v2=v2.to(dev))
    sp = lambda t_: t_.float().reshape(B, -1, H, 64).transpose(1, 2)
    ref = F.scaled_dot_product_attention(sp(q), sp(torch.cat([k1, k2], 1)), sp(torch.cat([v1, v2], 1)))
    assert _rel(out, ref.transpose(1, 2).reshape(B, Lq, D)) < 6e-3


# ------------------------------------------------------------------ elementwise
def test_norm_modulate_timestep_patch_final(dev):
    from ln3diff_b200 import ops
    from ln3diff_b200._lib import NORM_LAYER, NORM_NONE, NORM_RMS
    from oracle import dit as odit
    g = torch.Generator().manual_seed(9)
    x = torch.randn(300, 1024, generator=g) * 2 + 0.5
    sh = torch.randn(3, 6 * 1024, generator=g)
    out = ops.norm_modulate(x.to(dev), norm=NORM_LAYER, shift=sh.to(dev)[:, 0:1024], scale=sh.to(dev)[:, 1024:2048],
                            mod_rows=100)
    ref = odit.layer_norm(x) * (1 + sh[:, 1024:2048].repeat_interleave(100, 0)) + sh[:, :1024].repeat_interleave(100, 0)
    assert _rel(out, ref) < 4e-3
    w = torch.randn(768, generator=g)
    x7 = torch.randn(77, 768, generator=g)
    assert _rel(ops.norm_modulate(x7.to(dev), norm=NORM_RMS, weight=w.to(dev), eps=1e-5), odit.rms_norm(x7, w)) < 4e-3
    assert _rel(ops.norm_modulate(x7.to(dev), norm=NORM_NONE, act=ops.ACT_SILU), F.silu(x7)) < 4e-3
    t = torch.tensor([0.0, 1.0, 17.0, 999.0, 0.37])
    assert _rel(ops.timestep_embedding(t.to(dev)), odit.timestep_embedding(t)) < 4e-3
    sd = {"x_embedder.proj.weight": torch.randn(768, 4, 2, 2, generator=g), "x_embedder.proj.bias": torch.randn(768, generator=g)}
    xin, pos = torch.randn(2, 12, 32, 32, generator=g), torch.randn(1, 768, 768, generator=g)
    out = ops.patch_embed(xin.to(dev), sd["x_embedder.proj.weight"].to(dev), sd["x_embedder.proj.bias"].to(dev), pos.to(dev))
    assert _rel(out, odit.patch_embed_rollout(sd, xin) + pos) < 1e-6
    tok = torch.randn(2, 768, 768, generator=g)
    shift, scale = torch.randn(2, 768, generator=g), torch.randn(2, 768, generator=g)
    wf, bfin = torch.randn(16, 768, generator=g) * 0.05, torch.randn(16, generator=g)
    ref = odit.unpatchify_rollout(F.linear(odit.layer_norm(tok) * (1 + scale[:, None]) + shift[:, None], wf, bfin), 4)
    out = ops.final_layer(tok.to(dev), shift.to(dev), scale.to(dev), wf.to(dev), bfin.to(dev), 32)
    assert _rel(out, ref) < 1e-5


def test_sampler_update_kernel(dev):
    from ln3diff_b200 import ops
    g = torch.Generator().manual_seed(2)
    x, m0, m1, nz = (torch.randn(3, 12, 32, 32, generator=g) for _ in range(4))
    cf = torch.randn(3, 4, generator=g)
    c = cf[:, :, None, None, None]
    ref = c[:, 0] * x + c[:, 1] * m0 + c[:, 2] * m1 + c[:, 3] * nz
    out = ops.sampler_affine_update(x.to(dev), cf.to(dev), m0.to(dev), m1.to(dev), nz.to(dev))
    assert _rel(out, ref) < 1e-6
    out = ops.sampler_affine_update(x.to(dev), cf.to(dev), m0.to(dev))
    assert _rel(out, c[:, 0] * x + c[:, 1] * m0) < 1e-6


# ------------------------------------------------------------------ DiT forward + samplers
def test_dit_forward_matches_reference_golden(dev, golden):
    """CUDA DiT-B/2 forward vs the REFERENCE's own output (tests/golden/dit_t23d.npz)."""
    from ln3diff_b200.dit.dit_models_xformers import TextCondDiTBlock
    from ln3diff_b200.dit.dit_trilatent import DiT_models
    from oracle import dit as odit
    from oracle import fixtures as fx
    m = DiT_models["DiT-B/2"](input_size=32, num_classes=0, learn_sigma=False, in_channels=4,
                              context_dim=768, roll_out=True, vit_blk=TextCondDiTBlock)
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    m.load_state_dict(odit.synth_state_dict(shapes, seed=7, keep={"pos_embed": m.state_dict()["pos_embed"]}))
    m = m.to(dev)
    x, t, ctx = fx.dit_inputs()
    out = m(x.to(dev), t.to(dev), {"crossattn": ctx.to(dev)})
    assert out.dtype == torch.float32 and out.is_contiguous() and out.shape == (2, 12, 32, 32)
    assert _rel(out, golden("dit_t23d.npz")["out"]) < 2e-2


def test_edm_cfg_pipeline_vs_oracle(dev):
    """DiT-B/2, 4 Euler-EDM+CFG steps: fused pipeline and the mirrored sampler classes vs the oracle."""
    from ln3diff_b200 import pipeline
    from ln3diff_b200.sgm.modules.diffusionmodules.denoiser import DiscreteDenoiser
    from ln3diff_b200.sgm.modules.diffusionmodules.sampling import EulerEDMSampler
    from ln3diff_b200.utils import build_t23d
    from oracle import dit as odit
    from oracle import samplers as osmp
    m = build_t23d("DiT-B/2")
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(41)
    x0 = torch.randn(2, 12, 32, 32, generator=g)
    c = {"crossattn": torch.randn(2, 77, 768, generator=g)}
    uc = {"crossattn": torch.zeros(2, 77, 768)}
    ref = osmp.euler_edm_cfg_sample(lambda xi, ti, cc: odit.dit_t23d_forward(sd, "DiT-B/2", xi, ti, cc["crossattn"]),
                                    x0.clone(), c, uc, 4, 6.5)
    m = m.to(dev)
    cd, ucd = {"crossattn": c["crossattn"].to(dev)}, {"crossattn": uc["crossattn"].to(dev)}
    out = pipeline.sample_t23d(m, x0.to(dev), cd, ucd, 4, 6.5)
    assert _rel(out, ref) < 2e-2
    # the shared per-step modulation table (one adaLN row per step) is the same arithmetic as the per-forward path
    os.environ["LN3_SHARED_MODULATION"] = "0"
    try:
        out_per_forward = pipeline.sample_t23d(m, x0.to(dev), cd, ucd, 4, 6.5)
    finally:
        del os.environ["LN3_SHARED_MODULATION"]
    assert torch.equal(out, out_per_forward)
    disc = {"target": "sgm.modules.diffusionmodules.discretizer.LegacyDDPMDiscretization"}
    s = EulerEDMSampler(discretization_config=disc, num_steps=4, device=str(dev), guider_config={
        "target": "sgm.modules.diffusionmodules.guiders.VanillaCFG", "params": {"scale": 6.5}})
    d = DiscreteDenoiser(scaling_config={"target": "sgm.modules.diffusionmodules.denoiser_scaling.EpsScaling"},
                         num_idx=1000, discretization_config=disc).to(dev)
    out2 = s(lambda i, sg, cc: d(m, i, sg, cc), x0.clone().to(dev), cd, ucd)
    assert _rel(out2, ref) < 2e-2
    assert _rel(out2, out) < 1e-2


def test_ddpm_p_sample_loop_config1(dev):
    """BASELINE configs[0]: DiT-B/2, SpacedDiffusion('10') p_sample_loop, batch 1, vs the oracle."""
    from ln3diff_b200.guided_diffusion import gaussian_diffusion as gd
    from ln3diff_b200.guided_diffusion.respace import SpacedDiffusion, space_timesteps
    from ln3diff_b200.utils import build_t23d
    from oracle import dit as odit
    from oracle import samplers as osmp
    m = build_t23d("DiT-B/2")
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(1)
    noise = torch.randn(1, 12, 32, 32, generator=g)
    ctx = torch.randn(1, 77, 768, generator=torch.Generator().manual_seed(2))
    step_noise = [torch.randn(1, 12, 32, 32, generator=g) for _ in range(10)]
    tab = osmp.DDPMTables(osmp.linear_betas(1000), osmp.space_timesteps(1000, "10"))
    ref = osmp.ddpm_p_sample_loop(lambda xx, tt, cc: odit.dit_t23d_forward(sd, "DiT-B/2", xx, tt, cc),
                                  (1, 12, 32, 32), tab, noise, step_noise, cond=ctx)
    m = m.to(dev)
    diff = SpacedDiffusion(use_timesteps=space_timesteps(1000, "10"), betas=gd.get_named_beta_schedule("linear", 1000),
                           model_mean_type=gd.ModelMeanType.EPSILON, model_var_type=gd.ModelVarType.FIXED_LARGE,
                           loss_type=gd.LossType.MSE)

    class Engine:  # what TrainLoop.apply_model_inference does: call the denoiser with the context
        def apply_model_inference(self, x, t, c, **kw):
            return m(x, t, c)

    it = iter(step_noise)
    orig = torch.randn_like
    torch.randn_like = lambda v: next(it).to(v.device)
    try:
        out = diff.p_sample_loop(Engine(), (1, 12, 32, 32), cond=ctx.to(dev), noise=noise.to(dev),
                                 clip_denoised=False, device=dev)
    finally:
        torch.randn_like = orig
    assert _rel(out, ref) < 2e-2


# ------------------------------------------------------------------ renderer
def _render_cuda(dev, planes, osg, o, d, nc, nf, **kw):
    from ln3diff_b200 import ops
    pcl = ops.planes_to_channels_last(planes[None].contiguous().to(dev))
    return ops.render_views(pcl, o.contiguous().to(dev), d.contiguous().to(dev), nc.contiguous().to(dev),
                            nf.contiguous().to(dev), tuple(t.to(dev) for t in osg), views_per_obj=o.shape[0], **kw)


def test_render_matches_reference_golden(dev, golden):
    """Fused CUDA renderer vs the REFERENCE's ImportanceRenderer outputs (tests/golden/render.npz)."""
    from oracle import fixtures as fx
    g = golden("render.npz")
    res = 24
    planes, osg, nc, nf = fx.render_inputs(res)
    o = torch.stack([torch.from_numpy(g[f"ray_o_{v}"]) for v in range(2)])
    d = torch.stack([torch.from_numpy(g[f"ray_d_{v}"]) for v in range(2)])
    r = _render_cuda(dev, planes, osg, o, d, nc, nf)
    for v in range(2):
        assert _rel(r["rgb"][v].t(), g[f"rgb_{v}"]) < 1e-3          # north_star tolerance on pixels
        assert _rel(r["rgb"][v].t(), g[f"rgb_{v}"]) < 2e-5          # what the fp32 kernel actually achieves
        assert _rel(r["depth"][v].t(), g[f"depth_{v}"]) < 2e-5
        assert _rel(r["weights"][v].t(), g[f"weights_{v}"]) < 2e-5


def test_render_bookkeeping_and_rays_vs_oracle(dev, golden):
    from ln3diff_b200 import ops
    from oracle import fixtures as fx
    from oracle import render as orender
    cams = torch.from_numpy(golden("cameras.npz")["objv_eval_pose"])[:3]
    res = 32
    o_ref, d_ref = orender.generate_rays(cams[:, :16].reshape(-1, 4, 4), cams[:, 16:].reshape(-1, 3, 3), res)
    o, d = ops.generate_rays(cams.to(dev).contiguous(), res)
    assert torch.equal(o.cpu(), o_ref)                              # origins + ray order m = y*W + x: exact
    assert (d.cpu() - d_ref).abs().max() < 3e-7
    planes, osg, nc, nf = fx.render_inputs(res, n_views=3)
    r = _render_cuda(dev, planes, osg, o_ref, d_ref, nc, nf, debug=True)
    M = res * res
    n_bad_idx = n_bad_ord = 0
    for v in range(3):
        dbg = orender.render_rays(planes, osg, o_ref[v], d_ref[v], orender.OBJAVERSE_OPTS, nc[v], nf[v], return_debug=True)
        inb = r["inbox"].cpu()[v * M:(v + 1) * M].bool()
        assert torch.equal(inb[:, :64], dbg["inbox_coarse"])        # integer bookkeeping: bit-exact
        zf = r["z_fine"].cpu()[v * M:(v + 1) * M]
        assert (zf - dbg["z_fine"]).abs().max() < 5e-6
        # in-box of the fine samples / searchsorted / sort permutation depend on float cdf / depth
        # values that differ in the last ulp (scan order): allow ties only
        assert (inb[:, 64:] != dbg["inbox_fine"]).sum() <= 2
        n_bad_idx += int((r["inds"].cpu()[v * M:(v + 1) * M].long() != dbg["inds"]).sum())
        n_bad_ord += int((r["order"].cpu()[v * M:(v + 1) * M].long() != dbg["order"]).sum())
    assert n_bad_idx <= 3 * M * 64 * 2e-5 + 2
    assert n_bad_ord <= 3 * M * 128 * 2e-5 + 2


def test_render_edge_cases(dev):
    from oracle import fixtures as fx
    from oracle import render as orender
    res = 8
    planes, osg, nc, nf = fx.render_inputs(res, n_views=2)
    miss_o = torch.tensor([[3.0, 3.0, 3.0]]).repeat(res * res, 1)
    miss_d = F.normalize(torch.tensor([[1.0, 0.2, 0.1]]), dim=1).repeat(res * res, 1)
    in_o = torch.zeros(res * res, 3)
    in_d = F.normalize(torch.randn(res * res, 3, generator=torch.Generator().manual_seed(3)), dim=1)
    o, d = torch.stack([miss_o, in_o]), torch.stack([miss_d, in_d])
    r = _render_cuda(dev, planes, osg, o, d, nc, nf)                # group_size 1: per-view reductions
    for v in range(2):
        ref = orender.render_rays(planes, osg, o[v], d[v], orender.OBJAVERSE_OPTS, nc[v], nf[v])
        assert torch.isfinite(r["rgb"][v]).all()
        assert (r["rgb"][v].t().cpu() - ref["rgb"]).abs().max() < 1e-4
        assert (r["depth"][v].t().cpu() - ref["depth"]).abs().max() < 1e-4
        assert (r["weights"][v].t().cpu() - ref["weights"]).abs().max() < 1e-4


def test_render_full_size_properties(dev):
    """BASELINE config 3 size (128x128, 16 views): size-independent properties -- outputs in range,
    weights in [0,1], white background where nothing is hit, determinism, and view-batch
    independence (rendering views together == one at a time)."""
    from ln3diff_b200 import ops
    from ln3diff_b200.utils import orbit_cameras
    g = torch.Generator().manual_seed(4)
    V, res = 16, 128
    planes = (5 * torch.randn(1, 3, 32, 128, 128, generator=g)).to(dev)
    osg = [torch.randn(64, 32, generator=g), torch.randn(64, generator=g) * 0.1,
           torch.randn(4, 64, generator=g), torch.randn(4, generator=g) * 0.1]
    osg[3][0] += 2.0
    osg = tuple(t.to(dev) for t in osg)
    M = res * res
    nc, nf = torch.rand(V, M, 64, generator=g).to(dev), torch.rand(V, M, 64, generator=g).to(dev)
    pcl = ops.planes_to_channels_last(planes)
    o, d = ops.generate_rays(orbit_cameras(V).to(dev), res)
    r = ops.render_views(pcl, o, d, nc, nf, osg, views_per_obj=V)
    assert torch.isfinite(r["rgb"]).all() and torch.isfinite(r["depth"]).all()
    assert r["rgb"].min() >= -1.003 and r["rgb"].max() <= 1.003
    assert r["weights"].min() >= 0 and r["weights"].max() <= 1 + 1e-5
    empty = r["weights"][:, 0] < 1e-7
    assert empty.any() and (r["rgb"].permute(0, 2, 1)[empty] - 1).abs().max() < 1e-5
    r2 = ops.render_views(pcl, o, d, nc, nf, osg, views_per_obj=V)
    assert torch.equal(r["rgb"], r2["rgb"])                          # deterministic
    one = ops.render_views(pcl, o[5:6].contiguous(), d[5:6].contiguous(), nc[5:6].contiguous(),
                           nf[5:6].contiguous(), osg, views_per_obj=1)
    assert torch.equal(one["rgb"][0], r["rgb"][5]) and torch.equal(one["depth"][0], r["depth"][5])


# ------------------------------------------------------------------ VAE decoder
def test_decoder_conv_ops(dev):
    from ln3diff_b200 import ops
    g = torch.Generator().manual_seed(12)
    x = torch.randn(2, 48, 20, 24, generator=g)                  # NCHW: C=48, H=20, W=24
    w = torch.randn(40, 48, 3, 3, generator=g) * 0.1
    b = torch.randn(40, generator=g)
    gam, bet = 1 + 0.1 * torch.randn(48, generator=g), 0.1 * torch.randn(48, generator=g)
    xh = x.permute(0, 2, 3, 1).contiguous().to(dev)              # NHWC
    pk = lambda ww: ww.permute(2, 3, 1, 0).reshape(-1, ww.shape[1], ww.shape[0]).contiguous().to(dev)
    gn = ops.groupnorm_stats(xh, gam.to(dev), bet.to(dev), groups=8)
    ref_n = F.group_norm(x, 8, gam, bet, eps=1e-6)
    ref = F.conv2d(ref_n * torch.sigmoid(ref_n), w, b, padding=1)
    out = ops.conv_nhwc(xh, pk(w), b.to(dev), ksize=3, gn=gn, swish=True)
    assert _rel(out.permute(0, 3, 1, 2), ref) < 1e-5
    ref_up = F.conv2d(F.interpolate(x, scale_factor=2.0, mode="nearest"), w, b, padding=1)
    res = torch.randn(2, 40, 40, 48, generator=g)                # NCHW: Cout=40, 2H=40, 2W=48
    out = ops.conv_nhwc(xh, pk(w), b.to(dev), ksize=3, upsample=True, residual=res.permute(0, 2, 3, 1).contiguous().to(dev))
    assert _rel(out.permute(0, 3, 1, 2), ref_up + res) < 1e-5
    # tensor-core (TF32) 3x3 path: ragged tiles (20x24), Cin = 48 (3 chunks), Cout = 40 (tail of a 64-wide
    # tile), fused GroupNorm + swish, fused upsample + residual; and a 32-channel output (the other template)
    out_tf = ops.conv_nhwc(xh, pk(w), b.to(dev), ksize=3, gn=gn, swish=True, tf32=True)
    assert _rel(out_tf.permute(0, 3, 1, 2), ref) < 2e-3
    out_tf = ops.conv_nhwc(xh, pk(w), b.to(dev), ksize=3, upsample=True, tf32=True,
                           residual=res.permute(0, 2, 3, 1).contiguous().to(dev))
    assert _rel(out_tf.permute(0, 3, 1, 2), ref_up + res) < 2e-3
    w32 = torch.randn(32, 48, 3, 3, generator=g) * 0.1
    assert _rel(ops.conv_nhwc(xh, pk(w32), None, ksize=3, tf32=True).permute(0, 3, 1, 2), F.conv2d(x, w32, padding=1)) < 2e-3
    w1 = torch.randn(40, 48, 1, 1, generator=g) * 0.1
    assert _rel(ops.conv_nhwc(xh, pk(w1), None, ksize=1).permute(0, 3, 1, 2), F.conv2d(x, w1)) < 1e-5
    q, k, v = (torch.randn(3, 256, 128, generator=g) for _ in range(3))
    ref = torch.softmax(q @ k.transpose(1, 2) * 128 ** -0.5, -1) @ v
    assert _rel(ops.attn_single_head(q.to(dev), k.to(dev), v.to(dev)), ref) < 1e-5
    for (n_, L_, C_) in [(2, 200, 64), (1, 37, 32), (2, 5, 128)]:      # ragged key blocks / query groups
        q, k, v = (torch.randn(n_, L_, C_, generator=g) for _ in range(3))
        ref = torch.softmax(q @ k.transpose(1, 2) * C_ ** -0.5, -1) @ v
        assert _rel(ops.attn_single_head(q.to(dev), k.to(dev), v.to(dev)), ref) < 1e-5


def test_vae_decoder_matches_reference_golden(dev, golden):
    """CUDA decode (DiT2 tcgen05 blocks + NHWC conv kernels) vs the REFERENCE's modules
    (tests/golden/decoder.npz), and the same through the reference-named entry points."""
    from ln3diff_b200.utils import build_ae_decoder
    from oracle import fixtures as fx
    g = golden("decoder.npz")
    m = build_ae_decoder(fx.DECODER_ARCH)
    sd = m.state_dict()
    shapes = {k: tuple(v.shape) for k, v in sd.items()
              if k.startswith(("superresolution.ldm_upsample", "superresolution.conv_sr", "vit_decoder"))}
    sd.update(fx.decoder_state_dict(shapes))
    m.load_state_dict(sd)
    m = m.to(dev)
    lat = fx.decoder_latent().to(dev)
    cl = m.decode_to_channels_last(lat, in_mul=fx.SCALING_DIVIDER)           # (1, 3, 128, 128, 32)
    y = cl.permute(0, 1, 4, 2, 3).reshape(1, 96, 128, 128)
    assert _rel(y[:, :, 40:56, 40:56], g["crop"]) < 2e-2                     # bf16 DiT2 blocks
    assert _rel(y.abs().mean(dim=(0, 2, 3)), g["chan_absmean"]) < 1e-2
    ret = m.vit_decode_postprocess(m.vit_decode_backbone({"latent_normalized_2Ddiffusion": lat * fx.SCALING_DIVIDER}), {})
    assert ret["latent_after_vit"].shape == (1, 96, 128, 128)
    assert _rel(ret["latent_after_vit"], y) < 1e-3


def test_latent_to_pixels_end_to_end(dev, golden):
    """latent -> decode -> Triplane.forward(planes, c) through the mirrored classes vs the oracle
    chain (decoder oracle -> render oracle) with identical explicit noise."""
    from ln3diff_b200.utils import build_ae_decoder
    from oracle import decoder as odec
    from oracle import fixtures as fx
    from oracle import render as orender
    m = build_ae_decoder(fx.DECODER_ARCH, image_size=32)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    lat = fx.decoder_latent()
    cam = torch.from_numpy(golden("cameras.npz")["objv_eval_pose"])[5:6]
    res = 32
    planes_ref = odec.vae_decode(sd, fx.DECODER_ARCH, lat, fx.SCALING_DIVIDER)
    osg = tuple(sd[f"triplane_decoder.decoder.net.{i}.{n}"] for i, n in ((0, "weight"), (0, "bias"), (2, "weight"), (2, "bias")))
    # the mirror draws its noise with torch.rand_like / torch.rand on the device: intercept both
    gen = torch.Generator().manual_seed(77)
    nc, nf = torch.rand(1, res * res, 64, 1, generator=gen), torch.rand(res * res, 64, generator=gen)
    ref = orender.render_view(planes_ref.reshape(3, 32, 128, 128), osg, cam[0], res, orender.OBJAVERSE_OPTS,
                              nc[0, :, :, 0], nf)
    m = m.to(dev)
    ret = m.vit_decode_postprocess(lat.to(dev) * fx.SCALING_DIVIDER, {})
    orl, orr = torch.rand_like, torch.rand
    torch.rand_like = lambda t_, *a, **k: nc.to(t_.device).reshape(t_.shape)
    torch.rand = lambda *s, **k: nf.to(k.get("device", "cpu")).reshape(*s)
    try:
        out = m.triplane_decode(ret, cam.to(dev))
    finally:
        torch.rand_like, torch.rand = orl, orr
    assert set(("image_raw", "image_depth", "weights_samples", "image_mask", "feature_image")) <= set(out.keys())
    assert out["image_raw"].shape == (1, 3, res, res)
    # bf16 DiT2 features feed an fp32 renderer: pixels follow the decoder tolerance
    assert _rel(out["image_raw"][0], ref["image_raw"]) < 3e-2
    assert _rel(out["image_mask"][0], ref["image_mask"]) < 3e-2


# ------------------------------------------------------------------ I23D (flow matching)
def test_gemm_head_rmsnorm(dev):
    from ln3diff_b200 import ops
    from oracle import dit as odit
    g = torch.Generator().manual_seed(17)
    M, D, H = 300, 256, 4
    a = (torch.randn(M, 128, generator=g) * 0.5).bfloat16()
    w = (torch.randn(3 * D, 128, generator=g) * 0.1).bfloat16()
    b = torch.randn(3 * D, generator=g)
    nw = 1 + 0.1 * torch.randn(2, 64, generator=g)
    ref = (a.float() @ w.float().t() + b).reshape(M, 3, H, 64)
    ref[:, 0] = odit.rms_norm(ref[:, 0], nw[0], 1e-5)
    ref[:, 1] = odit.rms_norm(ref[:, 1], nw[1], 1e-5)
    out = ops.gemm(a.to(dev), w.to(dev), b.to(dev), head_norm=nw.to(dev), head_norm_sec_cols=D)
    assert _rel(out, ref.reshape(M, 3 * D)) < 4e-3


def test_dit_i23d_forward_matches_reference_golden(dev, golden):
    from ln3diff_b200.utils import build_i23d
    from oracle import fixtures as fx
    g = golden("dit_i23d.npz")
    m = build_i23d(fx.I23D_ARCH)
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    m.load_state_dict(fx.i23d_state_dict(shapes, m.state_dict()["pos_embed"]))
    m = m.to(dev)
    x, t, ctx = fx.i23d_inputs()
    cd = {k: v.to(dev) for k, v in ctx.items()}
    out = m(x.to(dev), t.to(dev), cd)
    assert out.dtype == torch.float32 and out.shape == (2, 12, 32, 32)
    assert _rel(out, g["out"]) < 2e-2
    assert _rel(m.forward_with_cfg(x.to(dev), t.to(dev), cd, 4.0), g["out_cfg"]) < 3e-2


def test_flow_euler_cfg_sampler_vs_oracle(dev):
    """BASELINE configs[3] plumbing at small size: Sampler.sample_ode('euler') + forward_with_cfg."""
    from ln3diff_b200.transport import Sampler, create_transport
    from ln3diff_b200.utils import build_i23d
    from oracle import dit as odit
    from oracle import samplers as osmp
    m = build_i23d("DiT-PixArt-B/2")
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    g = torch.Generator().manual_seed(42)
    z = torch.randn(1, 12, 32, 32, generator=g)
    c = {"vector": torch.randn(1, 768, generator=g), "crossattn": torch.randn(1, 256, 2048, generator=g)}
    ctx = {k: torch.cat([v, torch.zeros_like(v)]) for k, v in c.items()}            # cond first, uc = 0
    steps = 5
    ref = osmp.flow_ode_cfg_sample(lambda xx, tt, cc: odit.dit_i23d_pixart_forward(sd, "DiT-PixArt-B/2", xx, tt, cc),
                                   z, ctx, 4.0, steps)
    m = m.to(dev)
    fn = Sampler(create_transport(snr_type="lognorm")).sample_ode(sampling_method="euler", num_steps=steps)
    traj = fn(torch.cat([z, z]).to(dev), m.forward_with_cfg, context={k: v.to(dev) for k, v in ctx.items()}, cfg_scale=4.0)
    assert traj.shape == (steps, 2, 12, 32, 32)
    assert _rel(traj[-1].chunk(2)[0], ref) < 2e-2


def test_decode_and_render_pipeline_vs_oracle(dev, golden):
    """pipeline.decode_and_render (decode once, all views in one launch) vs the oracle chain."""
    from ln3diff_b200 import pipeline
    from ln3diff_b200.utils import build_ae_decoder
    from oracle import decoder as odec
    from oracle import fixtures as fx
    from oracle import render as orender
    m = build_ae_decoder(fx.DECODER_ARCH, image_size=32)
    sd = {k: v.clone() for k, v in m.state_dict().items()}
    lat = fx.decoder_latent()
    cams = torch.from_numpy(golden("cameras.npz")["objv_eval_pose"])[[2, 9]]
    res, V = 32, 2
    gen = torch.Generator().manual_seed(5)
    nc, nf = torch.rand(V, res * res, 64, generator=gen), torch.rand(V, res * res, 64, generator=gen)
    planes_ref = odec.vae_decode(sd, fx.DECODER_ARCH, lat, fx.SCALING_DIVIDER).reshape(3, 32, 128, 128)
    osg = tuple(sd[f"triplane_decoder.decoder.net.{i}.{n}"] for i, n in ((0, "weight"), (0, "bias"), (2, "weight"), (2, "bias")))
    m = m.to(dev)
    out = pipeline.decode_and_render(m, lat.to(dev), cams.to(dev), res, fx.SCALING_DIVIDER, noise=(nc.to(dev), nf.to(dev)))
    assert out["image_raw"].shape == (1, V, 3, res, res)
    for v in range(V):
        ref = orender.render_view(planes_ref, osg, cams[v], res, orender.OBJAVERSE_OPTS, nc[v], nf[v])
        assert _rel(out["image_raw"][0, v], ref["image_raw"]) < 3e-2       # bf16 DiT2 features upstream
        assert _rel(out["image_mask"][0, v], ref["image_mask"]) < 3e-2


def test_query_points_vs_reference_golden(dev, golden):
    """ln3_query_points (explicit points and in-kernel lattice) vs the reference's _run_model outputs, and
    the mirror's forward_points / triplane_decode_grid entry points."""
    from ln3diff_b200 import ops
    from oracle import fixtures as fx
    from oracle import render as orender
    g = golden("points.npz")
    planes, osg, _, _ = fx.render_inputs(8)
    cl = ops.planes_to_channels_last(planes[None].to(dev).contiguous())
    osg_d = tuple(t.to(dev).contiguous() for t in osg)
    sigma, rgb = ops.query_points(cl, osg_d, points=torch.from_numpy(g["points"])[None].to(dev).contiguous())
    assert _rel(sigma[0], g["sigma"]) < 1e-5 and _rel(rgb[0], g["rgb"]) < 1e-5
    G = int(g["grid_size"])
    sigma, rgb = ops.query_points(cl, osg_d, grid_size=G)
    assert _rel(sigma[0], g["grid_sigma"]) < 1e-5 and _rel(rgb[0], g["grid_rgb"]) < 1e-5
    # two objects, a lattice that is not a multiple of the warp size, non-default aabb: against the oracle
    planes2 = torch.stack([planes, planes.flip(0) * 0.5])
    cl2 = ops.planes_to_channels_last(planes2.to(dev).contiguous())
    lo, hi = (-0.3, -0.45, -0.2), (0.45, 0.1, 0.4)
    sigma, rgb = ops.query_points(cl2, osg_d, grid_size=7, aabb_min=lo, aabb_max=hi)
    pts = orender.grid_points(lo, hi, 7)
    for i in range(2):
        r_rgb, r_sigma = orender.run_model_points(planes2[i], osg, pts, 0.9)
        assert _rel(sigma[i], r_sigma) < 1e-5 and _rel(rgb[i], r_rgb) < 1e-5
    # full-size property: the 192^3 mesh-extraction lattice of one 128x128 object runs and is finite
    big = ops.planes_to_channels_last((torch.randn(1, 3, 32, 128, 128) * 2).to(dev))
    sigma, rgb = ops.query_points(big, osg_d, grid_size=192)
    assert sigma.shape == (1, 192 ** 3, 1) and torch.isfinite(sigma).all() and torch.isfinite(rgb).all()
    assert float(rgb.min()) >= -0.001 - 1e-6 and float(rgb.max()) <= 1.001 + 1e-6


def test_decoder_grid_entry_points(dev, golden):
    """RodinSR...ditDecoder.triplane_decode_grid / forward_points (vit_triplane.py:2009-2120 mirrors)."""
    from ln3diff_b200.utils import build_ae_decoder
    from oracle import fixtures as fx
    from oracle import render as orender
    m = build_ae_decoder(fx.DECODER_ARCH, image_size=32).to(dev)
    m.rendering_kwargs["osg_mlp_tf32"] = False          # exact fp32 MLP for the 1e-5 comparisons below
    planes = torch.randn(2, 96, 16, 16, generator=torch.Generator().manual_seed(3)) * 3
    out = m.triplane_decode_grid({"latent_after_vit": planes.to(dev)}, 6)
    assert out["sigma"].shape == (2, 6, 6, 6, 1) and out["rgb"].shape == (2, 6, 6, 6, 3)
    osg = tuple(t.cpu() for t in m.triplane_decoder.decoder.raw_parameters())
    pts = orender.grid_points([-0.45] * 3, [0.45] * 3, 6)
    for i in range(2):
        r_rgb, r_sigma = orender.run_model_points(planes[i].reshape(3, 32, 16, 16), osg, pts, 0.9)
        assert _rel(out["sigma"][i].reshape(-1, 1), r_sigma) < 1e-5 and _rel(out["rgb"][i].reshape(-1, 3), r_rgb) < 1e-5
    fp = m.forward_points(planes.to(dev), pts[None].repeat(2, 1, 1).to(dev))
    assert _rel(fp["sigma"], out["sigma"].reshape(2, -1, 1)) < 1e-6
    aabb = torch.tensor([[[-0.45] * 3, [0.45] * 3], [[-0.2] * 3, [0.3] * 3]])
    out2 = m.triplane_decode_grid({"latent_after_vit": planes.to(dev)}, 5, aabb=aabb)
    r_rgb, r_sigma = orender.run_model_points(planes[1].reshape(3, 32, 16, 16), osg, orender.grid_points([-0.2] * 3, [0.3] * 3, 5), 0.9)
    assert _rel(out2["sigma"][1].reshape(-1, 1), r_sigma) < 1e-5


def test_render_tf32_mlp_within_north_star_tolerance(dev, golden):
    """The tensor-core (TF32 operands, fp32 accumulate) OSG MLP path: pixels within the north-star 1e-3
    rel-L2 of the REFERENCE's renderer; ray bookkeeping (in-box masks) unchanged from the exact path."""
    from ln3diff_b200 import ops
    from oracle import fixtures as fx
    g = golden("render.npz")
    planes, osg, nc, nf = fx.render_inputs(24)
    o = torch.stack([torch.from_numpy(g[f"ray_o_{v}"]) for v in range(2)])
    d = torch.stack([torch.from_numpy(g[f"ray_d_{v}"]) for v in range(2)])
    r = _render_cuda(dev, planes, osg, o, d, nc, nf, mlp_tf32=True, debug=True)
    rx = _render_cuda(dev, planes, osg, o, d, nc, nf, mlp_tf32=False, debug=True)
    for v in range(2):
        assert _rel(r["rgb"][v].t(), g[f"rgb_{v}"]) < 1e-3
        assert _rel(r["depth"][v].t(), g[f"depth_{v}"]) < 1e-3
        assert _rel(r["weights"][v].t(), g[f"weights_{v}"]) < 1e-3
    assert torch.equal(r["inbox"][:, :64], rx["inbox"][:, :64])       # coarse in-box masks: independent of the MLP
    gp = golden("points.npz")
    cl = ops.planes_to_channels_last(fx.render_inputs(8)[0][None].to(dev).contiguous())
    sigma, rgb = ops.query_points(cl, tuple(t.to(dev) for t in osg), points=torch.from_numpy(gp["points"])[None].to(dev),
                                  mlp_tf32=True)
    assert _rel(sigma[0], gp["sigma"]) < 1e-3 and _rel(rgb[0], gp["rgb"]) < 1e-3
    print("tf32 rel-L2: rgb", _rel(r["rgb"][0].t(), g["rgb_0"]), "sigma(points)", _rel(sigma[0], gp["sigma"]))


def test_dit_t23d_pixart_forward_matches_reference_golden(dev, golden):
    """DiT_models['DiT-PixelArt-B/2'] (shared adaLN + tables, per-block RMS-normed text K/V) vs the reference."""
    from ln3diff_b200.dit.dit_trilatent import DiT_models
    from oracle import fixtures as fx
    g = golden("dit_t23d_pixart.npz")
    m = DiT_models[fx.T23D_PIXART_ARCH](input_size=32, num_classes=0, learn_sigma=False, in_channels=4,
                                        context_dim=768, roll_out=True)
    shapes = {k: tuple(v.shape) for k, v in m.state_dict().items()}
    m.load_state_dict(fx.i23d_state_dict(shapes, m.state_dict()["pos_embed"]))
    m = m.to(dev)
    x, t, ctx = fx.t23d_pixart_inputs()
    cd = {k: v.to(dev) for k, v in ctx.items()}
    out = m(x.to(dev), t.to(dev), cd)
    assert out.dtype == torch.float32 and out.shape == (2, 12, 32, 32)
    assert _rel(out, g["out"]) < 2e-2
    assert _rel(m.forward_with_cfg(x.to(dev), t.to(dev), cd, 6.5), g["out_cfg"]) < 3e-2


def test_closed_form_uncond_cross_attention(dev, monkeypatch):
    """Samples whose context tokens are all identical (the zero-embedding CFG half) skip the cross-attention
    q GEMM / FMHA / out GEMM: softmax over identical keys is uniform, the output is to_out(v_row).  The
    closed form must agree with the full computation to bf16 rounding, for both CFG batch layouts."""
    from ln3diff_b200.utils import build_t23d
    m = build_t23d("DiT-B/2").to(dev)
    g = torch.Generator().manual_seed(21)
    x = torch.randn(4, 12, 32, 32, generator=g).to(dev)
    t = torch.tensor([3.0, 500.0, 3.0, 500.0]).to(dev)
    c = torch.randn(2, 77, 768, generator=g)
    for ctx, rows in ((torch.cat([torch.zeros_like(c), c]), (2, 4)), (torch.cat([c, torch.zeros_like(c)]), (0, 2)),
                      (torch.cat([c, c]), (0, 4))):
        ctx = ctx.to(dev)
        monkeypatch.setenv("LN3_UNCOND_CLOSED_FORM", "1")
        m._ctx_cache.clear()
        fast = m(x, t, ctx).clone()
        assert m._ctx_cache.value["rows"] == rows
        # the attended-rows-only residual pass is a pure re-scheduling of the same fp32 operations: bit-identical
        monkeypatch.setenv("LN3_SPLIT_RESID_PASS", "0")
        m._graphs.clear()
        assert torch.equal(m(x, t, ctx), fast)
        monkeypatch.delenv("LN3_SPLIT_RESID_PASS")
        m._graphs.clear()
        monkeypatch.setenv("LN3_UNCOND_CLOSED_FORM", "0")
        m._ctx_cache.clear()
        full = m(x, t, ctx).clone()
        assert m._ctx_cache.value["rows"] == (0, 4) and m._ctx_cache.value["oconst"] is None
        assert _rel(fast, full) < 3e-3
    m._ctx_cache.clear()


@pytest.mark.parametrize("M,N,K,act", [(12288, 1024, 1024, 0), (6144, 1024, 1024, 0), (12288, 1024, 4096, 0),
                                       (12288, 3072, 1024, 0), (12288, 4096, 1024, 1), (5000, 1024, 512, 0),
                                       (2560, 2048, 256, 0)])
def test_gemm_streamk_tail(dev, M, N, K, act, monkeypatch):
    """Opt-in stream-K tail of the CTA-pair GEMM (LN3_GEMM_STREAMK=1): shapes whose tile count is not a
    multiple of the pair count split their last tiles along K (fp32 partial sums through the workspace).
    Result vs fp32 reference, repeated launches (the flags must return to zero)."""
    from ln3diff_b200 import ops
    monkeypatch.setenv("LN3_GEMM_STREAMK", "1")
    g = torch.Generator().manual_seed(M + N + K)
    a = (torch.randn(M, K, generator=g) * 0.5).bfloat16().to(dev)
    w = (torch.randn(N, K, generator=g) * 0.05).bfloat16().to(dev)
    b = torch.randn(N, generator=g).to(dev)
    ref = a.float() @ w.float().t() + b
    if act == 1:
        ref = F.gelu(ref)
    outs = [ops.gemm(a, w, b, act=act).float() for _ in range(3)]
    assert _rel(outs[0], ref) < 4e-3
    assert torch.equal(outs[0], outs[1]) and torch.equal(outs[1], outs[2])
    assert int(ops._gemm_workspace(a.device)[:1024].view(torch.int32).abs().sum()) == 0   # flags self-reset
    o32 = ops.gemm(a, w, b, act=act, out_kind=ops.OUT_F32) if act == 0 else None
    if o32 is not None:
        assert _rel(o32, ref) < 1e-5


def test_dit_full_size_properties(dev, monkeypatch):
    """BASELINE configs[1] size (DiT-L/2, 16 samples per forward), where the CPU oracle is too slow: properties
    that do not depend on a reference output.  (1) samples are independent: permuting the batch permutes the
    output bit-exactly (every kernel reduces each row in a fixed order); (2) a CUDA-graph replay equals the
    eager launch sequence bit-exactly; (3) a sample's output does not depend on its batch neighbours; (4) the
    CFG combination of the fused sampler update equals uc + s (c - uc) on the forward's own outputs."""
    from ln3diff_b200 import ops
    from ln3diff_b200.utils import build_t23d
    m = build_t23d("DiT-L/2", device=dev)
    g = torch.Generator().manual_seed(11)
    x = torch.randn(16, 12, 32, 32, generator=g).to(dev)
    t = torch.randint(0, 1000, (16,), generator=g).float().to(dev)
    ctx = torch.randn(16, 77, 768, generator=g).to(dev)
    out = m(x, t, ctx).clone()
    assert torch.isfinite(out).all() and out.shape == (16, 12, 32, 32)
    perm = torch.randperm(16, generator=g).to(dev)
    assert torch.equal(m(x[perm].contiguous(), t[perm].contiguous(), ctx[perm].contiguous()), out[perm])
    gr = m.capture_graph(16, ctx)
    assert m.capture_graph(16, ctx) is gr                     # cached per launch-sequence shape, not re-captured
    gr.x.copy_(x)
    gr.t.copy_(t)
    gr.in_scale.fill_(1.0)
    gr.replay()
    assert torch.equal(gr.out, out)
    monkeypatch.setenv("LN3_CUDA_GRAPH", "0")                   # the eager launch sequence, bit for bit
    assert torch.equal(m(x, t, ctx), out)
    monkeypatch.delenv("LN3_CUDA_GRAPH")
    x2 = x.clone()
    x2[1:] = torch.randn(15, 12, 32, 32, generator=g).to(dev)           # change every neighbour of sample 0
    assert torch.equal(m(x2, t, ctx)[0], out[0])
    coef = torch.tensor([[0.7, 1.0 - 6.5, 6.5, 0.0]] * 8).to(dev)          # x' = 0.7 x + (1-s) uc + s c
    upd = ops.sampler_affine_update(x[:8].contiguous(), coef, out[:8].contiguous(), out[8:].contiguous())
    assert _rel(upd, 0.7 * x[:8] + out[:8] + 6.5 * (out[8:] - out[:8])) < 1e-6


def test_closed_form_uncond_cross_attention_pixart_models(dev, monkeypatch):
    """Same identity in the PixArt-style denoisers (T23D DiT_TriLatent_PixelArt, I23D DiT_I23D_PixelArt): an
    all-zero unconditional half has identical (zero) text / CLIP tokens."""
    from ln3diff_b200.dit.dit_trilatent import DiT_models
    from ln3diff_b200.utils import build_i23d
    from oracle import fixtures as fx
    g = torch.Generator().manual_seed(23)
    x = torch.randn(4, 12, 32, 32, generator=g).to(dev)
    mt = DiT_models[fx.T23D_PIXART_ARCH](input_size=32, num_classes=0, learn_sigma=False, in_channels=4,
                                         context_dim=768, roll_out=True)
    shapes = {k: tuple(v.shape) for k, v in mt.state_dict().items()}
    mt.load_state_dict(fx.i23d_state_dict(shapes, mt.state_dict()["pos_embed"]))
    mi = build_i23d(fx.I23D_ARCH)
    cases = [(mt.to(dev), torch.tensor([3.0, 500.0, 3.0, 500.0]),
              {"vector": torch.randn(2, 768, generator=g), "crossattn": torch.randn(2, 77, 768, generator=g)}),
             (mi.to(dev), torch.tensor([0.1, 0.8, 0.1, 0.8]),
              {"vector": torch.randn(2, 768, generator=g), "crossattn": torch.randn(2, 256, 2048, generator=g)})]
    for m, t, c in cases:
        ctx = {k: torch.cat([v, torch.zeros_like(v)]).to(dev) for k, v in c.items()}     # cond first, uc = 0
        monkeypatch.setenv("LN3_UNCOND_CLOSED_FORM", "1")
        m._ctx_cache.clear()
        fast = m(x, t.to(dev), ctx).clone()
        assert m._ctx_cache.value["rows"] == (0, 2)
        monkeypatch.setenv("LN3_SPLIT_RESID_PASS", "0")
        m._graphs.clear()
        assert torch.equal(m(x, t.to(dev), ctx), fast)
        monkeypatch.delenv("LN3_SPLIT_RESID_PASS")
        m._graphs.clear()
        monkeypatch.setenv("LN3_UNCOND_CLOSED_FORM", "0")
        m._ctx_cache.clear()
        full = m(x, t.to(dev), ctx).clone()
        assert m._ctx_cache.value["oconst"] is None
        assert _rel(fast, full) < 3e-3
        m._ctx_cache.clear()
