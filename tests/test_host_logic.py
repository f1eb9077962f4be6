"""CPU: host-side mirrors (schedules, sampler loops, registries, state_dict surface) against the
oracle / golden fixtures.  CUDA-only fast paths are not taken on CPU tensors."""
import numpy as np
import torch

from oracle import fixtures as fx
from oracle import samplers as osmp


def test_state_dict_surface_matches_reference_names():
    from ln3diff_b200.utils import build_t23d
    m = build_t23d("DiT-B/2")
    keys = set(m.state_dict().keys())
    for k in ("pos_embed", "x_embedder.proj.weight", "t_embedder.mlp.0.weight", "t_embedder.mlp.2.bias",
              "clip_text_proj.y_proj.fc1.weight", "blocks.0.attn.qkv.weight", "blocks.0.attn.proj.bias",
              "blocks.0.mlp.mlp.0.weight", "blocks.0.mlp.mlp.1.bias", "blocks.0.mlp.mlp.2.weight",
              "blocks.0.mlp.mlp.3.bias", "blocks.0.adaLN_modulation.1.weight",
              "blocks.0.cross_attn.to_q.weight", "blocks.0.cross_attn.to_out.0.bias",
              "final_layer.linear.weight", "final_layer.adaLN_modulation.1.bias"):
        assert k in keys, k
    assert m.state_dict()["blocks.11.attn.qkv.weight"].shape == (2304, 768)
    assert sum(p.numel() for p in m.parameters()) == 159_626_512  # 159.6 M (SURVEY appendix A)


def test_sgm_mirror_matches_golden(golden):
    from ln3diff_b200.sgm.modules.diffusionmodules.denoiser import DiscreteDenoiser
    from ln3diff_b200.sgm.modules.diffusionmodules.sampling import EulerEDMSampler
    g = golden("samplers.npz")
    disc = {"target": "sgm.modules.diffusionmodules.discretizer.LegacyDDPMDiscretization"}
    s = EulerEDMSampler(discretization_config=disc, num_steps=10, device="cpu", guider_config={
        "target": "sgm.modules.diffusionmodules.guiders.VanillaCFG", "params": {"scale": 6.5}})
    d = DiscreteDenoiser(scaling_config={"target": "sgm.modules.diffusionmodules.denoiser_scaling.EpsScaling"},
                         num_idx=1000, discretization_config=disc)
    assert torch.equal(d.sigmas, torch.from_numpy(g["denoiser_sigmas"]))
    toy = fx.toy_network()
    x0, c, uc, *_ = fx.sampler_inputs()
    out = s(lambda i, sg, cc: d(toy, i, sg, cc), x0.clone(), c, uc)
    assert torch.equal(out, torch.from_numpy(g["sgm"]))


def test_ddpm_mirror_matches_golden(golden):
    from ln3diff_b200.guided_diffusion import gaussian_diffusion as gd
    from ln3diff_b200.guided_diffusion.respace import SpacedDiffusion, space_timesteps
    g = golden("samplers.npz")
    toy = fx.toy_network()
    _, c, _, noise, step_noise, _ = fx.sampler_inputs()
    diff = SpacedDiffusion(use_timesteps=space_timesteps(1000, "10"),
                           betas=gd.get_named_beta_schedule("linear", 1000),
                           model_mean_type=gd.ModelMeanType.EPSILON, model_var_type=gd.ModelVarType.FIXED_LARGE,
                           loss_type=gd.LossType.MSE)
    assert np.array_equal(diff.betas, g["ddpm_betas10"])

    class M:
        def apply_model_inference(self, x, t, cc, **kw):
            return toy(x, t * 1000, cc)

    it = iter(step_noise)
    orig = torch.randn_like
    torch.randn_like = lambda v: next(it)
    try:
        out = diff.p_sample_loop(M(), (2, 12, 32, 32), cond=c["crossattn"], noise=noise, clip_denoised=False,
                                 device="cpu")
    finally:
        torch.randn_like = orig
    assert torch.equal(out, torch.from_numpy(g["ddpm"]))
    # the fused-kernel coefficient table reproduces the same update: a x + w0 eps + s noise
    tab = diff._step_coef_table("cpu")
    t = torch.tensor([5, 5])
    x = noise
    eps = toy(x, torch.tensor([0.5, 0.5]) * 1000, c["crossattn"])
    class E:
        def apply_model_inference(self, xx, tt, cc, **kw):
            return eps
    ref = diff.p_mean_variance(E(), x, t, clip_denoised=False)
    cf = tab[t]
    fused = cf[:, 0, None, None, None] * x + cf[:, 1, None, None, None] * eps
    assert torch.allclose(fused, ref["mean"], rtol=1e-5, atol=1e-5)
    assert torch.allclose(cf[:, 3], torch.exp(0.5 * ref["log_variance"][:, 0, 0, 0]), rtol=1e-6)
    assert float(tab[0, 3]) == 0.0


def test_flow_mirror_matches_golden(golden):
    from ln3diff_b200.transport import Sampler, create_transport
    g = golden("samplers.npz")
    toy = fx.toy_network()
    _, c, uc, _, _, z = fx.sampler_inputs()
    fn = Sampler(create_transport(snr_type="lognorm")).sample_ode(sampling_method="euler", num_steps=10)
    ctx = {"crossattn": torch.cat([c["crossattn"], uc["crossattn"]])}

    def fwd_cfg(x, t, context, cfg_scale):
        e = toy(x, t * 1000, context)
        ce, ue = torch.split(e, len(e) // 2, dim=0)
        h = ue + cfg_scale * (ce - ue)
        return torch.cat([h, h], 0)

    traj = fn(torch.cat([z, z], 0), fwd_cfg, context=ctx, cfg_scale=4.0)
    assert traj.shape == (10, 4, 12, 32, 32)
    assert torch.equal(traj[-1].chunk(2)[0], torch.from_numpy(g["flow"]))


def test_fused_edm_tables_reproduce_the_reference_step():
    """pipeline.edm_cfg_tables: x' = x + w_u net_u + w_c net_c equals the reference loop (toy net)."""
    from ln3diff_b200 import pipeline
    toy = fx.toy_network()
    x0, c, uc, *_ = fx.sampler_inputs()
    B = x0.shape[0]
    tabs = pipeline.edm_cfg_tables(10, 6.5, B, "cpu")
    x = x0 * tabs["init_scale"]
    ctx = {"crossattn": torch.cat((uc["crossattn"], c["crossattn"]), 0)}
    for i in range(10):
        x2 = torch.cat([x, x], 0) * tabs["c_in"][i][:, None, None, None]
        net = toy(x2, tabs["t_idx"][i], ctx)
        cf = tabs["coef"][i]
        x = (cf[:, 0, None, None, None] * x + cf[:, 1, None, None, None] * net[:B]
             + cf[:, 2, None, None, None] * net[B:])
    ref = osmp.euler_edm_cfg_sample(toy, x0.clone(), c, uc, 10, 6.5)
    assert ((x - ref).norm() / ref.norm()).item() < 1e-5


def test_orbit_cameras_are_valid_rigid_transforms():
    from ln3diff_b200.utils import orbit_cameras
    cams = orbit_cameras(5)
    R = cams[:, :16].reshape(5, 4, 4)[:, :3, :3]
    assert torch.allclose(R @ R.transpose(1, 2), torch.eye(3).expand(5, 3, 3), atol=1e-5)
    assert torch.allclose(torch.linalg.det(R), torch.ones(5), atol=1e-5)


def test_overlay_routes_reference_import_names(tmp_path):
    """ln3diff_b200.overlay: the reference's import names of the mirrored modules resolve to this package,
    everything else keeps resolving to the (here: fake) reference checkout on sys.path."""
    import importlib
    import sys
    from ln3diff_b200 import overlay
    for pkg in ("dit", "sgm/modules/diffusionmodules", "nsr/volumetric_rendering", "guided_diffusion"):
        d = tmp_path
        for part in pkg.split("/"):
            d = d / part
            d.mkdir(exist_ok=True)
            (d / "__init__.py").write_text("")
    (tmp_path / "dit" / "norm.py").write_text("WHO = 'reference'\n")
    (tmp_path / "dit" / "dit_trilatent.py").write_text("WHO = 'reference'\n")
    (tmp_path / "nsr" / "train_util_diffusion.py").write_text("WHO = 'reference'\n")
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k.split(".")[0] in ("dit", "sgm", "nsr", "guided_diffusion", "transport")}
    sys.path.insert(0, str(tmp_path))
    overlay.install()
    try:
        import ln3diff_b200.dit.dit_trilatent as mirror
        assert importlib.import_module("dit.dit_trilatent") is mirror                 # mirrored name -> this package
        assert importlib.import_module("dit.dit_trilatent").DiT_models is mirror.DiT_models
        assert importlib.import_module("dit.norm").WHO == "reference"                 # not mirrored -> reference file
        assert importlib.import_module("nsr.train_util_diffusion").WHO == "reference"
        s = importlib.import_module("sgm.modules.diffusionmodules.sampling")
        assert s.__name__ == "ln3diff_b200.sgm.modules.diffusionmodules.sampling" and hasattr(s, "EulerEDMSampler")
        r = importlib.import_module("nsr.volumetric_rendering.renderer")
        assert r.ImportanceRenderer.__module__.startswith("ln3diff_b200.")
        t = importlib.import_module("transport")
        assert hasattr(t, "create_transport") and importlib.import_module("transport.transport").__name__.startswith("ln3diff_b200.")
        from guided_diffusion.respace import SpacedDiffusion                          # noqa: F401  (from-import form)
        assert SpacedDiffusion.__module__.startswith("ln3diff_b200.")
    finally:
        overlay.uninstall()
        sys.path.remove(str(tmp_path))
        for k in list(sys.modules):
            if k.split(".")[0] in ("dit", "sgm", "nsr", "guided_diffusion", "transport"):
                del sys.modules[k]
        sys.modules.update(saved)
    assert overlay._finder is None


def test_identical_token_row_detection(monkeypatch):
    """dit_trilatent._attention_rows: which samples of a CFG batch still need real cross-attention."""
    import torch
    from ln3diff_b200.dit.dit_trilatent import _attention_rows
    g = torch.Generator().manual_seed(0)
    c = torch.randn(3, 5, 8, generator=g)
    same = torch.randn(3, 1, 8, generator=g).expand(3, 5, 8)                 # identical tokens within a sample
    assert _attention_rows(torch.cat([same, c])) == (3, 6)                   # sgm VanillaCFG order (uc, c)
    assert _attention_rows(torch.cat([c, same])) == (0, 3)                   # forward_with_cfg order (c, uc)
    assert _attention_rows(torch.cat([same, c, same])) == (3, 6)             # prefix and suffix
    assert _attention_rows(torch.cat([same, same])) == (6, 6)                # nothing needs attention
    assert _attention_rows(torch.cat([c, c])) is None                        # nothing to skip
    assert _attention_rows(torch.cat([c[:1], same[:1], c[1:]])) is None      # identical sample in the middle: no
    assert _attention_rows(c[:, :1]) is None                                 # a single token is not "identical tokens"
    almost = same.clone()
    almost[1, 2, 3] += 1e-6
    assert _attention_rows(torch.cat([almost, c])) is None                   # exact comparison, nothing assumed
    monkeypatch.setenv("LN3_UNCOND_CLOSED_FORM", "0")
    assert _attention_rows(torch.cat([same, c])) is None


_SCRIPT_UTIL_CHECKOUT = {
    # a stand-in checkout laid out like the reference's: its script_util modules import mirrored and
    # non-mirrored names side by side, as the reference's guided_diffusion/ and nsr/script_util.py do
    "dit/dit_models_xformers.py": "class TextCondDiTBlock:\n    pass\n\n\nclass ImageCondDiTBlock:\n    pass\n",
    "dit/dit_trilatent.py": "DiT_models = {}\n",
    "dit/dit_i23d.py": "DiT_models = {}\n",
    "nsr/triplane.py": "class Triplane:\n    pass\n\n\nclass Triplane_fg_bg_plane(Triplane):\n    pass\n",
    "vit/vit_triplane.py": "from nsr.triplane import Triplane  # noqa: F401  (re-export)\n\n\n"
                           "class ViTTriplaneDecomposed:\n    pass\n",
    "ldm/modules/diffusionmodules/model.py": "class Encoder:\n    pass\n\n\nclass MVEncoder(Encoder):\n    pass\n",
    "nsr/script_util.py": "from vit.vit_triplane import Triplane, ViTTriplaneDecomposed  # noqa: F401\n"
                          "from nsr.triplane import Triplane_fg_bg_plane  # noqa: F401\n"
                          "from ldm.modules.diffusionmodules.model import Encoder, MVEncoder  # noqa: F401\n",
    "guided_diffusion/script_util.py": '''\
from . import gaussian_diffusion as gd
from .respace import SpacedDiffusion, space_timesteps
from dit.dit_models_xformers import TextCondDiTBlock, ImageCondDiTBlock  # noqa: F401
from dit.dit_trilatent import DiT_models as DiT_models_t23d
from dit.dit_i23d import DiT_models as DiT_models_i23d


def model_and_diffusion_defaults():
    return dict(create_dit=False, i23d=False, dit_model_arch="DiT-L/2", context_dim=768, roll_out=False,
                denoise_in_channels=4, denoise_out_channels=4, diffusion_input_size=32, learn_sigma=False,
                mixed_prediction=False, diffusion_steps=1000, timestep_respacing="")


def create_model_and_diffusion(create_dit, i23d, dit_model_arch, context_dim, roll_out, denoise_in_channels,
                               diffusion_input_size, learn_sigma, diffusion_steps, timestep_respacing, **kw):
    assert create_dit
    common = dict(input_size=diffusion_input_size, num_classes=0, learn_sigma=learn_sigma,
                  in_channels=denoise_in_channels, context_dim=context_dim, roll_out=roll_out)
    if i23d:
        model = DiT_models_i23d[dit_model_arch](pooling_ctx_dim=768, **common)
    else:
        model = DiT_models_t23d[dit_model_arch](vit_blk=TextCondDiTBlock, **common)
    diffusion = SpacedDiffusion(use_timesteps=space_timesteps(diffusion_steps, timestep_respacing or str(diffusion_steps)),
                                betas=gd.get_named_beta_schedule("linear", diffusion_steps),
                                model_mean_type=gd.ModelMeanType.EPSILON, model_var_type=gd.ModelVarType.FIXED_LARGE,
                                loss_type=gd.LossType.MSE)
    return model, diffusion
''',
}


def test_overlay_lets_the_reference_script_utils_import(tmp_path):
    """With the hook installed, a checkout's `guided_diffusion/script_util.py` and `nsr/script_util.py` laid out
    like the reference's import: mirrored names resolve to this package, the names the mirrors do not define
    (ViTTriplaneDecomposed, Encoder, MVEncoder, ImageCondDiTBlock, Triplane_fg_bg_plane) fall back to the
    checkout's files, and the checkout's own factory builds the mirrors."""
    import importlib
    import sys
    import pytest
    for rel, text in _SCRIPT_UTIL_CHECKOUT.items():
        d = tmp_path
        for part in rel.split("/")[:-1]:
            d = d / part
            d.mkdir(exist_ok=True)
            (d / "__init__.py").touch()
        (tmp_path / rel).write_text(text)
    prefixes = ("dit", "sgm", "nsr", "guided_diffusion", "transport", "vit", "ldm")
    saved = {k: sys.modules.pop(k) for k in list(sys.modules) if k.split(".")[0] in prefixes}
    saved_path = list(sys.path)
    from ln3diff_b200 import overlay
    sys.path.insert(0, str(tmp_path))
    overlay.install()
    try:
        g = importlib.import_module("guided_diffusion.script_util")
        n = importlib.import_module("nsr.script_util")
        assert g.SpacedDiffusion.__module__.startswith("ln3diff_b200.")
        assert g.TextCondDiTBlock.__module__.startswith("ln3diff_b200.")
        assert g.DiT_models_t23d["DiT-L/2"].__module__.startswith("ln3diff_b200.")
        assert g.DiT_models_i23d["DiT-PixArt-L/2"].__module__.startswith("ln3diff_b200.")
        assert g.ImageCondDiTBlock.__module__ == "dit.dit_models_xformers"            # reference fallback
        assert n.Triplane.__module__.startswith("ln3diff_b200.")                      # re-export resolved to the mirror
        assert n.ViTTriplaneDecomposed.__module__ == "vit.vit_triplane"
        assert n.Encoder.__module__ == "ldm.modules.diffusionmodules.model" and n.MVEncoder is not None
        assert n.Triplane_fg_bg_plane.__module__ == "nsr.triplane"
        with pytest.raises(AttributeError):
            importlib.import_module("dit.dit_trilatent").no_such_name
        # the checkout's own factory, unmodified, now builds the mirrors
        d = g.model_and_diffusion_defaults()
        d.update(dict(create_dit=True, dit_model_arch="DiT-B/2", context_dim=768, roll_out=True, denoise_in_channels=4,
                      denoise_out_channels=4, diffusion_input_size=32, learn_sigma=False, mixed_prediction=False,
                      timestep_respacing="10"))
        model, diffusion = g.create_model_and_diffusion(**d)
        assert type(model).__module__ == "ln3diff_b200.dit.dit_trilatent" and type(model).__name__ == "DiT_TriLatent"
        assert type(diffusion).__module__ == "ln3diff_b200.guided_diffusion.respace" and diffusion.num_timesteps == 10
        d.update(dict(i23d=True, dit_model_arch="DiT-PixArt-B/2", context_dim=1024))
        model, _ = g.create_model_and_diffusion(**d)
        assert type(model).__module__ == "ln3diff_b200.dit.dit_i23d"
    finally:
        overlay.uninstall()
        for k in list(sys.modules):
            if k.split(".")[0] in prefixes:
                del sys.modules[k]
        sys.modules.update(saved)
        sys.path[:] = saved_path
    import ln3diff_b200.dit.dit_trilatent as mirror
    assert "__getattr__" not in mirror.__dict__


def test_dopri5_restatement_solves_known_odes():
    """transport/dopri5.py (restated torchdiffeq dopri5; parity unpinned): closed-form ODEs within a small multiple
    of the tolerance, interpolated output grid, FSAL function-evaluation count (2 for the initial step + 6 per
    attempted step), no step shrink after an accepted step."""
    import math
    from ln3diff_b200.transport.dopri5 import odeint_dopri5
    st = {}
    grid = torch.linspace(0, 1, 11)
    y = odeint_dopri5(lambda t, v: -v, torch.ones(4, dtype=torch.float64), grid, rtol=1e-6, atol=1e-9, stats=st)
    assert y.shape == (11, 4) and torch.equal(y[0], torch.ones(4, dtype=torch.float64))
    assert (y[:, 0] - torch.exp(-grid.double())).abs().max() < 1e-6
    assert st["nfe"] == 2 + 6 * (st["accepted"] + st["rejected"])
    st = {}
    grid = torch.linspace(0, 2, 50)
    y = odeint_dopri5(lambda t, v: math.cos(5 * t) * v, torch.ones(3), grid, rtol=1e-3, atol=1e-6, stats=st)
    assert (y[:, 0] - torch.exp(torch.sin(5 * grid) / 5)).abs().max() < 1e-2 and st["rejected"] >= 1
    # a linear field is integrated exactly by any step: error ratio 0 -> the step grows by ifactor
    y = odeint_dopri5(lambda t, v: torch.full_like(v, 2.0), torch.zeros(2), [0.0, 0.5, 3.0])
    assert torch.allclose(y[:, 0], torch.tensor([0.0, 1.0, 6.0]), atol=1e-5)


def test_sample_ode_default_runs_dopri5_on_cpu_model():
    """`Sampler(transport).sample_ode()` with the reference's DEFAULT arguments (dopri5, 50 points, atol 1e-6,
    rtol 1e-3) runs through the mirror with a closed-form velocity field."""
    from ln3diff_b200.transport import Sampler, create_transport
    fn = Sampler(create_transport(snr_type="lognorm")).sample_ode()
    x0 = torch.randn(2, 3, generator=torch.Generator().manual_seed(0))
    traj = fn(x0, lambda x, t, **kw: -x * t[:, None])
    assert traj.shape == (50, 2, 3)
    assert torch.allclose(traj[-1], x0 * torch.exp(torch.tensor(-0.5)), atol=2e-3)


def test_general_conditioner_routing_cpu():
    """GeneralConditioner host logic (reference sgm/modules/encoders/modules.py:80-190) with stand-in embedders."""
    import torch
    from ln3diff_b200.sgm.modules.encoders.modules import AbstractEmbModel, GeneralConditioner

    class Tok(AbstractEmbModel):
        def __init__(self, d, pooled):
            super().__init__()
            self.d, self.pooled = d, pooled

        def forward(self, x):
            t = x[:, None, None].expand(-1, 5, self.d).float() + 1
            return (t, t[:, 0]) if self.pooled else t

    a, b = Tok(4, True), Tok(6, False)
    a._emb_config = {"input_key": "caption", "ucg_rate": 0.1}
    b._emb_config = {"input_key": "img", "ucg_rate": 0.0}
    cond = GeneralConditioner([a, b])
    batch = {"caption": torch.arange(3), "img": torch.arange(3) * 10}
    c, uc = cond.get_unconditional_conditioning(batch, force_uc_zero_embeddings=["caption"])
    assert c["crossattn"].shape == (3, 5, 10) and c["vector"].shape == (3, 4)      # crossattn concatenated on dim 2
    assert torch.equal(c["crossattn"][..., :4], batch["caption"][:, None, None].expand(-1, 5, 4).float() + 1)
    assert float(uc["crossattn"][..., :4].abs().max()) == 0 and torch.equal(uc["crossattn"][..., 4:], c["crossattn"][..., 4:])
    assert float(uc["vector"].abs().max()) == 0 and a.ucg_rate == 0.1
    import pytest
    with pytest.raises(KeyError):
        bad = Tok(4, False)
        bad._emb_config = {}
        GeneralConditioner([bad])


def test_conditioner_embedders_build_from_reference_layouts_and_refuse_cpu():
    """The three embedders accept state dicts in the key layout the reference objects hold (`transformer.*`,
    `model.visual.*`, dinov2 hub names under `model.`); there is no CPU fallback behind them."""
    import pytest
    import torch
    from ln3diff_b200.sgm.modules.encoders.modules import (FrozenCLIPEmbedder, FrozenDinov2ImageEmbedder,
                                                           FrozenOpenCLIPImageEmbedder)
    from oracle import conditioners as oc
    _, sd = oc.clip_text(depth=2)
    te = FrozenCLIPEmbedder(device="cpu", always_return_pooled=True, state_dict=sd)
    assert len(te.tower.layers) == 2 and te.tower.causal and te.token_embedding.shape == (49408, 768)
    assert te.tower.layers[0].qkv_w.shape == (3 * 768, 768) and te.tower.layers[0].qkv_w.dtype == torch.bfloat16
    _, sdv = oc.clip_vision(depth=1, width=256, mlp=1024, embed=128)
    ce = FrozenOpenCLIPImageEmbedder(device="cpu", output_tokens=True, state_dict=sdv)
    assert ce._conv_w.shape == (256, 640) and ce._embed_dim == 128 and ce.positional_embedding.shape == (257, 256)
    _, sdd = oc.dinov2_reg(depth=1, width=256)
    de = FrozenDinov2ImageEmbedder(device="cpu", state_dict=sdd)
    assert de.register_tokens.shape == (1, 4, 256) and de.tower.layers[0].ls1.shape == (1, 256)
    assert de.interpolate_pos_encoding(16).shape == (1, 257, 256)
    assert de.interpolate_pos_encoding(8).shape == (1, 65, 256)           # bicubic down-interpolation of the table
    if not torch.cuda.is_available():
        with pytest.raises(ValueError, match="CUDA"):
            te(torch.zeros(1, 77, dtype=torch.long))
        with pytest.raises(ValueError, match="CUDA"):
            de(torch.zeros(1, 3, 224, 224))
        from ln3diff_b200 import mesh
        with pytest.raises(ValueError, match="CUDA"):
            mesh.marching_cubes(torch.zeros(4, 4, 4), 0.0)


def test_gelu_polynomial_error_bounds_cpu():
    """The packed-polynomial erf-GELU of the fc1 epilogue (csrc/common.cuh: gelu_erf_poly2), restated in float32 numpy
    with the coefficients parsed from the source: the documented error bounds hold."""
    import math
    import os
    import re
    import numpy as np
    src = open(os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "ln3diff_b200", "csrc", "common.cuh")).read()
    body = src[src.index("void gelu_erf_poly2("):]
    body = body[:body.index("asm(\"fma.rn.sat.f32")]
    coef = [float(c) for c in re.findall(r"pk2\((-?\d\.\d+e[+-]\d+)f,", body)]     # Horner order: highest degree first
    assert len(coef) == 9
    x = np.linspace(-8, 8, 200001).astype(np.float32)
    u = np.minimum(x * x, np.float32(16.0)).astype(np.float32)
    q = np.full_like(x, np.float32(coef[0]))
    for c in coef[1:]:
        q = (q * u + np.float32(c)).astype(np.float32)
    phi = np.clip((x * q + np.float32(0.5)).astype(np.float32), 0.0, 1.0).astype(np.float32)
    g = (x * phi).astype(np.float32)
    ref = np.array([0.5 * v * (1.0 + math.erf(v / math.sqrt(2.0))) for v in x.astype(np.float64)])
    err = np.abs(g - ref)
    inside = np.abs(x) < 3.99
    assert err[inside].max() < 1.2e-5
    assert err.max() < 1.4e-4                                   # the flush to 0 just below x = -4
    big = np.abs(ref) > 1e-2
    assert (err[big] / np.abs(ref[big])).max() < 6e-4
    assert np.all(g[x > 4.01] == x[x > 4.01]) and np.all(g[x < -4.01] == 0)


def test_conditioner_never_substitutes_random_weights_silently():
    """Without state_dict= the embedders call the reference's loaders; offline those fail, and that is an error."""
    import pytest
    from ln3diff_b200.sgm.modules.encoders.modules import FrozenDinov2ImageEmbedder, FrozenOpenCLIPImageEmbedder
    with pytest.raises(RuntimeError, match="pretrained loader failed"):
        FrozenOpenCLIPImageEmbedder(device="cpu")          # open_clip is not installed
    with pytest.raises(RuntimeError, match="pretrained loader failed"):
        FrozenDinov2ImageEmbedder(device="cpu")            # torch.hub needs the network
    m = FrozenDinov2ImageEmbedder(device="cpu", random_init=True, depth=1, width=128)
    assert len(m.tower.layers) == 1
