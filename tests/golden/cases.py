"""Shared description of the golden cases (pure data, no reference / product imports).

``make_golden.py`` instantiates these with the *reference* classes to produce the ``.npz`` fixtures;
the tests instantiate the same cases with the product classes, the oracle and the CUDA engine.
"""
import torch

# ---------------------------------------------------------------- denoiser forward cases
# name -> (class name, ctor kwargs, x shape (without batch), t kind, cond shape or None, oracle kwargs)
NETS = {
    "janner_cfg2": dict(
        cls="JannerUNet1d", ctor=dict(in_dim=14, model_dim=32, emb_dim=32, kernel_size=5, dim_mult=[1, 2, 2, 2]),
        x=(32, 14), t="long", cond=None,
        oracle=dict(fn="janner_unet", emb_dim=32, kernel_size=5, n_stages=4)),
    "janner_kitchen_cond": dict(
        cls="JannerUNet1d", ctor=dict(in_dim=6, model_dim=16, emb_dim=16, kernel_size=3, dim_mult=[1, 4, 2]),
        x=(8, 6), t="float", cond=(16,),
        oracle=dict(fn="janner_unet", emb_dim=16, kernel_size=3, n_stages=3)),
    "chi_small": dict(
        cls="ChiUNet1d", ctor=dict(act_dim=7, obs_dim=20, To=2, model_dim=64, emb_dim=64, kernel_size=5,
                                   dim_mult=[1, 2, 2]),
        x=(16, 7), t="long", cond=(2, 20),
        oracle=dict(fn="chi_unet", emb_dim=64, kernel_size=5, n_stages=3)),
    "chi_cm_fourier": dict(
        cls="ChiUNet1d", ctor=dict(act_dim=3, obs_dim=5, To=2, model_dim=32, emb_dim=32, kernel_size=5,
                                   dim_mult=[1, 2, 2], timestep_emb_type="untrainable_fourier"),
        x=(8, 3), t="float", cond=(2, 5),
        oracle=dict(fn="chi_unet", emb_dim=32, kernel_size=5, n_stages=3, emb_kind="untrainable_fourier")),
    "dit_small": dict(
        cls="DiT1d", ctor=dict(in_dim=9, emb_dim=32, d_model=64, n_heads=2, depth=2, timestep_emb_type="fourier"),
        x=(10, 9), t="float", cond=(32,),
        oracle=dict(fn="dit1d", emb_dim=32, d_model=64, n_heads=2, depth=2, emb_kind="fourier")),
    "dit_pos_uncond": dict(
        cls="DiT1d", ctor=dict(in_dim=4, emb_dim=16, d_model=32, n_heads=1, depth=1),
        x=(7, 4), t="long", cond=None,
        oracle=dict(fn="dit1d", emb_dim=16, d_model=32, n_heads=1, depth=1)),
    "idql_small": dict(
        cls="IDQLMlp", ctor=dict(obs_dim=11, act_dim=3, emb_dim=32, hidden_dim=64, n_blocks=2),
        x=(3,), t="long", cond=(11,),
        oracle=dict(fn="idql_mlp", emb_dim=32, obs_dim=11, n_blocks=2)),
    "dvinv_small": dict(
        cls="DVInvMlp", ctor=dict(obs_dim=5, act_dim=3, emb_dim=16, hidden_dim=64),
        x=(3,), t="long", cond=(10,),
        oracle=dict(fn="dvinv_mlp", emb_dim=16)),
    "sfbc_small": dict(
        cls="SfBCUNet", ctor=dict(act_dim=3, emb_dim=32, hidden_dims=[64, 32, 32]),
        x=(3,), t="float", cond=(32,),
        oracle=dict(fn="sfbc_unet", emb_dim=32, n_layers=3)),
    "sfbc_uncond": dict(
        cls="SfBCUNet", ctor=dict(act_dim=6, emb_dim=16, hidden_dims=[32, 16]),
        x=(6,), t="float", cond=None,
        oracle=dict(fn="sfbc_unet", emb_dim=16, n_layers=2)),
    "pearce_small": dict(
        cls="PearceMlp", ctor=dict(act_dim=3, To=2, emb_dim=32, hidden_dim=64),
        x=(3,), t="float", cond=(2, 32),
        oracle=dict(fn="pearce_mlp", emb_dim=32, To=2)),
    "pearce_uncond_long_t": dict(
        cls="PearceMlp", ctor=dict(act_dim=6, To=1, emb_dim=16, hidden_dim=32),
        x=(6,), t="long", cond=None,
        oracle=dict(fn="pearce_mlp", emb_dim=16, To=1)),
    "dql_cfg1": dict(
        cls="DQLMlp", ctor=dict(obs_dim=11, act_dim=3, emb_dim=64),
        x=(3,), t="long", cond=(11,),
        oracle=dict(fn="dql_mlp", emb_dim=64, obs_dim=11)),
}
NET_BATCH = 3


def module_names(m):
    """(public instance attribute names, names the class defines below nn.Module) of a module, both sorted: what an instance
    offers the lowering besides its sub-modules, parameters and buffers."""
    mro = type(m).__mro__
    own = {k for base in mro[:mro.index(torch.nn.Module)] for k in vars(base) if not (k.startswith("__") and k.endswith("__"))}
    return sorted(k for k in vars(m) if not k.startswith("_")), sorted(own)


def net_inputs(case: dict, seed: int = 1):
    g = torch.Generator().manual_seed(seed)
    x = torch.randn((NET_BATCH, *case["x"]), generator=g)
    if case["t"] == "long":
        t = torch.tensor([0, 7, 63][:NET_BATCH], dtype=torch.long)
    else:
        t = torch.tensor([0.001, 0.37, 0.9946][:NET_BATCH], dtype=torch.float32)
    cond = None if case["cond"] is None else torch.randn((NET_BATCH, *case["cond"]), generator=g)
    return x, t, cond


# ---------------------------------------------------------------- sampler cases
SOLVERS = ["ddpm", "ddim", "ode_dpmsolver_1", "ode_dpmsolver++_1", "ode_dpmsolver++_2M",
           "sde_dpmsolver_1", "sde_dpmsolver++_1", "sde_dpmsolver++_2M"]

# tiny denoisers used under the samplers (fast on CPU, exercise mask/clip shapes)
SAMPLER_NETS = {
    "janner_tiny": dict(
        cls="JannerUNet1d", ctor=dict(in_dim=5, model_dim=8, emb_dim=8, kernel_size=3, dim_mult=[1, 2]),
        x=(8, 5), oracle=dict(fn="janner_unet", emb_dim=8, kernel_size=3, n_stages=2)),
    "dql_tiny": dict(
        cls="DQLMlp", ctor=dict(obs_dim=4, act_dim=3, emb_dim=16),
        x=(3,), oracle=dict(fn="dql_mlp", emb_dim=16, obs_dim=4)),
    "pearce_tiny": dict(
        cls="PearceMlp", ctor=dict(act_dim=3, To=1, emb_dim=8, hidden_dim=32),
        x=(3,), oracle=dict(fn="pearce_mlp", emb_dim=8, To=1)),
    "sfbc_tiny": dict(
        cls="SfBCUNet", ctor=dict(act_dim=3, emb_dim=8, hidden_dims=[32, 16]),
        x=(3,), oracle=dict(fn="sfbc_unet", emb_dim=8, n_layers=2)),
    "dvinv_tiny": dict(
        cls="DVInvMlp", ctor=dict(obs_dim=2, act_dim=3, emb_dim=8, hidden_dim=32),
        x=(3,), oracle=dict(fn="dvinv_mlp", emb_dim=8)),
}
SAMPLER_BATCH = 6


def sampler_cases():
    """Yield (name, spec).  Every solver x {discrete S==T (duplicated index, r=inf), discrete S<T with
    Diffusion-X, continuous} x predict_noise, plus CFG / warm-start / schedule variants."""
    out = {}
    for sv in SOLVERS:
        tag = sv.replace("+", "p")
        for pn in (True, False):
            p = "eps" if pn else "x0"
            out[f"disc_dup_{tag}_{p}"] = dict(
                kind="discrete", net="janner_tiny", solver=sv, predict_noise=pn, T=10, steps=10,
                fix_mask="first_row", clip=True, w_cfg=0.0, cond=None, temperature=0.5)
            out[f"disc_dx_{tag}_{p}"] = dict(
                kind="discrete", net="dql_tiny", solver=sv, predict_noise=pn, T=50, steps=4, diffusion_x=2,
                fix_mask=None, clip=True, w_cfg=1.0, cond="obs", temperature=1.0, step_schedule="quad")
            out[f"cont_{tag}_{p}"] = dict(
                kind="continuous", net="janner_tiny", solver=sv, predict_noise=pn, steps=5,
                fix_mask="first_row", clip=pn, w_cfg=1.0, cond="emb", temperature=0.5, schedule="linear")
    out["cont_cfg2branch_2M"] = dict(
        kind="continuous", net="janner_tiny", solver="ode_dpmsolver++_2M", predict_noise=True, steps=6,
        fix_mask="first_row", clip=True, w_cfg=2.5, cond="mlp", temperature=0.5, schedule="linear")
    out["disc_cfg2branch_ddpm"] = dict(
        kind="discrete", net="dql_tiny", solver="ddpm", predict_noise=True, T=20, steps=5,
        fix_mask=None, clip=True, w_cfg=1.7, cond="obs", temperature=1.0)
    out["disc_warm_ddim"] = dict(
        kind="discrete", net="janner_tiny", solver="ddim", predict_noise=True, T=40, steps=4,
        fix_mask="first_row", clip=False, w_cfg=0.0, cond=None, temperature=1.0, warm=0.5,
        step_schedule="quad_cos")
    out["cont_warm_sde"] = dict(
        kind="continuous", net="janner_tiny", solver="sde_dpmsolver++_1", predict_noise=False, steps=4,
        fix_mask=None, clip=True, w_cfg=0.0, cond=None, temperature=1.0, warm=0.4,
        step_schedule="cat_cos_continuous")
    # the SfBC / Decision-Veteran patterns: continuous-time SDE sampler over the U-shaped residual MLP (condition = an embedding
    # added to the time code) and over the inverse-dynamics MLP (condition = two stacked observations)
    out["cont_sfbc_2M_eps"] = dict(
        kind="continuous", net="sfbc_tiny", solver="ode_dpmsolver++_2M", predict_noise=True, steps=5,
        fix_mask=None, clip=True, w_cfg=1.0, cond="emb", temperature=1.0, schedule="linear")
    out["disc_dvinv_ddpm_x0"] = dict(
        kind="discrete", net="dvinv_tiny", solver="ddpm", predict_noise=False, T=8, steps=8,
        fix_mask=None, clip=True, w_cfg=1.0, cond="obs", temperature=1.0)
    return out


def edm_cases():
    """ContinuousEDM.sample cases: both solvers x {plain, clip + fix_mask + Diffusion-X, two-branch CFG, warm start}."""
    out = {}
    for sv in ("euler", "heun"):
        out[f"edm_{sv}_plain"] = dict(net="janner_tiny", solver=sv, steps=5, fix_mask=None, clip=False, w_cfg=0.0, cond=None,
                                      temperature=1.0)
        out[f"edm_{sv}_mask_clip_dx"] = dict(net="janner_tiny", solver=sv, steps=4, fix_mask="first_row", clip=True, w_cfg=1.0,
                                             cond="emb", temperature=0.5, diffusion_x=2)
        out[f"edm_{sv}_cfg2branch"] = dict(net="dql_tiny", solver=sv, steps=6, fix_mask=None, clip=True, w_cfg=1.7, cond="obs",
                                           temperature=1.0)
    out["edm_heun_warm"] = dict(net="janner_tiny", solver="heun", steps=4, fix_mask="first_row", clip=False, w_cfg=0.0, cond=None,
                                temperature=1.0, warm=0.4)
    return out


def legacy_cases():
    """Legacy DDPM class (ddpm.py): ancestral sampling and Diffusion-X (sample_x), both parameterisations."""
    return {
        "ddpm_eps_mask_clip": dict(net="janner_tiny", predict_noise=True, T=10, fix_mask="first_row", clip=True, w_cfg=1.0, cond="emb",
                                   temperature=0.5, extra=0, beta_schedule="cosine"),
        "ddpm_x0_linear": dict(net="janner_tiny", predict_noise=False, T=8, fix_mask=None, clip=True, w_cfg=0.0, cond=None,
                               temperature=1.0, extra=0, beta_schedule="linear"),
        "ddpm_x_eps_extra": dict(net="dql_tiny", predict_noise=True, T=6, fix_mask=None, clip=True, w_cfg=1.0, cond="obs",
                                 temperature=1.0, extra=3, beta_schedule="cosine"),
        "ddpm_x_x0_cfg2branch": dict(net="dql_tiny", predict_noise=False, T=6, fix_mask=None, clip=False, w_cfg=1.6, cond="obs",
                                     temperature=1.0, extra=2, beta_schedule="cosine"),
        # the Diffusion-BC pattern (pipelines/dbc_*.py): legacy DDPM over PearceMlp, observation embedding as condition, sample_x
        "ddpm_x_pearce_dbc": dict(net="pearce_tiny", predict_noise=True, T=8, fix_mask=None, clip=True, w_cfg=1.0, cond="emb",
                                  temperature=1.0, extra=2, beta_schedule="cosine"),
    }


def rf_cases():
    """Rectified flow (rectifiedflow.py): discrete and continuous time, CFG regimes, Diffusion-X repeats, warm start, final clip."""
    return {
        "rf_disc_plain": dict(kind="discrete", net="janner_tiny", T=20, steps=5, fix_mask="first_row", clip=False, w_cfg=0.0, cond=None,
                              temperature=0.5),
        "rf_disc_cond_clip_dx": dict(kind="discrete", net="dql_tiny", T=30, steps=4, fix_mask=None, clip=True, w_cfg=1.0, cond="obs",
                                     temperature=1.0, diffusion_x=2, step_schedule="quad"),
        "rf_cont_cfg2branch": dict(kind="continuous", net="janner_tiny", steps=6, fix_mask="first_row", clip=True, w_cfg=2.0, cond="emb",
                                   temperature=1.0),
        "rf_cont_warm": dict(kind="continuous", net="janner_tiny", steps=4, fix_mask=None, clip=False, w_cfg=0.0, cond=None,
                             temperature=1.0, warm=0.4),
    }


def legacy_edm_cases():
    """Legacy EDM class (edm.py): Euler / Heun over the descending Karras grid, CFG regimes, fix_mask, sample_x extra steps."""
    return {
        "ledm_euler_plain": dict(net="janner_tiny", solver="euler", steps=5, fix_mask=None, w_cfg=0.0, cond=None, extra=0),
        "ledm_heun_mask_cond": dict(net="janner_tiny", solver="heun", steps=6, fix_mask="first_row", w_cfg=1.0, cond="emb", extra=0),
        "ledm_heun_cfg2branch_x": dict(net="dql_tiny", solver="heun", steps=4, fix_mask=None, w_cfg=1.5, cond="obs", extra=3),
    }


def guided_cases():
    """Classifier-guided sampling (diffusionsde.py:153-173, :597-606) with cleandiffuser_b200.testing.ToyClassifier attached:
    the Diffuser pattern (x0-prediction, DDPM, fix_mask, w_cg = 0.3) and eps-prediction with a condition branch."""
    return {
        "cg_disc_ddpm_x0": dict(kind="discrete", net="janner_tiny", solver="ddpm", predict_noise=False, T=10, steps=10,
                                fix_mask="first_row", clip=False, w_cfg=0.0, cond=None, temperature=0.5, w_cg=0.3),
        "cg_disc_ddim_eps_clip": dict(kind="discrete", net="janner_tiny", solver="ddim", predict_noise=True, T=20, steps=5,
                                      fix_mask="first_row", clip=True, w_cfg=0.0, cond=None, temperature=1.0, w_cg=0.7),
        "cg_cont_2M_eps_cond": dict(kind="continuous", net="janner_tiny", solver="ode_dpmsolver++_2M", predict_noise=True, steps=5,
                                    fix_mask=None, clip=True, w_cfg=1.0, cond="emb", temperature=0.5, schedule="linear", w_cg=0.4),
    }


def sampler_inputs(spec: dict, seed: int = 1):
    """prior / condition / masks for a sampler case (deterministic)."""
    g = torch.Generator().manual_seed(seed)
    net = SAMPLER_NETS[spec["net"]]
    xs = net["x"]
    prior = torch.zeros((SAMPLER_BATCH, *xs))
    fix_mask = None
    if spec.get("fix_mask") == "first_row":
        fix_mask = torch.zeros(xs)
        fix_mask[0, :3] = 1.
        prior[:, 0, :3] = torch.randn((SAMPLER_BATCH, 3), generator=g)
    cond = None
    if spec["cond"] == "obs":
        cond = torch.randn((SAMPLER_BATCH, 4), generator=g)
    elif spec["cond"] == "emb":
        cond = torch.randn((SAMPLER_BATCH, 8), generator=g)
    elif spec["cond"] == "mlp":
        cond = torch.rand((SAMPLER_BATCH, 1), generator=g)
    x_max = x_min = None
    if spec.get("clip"):
        x_max = torch.ones((1, *xs)) * 1.0
        x_min = torch.ones((1, *xs)) * -1.0
    warm = None
    if spec.get("warm") is not None:
        warm = torch.randn((SAMPLER_BATCH, *xs), generator=g) * 0.5
    return dict(prior=prior, fix_mask=fix_mask, cond=cond, x_max=x_max, x_min=x_min, warm=warm)
