"""Generate the golden fixtures by running the UNMODIFIED reference (CPU, fp32).

    python tests/golden/make_golden.py            # needs /root/reference; writes tests/golden/*.npz

The reference's own tests contain no numeric vectors for the sampling path (SURVEY 8c), so these
files are the pins: reference class + synthetic weights (``cleandiffuser_b200.testing.synth_state_dict``,
a recipe over the state-dict template, so no weights need to be stored) + fixed inputs (+ a recorded
noise tape for samplers) -> outputs.  /root/reference is only ever read here, never at test time.
"""
import os
import sys

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
sys.path.insert(0, "/root/reference")

import cases  # noqa: E402
from cleandiffuser_b200.testing import NoiseTape, ToyClassifier, state_checksum, synth_state_dict  # noqa: E402

import cleandiffuser.nn_diffusion as ref_nn  # noqa: E402
import cleandiffuser.nn_condition as ref_cond  # noqa: E402
from cleandiffuser.diffusion import ContinuousDiffusionSDE, DiscreteDiffusionSDE  # noqa: E402
from cleandiffuser.diffusion.consistency_model import ContinuousConsistencyModel  # noqa: E402
from cleandiffuser.diffusion.newedm import ContinuousEDM  # noqa: E402
from cleandiffuser.utils import (SUPPORTED_NOISE_SCHEDULES, SUPPORTED_SAMPLING_STEP_SCHEDULE,  # noqa: E402
                                 SUPPORTED_TIMESTEP_EMBEDDING, SinusoidalEmbedding)


def build_net(case):
    net = getattr(ref_nn, case["cls"])(**case["ctor"])
    sd = synth_state_dict(net.state_dict(), seed=0)
    net.load_state_dict(sd)
    return net.eval(), sd


def gen_nets():
    out = {}
    for name, case in cases.NETS.items():
        net, sd = build_net(case)
        x, t, cond = cases.net_inputs(case)
        with torch.no_grad():
            y = net(x, t, cond)
        out[name + "/y"] = y.numpy()
        out[name + "/checksum"] = np.array(state_checksum(sd))
        out[name + "/keys"] = np.array(["%s|%s" % (k, ",".join(map(str, v.shape))) for k, v in sd.items()])
    np.savez_compressed(os.path.join(HERE, "nets.npz"), **out)
    print("nets.npz", len(out))


def gen_tables():
    out = {}
    for T in (5, 10, 100):
        grid = torch.linspace(1e-3, 1.0, T)
        for kind in ("linear", "cosine"):
            a, s = SUPPORTED_NOISE_SCHEDULES[kind]["forward"](grid)
            out[f"alpha/{kind}/{T}"], out[f"sigma/{kind}/{T}"] = a.numpy(), s.numpy()
    for name, fn in SUPPORTED_SAMPLING_STEP_SCHEDULE.items():
        for (T, S) in ((100, 100), (100, 20), (1000, 7)):
            span = [1e-3, 0.9946] if name.endswith("continuous") else T
            out[f"steps/{name}/{T}_{S}"] = fn(span, S).numpy()
    tl, tf = torch.tensor([0, 3, 99]), torch.tensor([0.001, 0.5, 1.0])
    for kind in ("positional", "untrainable_positional"):
        emb = SUPPORTED_TIMESTEP_EMBEDDING[kind](32)
        out[f"emb/{kind}/long"], out[f"emb/{kind}/float"] = emb(tl).numpy(), emb(tf).numpy()
    out["emb/sinusoidal/long"] = SinusoidalEmbedding(32)(torch.arange(10)).numpy()
    out["emb/sinusoidal/float"] = SinusoidalEmbedding(32)(torch.arange(10).float()).numpy()
    np.savez_compressed(os.path.join(HERE, "tables.npz"), **out)
    print("tables.npz", len(out))


def build_condition(spec):
    if spec["cond"] == "mlp":
        nc = ref_cond.MLPCondition(1, 8, [8], torch.nn.SiLU(), dropout=0.25)
        nc.load_state_dict(synth_state_dict(nc.state_dict(), seed=3))
        return nc
    if spec["cond"] in ("obs", "emb"):
        return ref_cond.IdentityCondition(dropout=0.0)
    return None


def gen_samplers():
    out = {}
    for name, spec in cases.sampler_cases().items():
        net, _ = build_net(cases.SAMPLER_NETS[spec["net"]])
        inp = cases.sampler_inputs(spec)
        common = dict(nn_condition=build_condition(spec), fix_mask=inp["fix_mask"], x_max=inp["x_max"],
                      x_min=inp["x_min"], predict_noise=spec["predict_noise"], device="cpu",
                      noise_schedule=spec.get("schedule", "cosine"))
        if spec["kind"] == "discrete":
            agent = DiscreteDiffusionSDE(net, diffusion_steps=spec["T"], **common)
            sched = spec.get("step_schedule", "uniform")
        else:
            agent = ContinuousDiffusionSDE(net, **common)
            sched = spec.get("step_schedule", "uniform_continuous")
        agent.model_ema.eval()
        kw = dict(solver=spec["solver"], n_samples=cases.SAMPLER_BATCH, sample_steps=spec["steps"],
                  sample_step_schedule=sched, use_ema=True, temperature=spec["temperature"],
                  condition_cfg=inp["cond"], w_cfg=spec["w_cfg"],
                  diffusion_x_sampling_steps=spec.get("diffusion_x", 0))
        if inp["warm"] is not None:
            kw.update(warm_start_reference=inp["warm"], warm_start_forward_level=spec["warm"])
        tape = NoiseTape()
        with tape.active(), torch.no_grad():
            x0, log = agent.sample(inp["prior"], **kw)
        out[name + "/x0"] = x0.numpy()
        for j, z in enumerate(tape.draws):
            out[f"{name}/z{j}"] = z.numpy()
        out[name + "/n_draws"] = np.array(len(tape.draws))
    np.savez_compressed(os.path.join(HERE, "samplers.npz"), **out)
    print("samplers.npz", len(out))


def gen_consistency():
    out = {}
    case = cases.NETS["chi_cm_fourier"]
    for steps in (1, 3):
        net, _ = build_net(case)
        cm = ContinuousConsistencyModel(net, ref_cond.IdentityCondition(dropout=0.0),
                                        x_max=torch.ones(1, 8, 3), x_min=-torch.ones(1, 8, 3), device="cpu")
        g = torch.Generator().manual_seed(5)
        prior = torch.zeros(4, 8, 3)
        cond = torch.randn((4, 2, 5), generator=g)
        tape = NoiseTape()
        with tape.active(), torch.no_grad():
            x0, _ = cm.sample(prior, n_samples=4, sample_steps=steps, condition_cfg=cond, w_cfg=1.0)
        out[f"cm{steps}/x0"], out[f"cm{steps}/cond"] = x0.numpy(), cond.numpy()
        for j, z in enumerate(tape.draws):
            out[f"cm{steps}/z{j}"] = z.numpy()
        out[f"cm{steps}/n_draws"] = np.array(len(tape.draws))
    np.savez_compressed(os.path.join(HERE, "consistency.npz"), **out)
    print("consistency.npz", len(out))


def gen_guided():
    out = {}
    for name, spec in cases.guided_cases().items():
        ncase = cases.SAMPLER_NETS[spec["net"]]
        net, _ = build_net(ncase)
        inp = cases.sampler_inputs(spec)
        common = dict(nn_condition=build_condition(spec), fix_mask=inp["fix_mask"], x_max=inp["x_max"], x_min=inp["x_min"],
                      predict_noise=spec["predict_noise"], device="cpu", noise_schedule=spec.get("schedule", "cosine"),
                      classifier=ToyClassifier(ncase["x"]))
        if spec["kind"] == "discrete":
            agent = DiscreteDiffusionSDE(net, diffusion_steps=spec["T"], **common)
            sched = "uniform"
        else:
            agent = ContinuousDiffusionSDE(net, **common)
            sched = "uniform_continuous"
        agent.model_ema.eval()
        tape = NoiseTape()
        with tape.active():
            x0, log = agent.sample(inp["prior"], solver=spec["solver"], n_samples=cases.SAMPLER_BATCH, sample_steps=spec["steps"],
                                   sample_step_schedule=sched, use_ema=True, temperature=spec["temperature"],
                                   condition_cfg=inp["cond"], w_cfg=spec["w_cfg"], w_cg=spec["w_cg"])
        out[name + "/x0"] = x0.detach().numpy()
        if log.get("log_p") is not None:
            out[name + "/log_p"] = log["log_p"].detach().numpy()
        for j, z in enumerate(tape.draws):
            out[f"{name}/z{j}"] = z.numpy()
        out[name + "/n_draws"] = np.array(len(tape.draws))
    np.savez_compressed(os.path.join(HERE, "guided.npz"), **out)
    print("guided.npz", len(out))


def gen_legacy():
    from cleandiffuser.diffusion.ddpm import DDPM
    out = {}
    for name, spec in cases.legacy_cases().items():
        net, _ = build_net(cases.SAMPLER_NETS[spec["net"]])
        inp = cases.sampler_inputs(spec)
        agent = DDPM(net, build_condition(spec), fix_mask=inp["fix_mask"], x_max=inp["x_max"], x_min=inp["x_min"],
                     predict_noise=spec["predict_noise"], diffusion_steps=spec["T"], beta_schedule=spec["beta_schedule"], device="cpu")
        agent.model_ema.eval()
        kw = dict(n_samples=cases.SAMPLER_BATCH, sample_steps=spec["T"], use_ema=True, temperature=spec["temperature"],
                  condition_cfg=inp["cond"], w_cfg=spec["w_cfg"])
        tape = NoiseTape()
        with tape.active(), torch.no_grad():
            if spec["extra"]:
                x0, log = agent.sample_x(inp["prior"], extra_sample_steps=spec["extra"], **kw)
            else:
                x0, log = agent.sample(inp["prior"], **kw)
        out[name + "/x0"] = x0.numpy()
        for j, z in enumerate(tape.draws):
            out[f"{name}/z{j}"] = z.numpy()
        out[name + "/n_draws"] = np.array(len(tape.draws))
    np.savez_compressed(os.path.join(HERE, "legacy.npz"), **out)
    print("legacy.npz", len(out))


def gen_rf():
    from cleandiffuser.diffusion.rectifiedflow import ContinuousRectifiedFlow, DiscreteRectifiedFlow
    out = {}
    for name, spec in cases.rf_cases().items():
        net, _ = build_net(cases.SAMPLER_NETS[spec["net"]])
        inp = cases.sampler_inputs(spec)
        common = dict(nn_condition=build_condition(spec), fix_mask=inp["fix_mask"], x_max=inp["x_max"], x_min=inp["x_min"], device="cpu")
        if spec["kind"] == "discrete":
            agent, sched = DiscreteRectifiedFlow(net, diffusion_steps=spec["T"], **common), spec.get("step_schedule", "uniform")
        else:
            agent, sched = ContinuousRectifiedFlow(net, **common), spec.get("step_schedule", "uniform_continuous")
        agent.model_ema.eval()
        kw = dict(n_samples=cases.SAMPLER_BATCH, sample_steps=spec["steps"], sample_step_schedule=sched, use_ema=True,
                  temperature=spec["temperature"], condition_cfg=inp["cond"], w_cfg=spec["w_cfg"],
                  diffusion_x_sampling_steps=spec.get("diffusion_x", 0))
        if inp["warm"] is not None:
            kw.update(warm_start_reference=inp["warm"], warm_start_forward_level=spec["warm"])
        tape = NoiseTape()
        with tape.active(), torch.no_grad():
            x0, log = agent.sample(inp["prior"], **kw)
        out[name + "/x0"] = x0.numpy()
        for j, z in enumerate(tape.draws):
            out[f"{name}/z{j}"] = z.numpy()
        out[name + "/n_draws"] = np.array(len(tape.draws))
    np.savez_compressed(os.path.join(HERE, "rf.npz"), **out)
    print("rf.npz", len(out))


def gen_legacy_edm():
    from cleandiffuser.diffusion.edm import EDM
    out = {}
    for name, spec in cases.legacy_edm_cases().items():
        net, _ = build_net(cases.SAMPLER_NETS[spec["net"]])
        inp = cases.sampler_inputs(dict(spec, clip=False))
        agent = EDM(net, build_condition(spec), fix_mask=inp["fix_mask"], device="cpu")
        agent.model_ema.eval()
        kw = dict(n_samples=cases.SAMPLER_BATCH, sample_steps=spec["steps"], use_ema=True, solver=spec["solver"],
                  condition_cfg=inp["cond"], w_cfg=spec["w_cfg"])
        tape = NoiseTape()
        with tape.active(), torch.no_grad():
            if spec["extra"]:
                x0, log = agent.sample_x(inp["prior"], extra_sample_steps=spec["extra"], **kw)
            else:
                x0, log = agent.sample(inp["prior"], **kw)
        out[name + "/x0"] = x0.numpy()
        for j, z in enumerate(tape.draws):
            out[f"{name}/z{j}"] = z.numpy()
        out[name + "/n_draws"] = np.array(len(tape.draws))
    np.savez_compressed(os.path.join(HERE, "legacy_edm.npz"), **out)
    print("legacy_edm.npz", len(out))


def gen_edm():
    out = {}
    for name, spec in cases.edm_cases().items():
        net, _ = build_net(cases.SAMPLER_NETS[spec["net"]])
        inp = cases.sampler_inputs(spec)
        agent = ContinuousEDM(net, build_condition(spec), fix_mask=inp["fix_mask"], x_max=inp["x_max"], x_min=inp["x_min"],
                              device="cpu")
        agent.model_ema.eval()
        kw = dict(solver=spec["solver"], n_samples=cases.SAMPLER_BATCH, sample_steps=spec["steps"], use_ema=True,
                  temperature=spec["temperature"], condition_cfg=inp["cond"], w_cfg=spec["w_cfg"],
                  diffusion_x_sampling_steps=spec.get("diffusion_x", 0))
        if inp["warm"] is not None:
            kw.update(warm_start_reference=inp["warm"], warm_start_forward_level=spec["warm"])
        tape = NoiseTape()
        with tape.active(), torch.no_grad():
            x0, log = agent.sample(inp["prior"], **kw)
        out[name + "/x0"] = x0.numpy()
        for j, z in enumerate(tape.draws):
            out[f"{name}/z{j}"] = z.numpy()
        out[name + "/n_draws"] = np.array(len(tape.draws))
    np.savez_compressed(os.path.join(HERE, "edm.npz"), **out)
    print("edm.npz", len(out))


def module_tree(net):
    """[path, class module, class name, {param: shape}, {buffer: shape}, {plain attribute: value}, public attribute names,
    class-defined names] per sub-module, in ``named_modules`` order: everything structural the lowering can read from an
    instance.  The two name lists are recorded for the reference's own classes only (None for torch classes)."""
    plain = (int, float, bool, str, type(None))
    rows = []
    for path, m in net.named_modules():
        attrs = {k: list(v) if isinstance(v, tuple) else v for k, v in vars(m).items()
                 if not k.startswith("_") and k != "training"
                 and (isinstance(v, plain) or isinstance(v, (tuple, list)) and all(isinstance(e, plain) for e in v))}
        names = cases.module_names(m) if type(m).__module__.startswith("cleandiffuser.") else (None, None)
        rows.append([path, type(m).__module__, type(m).__name__,
                     {k: list(p.shape) for k, p in m.named_parameters(recurse=False)},
                     {k: list(b.shape) for k, b in m.named_buffers(recurse=False)}, attrs, *names])
    return rows


def diffusion_layout():
    """{module: {class name: defining module}} for ``cleandiffuser.diffusion`` and each of its sub-modules: every
    reference class bound there, defined or imported."""
    import importlib
    import pkgutil
    import cleandiffuser.diffusion as pkg
    layout = {}
    for name in [pkg.__name__] + [f"{pkg.__name__}.{m.name}" for m in pkgutil.iter_modules(pkg.__path__)]:
        mod = importlib.import_module(name)
        layout[name] = {k: v.__module__ for k, v in vars(mod).items()
                        if isinstance(v, type) and v.__module__.startswith("cleandiffuser.")}
    return layout


def gen_reference_modules():
    """The module trees of the reference's own backbone instances (the NETS cases and the sampler nets) and the layout of
    its ``diffusion`` package, so that tests/test_reference_instances_cpu.py can rebuild instances with the reference's
    structure and class identity, and a package with the reference's layout for ``install()``."""
    import json
    out = {}
    for name, case in list(cases.NETS.items()) + [("sampler/" + k, v) for k, v in cases.SAMPLER_NETS.items()]:
        out[name] = np.array(json.dumps(module_tree(getattr(ref_nn, case["cls"])(**case["ctor"])), separators=(",", ":")))
    out["layout/diffusion"] = np.array(json.dumps(diffusion_layout(), separators=(",", ":")))
    np.savez_compressed(os.path.join(HERE, "reference_modules.npz"), **out)
    print("reference_modules.npz", len(out))


if __name__ == "__main__":
    torch.set_num_threads(1)
    only = sys.argv[1:]
    for fn in (gen_tables, gen_nets, gen_samplers, gen_consistency, gen_edm, gen_guided, gen_legacy, gen_rf, gen_legacy_edm,
               gen_reference_modules):
        if not only or fn.__name__[4:] in only:
            fn()
