"""Drop-in boundary against the reference's own classes (SURVEY 8b): modules built from the reference's classes must lower
to the engine's operator program with no fallback, and ``cleandiffuser_b200.install()`` must let the call sequence of a
pipeline that imports from ``cleandiffuser`` run on this package's sampler classes.

The reference's instances are stood in for by instances with the reference's structure AND class identity:
``tests/golden/reference_modules.npz`` holds the module tree of the reference's own instance of every case (written by
``make_golden.py::gen_reference_modules``: module paths, class modules and names, parameter and buffer shapes, plain
attributes).  This package's module of the same case is checked against that tree, then every sub-module the reference
defines is re-classed to a class of the reference's name and module that derives from ``nn.Module`` only, so that the
lowering can only recognise it the way it recognises a reference instance (structurally), never through this package's
classes.  The lowered programs run on the numpy interpreter of the ABI (tests/emulator.py); the kernels are the same ones
the GPU parity tests check.

The same fixture records the layout of the reference's ``cleandiffuser.diffusion`` package (which module binds which
class, and where each class is defined).  ``install()`` runs against a stand-in package built from that record, not from
the overlay's own target list.  The pipeline's call sequence there uses a toy classifier in place of the reference's
CumRewClassifier over HalfJannerUNet1d and leaves out ``report_parameters``, so the reference's real classifier path is
not covered here.
"""
import json
import os
import sys
import types

import numpy as np
import pytest
import torch
from torch import nn

import cases
import emulator
from cleandiffuser_b200 import nn_diffusion as pnn
from cleandiffuser_b200 import overlay
from cleandiffuser_b200.engine import runtime
from cleandiffuser_b200.testing import ToyClassifier, synth_state_dict

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TREES = np.load(os.path.join(ROOT, "tests", "golden", "reference_modules.npz"), allow_pickle=False)
_FOREIGN = {}


def _foreign_class(cls, module, name):
    """A class named ``module.name`` deriving from nn.Module only, with the methods of ``cls`` (and of its bases below
    nn.Module)."""
    key = (cls, module, name)
    if key not in _FOREIGN:
        ns = {}
        for base in reversed(cls.__mro__[:cls.__mro__.index(nn.Module)]):
            ns.update({k: v for k, v in vars(base).items() if k not in ("__dict__", "__weakref__")})
        ns.update(__module__=module, __qualname__=name)
        _FOREIGN[key] = type(name, (nn.Module,), ns)
    return _FOREIGN[key]


def reference_instance(tree_name, net):
    """This package's module ``net``, checked against the reference's recorded tree ``tree_name`` and re-classed to it.
    The re-classed modules keep this package's attributes and methods; the check makes sure those are exactly the names the
    reference's instance has."""
    tree = json.loads(str(TREES[tree_name]))
    mods = list(net.named_modules())
    assert [p for p, _ in mods] == [row[0] for row in tree], "module paths differ from the reference's"
    for (path, m), (_, module, name, params, buffers, attrs, attr_names, own_names) in zip(mods, tree):
        assert {k: list(p.shape) for k, p in m.named_parameters(recurse=False)} == params, path
        assert {k: list(b.shape) for k, b in m.named_buffers(recurse=False)} == buffers, path
        for k, v in attrs.items():
            got = getattr(m, k)
            assert (list(got) if isinstance(got, tuple) else got) == v, (path, k, got, v)
        if module.startswith("cleandiffuser."):
            # nothing more and nothing less than the reference's class offers: instance attributes, methods
            assert list(cases.module_names(m)) == [attr_names, own_names], (path, cases.module_names(m), attr_names, own_names)
            m.__class__ = _foreign_class(type(m), module, name)
        else:                                          # a torch class: the reference uses it as it is
            assert (type(m).__module__, type(m).__name__) == (module, name), path
    return net


@pytest.fixture()
def ref(monkeypatch):
    """Builds reference-identity instances; the engine runs on the emulator, and any fallback to the PyTorch loop raises."""
    monkeypatch.setattr(runtime, "_device_ok", lambda device: True)
    monkeypatch.setattr(runtime, "_make_handle", lambda device, ops, n: emulator.Handle(ops, n))
    monkeypatch.setenv("CDS_BACKEND", "cuda")
    return reference_instance


@pytest.mark.parametrize("math", ["fp32", "tf32"])
@pytest.mark.parametrize("name", list(cases.NETS))
def test_reference_backbone_instances_lower_without_fallback(golden, ref, name, math, monkeypatch):
    """JannerUNet1d / ChiUNet1d / DiT1d / DQLMlp ... with the reference's class identity through ``engine_forward``."""
    monkeypatch.setenv("CDS_MATH", math)
    case = cases.NETS[name]
    net = ref(name, getattr(pnn, case["cls"])(**case["ctor"])).eval()
    assert type(net).__module__.startswith("cleandiffuser.") and not isinstance(net, getattr(pnn, case["cls"]))
    net.load_state_dict(synth_state_dict(net.state_dict(), seed=0))
    x, t, cond = cases.net_inputs(case)
    want = golden["nets"][name + "/y"]
    for i in range(cases.NET_BATCH):
        y = runtime.engine_forward(net, x, t[i:i + 1], cond)           # raises lower.Unsupported if anything is not recognised
        err = np.abs(y[i].numpy() - want[i])
        if math == "fp32":
            assert err.max() < 2e-5, (name, i, err.max())
        else:
            assert err.max() < 2e-2 and err.mean() < 2e-3, (name, i, err.max(), err.mean())


def test_reference_instances_inside_product_sampler(golden, ref):
    """A reference-identity JannerUNet1d handed to this package's DiscreteDiffusionSDE: engine call, no fallback, golden result."""
    from common import tape_of
    from cleandiffuser_b200.diffusion import DiscreteDiffusionSDE
    from cleandiffuser_b200.testing import NoiseTape
    name = "disc_dup_ddpm_x0"
    spec = cases.sampler_cases()[name]
    ncase = cases.SAMPLER_NETS[spec["net"]]
    net = ref("sampler/" + spec["net"], getattr(pnn, ncase["cls"])(**ncase["ctor"])).eval()
    net.load_state_dict(synth_state_dict(net.state_dict(), seed=0))
    inp = cases.sampler_inputs(spec)
    agent = DiscreteDiffusionSDE(net, None, fix_mask=inp["fix_mask"], x_max=inp["x_max"], x_min=inp["x_min"],
                                 predict_noise=spec["predict_noise"], diffusion_steps=spec["T"], device="cpu")
    before, fb = runtime.STATS["engine_calls"], runtime.STATS["fallbacks"]
    os.environ["CDS_MATH"] = "fp32"
    tape = NoiseTape(tape_of(golden["samplers"], name))
    with tape.active(), torch.no_grad():
        x0, _ = agent.sample(inp["prior"], solver=spec["solver"], n_samples=cases.SAMPLER_BATCH, sample_steps=spec["steps"],
                             temperature=spec["temperature"], w_cfg=spec["w_cfg"])
    assert runtime.STATS["engine_calls"] == before + 1 and runtime.STATS["fallbacks"] == fb
    np.testing.assert_allclose(x0.numpy(), golden["samplers"][name + "/x0"], rtol=1e-4, atol=3e-4)


# the hot-path sampler classes the overlay hands to this package (cleandiffuser_b200/overlay.py): rebound in
# ``cleandiffuser.diffusion`` and in the sub-module that defines each, nowhere else
SAMPLERS = {"DiscreteDiffusionSDE", "ContinuousDiffusionSDE", "ContinuousConsistencyModel", "ContinuousEDM", "DDPM", "EDM",
            "DiscreteRectifiedFlow", "ContinuousRectifiedFlow"}


@pytest.fixture()
def standin_reference(monkeypatch):
    """A ``cleandiffuser`` package with the reference's ``diffusion`` layout as recorded in the fixture: the same modules,
    each binding the same class names, defined there or imported from the same defining module; plus
    ``nn_diffusion.JannerUNet1d`` building reference-identity instances.  Yields {(module, name): original class}."""
    layout = json.loads(str(TREES["layout/diffusion"]))
    made, classes = {}, {}

    def module(name):
        if name not in made:
            mod = types.ModuleType(name)
            mod.__path__ = []                          # every level may hold sub-modules
            made[name] = mod
            if "." in name:
                parent, leaf = name.rsplit(".", 1)
                setattr(module(parent), leaf, mod)
        return made[name]

    originals = {}
    for mod_name, names in layout.items():
        for n, home in names.items():
            cls = classes.setdefault((home, n), type(n, (), {"__module__": home}))
            setattr(module(mod_name), n, cls)
            originals[mod_name, n] = cls
    # the reference's tree of this constructor call is the janner_cfg2 case's
    module("cleandiffuser.nn_diffusion").JannerUNet1d = lambda *a, **kw: reference_instance("janner_cfg2", pnn.JannerUNet1d(*a, **kw))
    for k in [k for k in sys.modules if k == "cleandiffuser" or k.startswith("cleandiffuser.")]:
        monkeypatch.delitem(sys.modules, k)
    for k, mod in made.items():
        monkeypatch.setitem(sys.modules, k, mod)
    yield originals
    overlay.uninstall()


class TrainableToyClassifier(ToyClassifier):
    """ToyClassifier with the reference classifier's ``update`` (cleandiffuser/classifier/base.py:47-58): one MSE step of
    log p towards the target."""

    def __init__(self, x_shape):
        super().__init__(x_shape)
        self.optim = torch.optim.Adam(self.model.parameters(), lr=1e-3)

    def update(self, x, noise, y):
        loss = ((self.logp(x, noise) - y) ** 2).mean()
        self.optim.zero_grad()
        loss.backward()
        self.optim.step()
        return {"loss": loss.item()}


def test_install_overlay_runs_the_diffuser_pipeline_call_sequence(standin_reference, monkeypatch):
    """``install()`` rebinds exactly the sampler classes of the reference's recorded layout (in ``cleandiffuser.diffusion``
    and in each class's defining sub-module) and leaves every other binding alone; the diffuser pipeline's call sequence
    (pipelines/diffuser_d4rl_mujoco.py:39-66 construction, :75-90 one training step of each, :136-148 guided inference over
    candidates and selection) runs on this package's sampler through the names it imports from ``cleandiffuser``;
    ``uninstall()`` restores every original binding.  The classifier is a toy one (TrainableToyClassifier) in place of the
    pipeline's CumRewClassifier over HalfJannerUNet1d, and the pipeline's ``report_parameters`` call is left out: neither
    is part of this package, so this test does not cover the reference's real classifier path."""
    import cleandiffuser_b200
    monkeypatch.setenv("CDS_BACKEND", "auto")
    patched = cleandiffuser_b200.install()
    layout = json.loads(str(TREES["layout/diffusion"]))
    want = {(m, n) for m, names in layout.items() for n, home in names.items()
            if n in SAMPLERS and m in ("cleandiffuser.diffusion", home)}
    assert sorted(patched) == sorted(f"{m}.{n}" for m, n in want)
    for (m, n), orig in standin_reference.items():
        now = getattr(sys.modules[m], n)
        assert now is getattr(cleandiffuser_b200.diffusion, n) if (m, n) in want else now is orig, (m, n)
    from cleandiffuser.diffusion import DiscreteDiffusionSDE
    from cleandiffuser.nn_diffusion import JannerUNet1d
    assert DiscreteDiffusionSDE is cleandiffuser_b200.diffusion.DiscreteDiffusionSDE

    obs_dim, act_dim, horizon, model_dim, dim_mult = 11, 3, 32, 32, [1, 2, 2, 2]
    nn_diffusion = JannerUNet1d(obs_dim + act_dim, model_dim=model_dim, emb_dim=model_dim, dim_mult=dim_mult,
                                timestep_emb_type="positional", attention=False, kernel_size=5)
    assert type(nn_diffusion).__module__.startswith("cleandiffuser.")
    fix_mask = torch.zeros((horizon, obs_dim + act_dim))
    fix_mask[0, :obs_dim] = 1.
    loss_weight = torch.ones((horizon, obs_dim + act_dim))
    loss_weight[0, obs_dim:] = 10.
    agent = DiscreteDiffusionSDE(nn_diffusion, None, fix_mask=fix_mask, loss_weight=loss_weight,
                                 classifier=TrainableToyClassifier((horizon, obs_dim + act_dim)), ema_rate=0.9999,
                                 device="cpu", diffusion_steps=20, predict_noise=False)
    g = torch.Generator().manual_seed(0)
    x, R = torch.randn(8, horizon, obs_dim + act_dim, generator=g), torch.randn(8, 1, generator=g)
    log = agent.update(x)
    assert "loss" in log
    log = agent.update_classifier(x, R)
    assert "loss" in log
    agent.eval()
    num_envs, num_candidates = 2, 4
    prior = torch.zeros((num_envs, horizon, obs_dim + act_dim))
    prior[:, 0, :obs_dim] = torch.randn(num_envs, obs_dim, generator=g)
    traj, log = agent.sample(prior.repeat(num_candidates, 1, 1), solver="ddpm", n_samples=num_candidates * num_envs,
                             sample_steps=20, use_ema=True, w_cg=0.3, temperature=0.5)
    logp = log["log_p"].view(num_candidates, num_envs, -1).sum(-1)
    idx = logp.argmax(0)
    act = traj.view(num_candidates, num_envs, horizon, -1)[idx, torch.arange(num_envs), 0, obs_dim:]
    assert act.shape == (num_envs, act_dim) and torch.isfinite(traj).all()
    assert torch.equal(traj[:, 0, :obs_dim], prior.repeat(num_candidates, 1, 1)[:, 0, :obs_dim])

    cleandiffuser_b200.uninstall()
    for (m, n), orig in standin_reference.items():
        assert getattr(sys.modules[m], n) is orig, (m, n)
