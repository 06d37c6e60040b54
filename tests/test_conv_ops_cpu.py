"""CPU side of the operator-level conv tests (tests/test_conv_ops_gpu.py):

  * discrimination: the tolerance of tests/op_reference.py rejects the output of a kernel with a plausible defect, modelled as a
    mutation of the fp64 reference (nothing runs on a GPU);
  * the CPU interpreter the lowering tests trust (tests/emulator.py) agrees with the fp64 reference on small versions of the cases;
  * coverage: the case list reaches every (KC, N, SPLIT) instantiation of conv_tc (CDS_TC_VARIANTS, conv_tc.cuh:1470) and every
    epilogue lane, according to the Python mirror of the kernel choice in op_reference.py."""
import ctypes as C

import numpy as np
import pytest
import torch

import emulator
import op_reference as R
from cleandiffuser_b200.engine import cabi


def _as_kernel_output(ref, out_dtype):
    """what a correct kernel could store: the reference rounded to the output type, plus fp32-level noise"""
    g = torch.Generator().manual_seed(0)
    y = ref + 0.2 * R.A_ABS * ref.pow(2).mean().sqrt() * torch.randn(ref.shape, generator=g, dtype=torch.float64)
    if out_dtype == cabi.TF32:
        return R.tf32_round(y.float()).double()
    if out_dtype == cabi.BF16:
        return y.to(torch.bfloat16).double()
    return y.float().double()


_DEFECTS = [
    ("drop_last_res", R.ConvCase("d_res", R.TF, B=7, L_in=16, L_out=16, C_in=32, C_out=64, taps=3, pad=1, groups=8, act=R.MISH,
                                 res="id")),
    ("edge_unpadded", R.ConvCase("d_pad", R.TF, B=5, L_in=8, L_out=8, C_in=32, C_out=64, taps=5, pad=2, groups=8, act=R.MISH)),
    ("edge_unpadded", R.ConvCase("d_pad_bf16", R.BF, B=5, L_in=32, L_out=32, C_in=64, C_out=32, taps=5, pad=2)),
    ("phase_shift", R.ConvCase("d_phase", R.TF, B=5, L_in=8, L_out=8, C_in=32, C_out=64, taps=3, pad=1, phases=2,
                               act=R.GELU_T)),
    ("col_tile_bias:160", R.ConvCase("d_coltile", R.TF, B=300, L_in=1, L_out=1, C_in=64, C_out=320)),
    ("prev_step", R.ConvCase("d_step", R.TF, B=9, L_in=16, L_out=16, C_in=32, C_out=64, taps=3, pad=1, groups=8, act=R.MISH,
                             shift="s")),
    ("prev_step", R.ConvCase("d_step_bf16", R.BF, B=9, L_in=8, L_out=8, C_in=64, C_out=128, taps=3, pad=1, act=R.SILU)),
    ("gn_single_pass", R.ConvCase("d_gn32", R.TF, B=6, L_in=32, L_out=32, C_in=32, C_out=64, taps=3, pad=1, groups=8,
                                  act=R.MISH, gn_offset=256)),
    ("gn_single_pass", R.ConvCase("d_gn4", R.TF, B=6, L_in=4, L_out=4, C_in=64, C_out=1024, taps=3, pad=1, groups=8,
                                  act=R.MISH, gn_offset=256)),
]


@pytest.mark.parametrize("defect,case", _DEFECTS, ids=[f"{d}-{c.name}" for d, c in _DEFECTS])
def test_tolerance_rejects_defect(defect, case):
    d = R.make_data(case, seed=3)
    ref, gn = R.conv_ref(case, d)
    good = _as_kernel_output(ref, case.odt)
    ok = R.excess(good, ref, case.odt, gn)
    assert ok <= 1.0, f"a correct output fails the tolerance ({ok:.2f})"
    bad, _ = R.conv_ref(case, d, defect=defect)
    ex = R.excess(_as_kernel_output(bad, case.odt), ref, case.odt, gn)
    print(f"{defect:18s} {case.name:12s} correct {ok:.3f}  defect {ex:.1f} x tolerance")
    assert ex > 1.0, f"defect {defect} passes the tolerance ({ex:.3f})"


def test_tf32_tolerance_is_far_tighter_than_the_network_tolerance():
    c = R.ConvCase("t", R.TF, B=5, L_in=16, L_out=16, C_in=32, C_out=64, taps=3, pad=1, groups=8, act=R.MISH)
    ref, gn = R.conv_ref(c, R.make_data(c))
    rms = ref.pow(2).mean().sqrt().item()
    # the absolute part of the bound is ~2000 x inside the 2e-2 max error the golden-net tests allow in TF32
    assert R.A_ABS * rms < 2e-2 / 100


# ------------------------------------------------------------------------------------------------------ emulator cross-check
def _host_op(c: R.ConvCase, d, keep):
    """cds_conv_op over host tensors (the emulator reads raw host pointers), dense views"""
    def hold(t):
        t = t.contiguous()
        keep.append(t)
        return t

    def ptr(t):
        return hold(t).data_ptr()

    def bf(t):
        return hold(t.to(torch.bfloat16)).data_ptr()

    op = cabi.Op()
    op.kind = cabi.OP_CONV
    k = op.u.conv
    k.batch, k.L_in, k.L_out, k.C_in, k.C_out = c.B, c.L_in, c.L_out, c.C_in, c.C_out
    k.taps, k.stride, k.pad, k.phases, k.math = c.taps, c.stride, c.pad, c.phases, c.math
    k.in_batch_mod, k.res_batch_mod, k.sample_row_div = c.in_batch_mod, c.res_batch_mod, c.sample_row_div
    idt = c.in_dt
    k.in_ = bf(d["x"]) if idt == cabi.BF16 else ptr(d["x"])
    k.in_bstride, k.in_lstride, k.in_dtype = c.L_in * c.C_in, c.C_in, idt
    if c.tc:
        wp = d["w"].permute(2, 0, 1)
        k.w = bf(wp) if idt == cabi.BF16 else ptr(wp)
    else:
        k.w = ptr(d["w"].permute(2, 1, 0))
    for key in ("bias", "scale", "shift"):
        v = getattr(k, key)
        if key + "_step" in d:
            v.step, v.step_stride = ptr(d[key + "_step"]), c.C_out
        if key + "_sample" in d:
            v.sample, v.sample_stride = ptr(d[key + "_sample"]), c.C_out
    k.act = c.act
    if c.groups:
        k.groups, k.gn_gamma, k.gn_beta, k.gn_eps = c.groups, ptr(d["gamma"]), ptr(d["beta"]), R.GN_EPS
    if "id" in c.res:
        rdt = cabi.BF16 if idt == cabi.BF16 else cabi.F32
        k.res = bf(d["res"]) if rdt == cabi.BF16 else ptr(d["res"])
        k.res_bstride, k.res_lstride, k.res_dtype = (0 if c.res_bstride0 else c.L_out * c.C_out), c.C_out, rdt
    if "sc" in c.res:
        k.res_in = bf(d["res_in"]) if idt == cabi.BF16 else ptr(d["res_in"])
        k.res_in_bstride, k.res_in_lstride, k.res_C, k.res_in_dtype = c.L_out * c.res_C, c.res_C, c.res_C, idt
        rw = d["res_w"] if c.tc else d["res_w"].t()
        k.res_w = bf(rw) if idt == cabi.BF16 else ptr(rw)
        k.res_bias = ptr(d["res_bias"])
    out = torch.zeros(c.B, c.L_out * c.phases, c.C_out, dtype=torch.bfloat16 if c.odt == cabi.BF16 else torch.float32)
    keep.append(out)
    k.out, k.out_bstride, k.out_lstride, k.out_dtype = out.data_ptr(), c.L_out * c.phases * c.C_out, c.C_out, c.odt
    return op, out


def _small(c: R.ConvCase):
    T = 128 // c.L_out
    B = max(c.in_batch_mod, c.res_batch_mod, 2) + 1 if (c.in_batch_mod or c.res_batch_mod) else min(T + 1, 5)
    return c.with_(B=B * 2 if c.in_batch_mod else B, in_pad=0, in_coff=0, out_pad=0, sample_pad=0, gn_offset=0, env=())


_EMU = [c for c in R.conv_cases() if c.C_out * c.C_in <= 512 * 64 and not c.name.endswith("_ps0")][::2]


@pytest.mark.parametrize("case", _EMU, ids=[c.name for c in _EMU])
def test_emulator_agrees_with_fp64_reference(case):
    c = _small(case)
    d = R.make_data(c, seed=5)
    keep = []
    op, out = _host_op(c, d, keep)
    with np.errstate(over="ignore"):
        emulator.run_conv(op.u.conv, c.iter)
    ref, gn = R.conv_ref(c, d)
    # the interpreter computes in fp32 between the fp64 GEMM and GroupNorm; Mish / GELU in numpy float32
    ex = R.excess(out.double(), ref, c.odt, gn, a=4 * R.A_ABS)
    assert ex <= 1.0, ex


def test_emulator_lnmod_agrees_with_fp64_reference():
    g = torch.Generator().manual_seed(2)
    B, L, C_ = 3, 5, 96
    x = torch.randn(B * L, C_, generator=g) * 2 + 1
    sh, sc = torch.randn(B, C_, generator=g), torch.randn(B, C_, generator=g)
    out = torch.zeros(B * L, C_)
    op = cabi.Op()
    m = op.u.lnmod
    m.batch, m.L, m.C, m.eps = B, L, C_, 1e-6
    m.in_, m.out, m.shift, m.scale, m.mod_bstride, m.out_dtype = x.data_ptr(), out.data_ptr(), sh.data_ptr(), sc.data_ptr(), C_, cabi.F32
    emulator.run_lnmod(m)
    assert R.excess(out.double(), R.lnmod_ref(x, sh, sc, L), cabi.F32) <= 1.0


# ------------------------------------------------------------------------------------------------------------------ coverage
def test_cases_reach_every_tc_variant_and_lane():
    cases = [c for c in R.conv_cases() if c.expect == "tc"]
    reached = {}
    for c in cases:
        g = R.tc_geometry(c)
        reached.setdefault((g["kc"], g["n"], g["split"], c.math), c.name)
    # TF32 never splits a 64-column layer (conv_tc_pick_split, :1264): (KC, 32, 2) is a bf16-only instantiation
    tf32_unreachable = {(64, 32, 2), (32, 32, 2)}
    for v in R.TC_VARIANTS:
        mode = R.BF if v in tf32_unreachable else R.TF
        key = v + (mode,)
        assert key in reached, f"no case reaches conv_tc<KC={v[0]}, N={v[1]}, SPLIT={v[2]}> in {'bf16' if mode == R.BF else 'tf32'}"
        print(f"KC={v[0]:2d} N={v[1]:3d} SPLIT={v[2]} {'BF16' if mode == R.BF else 'TF32'}: {reached[key]}")
    lanes = {}
    for c in cases:
        lanes.setdefault((R.tc_lane(c), c.math), c.name)
    for lane in ("fast", "plain", "gated", "table", "wide_gn", "generic"):
        assert (lane, R.TF) in lanes, lane
        print(f"lane {lane:8s} TF32: {lanes[(lane, R.TF)]}")
    kinds = {c.expect for c in R.conv_cases()}
    assert kinds == {"tc", "ps", "simt"}
    persistent = [c.name for c in R.conv_cases() if any(r == "persist" for r, _ in R.regimes(c))]
    assert {R.tc_lane(c) for c in R.conv_cases() if c.name in persistent} >= {"fast", "plain", "gated", "table", "wide_gn", "generic"}
