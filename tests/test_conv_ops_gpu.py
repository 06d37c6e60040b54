"""Operator-level parity of CDS_OP_CONV (conv_tc / conv_ps / conv_simt), CDS_OP_LNMOD and the fused Linear + LayerNorm kernel
against the fp64 reference of tests/op_reference.py, one operator through cabi.run_op / a 2-operator plan at a time.

Every conv case checks, per batch regime:
  1. every guard word around the output (pad channels between rows, trajectories past the batch, head and tail of the allocation)
     is bit-identical after the run: stray stores become assertion failures without faulting;
  2. the output is within the tolerance stated in tests/op_reference.py;
  3. CDS_TF32 outputs are TF32-representable;
  4. a second run writes the same bits;
  5. the kernel that ran and the tiles each CTA ran (cds_debug_trace, slot 5 of the per-CTA timeline, csrc/conv_tc.cuh:72): conv_tc
     cases cover every row x column tile exactly once, and persistent cases give every CTA >= 6 tiles, so that both accumulator
     buffers reach their third use; conv_ps launches one tile per CTA; conv_simt cases record no tensor-core launch."""
import ctypes as C
import os
import zlib

import pytest
import torch

import op_reference as R
from cleandiffuser_b200.engine import cabi

pytestmark = pytest.mark.gpu

SENT32 = 0x7FBADBAD          # NaN bit patterns: an element the kernel failed to write also fails the value check
SENT16 = 0x7FBB
POISON = 1.0e4               # pad channels / extra trajectories of INPUT views: reading them shows up as a huge error
SLOTS = 64
HEAD = 64                    # elements of guard before every view (keeps 16-byte alignment)


class _Env:
    def __init__(self, pairs):
        self.pairs, self.old = dict(pairs), {}

    def __enter__(self):
        for k, v in self.pairs.items():
            self.old[k] = os.environ.get(k)
            os.environ[k] = v

    def __exit__(self, *a):
        for k, v in self.old.items():
            if v is None:
                os.environ.pop(k, None)
            else:
                os.environ[k] = v


def _tdt(dt):
    return torch.bfloat16 if dt == cabi.BF16 else torch.float32


def _view_buffer(vals, n_traj, lstride, coff, dt, fill):
    """one allocation: HEAD guard elements, n_traj trajectories of rows with `lstride` elements (data at channel offset `coff`),
    tail; returns (flat tensor, element offset of the view, bstride)"""
    L, Cv = vals.shape[1], vals.shape[2]
    bstride = L * lstride
    flat = torch.full((HEAD + n_traj * bstride + HEAD,), fill, dtype=_tdt(dt))
    body = flat[HEAD:HEAD + n_traj * bstride].view(n_traj, L, lstride)
    body[:vals.shape[0], :, coff:coff + Cv] = vals.to(_tdt(dt))
    return flat.cuda(), HEAD + coff, bstride


def _ptr(t, off=0):
    return t.data_ptr() + off * t.element_size()


def _vecs(d, key, c, keep):
    v = cabi.Vec()
    if key + "_step" in d:
        t = d[key + "_step"].cuda()
        keep.append(t)
        v.step, v.step_stride = t.data_ptr(), t.shape[1]
    if key + "_sample" in d:
        s = d[key + "_sample"]
        stride = c.C_out + c.sample_pad
        t = torch.zeros(s.shape[0] * stride + 4, dtype=torch.float32)
        t[:s.shape[0] * stride].view(s.shape[0], stride)[:, :c.C_out] = s
        t = t.cuda()
        keep.append(t)
        v.sample, v.sample_stride = t.data_ptr(), stride
    return v


class Built:
    """device buffers and the cds_conv_op of one case"""

    def __init__(self, c: R.ConvCase, d):
        keep = []
        op = cabi.Op()
        op.kind = cabi.OP_CONV
        k = op.u.conv
        k.batch, k.L_in, k.L_out, k.C_in, k.C_out = c.B, c.L_in, c.L_out, c.C_in, c.C_out
        k.taps, k.stride, k.pad, k.phases = c.taps, c.stride, c.pad, c.phases
        k.in_batch_mod, k.res_batch_mod, k.sample_row_div = c.in_batch_mod, c.res_batch_mod, c.sample_row_div
        k.math = c.math
        idt = c.in_dt
        # input: pad channels, a channel-offset view, extra (poisoned) trajectories past the ones the op may read
        x = d["x"]
        in_l = c.in_coff + c.C_in + c.in_pad
        xb, xo, xbs = _view_buffer(x, x.shape[0] + 2, in_l, c.in_coff, idt, POISON)
        keep.append(xb)
        k.in_, k.in_bstride, k.in_lstride, k.in_dtype = _ptr(xb, xo), xbs, in_l, idt
        # weights packed from the PyTorch layout (C_out*phases, C_in, taps) as cds.h:112-121 states
        w = d["w"]
        if c.tc:
            wp = w.permute(2, 0, 1).contiguous().to(_tdt(idt))      # [taps][C_out*phases][C_in]
        else:
            wp = w.permute(2, 1, 0).contiguous()                     # fp32 [taps*C_in][C_out*phases]
        wp = wp.cuda()
        keep.append(wp)
        k.w = wp.data_ptr()
        k.bias, k.scale, k.shift = _vecs(d, "bias", c, keep), _vecs(d, "scale", c, keep), _vecs(d, "shift", c, keep)
        k.act = c.act
        if c.groups:
            gm, bt = d["gamma"].cuda(), d["beta"].cuda()
            keep += [gm, bt]
            k.groups, k.gn_gamma, k.gn_beta, k.gn_eps = c.groups, gm.data_ptr(), bt.data_ptr(), R.GN_EPS
        rdt = c.act_dtype if c.tc else idt
        if "id" in c.res:
            r = d["res"]
            if c.name.startswith(("gated", "table")):
                rdt = cabi.F32
            rb, ro, rbs = _view_buffer(r, r.shape[0] + 1, c.C_out, 0, rdt, POISON)
            keep.append(rb)
            k.res, k.res_bstride, k.res_lstride, k.res_dtype = _ptr(rb, ro), (0 if c.res_bstride0 else rbs), c.C_out, rdt
        if "sc" in c.res:
            ri = d["res_in"]
            rib, rio, ribs = _view_buffer(ri, ri.shape[0] + 1, c.res_C, 0, idt, POISON)
            rw = d["res_w"] if c.tc else d["res_w"].t()
            rw = rw.contiguous().to(_tdt(idt)).cuda()
            rbias = d["res_bias"].cuda()
            keep += [rib, rw, rbias]
            k.res_in, k.res_in_bstride, k.res_in_lstride, k.res_C, k.res_in_dtype = _ptr(rib, rio), ribs, c.res_C, c.res_C, idt
            k.res_w, k.res_bias = rw.data_ptr(), rbias.data_ptr()
        # output: pad channels between rows, 2 guard trajectories past the batch, head and tail
        odt = c.odt
        Lo, out_l = c.L_out * c.phases, c.C_out + c.out_pad
        self.sent = SENT16 if odt == cabi.BF16 else SENT32
        ib = torch.int16 if odt == cabi.BF16 else torch.int32
        n = HEAD + (c.B + 2) * Lo * out_l + HEAD
        self.out = torch.full((n,), self.sent, dtype=ib, device="cuda")
        k.out, k.out_bstride, k.out_lstride, k.out_dtype = _ptr(self.out, HEAD), Lo * out_l, out_l, odt
        mask = torch.zeros(n, dtype=torch.bool)
        mask[HEAD:HEAD + c.B * Lo * out_l].view(c.B, Lo, out_l)[:, :, :c.C_out] = True
        self.written = mask.cuda()
        self.shape = (c.B, Lo, out_l)
        self.keep, self.op, self.c, self.odt = keep, op, c, odt

    def values(self):
        c = self.c
        body = self.out[HEAD:HEAD + c.B * self.shape[1] * self.shape[2]].view(self.shape)[:, :, :c.C_out]
        return body.view(torch.bfloat16).float() if self.odt == cabi.BF16 else body.view(torch.float32)

    def guards_intact(self):
        g = self.out[~self.written]
        return int((g != self.sent).sum().item()), g.numel()


def _run(b: Built, trace_cap=0):
    lib = cabi.load()
    buf = None
    if trace_cap:
        buf = torch.zeros(trace_cap * SLOTS, dtype=torch.int64, device="cuda")
        lib.cds_debug_trace(C.c_void_p(buf.data_ptr()), buf.numel(), 0)
    try:
        cabi.run_op(0, b.op, b.c.iter, torch.cuda.current_stream().cuda_stream)
        torch.cuda.synchronize()
    finally:
        grid = lib.cds_debug_trace(None, 0, -1) if trace_cap else 0
    tiles = buf.view(-1, SLOTS)[:grid, 5].cpu() if grid else None
    return grid, tiles


def _sms():
    return torch.cuda.get_device_properties(0).multi_processor_count


def _persistent_batch(c: R.ConvCase):
    """grid of a launch with more tiles than can be resident, then a batch giving every CTA >= 6 tiles, the last one ragged"""
    g = R.tc_geometry(c.with_(B=1))
    m_probe = (2 * _sms() + 1 + g["nct"] - 1) // g["nct"] + 1
    probe = c.with_(B=m_probe * g["T"])
    with _Env(c.env):
        grid, tiles = _run(Built(probe, R.make_data(probe, seed=1)), trace_cap=4 * _sms())
    assert 0 < grid < R.tc_geometry(probe)["tiles"], (grid, R.tc_geometry(probe))
    m_tiles = (6 * grid + grid // 2 + g["nct"] - 1) // g["nct"]
    return m_tiles * g["T"] - (g["T"] // 3 if g["T"] > 1 else 0), grid


REPORT = []


def _check_case(c: R.ConvCase, regime):
    d = R.make_data(c, seed=zlib.crc32(c.name.encode()) % 1000)
    with _Env(c.env):
        b = Built(c, d)
        grid, tiles = _run(b, trace_cap=8 * _sms() + 64)
        first = b.out.clone()
        _run(b)
    bad, total = b.guards_intact()
    assert bad == 0, f"{bad} of {total} guard words overwritten"
    assert torch.equal(first, b.out), "second run wrote different bits"
    y = b.values()
    if b.odt == cabi.TF32:
        assert int((y.contiguous().view(torch.int32) & 0x1FFF).abs().max()) == 0, "CDS_TF32 output not TF32-representable"
    ref, gn_term = R.conv_ref(c, d, device="cuda")
    ex = R.excess(y, ref, b.odt, gn_term)
    # ---- which kernel ran and how many tiles each CTA ran
    if c.expect == "simt":
        assert grid == 0, "a tensor-core launch served a CDS_MATH_FP32 op"
        info = ""
    elif c.expect == "ps":
        n_ps = (c.B + 127) // 128 * 4                  # 4 column tiles of C_out / 4 (conv_ps_width)
        assert grid == n_ps and int(tiles.sum()) == n_ps and int(tiles.min()) == 1, (grid, tiles)
        info = f"grid {grid}"
    else:
        geo = R.tc_geometry(c)
        assert grid > 0, "no conv_tc launch recorded"
        assert int(tiles.sum()) == geo["tiles"], (int(tiles.sum()), geo)
        info = f"grid {grid} tiles {geo['tiles']} per-CTA {int(tiles.min())}..{int(tiles.max())}"
        if regime == "persist":
            assert int(tiles.min()) >= 6, info
    REPORT.append((c.name, regime, c.B, ex, info))
    print(f"[conv-op] {c.name:48s} {regime:7s} B={c.B:6d} err/tol={ex:.3f} {info}")
    assert ex <= 1.0, f"max |y - ref| / tol = {ex:.3f}"


_CASES = [(c, reg, B) for c in R.conv_cases() for reg, B in R.regimes(c)]


@pytest.mark.parametrize("case,regime,B", _CASES, ids=[f"{c.name}-{r}" for c, r, _ in _CASES])
def test_conv_op_matches_fp64(case, regime, B):
    if regime == "persist":
        B, _ = _persistent_batch(case)
    _check_case(case.with_(B=B), regime)


# --------------------------------------------------------------------------------------------- CDS_OP_LNMOD and Linear + LN
def _lnmod_op(x, out, shift, scale, L, out_dtype, eps=1e-6):
    op = cabi.Op()
    op.kind = cabi.OP_LNMOD
    m = op.u.lnmod
    m.batch, m.L, m.C, m.eps = x.shape[0] // L, L, x.shape[1], eps
    m.in_, m.out, m.shift, m.scale, m.mod_bstride, m.out_dtype = x.data_ptr(), out.data_ptr(), shift.data_ptr(), scale.data_ptr(), \
        shift.stride(0), out_dtype
    return op


@pytest.mark.parametrize("C,L,B,out_dtype,misalign", [
    (128, 10, 37, cabi.TF32, 0),        # ln_rows_vec<16, 3>
    (192, 7, 5, cabi.F32, 0),           # <16, 3>
    (256, 32, 64, cabi.TF32, 0),        # <16, 6>
    (384, 3, 11, cabi.F32, 0),          # <16, 6>
    (320, 100, 13, cabi.TF32, 0),       # <32, kLnVec>
    (512, 16, 9, cabi.F32, 0),          # <32, kLnVec>
    (30, 10, 7, cabi.F32, 0),           # scalar path: C % 4 != 0
    (128, 10, 7, cabi.F32, 1),          # scalar path: misaligned rows
    (256, 16, 9, cabi.BF16, 0),         # bf16 output (scalar path)
    (700, 4, 3, cabi.F32, 0),           # scalar path, row not held in registers
])
def test_lnmod_op_matches_fp64(C, L, B, out_dtype, misalign):
    g = torch.Generator().manual_seed(C + L)
    rows = B * L
    xs = torch.randn(rows * C + misalign, generator=g) * 2 + 3
    x = xs.cuda()[misalign:].view(rows, C)
    shift, scale = (torch.randn(B, C, generator=g) * 0.3).cuda(), (torch.randn(B, C, generator=g) * 0.3).cuda()
    o_el = rows * C + 2 * HEAD + misalign
    out = torch.full((o_el,), SENT16 if out_dtype == cabi.BF16 else SENT32,
                     dtype=torch.int16 if out_dtype == cabi.BF16 else torch.int32, device="cuda")
    view = out[HEAD + misalign:HEAD + misalign + rows * C]
    op = _lnmod_op(x, view, shift, scale, L, out_dtype)
    cabi.run_op(0, op, 0, torch.cuda.current_stream().cuda_stream)
    torch.cuda.synchronize()
    keep = torch.ones(out.numel(), dtype=torch.bool, device="cuda")
    keep[HEAD + misalign:HEAD + misalign + rows * C] = False
    assert bool((out[keep] == out[0]).all()), "LayerNorm wrote outside its output"
    y = view.view(torch.bfloat16).float() if out_dtype == cabi.BF16 else view.view(torch.float32)
    if out_dtype == cabi.TF32:
        assert int((view & 0x1FFF).abs().max()) == 0
    ref = R.lnmod_ref(x, shift, scale, L).view(rows, C)
    ex = R.excess(y.view(rows, C), ref, out_dtype)
    print(f"[lnmod] C={C} L={L} B={B} dtype={out_dtype} misalign={misalign}: err/tol={ex:.3f}")
    assert ex <= 1.0, ex


def _linear_ln(form, C, L, B, ibm, fuse, graph):
    """[gated conv | table conv, lnmod] over B trajectories of L tokens as a 2-operator plan; returns (X, Y, launches per
    iteration, reference X, reference Y)"""
    g = torch.Generator().manual_seed(C * 7 + L)
    K = 64
    rows = B * L
    ar = ibm if ibm else rows
    a = torch.randn(ar, K, generator=g)
    w = torch.randn(C, K, generator=g) / K ** 0.5
    bias = torch.randn(R.N_STEPS, C, generator=g) * 0.3
    gate = torch.randn(B, C, generator=g) * 0.5
    res = torch.randn(L if form == "table" else rows, C, generator=g)
    shift, scale = torch.randn(B, C, generator=g) * 0.3, torch.randn(B, C, generator=g) * 0.3
    dev = [t.cuda() for t in (a, w, bias, gate, res, shift, scale)]
    a_d, w_d, bias_d, gate_d, res_d, shift_d, scale_d = dev
    X = torch.full((rows, C), float("nan"), device="cuda")
    Y = torch.full((rows, C), float("nan"), device="cuda")
    op = cabi.Op()
    op.kind = cabi.OP_CONV
    k = op.u.conv
    k.batch, k.L_in, k.L_out, k.C_in, k.C_out, k.taps, k.stride, k.pad, k.phases = rows, 1, 1, K, C, 1, 1, 0, 1
    k.in_batch_mod = ibm
    k.in_, k.in_bstride, k.in_lstride, k.in_dtype = a_d.data_ptr(), K, K, cabi.F32
    k.w = w_d.data_ptr()
    k.bias.step, k.bias.step_stride = bias_d.data_ptr(), C
    if form == "gated":
        k.scale.sample, k.scale.sample_stride = gate_d.data_ptr(), C
    k.res, k.res_bstride, k.res_lstride, k.res_dtype = res_d.data_ptr(), C, C, cabi.F32
    k.res_batch_mod = L if form == "table" else 0
    k.out, k.out_bstride, k.out_lstride = X.data_ptr(), C, C
    k.math, k.out_dtype, k.sample_row_div = cabi.MATH_TF32_TC, cabi.F32, L
    ln = _lnmod_op(X, Y, shift_d, scale_d, L, cabi.TF32)
    with _Env((("CDS_FUSE_LN", "1" if fuse else "0"),)):
        plan = cabi.Plan(0)
        plan.append([op, ln])
        plan.finalize(R.N_STEPS)
    plan.run(2, 1, torch.cuda.current_stream().cuda_stream, use_graph=graph)
    torch.cuda.synchronize()
    launches = plan.launches_per_iter()
    plan.close()
    tr = torch.arange(rows) // L
    ad = R.tf32_trunc(a).double()[torch.arange(rows) % ar]
    acc = ad @ R.tf32_trunc(w).double().t() + bias[2].double()
    xr = acc * gate.double()[tr] + res.double() if form == "gated" else acc + res.double()[torch.arange(rows) % L]
    yr = R.lnmod_ref(xr, shift, scale, L)
    return X, Y, launches, xr, yr


# (form, C_out, tokens per trajectory L, trajectories B, in_batch_mod): B * L rows, never a multiple of 128 (ragged last tile)
_LINLN = [("gated", 256, 32, 9, 0), ("gated", 320, 64, 15, 0), ("gated", 384, 100, 7, 0), ("gated", 512, 64, 17, 256),
          ("table", 320, 100, 10, 0), ("table", 256, 32, 13, 128), ("gated", 320, 64, "persist", 0),
          ("table", 512, 100, "persist", 0)]


@pytest.mark.parametrize("form,C,L,B,ibm", _LINLN)
def test_linear_layernorm_pair_matches_fp64(form, C, L, B, ibm):
    if B == "persist":
        B = 6 * _sms() * 128 // L + 1      # >= 6 row tiles per CTA even at one CTA per SM
    rows = B * L
    assert rows % 128 != 0
    for fuse, graph in ((True, True), (False, False), (True, False), (False, True)):
        X, Y, launches, xr, yr = _linear_ln(form, C, L, B, ibm, fuse, graph)
        assert launches == (2 if fuse else 3), (fuse, launches)
        ex_x = R.excess(X.cpu(), xr, cabi.F32)
        ex_y = R.excess(Y.cpu(), yr, cabi.TF32)
        assert int((Y.view(torch.int32) & 0x1FFF).abs().max()) == 0
        print(f"[linear-ln] {form} C={C} L={L} rows={rows} ibm={ibm} fused={fuse} graph={graph}: "
              f"X err/tol={ex_x:.3f} Y err/tol={ex_y:.3f}")
        assert ex_x <= 1.0 and ex_y <= 1.0, (ex_x, ex_y)
