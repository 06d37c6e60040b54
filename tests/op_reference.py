"""fp64 reference of the CDS_OP_CONV / CDS_OP_LNMOD operator contract (include/cds.h:98-136), for operator-level tests.

Written from the header, not from the lowering or the CPU interpreter (tests/emulator.py): the test packs the weights itself from
PyTorch-layout tensors, so a disagreement about the packing shows up as a failure instead of being shared by both sides.

Operands are modelled the way the hardware reads them, so that what is left between a kernel and this reference is fp32
accumulation order, the MUFU approximations and the rounding of the stored output:
  * CDS_MATH_TF32_TC: tcgen05 kind::tf32 ignores the low 13 mantissa bits of `in`, `w`, `res_in` and `res_w` (cds.h:71-74);
  * CDS_MATH_BF16_TC: the inputs are generated as bf16 values, which the MMA reads exactly;
  * CDS_MATH_FP32: the values are used unchanged.
Everything after the operands (bias, GroupNorm, activation, FiLM, residuals) is computed in float64 in exact form.

Tolerance, one formula for every case:   |y - ref| <= r_out * |ref| + A_ABS * rms(ref) + gn_term
  * r_out: the rounding of the stored value -- 2^-11 for CDS_TF32 (round to nearest, half an ulp of a 10-bit mantissa), 2^-8 for
    bf16 (half an ulp is 2^-9; the kernels also round products of bf16 activations), 0 for fp32;
  * A_ABS = 1e-5: fp32 accumulation of <= 1280 products (relative 2^-24 per step, random walk: ~ sqrt(1280) * 6e-8 = 2e-6 of the
    accumulator's scale), the bias add, ex2/rcp/rsqrt.approx (relative ~2^-22 each), and the cancellation of Mish's
    1 - 2/(e^2 + 2e + 2) form for negative inputs (absolute ~6e-8 * |y|).  Inputs are scaled so that rms(ref) is O(1); the
    operator-level error then sits near 1e-6, an order of magnitude inside the bound, and ~2000 x inside the network-level
    TF32 tolerance (2e-2) that used to be the only check of these kernels;
  * gn_term (GroupNorm layers only): the pre-normalisation value y = acc + bias is an fp32 number; when a group carries a large
    common offset, y itself cannot be closer than half an ulp of |y| to the exact value, and the normalisation multiplies that by
    rstd * |gamma|.  gn_term = 2 * 2^-24 * max|y| * rstd * |gamma| per group, i.e. the best any fp32 kernel can do.  For an offset
    of 256 sigma that is ~3e-5; single-pass raw moments in fp32 err by ~1e-2 there.
"""
import dataclasses
import math

import torch

from cleandiffuser_b200.engine import cabi

A_ABS = 1e-5
R_OUT = {cabi.F32: 0.0, cabi.TF32: 2.0 ** -11, cabi.BF16: 2.0 ** -8}
GN_EPS = 1e-5
N_STEPS = 3          # rows of every per-iteration table; cases run at iteration 2
ACT_NAMES = {cabi.ACT_NONE: "none", cabi.ACT_MISH: "mish", cabi.ACT_SILU: "silu", cabi.ACT_GELU_TANH: "gelu_tanh",
             cabi.ACT_MISH_SILU: "mish_silu", cabi.ACT_LEAKY_RELU: "leaky_relu", cabi.ACT_GELU_ERF: "gelu_erf"}


def tf32_trunc(x: torch.Tensor) -> torch.Tensor:
    """what tcgen05 kind::tf32 reads of an fp32 operand: the low 13 mantissa bits cleared"""
    return (x.to(torch.float32).contiguous().view(torch.int32) & ~0x1FFF).view(torch.float32)


def tf32_round(x: torch.Tensor) -> torch.Tensor:
    """fp32 -> nearest TF32, ties away from zero (cvt.rna.tf32.f32): how a CDS_TF32 tensor is written"""
    return ((x.to(torch.float32).contiguous().view(torch.int32) + 0x1000) & ~0x1FFF).view(torch.float32)


@dataclasses.dataclass
class ConvCase:
    """One CDS_OP_CONV invocation.  Vector parts: "" absent, "s" per-iteration step row, "b" per-trajectory sample row,
    "sb" both.  res: "" none, "id" identity residual, "sc" 1x1 shortcut conv, "id+sc" both."""
    name: str
    math: int
    B: int
    L_in: int
    L_out: int
    C_in: int
    C_out: int
    taps: int = 1
    stride: int = 1
    pad: int = 0
    phases: int = 1
    groups: int = 0
    act: int = cabi.ACT_NONE
    bias: str = "s"
    scale: str = ""
    shift: str = ""
    res: str = ""
    res_C: int = 0
    in_batch_mod: int = 0
    res_batch_mod: int = 0
    res_bstride0: bool = False      # identity residual read through res_bstride = 0 (one row for every trajectory)
    sample_row_div: int = 0
    out_dtype: int = -1             # -1: the mode's activation dtype
    in_dtype: int = -1              # -1: the mode's operand dtype (CDS_MATH_FP32 also reads bf16 activations)
    in_pad: int = 0                 # pad channels after each input row (in_lstride = in_coff + C_in + in_pad)
    in_coff: int = 0                # the input view starts this many channels into its rows
    out_pad: int = 0                # pad channels after each output row
    sample_pad: int = 0             # sample_stride = C_out + sample_pad (rows not 16-byte aligned when % 4 != 0)
    gn_offset: float = 0.0          # GroupNorm layers: add a common offset of this many group-sigmas to each group's bias
    amp: float = 1.0                # scale of the pre-activation (edge cases: +-100)
    iter: int = 2
    env: tuple = ()                 # (name, value) environment settings the kernel choice reads (CDS_NO_TMA_RES, CDS_PS ...)
    expect: str = "tc"              # kernel that must serve it: "tc" (conv_tc), "ps" (conv_ps), "simt" (conv_simt)
    persistent: bool = False        # resize the batch so that every CTA runs >= 6 tiles

    @property
    def tc(self):
        return self.math in cabi.TC_MODES

    @property
    def act_dtype(self):
        return {cabi.MATH_TF32_TC: cabi.TF32, cabi.MATH_BF16_TC: cabi.BF16}.get(self.math, cabi.F32)

    @property
    def odt(self):
        return self.act_dtype if self.out_dtype < 0 else self.out_dtype

    @property
    def in_dt(self):
        if self.in_dtype >= 0:
            return self.in_dtype
        return cabi.BF16 if self.math == cabi.MATH_BF16_TC else cabi.F32

    @property
    def N(self):
        return self.C_out * self.phases

    def with_(self, **kw):
        return dataclasses.replace(self, **kw)


def _owners(c: ConvCase):
    div = c.sample_row_div if c.sample_row_div > 1 else 1
    return (c.B + div - 1) // div


def make_data(c: ConvCase, seed: int = 0):
    """Host tensors of a case in PyTorch layout, seeded.  Activations are bf16-representable in BF16 mode; TF32-mode operands are
    arbitrary fp32 (the kernel truncates, the reference models it)."""
    g = torch.Generator().manual_seed(seed)
    rnd = lambda *s: torch.randn(*s, generator=g, dtype=torch.float64)
    bf = c.in_dt == cabi.BF16
    q = (lambda t: t.to(torch.bfloat16).to(torch.float32)) if bf else (lambda t: t.to(torch.float32))
    K = c.taps * c.C_in
    d = {}
    Bx = c.in_batch_mod if c.in_batch_mod > 0 else c.B
    d["x"] = q(rnd(Bx, c.L_in, c.C_in))
    # weight as nn.Conv1d / ConvTranspose-phase stacks: (C_out * phases, C_in, taps); scaled to unit-variance outputs
    d["w"] = q(rnd(c.N, c.C_in, c.taps) * (c.amp / math.sqrt(K)))
    own = _owners(c)
    for key in ("bias", "scale", "shift"):
        parts = getattr(c, key)
        base = 1.0 if key == "scale" else 0.0
        if "s" in parts:
            d[key + "_step"] = (base * (1.0 / (2 if "b" in parts else 1)) + 0.3 * rnd(N_STEPS, c.C_out)).to(torch.float32)
        if "b" in parts:
            d[key + "_sample"] = ((base / 2 if "s" in parts else base) + 0.3 * rnd(own, c.C_out)).to(torch.float32)
    if c.groups > 0:
        d["gamma"] = (1.0 + 0.2 * rnd(c.C_out)).to(torch.float32)
        d["beta"] = (0.2 * rnd(c.C_out)).to(torch.float32)
        if c.gn_offset:
            # a common offset per group, in units of the group's pre-norm sigma (~amp: unit-variance outputs)
            cpg = c.C_out // c.groups
            off = (c.gn_offset * c.amp * torch.tensor([(-1.0) ** gi for gi in range(c.groups)], dtype=torch.float64)).repeat_interleave(cpg)
            d["bias_step"] = (d["bias_step"].double() + off).to(torch.float32)
    Br = c.res_batch_mod if c.res_batch_mod > 0 else c.B
    if "id" in c.res:
        d["res"] = q(rnd(1 if c.res_bstride0 else Br, c.L_out, c.C_out))
    if "sc" in c.res:
        d["res_in"] = q(rnd(Br, c.L_out, c.res_C))
        d["res_w"] = q(rnd(c.C_out, c.res_C) / math.sqrt(c.res_C))
        d["res_bias"] = (0.2 * rnd(c.C_out)).to(torch.float32)
    return d


def act_ref(kind, x: torch.Tensor) -> torch.Tensor:
    """the seven activations of cds.h in exact float64 form"""
    if kind == cabi.ACT_NONE:
        return x
    if kind == cabi.ACT_MISH:
        return x * torch.tanh(torch.nn.functional.softplus(x, threshold=1e9))
    if kind == cabi.ACT_SILU:
        return x * torch.sigmoid(x)
    if kind == cabi.ACT_GELU_TANH:
        return 0.5 * x * (1 + torch.tanh(math.sqrt(2 / math.pi) * (x + 0.044715 * x ** 3)))
    if kind == cabi.ACT_MISH_SILU:
        m = act_ref(cabi.ACT_MISH, x)
        return m * torch.sigmoid(m)
    if kind == cabi.ACT_LEAKY_RELU:
        return torch.where(x > 0, x, 0.01 * x)
    if kind == cabi.ACT_GELU_ERF:
        return 0.5 * x * (1 + torch.erf(x / math.sqrt(2)))
    raise ValueError(kind)


def _vec(c, d, key, it, device):
    """vec(b, c) = step[iter] + sample[b / sample_row_div] as a (B, C_out) float64 tensor, or None"""
    out = None
    if key + "_step" in d:
        out = d[key + "_step"][it].double().to(device)[None].expand(c.B, -1)
    if key + "_sample" in d:
        div = c.sample_row_div if c.sample_row_div > 1 else 1
        smp = d[key + "_sample"].double().to(device)[torch.arange(c.B, device=device) // div]
        out = smp if out is None else out + smp
    return out


def _gn_single_pass_fp32(y, c):
    """GroupNorm statistics as single-pass raw moments in fp32, in the reduction order of conv_tc's fast lane: per-position sums over
    the group's channels in 4-wide steps, then a butterfly over the L positions.  Only for the discrimination test."""
    B, L, C = y.shape
    G = c.groups
    yg = y.to(torch.float32).reshape(B, L, G, C // G)
    s1 = torch.zeros(B, L, G, dtype=torch.float32, device=y.device)
    s2 = torch.zeros_like(s1)
    for k in range(0, C // G, 4):
        x = yg[..., k:k + 4]
        s1 = s1 + ((x[..., 0] + x[..., 1]) + (x[..., 2] + x[..., 3]))
        for j in range(4):
            s2 = torch.addcmul(s2, x[..., j], x[..., j])
    while s1.shape[1] > 1:
        h = s1.shape[1] // 2
        s1, s2 = s1[:, :h] + s1[:, h:], s2[:, :h] + s2[:, h:]
    inv = torch.tensor(1.0 / (L * (C // G)), dtype=torch.float32)
    mean = s1 * inv
    var = torch.clamp(s2 * inv - mean * mean, min=0)
    return mean.double(), var.double()


def conv_ref(c: ConvCase, d: dict, device="cpu", defect: str = ""):
    """out(b, l*phases + n / C_out, n % C_out) of cds.h:98-107 in float64 -> (B, L_out * phases, C_out).  Also returns the group
    term of the tolerance (per element) for GroupNorm layers, else None.

    `defect` builds the reference of a plausibly WRONG kernel (tests/test_conv_ops_cpu.py checks that the comparison rejects each):
    drop_last_res, edge_unpadded, phase_shift, col_tile_bias:<tile width>, prev_step, gn_single_pass."""
    dev = torch.device(device)
    B, N = c.B, c.N
    it = c.iter - 1 if defect == "prev_step" else c.iter
    x = d["x"]
    w = d["w"]                                                    # (N, C_in, taps)
    if c.math == cabi.MATH_TF32_TC:
        x, w = tf32_trunc(x), tf32_trunc(w)
    x = x.double().to(dev)
    w = w.double().to(dev)
    if c.in_batch_mod > 0:
        x = x[torch.arange(B, device=dev) % c.in_batch_mod]
    acc = torch.zeros(B, c.L_out, N, dtype=torch.float64, device=dev)
    lpos = torch.arange(c.L_out, device=dev)
    for tap in range(c.taps):
        pos = lpos * c.stride + tap - c.pad
        ok = (pos >= 0) & (pos < c.L_in)
        if defect == "edge_unpadded":                          # the out-of-range tap reads the edge position instead of zero
            pos, ok = pos.clamp(0, c.L_in - 1), torch.ones_like(ok)
        if ok.any():
            acc[:, ok] += torch.einsum("blk,nk->bln", x[:, pos[ok]], w[:, :, tap])
    chan = torch.arange(N, device=dev) % c.C_out
    y = acc
    bias = _vec(c, d, "bias", it, dev)
    if bias is not None:
        bcol = bias[:, chan]
        if defect.startswith("col_tile_bias"):                 # the second runtime column tile uses the first tile's constants
            tn = int(defect.split(":")[1])
            bcol = bcol.clone()
            bcol[:, tn:2 * tn] = bcol[:, :tn]
        y = y + bcol[:, None, :]
    gn_term = None
    if c.groups > 0:
        G, cpg = c.groups, c.C_out // c.groups
        yg = y.reshape(B, c.L_out, G, cpg)
        if defect == "gn_single_pass":
            mean, var = _gn_single_pass_fp32(y, c)
            mean, var = mean[..., None], var[..., None]
        else:
            mean = yg.mean(dim=(1, 3), keepdim=True)
            var = ((yg - mean) ** 2).mean(dim=(1, 3), keepdim=True)
        rstd = 1.0 / torch.sqrt(var + GN_EPS)
        gamma, beta = d["gamma"].double().to(dev), d["beta"].double().to(dev)
        y = ((yg - mean) * rstd).reshape(B, c.L_out, c.C_out) * gamma + beta
        ymax = yg.abs().amax(dim=(1, 3), keepdim=True)
        gn_term = (2 * 2.0 ** -24 * ymax * rstd).expand_as(yg).reshape(B, c.L_out, c.C_out) * gamma.abs()
    y = act_ref(c.act, y)
    scale, shift = _vec(c, d, "scale", it, dev), _vec(c, d, "shift", it, dev)
    if scale is not None:
        y = y * scale[:, None, chan]
    if shift is not None:
        y = y + shift[:, None, chan]
    Br = c.res_batch_mod if c.res_batch_mod > 0 else B
    rb = torch.arange(B, device=dev) % Br
    if "id" in c.res:
        r = d["res"].double().to(dev)
        r = r[torch.zeros(B, dtype=torch.long, device=dev)] if c.res_bstride0 else r[rb]
        if defect == "drop_last_res":
            r = r.clone()
            r[-1] = 0
        y = y + r
    if "sc" in c.res:
        rin, rw = d["res_in"], d["res_w"]
        if c.math == cabi.MATH_TF32_TC:
            rin, rw = tf32_trunc(rin), tf32_trunc(rw)
        y = y + torch.einsum("blk,nk->bln", rin.double().to(dev)[rb], rw.double().to(dev)) + d["res_bias"].double().to(dev)
    out = y.reshape(B, c.L_out, c.phases, c.C_out)
    if defect == "phase_shift":                                # phase 1 written one position late
        out = out.clone()
        out[:, 1:, 1] = out[:, :-1, 1].clone()
    out = out.reshape(B, c.L_out * c.phases, c.C_out)
    if gn_term is not None:
        gn_term = gn_term.reshape(B, c.L_out, 1, c.C_out).expand(B, c.L_out, c.phases, c.C_out).reshape(out.shape)
    return out, gn_term


def lnmod_ref(x, shift, scale, L, eps=1e-6):
    """LayerNorm(no affine) * (1 + scale) + shift, rows (B*L, C), per-trajectory (B, C) vectors; float64"""
    x = x.double()
    mean = x.mean(-1, keepdim=True)
    var = ((x - mean) ** 2).mean(-1, keepdim=True)
    tr = torch.arange(x.shape[0], device=x.device) // L
    return (x - mean) / torch.sqrt(var + eps) * (1 + scale.double()[tr]) + shift.double()[tr]


def tolerance(ref: torch.Tensor, out_dtype: int, extra=None, a: float = A_ABS):
    """per-element bound r_out |ref| + a rms(ref) (+ extra)"""
    rms = ref.pow(2).mean().sqrt().item()
    tol = R_OUT[out_dtype] * ref.abs() + a * max(rms, 1e-30)
    return tol if extra is None else tol + extra


def excess(y: torch.Tensor, ref: torch.Tensor, out_dtype: int, extra=None, a: float = A_ABS):
    """max |y - ref| / tolerance (<= 1 passes; NaN and inf count as failures)"""
    y = y.double().to(ref.device)
    err = (y - ref).abs()
    r = err / tolerance(ref, out_dtype, extra, a)
    r = torch.where(torch.isfinite(r), r, torch.full_like(r, float("inf")))
    return r.max().item()


# ---------------------------------------------------------------------------------------------------------------------------
# Python mirror of the tensor-core kernel choice (csrc/conv_tc.cuh).  Documentation that can drift: the GPU tests check the tile
# counts it predicts against what the kernel reports through cds_debug_trace.
TC_VARIANTS = [(64, 16, 1), (64, 32, 1), (64, 64, 1), (64, 128, 1), (64, 256, 1), (64, 32, 2), (64, 64, 2), (64, 128, 2),
               (64, 256, 2), (64, 256, 4), (64, 160, 1), (64, 192, 1),
               (32, 16, 1), (32, 32, 1), (32, 64, 1), (32, 128, 1), (32, 256, 1), (32, 32, 2), (32, 64, 2), (32, 128, 2)]   # :1470


def pick_kc(c: ConvCase):                                   # conv_tc_pick_kc, conv_tc.cuh:1179
    full = 32 if c.math == cabi.MATH_TF32_TC else 64
    wide = c.C_in % full == 0 and ("sc" not in c.res or c.res_C % full == 0)
    return 64 if wide else 32


def runtime_tile(n, kc):                                     # conv_tc_runtime_tile, :1190
    if n % 256 == 0:
        return 256
    if kc == 64 and n % 192 == 0:
        return 192
    if kc == 64 and n % 160 == 0:
        return 160
    return 128 if n % 128 == 0 else 64


def tc_width(c: ConvCase):                                   # conv_tc_width, :1196
    n = c.N
    if n in (32, 64, 128, 256):
        return n if (c.phases == 1 or c.C_out % 16 == 0) else 0
    if n in (512, 1024) and c.phases == 1:
        return n
    if n > 64 and n % 64 == 0 and c.groups == 0:
        tn = runtime_tile(n, pick_kc(c))
        if c.phases == 1 or c.C_out % tn == 0:
            return n
    if n < 32 and c.phases == 1 and c.taps == 1 and c.groups == 0 and not c.res:
        return 16 if n <= 16 else 32
    return 0


def pick_split(c: ConvCase, n_total, m_tiles):               # conv_tc_pick_split, :1256 (without the experiment switches)
    if n_total > 256:
        return n_total // 256
    if c.phases != 1 or n_total < 64:
        return 1
    if n_total >= 128:
        return 2
    if c.math == cabi.MATH_TF32_TC:
        return 1
    return 2 if m_tiles < 296 else 1


def tc_geometry(c: ConvCase):
    """(KC, N, SPLIT, column tiles, row tiles, tiles) of the conv_tc launch -- conv_tc_prepare, :1270"""
    T = 128 // c.L_out
    m_tiles = (c.B * c.L_out + 127) // 128
    n_total = tc_width(c)
    kc = pick_kc(c)
    fixed = n_total in (16, 32, 64, 128, 256) or (n_total in (512, 1024) and c.groups != 0)
    if fixed:
        split = pick_split(c, n_total, m_tiles)
        n, col_tiles = n_total // split, 1
    else:
        split, n = 1, runtime_tile(n_total, kc)
        col_tiles = n_total // n
    nct = split if split > 1 else col_tiles
    return dict(kc=kc, n=n, split=split, col_tiles=col_tiles, T=T, m_tiles=m_tiles, tiles=m_tiles * nct, nct=nct)


def ps_eligible(c: ConvCase):                                # conv_ps_eligible, conv_ps.cuh:389 (given conv_tc_eligible)
    return (c.tc and c.L_in == 4 and c.L_out == 4 and c.stride == 1 and c.phases == 1 and c.taps in (1, 3, 5)
            and c.pad == c.taps // 2 and c.groups == 8 and c.act == cabi.ACT_MISH and c.C_out in (128, 256)
            and c.C_in % 64 == 0 and ("sc" not in c.res or c.res_C % 64 == 0) and "b" not in c.bias and not c.scale
            and "b" not in c.shift and c.odt == c.act_dtype and c.in_batch_mod % 128 == 0 and c.res_batch_mod % 128 == 0
            and dict(c.env).get("CDS_PS") != "0")


def tc_lane(c: ConvCase):
    """which epilogue lane of conv_tc_kernel serves the case: fast (:468), gated / table / plain (:652-662), wide_gn (:1007) or
    generic; ignores the alignment conditions, which the cases below always meet unless they test the generic lane on purpose"""
    g = tc_geometry(c)
    N, kcols = g["n"], g["n"] * g["split"]
    has_gn = c.groups > 0
    smp = "b" in c.bias or "b" in c.scale or "b" in c.shift
    film = 2 if (smp or c.scale) else (1 if c.shift else 0)
    io_vec = tc_width(c) == c.N and c.C_out % 16 == 0
    add_res = "id" in c.res
    has_sc = "sc" in c.res
    out_tma = c.C_out % 16 == 0 and (c.out_pad * (2 if c.odt == cabi.BF16 else 4)) % 16 == 0 and not dict(c.env).get("CDS_NO_TMA_STORE")
    if (N >= 32 and g["col_tiles"] <= 1 and has_gn and c.act == cabi.ACT_MISH and film != 2 and c.phases == 1 and io_vec
            and c.odt == c.act_dtype and c.res_batch_mod == 0 and out_tma and kcols <= 256 and (N & (N - 1)) == 0):
        return "fast"
    if N >= 32 and not has_sc:
        if (not has_gn and c.act == cabi.ACT_NONE and c.scale == "b" and not c.shift and "b" not in c.bias and add_res
                and c.odt != cabi.BF16 and io_vec and c.phases == 1 and c.res_batch_mod == 0 and out_tma and c.sample_pad % 4 == 0):
            return "gated"
        if (not has_gn and film == 0 and not smp and add_res and c.res_batch_mod > 0 and c.act == cabi.ACT_NONE
                and c.odt != cabi.BF16 and io_vec and c.phases == 1 and out_tma):
            return "table"
        if (not has_gn and film == 0 and not smp and not add_res and io_vec and c.res_batch_mod == 0
                and c.act in (cabi.ACT_NONE, cabi.ACT_GELU_TANH)):
            return "plain"
    if has_gn and kcols // 8 > 32:
        return "wide_gn"
    return "generic"


def kernel_for(c: ConvCase):
    if not c.tc:
        return "simt"
    return "ps" if ps_eligible(c) else "tc"


# ---------------------------------------------------------------------------------------------------------------------------
# The case matrix of tests/test_conv_ops_gpu.py.  Every case runs in up to three batch regimes: "one" (a single ragged row tile),
# "multi" (several row tiles, the last one ragged) and "persist" (resized on the GPU so that every CTA runs >= 6 tiles).
TF, BF, FP = cabi.MATH_TF32_TC, cabi.MATH_BF16_TC, cabi.MATH_FP32
MISH, SILU, GELU_T, GELU_E = cabi.ACT_MISH, cabi.ACT_SILU, cabi.ACT_GELU_TANH, cabi.ACT_GELU_ERF


def _conv(name, math_, L, C_in, C_out, taps=1, **kw):
    kw.setdefault("pad", taps // 2)
    kw.setdefault("L_in", L * kw.get("stride", 1))
    return ConvCase(name=name, math=math_, B=1, L_out=L, C_in=C_in, C_out=C_out, taps=taps, **kw)


def _both(name, L, C_in_tf32, C_out, **kw):
    """the same layer in TF32 and in BF16 (bf16 rows hold twice the channels of an fp32 row of the same bytes)"""
    res_C = kw.pop("res_C", 0)
    return [_conv(name + "_tf32", TF, L, C_in_tf32, C_out, res_C=res_C, **kw),
            _conv(name + "_bf16", BF, L, 2 * C_in_tf32, C_out, res_C=2 * res_C, **kw)]


def conv_cases():
    gn = dict(groups=8, act=MISH)
    cs = []
    # ---- conv_tc fast lane: GN + Mish, film 0 / 1, identity residual through TMA / ld.global, shortcut conv with res_C != C_in
    cs += _both("fast_L32_c32_kc32_shift_res", 32, 16, 32, taps=5, shift="s", res="id", **gn)
    cs += _both("fast_L16_c64_kc64_idsc", 16, 64, 64, taps=5, res="id+sc", res_C=32, **gn)
    cs += _both("fast_L8_c128_kc32_shift_res", 8, 48, 128, taps=3, shift="s", res="id", **gn)
    cs += [_conv("fast_L4_c256_kc64_sc_tf32", TF, 4, 32, 256, taps=3, res="sc", res_C=64, **gn),      # (bf16 twin: conv_ps)
           _conv("fast_L4_c256_kc32_sc_bf16", BF, 4, 96, 256, taps=3, res="sc", res_C=64, **gn)]
    cs += _both("fast_L32_c32_kc64_shift", 32, 64, 32, taps=5, shift="s", **gn)
    cs += _both("fast_L8_c64_kc32_res_notma", 8, 16, 64, taps=5, res="id", env=(("CDS_NO_TMA_RES", "1"),), **gn)
    cs += _both("fast_L16_c128_kc64_shift_sc", 16, 64, 128, taps=5, shift="s", res="sc", res_C=96, **gn)
    cs += _both("fast_L4_c256_kc32_res", 4, 48, 256, taps=5, res="id", **gn)
    # ---- wide GroupNorm (C_out 512 / 1024: split 2 / 4, 64 / 128 channels per group), with and without per-trajectory FiLM
    cs += _both("wide_L16_c512_shift_res", 16, 64, 512, taps=5, shift="s", res="id", **gn)
    cs += _both("wide_L8_c1024_film", 8, 32, 1024, taps=3, scale="b", shift="b", **gn)
    cs += _both("wide_L8_c512_film_sc", 8, 32, 512, taps=3, scale="sb", shift="b", res="sc", res_C=64, **gn)
    # ---- GroupNorm with another activation (generic lane, the run(T, AX, F2) branch)
    cs += _both("gn_silu_L16_c64", 16, 32, 64, taps=3, groups=8, act=SILU, shift="s")
    cs += _both("gn_gelu_L32_c256_film", 32, 64, 256, taps=3, groups=8, act=GELU_T, scale="sb", shift="b")
    # ---- plain lane: act NONE / GELU_TANH, out F32 / TF32 / BF16, stride 2, two phases (4-D TMA store / direct stores)
    cs += _both("plain_stride2_L16_c64", 16, 32, 64, taps=3, stride=2)
    cs += _both("plain_phases2_L8_c64", 8, 32, 64, taps=3, phases=2, act=GELU_T)
    cs += _both("plain_phases2_L8_c64_notma", 8, 32, 64, taps=3, phases=2, env=(("CDS_NO_TMA_STORE", "1"),))
    cs += _both("plain_phases2_L16_c128_kc32", 16, 48, 128, taps=3, phases=2, act=GELU_T)
    cs += [_conv("plain_L8_c64_out_f32_tf32", TF, 8, 32, 64, taps=3, act=GELU_T, out_dtype=cabi.F32),
           _conv("plain_L8_c64_out_bf16_tf32", TF, 8, 32, 64, taps=3, out_dtype=cabi.BF16)]
    # runtime column tiles: 320 = 2 x 160, 384 = 3 x 128 (KC 32) / 2 x 192, 960 = 5 x 192, 1280 = 5 x 256, 192 = 3 x 64 (KC 32)
    cs += _both("coltile_tok_c320", 1, 64, 320, act=GELU_T)
    cs += _both("coltile_tok_c384_kc32", 1, 48, 384)
    cs += [_conv("coltile_tok_c960_tf32", TF, 1, 64, 960, out_dtype=cabi.F32),
           _conv("coltile_tok_c1280_tf32", TF, 1, 64, 1280, act=GELU_T),
           _conv("coltile_L16_c192_kc32_tf32", TF, 16, 16, 192, taps=3),
           _conv("coltile_tok_c512_kc32_tf32", TF, 1, 48, 512)]
    # ---- gated (gate x out + dense residual) and table (+ table[row % period]) forms over flattened token rows
    for div, C in ((37, 128), (64, 256), (100, 320)):
        cs.append(_conv(f"gated_div{div}_c{C}_tf32", TF, 1, 64, C, scale="b", res="id", sample_row_div=div, out_dtype=cabi.F32))
        cs.append(_conv(f"table_p{div}_c{C}_tf32", TF, 1, 64, C, res="id", res_batch_mod=div, out_dtype=cabi.F32))
    cs.append(_conv("gated_div64_c256_tf32out", TF, 1, 32, 256, scale="b", res="id", sample_row_div=64, out_dtype=cabi.TF32))
    # ---- generic lane: the other activations with step + sample scale and shift, unaligned FiLM rows, narrow heads, CFG halves,
    # strided views, per-trajectory residual rows
    cs += _both("gen_silu_L8_c64_film", 8, 32, 64, taps=3, act=SILU, scale="sb", shift="sb")
    cs += _both("gen_mishsilu_L16_c128_film_unaligned", 16, 32, 128, taps=3, act=cabi.ACT_MISH_SILU, scale="sb", shift="sb",
                sample_pad=1)
    cs += _both("gen_leaky_L8_c64_cfg", 8, 32, 64, taps=3, act=cabi.ACT_LEAKY_RELU, scale="s", shift="b", in_batch_mod=32)
    cs += _both("gen_gelu_erf_L4_c64_strided", 4, 32, 64, taps=3, act=GELU_E, bias="sb", in_pad=8, in_coff=8, out_pad=8)
    cs += _both("gen_film_bias_sample_tok", 1, 32, 128, act=SILU, bias="sb", scale="b", sample_row_div=37)
    for C_out, C_in in ((14, 32), (29, 16), (14, 16)):
        cs.append(_conv(f"head_c{C_out}_cin{C_in}_f32", TF, 16, C_in, C_out, out_dtype=cabi.F32, out_pad=3))
        cs.append(_conv(f"head_c{C_out}_cin{C_in}_tf32", TF, 16, C_in, C_out, out_dtype=cabi.TF32, out_pad=3))
    cs += _both("gen_gn_res_batch_mod", 8, 32, 64, taps=3, res="id", res_batch_mod=32, **gn)
    cs += _both("gen_gn_res_bstride0", 8, 32, 64, taps=3, res="id", res_bstride0=True, **gn)
    # ---- conv_ps (L = 4, C_out 128 / 256) and the same layers with CDS_PS=0 (then conv_tc serves them)
    for nm, cin, cout, taps, kw in (("ps_c64_128_k5_res", 64, 128, 5, dict(shift="s", res="id")),
                                    ("ps_c128_256_k3_sc", 128, 256, 3, dict(res="sc", res_C=64)),
                                    ("ps_c256_256_k1_cfg", 256, 256, 1, dict(in_batch_mod=128, res="id", res_batch_mod=128)),
                                    ("ps_c64_256_k5_idsc", 64, 256, 5, dict(shift="s", res="id+sc", res_C=128)),
                                    ("ps_c128_128_k3", 128, 128, 3, {})):
        for m in (TF, BF):
            c = _conv(f"{nm}_{'tf32' if m == TF else 'bf16'}", m, 4, cin, cout, taps=taps, **gn, **kw)
            cs += [c.with_(expect="ps"), c.with_(name=c.name + "_ps0", env=(("CDS_PS", "0"),))]
    # ---- conv_simt (CDS_MATH_FP32): fp32 and bf16 inputs, BN 32 / 64 / 128, GroupNorm, stride 2, two phases, shortcut conv
    cs += [_conv("simt_L32_c32_gn_sc", FP, 32, 14, 32, taps=5, shift="s", res="sc", res_C=14, **gn),
           _conv("simt_L16_stride2_bf16in", FP, 16, 32, 64, taps=3, stride=2, act=MISH, in_dtype=cabi.BF16, out_dtype=cabi.BF16),
           _conv("simt_L8_phases2", FP, 8, 32, 64, taps=3, phases=2, act=GELU_T),
           _conv("simt_L4_c256_gn_film_res", FP, 4, 64, 256, taps=3, scale="b", shift="b", res="id", **gn)]
    # ---- edges: pre-activations spanning +-100s (Mish's e = inf branch, flush to zero, the GELU tails)
    for act in (MISH, GELU_E, SILU, cabi.ACT_MISH_SILU):
        cs.append(_conv(f"edge_amp100_{ACT_NAMES[act]}_tf32", TF, 8, 32, 64, taps=3, act=act, amp=100.0, shift="s"))
    cs.append(_conv("edge_amp100_gelu_tanh_plain_tf32", TF, 8, 32, 64, taps=3, act=GELU_T, amp=100.0, out_dtype=cabi.F32))
    cs.append(_conv("edge_amp100_mish_bf16", BF, 8, 64, 64, taps=3, act=MISH, amp=100.0, shift="s"))
    # ---- GroupNorm with a large common offset (64 and 256 group sigmas in the bias) on every GroupNorm implementation
    for off in (64, 256):
        cs += [_conv(f"gnoff{off}_fast_L16_c64_tf32", TF, 16, 64, 64, taps=5, gn_offset=off, shift="s", **gn),
               _conv(f"gnoff{off}_fast_L32_c256_tf32", TF, 32, 32, 256, taps=3, gn_offset=off, **gn),
               _conv(f"gnoff{off}_generic_L8_c64_tf32", TF, 8, 32, 64, taps=3, gn_offset=off, scale="b", **gn),
               _conv(f"gnoff{off}_wide_L16_c512_tf32", TF, 16, 64, 512, taps=3, gn_offset=off, **gn),
               _conv(f"gnoff{off}_ps_c256_tf32", TF, 4, 64, 256, taps=3, gn_offset=off, expect="ps", **gn),
               _conv(f"gnoff{off}_ps_c128_bf16", BF, 4, 128, 128, taps=3, gn_offset=off, expect="ps", **gn),
               _conv(f"gnoff{off}_simt_L16_c64", FP, 16, 32, 64, taps=3, gn_offset=off, **gn)]
    for c in cs:
        assert kernel_for(c) == (c.expect if c.expect != "tc" or c.tc else "simt"), c.name
    return [c if c.tc else c.with_(expect="simt") for c in cs]


PERSISTENT = ("fast_L32_c32_kc32_shift_res", "fast_L16_c64_kc64_idsc", "fast_L8_c128_kc32_shift_res", "fast_L4_c256_kc64_sc",
              "fast_L8_c64_kc32_res_notma", "wide_L16_c512_shift_res", "wide_L8_c1024_film", "plain_phases2_L8_c64",
              "coltile_tok_c320", "coltile_tok_c960_tf32", "gated_div100_c320_tf32", "table_p37_c128_tf32",
              "gen_mishsilu_L16_c128_film_unaligned", "gen_gelu_erf_L4_c64_strided", "head_c29_cin16_tf32",
              "gen_gn_res_batch_mod", "gnoff256_fast_L16_c64_tf32")


def regimes(c: ConvCase):
    """batch sizes of the "one" and "multi" regimes; "persist" is sized on the GPU from the grid of a probe launch"""
    T = 128 // c.L_out
    if c.expect == "ps" or (c.tc and ps_eligible(c.with_(env=()))):
        one, multi = 100, 300                                # (conv_ps: tiles of 128 trajectories)
    else:
        one, multi = (T - 1 if T > 1 else 1), 3 * T + T // 2 + 1
    if c.in_batch_mod:
        one, multi = max(one, c.in_batch_mod) + 1, 3 * c.in_batch_mod
    if c.res_batch_mod:
        one, multi = max(one, c.res_batch_mod + 1), max(multi, 3 * c.res_batch_mod)
    out = [("one", one), ("multi", multi)]
    if c.math == TF and c.expect == "tc" and any(c.name.startswith(p) for p in PERSISTENT):
        out.append(("persist", 0))
    return out
