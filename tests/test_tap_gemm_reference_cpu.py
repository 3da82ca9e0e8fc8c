"""A float64 reference of the tcgen05 tap-GEMM (csrc/gemm_sm100.cu) and the comparator tests/test_gpu_tap_gemm.py
checks the kernel with, plus the CPU checks that make both trustworthy:
  - the reference, fed weights packed by the product's own loaders, computes what the oracle's causal Conv1d /
    ConvTranspose1d and the gated MLPs compute;
  - the comparator accepts a float32-accumulated computation of every sweep case, and rejects that computation once
    it carries any of a list of plausible kernel faults (a dropped tap, a shifted tap, missing K columns, a wrong
    channel modulus, an unwritten column chunk or row, gate and up swapped);
  - the ctypes descriptor of the test hook has the C layout, and its wrapper refuses undersized buffers.

The kernel (reference in parentheses):
  acc[b][m][n] = sum_tap sum_k A[b][m + shift[tap] + a_row0][k] * W[n][tap*Kp + k]   (float64; rows outside
  [0, a_rows) read as zero); then the epilogue with the kernel's bf16 rounding points:
    x = rnd(acc + bias[n % cmod]); x = rnd(x * scale); x = rnd(x + resid)   -> out_raw
    out_act = rnd(act(x))                               (SnakeBeta, GELU, or x itself)
    gated:  g, u = rnd(acc + bias) of the gate / up columns;  out_act = rnd(rnd(silu(g)) * u)
The kernel's admissible output is an interval carried through that chain: the fp32 accumulation may be off by
ACC_REL * S (S = sum |a| * |w|, the same sum with absolute values), every fp32 operation by 2^-23 of its magnitude,
every activation by its Lipschitz constant times the input's interval plus its evaluation error (the SFU sine and
exponential included); rounding maps an interval onto the bf16 grid points it covers.  So an element is off by at
most one bf16 ulp, and only where the exact value lies within the accumulation error of a rounding boundary.
ACC_REL = 2^-16 is 57x what a float32 emulation of the accumulation needs at K up to 6144 with 7 taps
(1.15 * 2^-24 * S worst case); separately, at most 0.5 % of the elements may differ from the rounded reference.
The float32 emulation differs in about 1e-4 of them; the tensor cores' accumulation and the SFU sine of the SnakeBeta
epilogue in up to 0.31 % (see MISMATCH_RATE), every one of them inside the interval."""
import ctypes
import dataclasses
import math
import os
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

ACT_NONE, ACT_SNAKE, ACT_GELU, ACT_SWIGLU_PAIR, ACT_SWIGLU_BLK8 = range(5)
GATED = (ACT_SWIGLU_PAIR, ACT_SWIGLU_BLK8)
ACC_REL = 2.0 ** -16       # accumulation error the comparator allows, relative to S = sum |a| * |w|
F32_REL = 2.0 ** -23       # one float32 rounding (2^-24) with margin
MISMATCH_RATE = 5e-3       # share of elements allowed to differ from the rounded reference (by one ulp); measured on
                           # the B200: up to 0.2 % for plain and gated outputs at K up to 6144, 0.31 % for SnakeBeta
                           # after 7-tap convolutions (profiles/tap_gemm_parity.txt)
SENTINEL = 0x7FA5          # bf16 NaN with a payload: what every output buffer holds before a launch
GUARD = 64                 # sentinel elements after the last batch slice of every output buffer


# ----------------------------------------------------------------------------------------------------- cases
@dataclasses.dataclass
class Case:
    """One tap-GEMM problem: geometry, epilogue and the buffer views it runs on."""
    name: str
    B: int
    T: int
    K: int
    N: int
    shifts: tuple = (0,)
    bn: int = 0                # 0: the production choice
    act: int = ACT_NONE
    cmod: int = 0              # 0: N
    bias: bool = True
    scale: bool = False
    resid: bool = False
    inplace: bool = False      # resid is out_raw itself (the talker prefill's residual stream)
    raw: bool = True
    actout: bool = False
    hist: int = 0              # history rows in front of every batch slice of A (streaming views)
    view: bool = False         # outputs / residual inside larger per-batch slices (explicit batch strides)
    snake_big: bool = False    # SnakeBeta arguments |x * exp(alpha)| up to ~1e3
    seed: int = 0
    ntaps: int = 0             # 0: len(shifts) (the refusal checks set it apart)

    @property
    def Kp(self):
        return (self.K + 63) // 64 * 64

    @property
    def taps(self):
        return self.ntaps or len(self.shifts)

    @property
    def act_width(self):
        return self.N // 2 if self.act in GATED else self.N


def _conv_shifts(k, dil):
    return tuple(-(k - 1 - j) * dil for j in range(k))


SHIFT_SETS = [(0,), (0, -1), (-2, -1, 0), _conv_shifts(7, 1), _conv_shifts(7, 3), _conv_shifts(7, 9),
              (-6, -5, -4, -3, -2, -1, 0, 1)]
EPILOGUES = [dict(act=ACT_NONE, scale=True, resid=True), dict(act=ACT_SNAKE, resid=True, actout=True),
             dict(act=ACT_SNAKE, raw=False, actout=True), dict(act=ACT_GELU, raw=False, actout=True),
             dict(act=ACT_NONE, bias=False, resid=True, inplace=True), dict(act=ACT_SWIGLU_PAIR, raw=False, actout=True),
             dict(act=ACT_SWIGLU_BLK8, raw=False, actout=True)]


def sweep_cases():
    """Every tile width from 16 to 256, each with a partial last N tile where one exists, crossed (not multiplied) with
    the T / B / K / tap / epilogue variants; then the named edge cases."""
    cases = []
    for i, bn in enumerate(range(16, 257, 16)):
        N = bn * (1 + i % 2) + 16 * (1 + i % 3)
        cases.append(Case(f"bn{bn}", B=(1, 3)[i % 2], T=(1, 4, 127, 128, 129, 300)[i % 6], K=(16, 48, 96, 192, 1536)[i % 5],
                          N=N, shifts=SHIFT_SETS[i % 7], bn=bn, seed=i, **EPILOGUES[i % 7]))
    cases += [
        Case("partial_n272", B=2, T=129, K=96, N=272, bn=256, act=ACT_SNAKE, resid=True, actout=True, seed=20),
        Case("convT_288_bn144", B=3, T=300, K=192, N=288, cmod=96, shifts=(0, -1), bn=144, act=ACT_SNAKE, actout=True, seed=21),
        Case("convT_288_pick", B=1, T=127, K=96, N=288, cmod=96, shifts=(0, -1), act=ACT_SNAKE, actout=True, seed=22),
        Case("c96_dil9_bn96", B=2, T=300, K=96, N=96, shifts=_conv_shifts(7, 9), bn=96, act=ACT_SNAKE, raw=False,
             actout=True, seed=23),
        Case("c96_resid_bn96", B=3, T=129, K=96, N=96, bn=96, act=ACT_SNAKE, resid=True, actout=True, seed=24),
        Case("t1_dil9", B=3, T=1, K=64, N=64, shifts=_conv_shifts(7, 9), act=ACT_SNAKE, raw=False, actout=True, seed=25),
        Case("snake_big_args", B=2, T=129, K=128, N=160, act=ACT_SNAKE, resid=True, actout=True, snake_big=True, seed=26),
        Case("gelu_pw1", B=3, T=128, K=64, N=256, act=ACT_GELU, raw=False, actout=True, seed=27),
        Case("none_scale_resid", B=2, T=300, K=1536, N=128, scale=True, resid=True, seed=28),
        Case("inplace_resid", B=1, T=300, K=256, N=512, bias=False, resid=True, inplace=True, seed=29),
        Case("swiglu_pair_bias", B=2, T=129, K=192, N=384, act=ACT_SWIGLU_PAIR, raw=False, actout=True, seed=30),
        Case("swiglu_blk8", B=1, T=37, K=256, N=1024, act=ACT_SWIGLU_BLK8, bias=False, raw=False, actout=True, seed=31),
        Case("many_tiles", B=3, T=300, K=64, N=512, bn=64, act=ACT_GELU, actout=True, seed=32),
        # streaming views: A = [B][hist + cap][K] read from row hist on, outputs / residual inside history buffers
        Case("hist_dil3", B=3, T=129, K=96, N=96, shifts=_conv_shifts(7, 3), hist=18, view=True, act=ACT_SNAKE,
             raw=False, actout=True, seed=33),
        Case("hist_dil9_t4", B=2, T=4, K=192, N=192, shifts=_conv_shifts(7, 9), hist=54, view=True, act=ACT_SNAKE,
             raw=False, actout=True, seed=34),
        Case("hist_convT", B=3, T=127, K=192, N=384, cmod=96, shifts=(0, -1), hist=1, view=True, act=ACT_SNAKE,
             actout=True, seed=35),
        Case("hist_preconv_resid", B=2, T=13, K=512, N=256, shifts=(-2, -1, 0), hist=2, view=True, scale=True,
             resid=True, seed=36),
        Case("view_gelu", B=3, T=40, K=64, N=256, view=True, act=ACT_GELU, actout=True, seed=37),
        Case("view_swiglu", B=2, T=33, K=128, N=256, view=True, act=ACT_SWIGLU_PAIR, raw=False, actout=True, seed=38),
    ]
    return cases


# ----------------------------------------------------------------------------------------------------- buffers
@dataclasses.dataclass
class Layout:
    """A [B][T][width] tensor inside one flat allocation: batch slices of `bs` elements, the tensor at element
    `offset` of each slice (rows in front = history, rows behind = a gap); output buffers (numel) add GUARD
    sentinel elements at the end."""
    B: int
    T: int
    width: int
    before: int = 0
    after: int = 0

    @property
    def bs(self):
        return (self.before + self.T + self.after) * self.width

    @property
    def offset(self):
        return self.before * self.width

    @property
    def numel(self):
        return self.B * self.bs + GUARD

    def view(self, flat):
        return flat[:self.B * self.bs].view(self.B, -1)[:, self.offset:self.offset + self.T * self.width].reshape(
            self.B, self.T, self.width)

    def mask(self, device="cpu"):
        m = torch.zeros(self.numel, dtype=torch.bool, device=device)
        self.view(m)[:] = True
        return m


def layouts(c: Case):
    """Layout of A (rows = hist + T + unread tail), resid, out_raw, out_act; the view cases use odd strides."""
    a = Layout(c.B, c.hist + c.T, c.K, 0, 3 if c.hist or c.view else 0)
    mk = (lambda w, pre, post: Layout(c.B, c.T, w, pre, post)) if c.view else (lambda w, pre, post: Layout(c.B, c.T, w))
    return a, mk(c.N, 5, 2), mk(c.N, 3, 1), mk(c.act_width, 7, 3)


def make_inputs(c: Case, device="cpu"):
    """Seeded inputs of a case as flat device buffers: A, W (its Kp padding random, so a column of A past K read as
    anything but zero shows), fp32 channel vectors, the residual.  Rows of A past hist + T are NaN: never to be read."""
    g = torch.Generator().manual_seed(1000 + c.seed)
    la, lr, _, _ = layouts(c)
    A = torch.full((la.B * la.bs,), float("nan"))
    A[:la.B * la.bs].view(c.B, -1)[:, :(c.hist + c.T) * c.K] = torch.randn(c.B, (c.hist + c.T) * c.K, generator=g)
    wstd = 1.0 / math.sqrt(c.K * c.taps)
    W = torch.randn(c.N, c.taps * c.Kp, generator=g) * wstd
    cm = c.cmod or c.N
    inp = {"A": A.bfloat16(), "W": W.bfloat16()}
    if c.bias:
        inp["bias"] = torch.randn(cm, generator=g) * 0.5
    if c.scale:
        inp["scale"] = (torch.rand(cm, generator=g) + 0.5) * torch.where(torch.rand(cm, generator=g) < 0.2, -1.0, 1.0)
    if c.act == ACT_SNAKE:
        lo, hi = (5.0, 6.9) if c.snake_big else (-1.0, 1.0)
        inp["snake_ea"] = torch.exp(torch.rand(cm, generator=g) * (hi - lo) + lo)
        inp["snake_ib"] = 1.0 / (torch.exp(torch.rand(cm, generator=g) * 2 - 1) + 1e-9)
    if c.resid:
        R = torch.full((lr.B * lr.bs,), float("nan"))
        lr.view(R)[:] = torch.randn(c.B, c.T, c.N, generator=g)
        inp["resid"] = R.bfloat16()
    return {k: v.to(device) for k, v in inp.items()}


def a_view(c: Case, A):
    """The [B][a_rows][K] rows the A tensor map covers."""
    la = layouts(c)[0]
    return A[:la.B * la.bs].view(c.B, -1)[:, :(c.hist + c.T) * c.K].reshape(c.B, c.hist + c.T, c.K)


# ----------------------------------------------------------------------------------------------------- reference
def bf16_grid(x):
    """Spacing of the bf16 grid at |x| (float64): 2^(e-8) for |x| in [2^(e-1), 2^e), subnormals 2^-133."""
    _, e = torch.frexp(x)
    return torch.ldexp(torch.ones_like(x), torch.clamp(e, min=-125) - 8)


def rnd(x):
    """float64 -> nearest bf16 value, ties to even (the kernel's cvt.rn.bf16.f32 on a float32 value is the same)."""
    u = bf16_grid(x)
    return torch.round(x / u) * u


def accumulate(A, W, T, Kp, shifts, a_row0=0):
    """float64 acc [B][T][N] and S = the same sum over |a| * |w|.  A: [B][a_rows][K]; W: [N][ntaps*Kp]."""
    B, a_rows, K = A.shape
    A64, W64 = A.double(), W.double()
    acc = torch.zeros(B, T, W.shape[0], dtype=torch.float64, device=A.device)
    S = torch.zeros_like(acc)
    m = torch.arange(T, device=A.device)
    for tap, sh in enumerate(shifts):
        rows = m + sh + a_row0
        ok = (rows >= 0) & (rows < a_rows)
        At = torch.zeros(B, T, K, dtype=torch.float64, device=A.device)
        At[:, ok] = A64[:, rows[ok]]
        Wt = W64[:, tap * Kp:tap * Kp + K]
        acc += At @ Wt.T
        S += At.abs() @ Wt.abs().T
    return acc, S


def _chan(v, N, cmod):
    return v.double()[torch.arange(N, device=v.device) % cmod]


def gelu(x):
    return 0.5 * x * (1.0 + torch.erf(x / math.sqrt(2.0)))


def silu(x):
    return x / (1.0 + torch.exp(-x))


def act_bounds(act, x, xlo, xhi, ea=None, ib=None):
    """(value at x, half-width) of the kernel's activation over the input interval [xlo, xhi] around x: Lipschitz
    constant times the input's distance plus the float32 / SFU evaluation error at the interval's largest |x|."""
    w = torch.maximum(xhi - x, x - xlo)
    xm = torch.maximum(xlo.abs(), xhi.abs())
    if act == ACT_SNAKE:
        # the argument x * exp(alpha) is a float32 product in the kernel as in PyTorch: a rounding point.  Then MUFU.SIN
        # (2^-21.4 on [-pi, pi]) after the Cody-Waite reduction (error ~2^-33 per period), and where the input is an
        # interval, the rounding of the argument at its other points
        a = (x * ea).float().double()
        am = xm * ea
        d_sin = 2.0 ** -21 + 2.0 ** -30 * am + torch.where(w > 0, 2 * F32_REL * am, torch.zeros_like(am))
        err = ib * (2 * d_sin + d_sin ** 2) + 2 * F32_REL * (xm + ib)
        return x + ib * torch.sin(a) ** 2, (1 + ib * ea) * w + err
    if act == ACT_GELU:
        return gelu(x), 1.13 * w + 2.0 ** -20 * xm
    if act in GATED:
        return silu(x), 1.1 * w + xm * (2.0 ** -21 + 2.0 ** -23 * xm) + 2.0 ** -140
    return x.clone(), w


def _round_interval(v, lo, hi):
    return rnd(v), rnd(lo), rnd(hi)


def reference(c: Case, inp):
    """name -> (rounded reference, lowest, highest admissible kernel value), float64 [B][T][width], for out_raw and
    out_act as the case writes them."""
    A = a_view(c, inp["A"])
    acc, S = accumulate(A, inp["W"], c.T, c.Kp, c.shifts, c.hist)
    cm = c.cmod or c.N
    x = acc + (_chan(inp["bias"], c.N, cm) if c.bias else 0.0)
    e = ACC_REL * S + F32_REL * x.abs()
    v, lo, hi = _round_interval(x, x - e, x + e)
    out = {}
    if c.act in GATED:
        if c.act == ACT_SWIGLU_PAIR:
            gi = torch.arange(0, c.N, 2)
        else:
            j = torch.arange(c.N // 2)
            gi = (j // 8) * 16 + j % 8
        gi = gi.to(v.device)
        ui = gi + (1 if c.act == ACT_SWIGLU_PAIR else 8)
        g, glo, ghi = v[..., gi], lo[..., gi], hi[..., gi]
        u, ulo, uhi = v[..., ui], lo[..., ui], hi[..., ui]
        s, d = act_bounds(c.act, g, glo, ghi)
        s, slo, shi = _round_interval(s, s - d, s + d)
        corners = torch.stack([slo * ulo, slo * uhi, shi * ulo, shi * uhi])
        plo, phi = corners.min(0).values, corners.max(0).values
        y = s * u
        out["out_act"] = _round_interval(y, plo - F32_REL * plo.abs(), phi + F32_REL * phi.abs())
        return out
    if c.scale:
        sc = _chan(inp["scale"], c.N, cm)
        p = torch.stack([lo * sc, hi * sc])
        plo, phi = p.min(0).values, p.max(0).values
        v, lo, hi = _round_interval(v * sc, plo - F32_REL * plo.abs(), phi + F32_REL * phi.abs())
    if c.resid:
        r = layouts(c)[1].view(inp["resid"]).double()
        x = v + r
        v, lo, hi = _round_interval(x, lo + r - F32_REL * (lo + r).abs(), hi + r + F32_REL * (hi + r).abs())
    if c.raw:
        out["out_raw"] = (v, lo, hi)
    if c.actout:
        out["out_act"] = activate(c, inp, v, lo, hi)
    return out


def activate(c: Case, inp, v, lo, hi):
    """out_act of a non-gated case from its pre-activation value v in [lo, hi]."""
    cm = c.cmod or c.N
    kw = {}
    if c.act == ACT_SNAKE:
        kw = dict(ea=_chan(inp["snake_ea"], c.N, cm), ib=_chan(inp["snake_ib"], c.N, cm))
    y, d = act_bounds(c.act, v, lo, hi, **kw)
    return _round_interval(y, y - d, y + d)


def compare(out, ref):
    """Check a kernel output (bf16 [B][T][width]) against (rounded reference, lo, hi): figures and the failures."""
    v, lo, hi = ref
    o = out.double()
    inside = (o >= lo) & (o <= hi)                                   # NaN -> outside
    bound = torch.maximum(torch.maximum(hi - v, v - lo), bf16_grid(v))
    ratio = ((o - v).abs() / bound).nan_to_num(nan=float("inf"))
    mism = (o != v)
    bad = (~inside).nonzero()
    return {"n": int(v.numel()), "n_outside": int(bad.shape[0]), "worst_ratio": float(ratio.max()) if v.numel() else 0.0,
            "mismatch_rate": float(mism.double().mean()) if v.numel() else 0.0,
            "first_outside": bad[:3].tolist(),
            "ok": bad.shape[0] == 0 and float(mism.double().mean()) <= MISMATCH_RATE}


def check_case(c: Case, inp, outs):
    """Compare every output of a case (dict name -> bf16 [B][T][width]); also out_act against the activation of the
    kernel's own out_raw where both exist.  Returns name -> figures."""
    ref = reference(c, inp)
    rep = {k: compare(outs[k], r) for k, r in ref.items()}
    if c.raw and c.actout:
        raw = outs["out_raw"].double()
        rep["out_act_vs_own_raw"] = compare(outs["out_act"], activate(c, inp, raw, raw, raw))
    return rep


# ----------------------------------------------------------------------------------------------------- emulation
def emulate(c: Case, inp, fault=None):
    """What the kernel computes, on the CPU: float32 accumulation (BLAS order), the float32 epilogue with the bf16
    rounding points.  `fault` injects one of the FAULTS below."""
    shifts = list(c.shifts)
    A = a_view(c, inp["A"]).float()
    W = inp["W"].float().clone()
    cm = c.cmod or c.N
    if fault == "drop_tap":
        shifts = shifts[:-1]
    elif fault == "shift_off_by_one":
        shifts[0] -= 1
    elif fault == "drop_last_k16":
        for t in range(c.taps):
            W[:, t * c.Kp + c.K - 16:t * c.Kp + c.K] = 0
    acc = torch.zeros(c.B, c.T, c.N)
    m = torch.arange(c.T)
    for tap, sh in enumerate(shifts):
        rows = m + sh + c.hist
        ok = (rows >= 0) & (rows < c.hist + c.T)
        At = torch.zeros(c.B, c.T, c.K)
        At[:, ok] = A[:, rows[ok]]
        acc += At @ W[:, tap * c.Kp:tap * c.Kp + c.K].T
    r16 = lambda t: t.bfloat16().float()  # noqa: E731
    ch = torch.arange(c.N) % (cm // 2 if fault == "wrong_cmod" else cm)
    x = acc + (inp["bias"].float()[ch] if c.bias else 0.0)
    x = r16(x)
    outs = {}
    if c.act in GATED:
        if c.act == ACT_SWIGLU_PAIR:
            g, u = x[..., 0::2], x[..., 1::2]
        else:
            xs = x.view(c.B, c.T, c.N // 16, 2, 8)
            g, u = xs[:, :, :, 0].reshape(c.B, c.T, -1), xs[:, :, :, 1].reshape(c.B, c.T, -1)
        if fault == "swap_gate_up":
            g, u = u, g
        outs["out_act"] = (r16(g / (1 + torch.exp(-g))) * u).bfloat16()
    else:
        if c.scale:
            x = r16(x * inp["scale"].float()[ch])
        if c.resid:
            x = r16(x + layouts(c)[1].view(inp["resid"]).float())
        if c.raw:
            outs["out_raw"] = x.bfloat16()
        if c.actout:
            if c.act == ACT_SNAKE:
                y = x + inp["snake_ib"].float()[ch] * torch.sin(x * inp["snake_ea"].float()[ch]) ** 2
            elif c.act == ACT_GELU:
                y = 0.5 * x * (1 + torch.erf(x * 0.70710678118654752))
            else:
                y = x
            outs["out_act"] = y.bfloat16()
    for k in outs:
        if fault == "unwritten_chunk":
            outs[k][0, :128, 16:32] = float("nan")
        elif fault == "drop_last_row":
            outs[k][:, -1] = float("nan")
    return outs


# ----------------------------------------------------------------------------------------------------- the hook
def out_buffers(c: Case, device):
    """Sentinel-filled flat bf16 buffers for out_raw / out_act (None where the case does not write one)."""
    _, _, lraw, lact = layouts(c)
    mk = lambda l: torch.full((l.numel,), SENTINEL, dtype=torch.int16, device=device).view(torch.bfloat16)  # noqa: E731
    return {"out_raw": mk(lraw) if c.raw else None, "out_act": mk(lact) if c.actout else None}


def launch(c: Case, inp, outs, max_ctas=0):
    """One q3_debug_tap_gemm launch of case c on the current stream.  Every buffer is checked against what the
    descriptor lets the kernel touch first, so a wrong test raises here instead of reaching the device."""
    from qwen3_tts_b200 import _lib
    la, lr, lraw, lact = layouts(c)
    cm = c.cmod or c.N

    def need(name, t, n, dtype):
        if t is None:
            raise ValueError(f"{c.name}: {name} missing")
        if t.dtype != dtype or not t.is_contiguous() or t.dim() != 1 or t.numel() < n:
            raise ValueError(f"{c.name}: {name} must be a flat contiguous {dtype} tensor of >= {n} elements, "
                             f"got {t.dtype} {tuple(t.shape)}")
        return t.data_ptr()

    d = _lib.TapGemmDesc()
    d.B, d.T, d.K, d.N, d.Kp, d.ntaps, d.bn, d.act, d.cmod, d.max_ctas = c.B, c.T, c.K, c.N, c.Kp, c.taps, c.bn, c.act, c.cmod, max_ctas
    for i, sh in enumerate(c.shifts[:8]):
        d.shifts[i] = sh
    d.a = need("A", inp["A"], la.B * la.bs, torch.bfloat16)
    d.a_bs, d.a_rows, d.a_row0 = (la.bs, c.hist + c.T, c.hist) if c.hist or c.view else (0, 0, 0)
    d.w = need("W", inp["W"].reshape(-1), c.N * c.taps * c.Kp, torch.bfloat16)
    for name, on in (("bias", c.bias), ("scale", c.scale), ("snake_ea", c.act == ACT_SNAKE), ("snake_ib", c.act == ACT_SNAKE)):
        if on:
            setattr(d, name, need(name, inp[name], cm, torch.float32))
    if c.resid:
        src, lres = (outs["out_raw"], lraw) if c.inplace else (inp["resid"], lr)
        d.resid = need("resid", src[lres.offset:], (c.B - 1) * lres.bs + c.T * c.N, torch.bfloat16)
        d.resid_bs = lres.bs if c.view else 0
    for name, l, on in (("out_raw", lraw, c.raw), ("out_act", lact, c.actout)):
        if on:
            t = outs[name]
            if t is None or t.numel() != l.numel:
                raise ValueError(f"{c.name}: {name} must be the case's sentinel buffer of {l.numel} elements")
            setattr(d, name, need(name, t[l.offset:], (c.B - 1) * l.bs + c.T * l.width, torch.bfloat16))
            setattr(d, "raw_bs" if name == "out_raw" else "act_bs", l.bs if c.view else 0)
    lib = _lib.load()
    stream = torch.cuda.current_stream().cuda_stream
    _lib.check(lib.q3_debug_tap_gemm(ctypes.byref(d), ctypes.c_void_p(stream)))


def run(c: Case, inp, max_ctas=0):
    """Fresh sentinel outputs (the residual copied in for in-place cases), one launch; returns the flat buffers."""
    outs = out_buffers(c, inp["A"].device)
    if c.inplace:
        layouts(c)[2].view(outs["out_raw"])[:] = layouts(c)[1].view(inp["resid"])
    launch(c, inp, outs, max_ctas)
    return outs


def test_wrapper_refuses_buffers_smaller_than_the_descriptor():
    c = CASES["hist_convT"]
    inp = make_inputs(c)
    outs = out_buffers(c, "cpu")
    for key, cut in (("A", 1), ("W", 1), ("bias", 1), ("snake_ib", 16)):
        bad = dict(inp)
        bad[key] = inp[key].reshape(-1)[:-cut]
        with pytest.raises(ValueError, match=key):
            launch(c, bad, outs)
    with pytest.raises(ValueError, match="out_act"):
        launch(c, inp, {"out_raw": outs["out_raw"], "out_act": outs["out_act"][:-1]})
    c2 = CASES["hist_preconv_resid"]
    inp2 = make_inputs(c2)
    inp2["resid"] = inp2["resid"][:layouts(c2)[1].B * layouts(c2)[1].bs - 1 - 2 * c2.N]
    with pytest.raises(ValueError, match="resid"):
        launch(c2, inp2, out_buffers(c2, "cpu"))


# fault -> the case it is injected into (one that has what the fault needs: taps, a cmod < N, a gated epilogue ...)
FAULTS = {"drop_tap": "hist_dil3", "shift_off_by_one": "c96_dil9_bn96", "drop_last_k16": "bn48",
          "wrong_cmod": "convT_288_bn144", "unwritten_chunk": "partial_n272", "swap_gate_up": "swiglu_pair_bias",
          "drop_last_row": "none_scale_resid"}

CASES = {c.name: c for c in sweep_cases()}


def test_case_names_are_unique_and_cover_the_sweep():
    cs = sweep_cases()
    assert len(CASES) == len(cs)
    assert {c.bn for c in cs} >= set(range(16, 257, 16))
    assert {c.T for c in cs} >= {1, 4, 127, 128, 129, 300} and {c.B for c in cs} >= {1, 3}
    assert {c.K for c in cs} >= {16, 48, 96, 192, 1536}
    assert {len(c.shifts) for c in cs} >= {1, 2, 3, 7, 8}
    assert {c.act for c in cs} == set(range(5))
    assert any(c.N % c.bn for c in cs if c.bn)                          # partial last N tiles
    assert any(c.cmod and c.cmod < c.N for c in cs)


def test_bf16_rounding_matches_torch():
    g = torch.Generator().manual_seed(0)
    x = torch.cat([torch.randn(100000, generator=g) * 10.0 ** torch.randint(-30, 30, (100000,), generator=g).float(),
                   torch.tensor([0.0, -0.0, 1.0 + 2 ** -8, 1.0 + 3 * 2 ** -8, 2.0 ** -130, -(2.0 ** -127)])])
    assert torch.equal(rnd(x.double()), x.bfloat16().double())


def test_reference_is_the_products_causal_conv1d():
    """Tap-major packing of CodecDecoder._conv_w with the decoder's shifts == oracle.codec.causal_conv1d."""
    from oracle import codec as OC
    from qwen3_tts_b200.codec import CodecDecoder
    g = torch.Generator().manual_seed(1)
    for k, dil, ci, co in ((7, 1, 96, 48), (7, 3, 40, 32), (7, 9, 16, 16), (3, 1, 72, 64)):
        T = 50
        x, w, b = torch.randn(2, ci, T, generator=g).double(), torch.randn(co, ci, k, generator=g).double(), torch.randn(co, generator=g).double()
        want = OC.causal_conv1d(x, w, b, dilation=dil).transpose(1, 2)
        acc, _ = accumulate(x.transpose(1, 2), CodecDecoder._conv_w(w).double(), T, (ci + 63) // 64 * 64, _conv_shifts(k, dil))
        torch.testing.assert_close(acc + b, want, rtol=0, atol=1e-12)


def test_reference_is_the_products_causal_conv_transpose1d():
    """CodecDecoder._convT_w as N = stride * Cout columns, taps {0, -1} (k = 2 * stride) or {0} (k = stride), bias by
    n % Cout (cmod = Cout) == oracle.codec.causal_conv_transpose1d."""
    from oracle import codec as OC
    from qwen3_tts_b200.codec import CodecDecoder
    g = torch.Generator().manual_seed(2)
    for stride, taps, ci, co in ((3, 2, 64, 32), (8, 2, 48, 16), (2, 1, 32, 32)):
        T = 20
        x = torch.randn(2, ci, T, generator=g).double()
        w = torch.randn(ci, co, taps * stride, generator=g).double()
        b = torch.randn(co, generator=g).double()
        want = OC.causal_conv_transpose1d(x, w, b, stride)                        # (B, co, T*stride)
        acc, _ = accumulate(x.transpose(1, 2), CodecDecoder._convT_w(w, stride).double(), T, (ci + 63) // 64 * 64,
                            (0, -1)[:taps])
        got = (acc + _chan(b, stride * co, co)).view(2, T, stride, co).permute(0, 3, 1, 2).reshape(2, co, T * stride)
        torch.testing.assert_close(got, want, rtol=0, atol=1e-12)


def _packed_codec_gate_up(cfg, W):
    from qwen3_tts_b200.codec import CodecDecoder
    d = object.__new__(CodecDecoder)
    d.cfg, d.device, d.max_frames, store = cfg, torch.device("cpu"), 8, {}
    d._put = lambda name, x, bf16: store.__setitem__(name, x)
    d._load(W)
    return store


def _packed_engine(cfg, W):
    from qwen3_tts_b200.engine import AREngine
    e = object.__new__(AREngine)
    e.cfg, e.device, e.max_ctx, store = cfg, torch.device("cpu"), 16, {}
    e.has_proj = "talker.code_predictor.small_to_mtp_projection.weight" in W
    e._put = lambda name, x: store.__setitem__(name, x)
    e._load(W)
    return store


@pytest.mark.parametrize("who", ["codec_pair", "talker_blk8"])
def test_reference_swiglu_is_the_products_gated_mlp(who):
    """The gated epilogues on the gate/up row interleaves the product's loaders write (the codec's (gate_i, up_i)
    pairs, the talker's blocks of 8) == silu(x gate^T) * (x up^T) with the kernel's rounding points."""
    from oracle import codec as OC
    from qwen3_tts_b200 import synthetic
    if who == "codec_pair":
        from tests.test_gpu_codec import _pkg_cfg, _small_cfg
        oc = _small_cfg()
        W = {k: v.bfloat16().float() for k, v in OC.random_weights(oc, seed=3).items()}
        packed = _packed_codec_gate_up(_pkg_cfg(oc), W)["tr.0.gate_up.w"]
        gate, up = W["pre_transformer.layers.0.mlp.gate_proj.weight"], W["pre_transformer.layers.0.mlp.up_proj.weight"]
        act = ACT_SWIGLU_PAIR
    else:
        cfg = synthetic.cfg_tiny()
        W = synthetic.random_tts_weights(cfg, device="cpu", seed=0)
        packed = _packed_engine(cfg, W)["talker.layers.1.gate_up"].float()
        gate = W["talker.model.layers.1.mlp.gate_proj.weight"].float()
        up = W["talker.model.layers.1.mlp.up_proj.weight"].float()
        act = ACT_SWIGLU_BLK8
    I, K = gate.shape
    c = Case("swiglu", B=1, T=9, K=K, N=2 * I, act=act, bias=False, raw=False, actout=True)
    x = torch.randn(1, 9, K, generator=torch.Generator().manual_seed(4)).bfloat16()
    Wp = torch.zeros(2 * I, c.Kp)
    Wp[:, :K] = packed[:, :K]
    got = reference(c, {"A": x.reshape(-1), "W": Wp})["out_act"][0]
    xd = x.double()
    want = rnd(rnd(silu(rnd(xd @ gate.double().T))) * rnd(xd @ up.double().T))
    assert torch.equal(got, want)


@pytest.mark.parametrize("name", list(CASES))
def test_comparator_accepts_float32_computation(name):
    c = CASES[name]
    inp = make_inputs(c)
    rep = check_case(c, inp, emulate(c, inp))
    for k, r in rep.items():
        assert r["ok"], (k, r)


@pytest.mark.parametrize("fault", list(FAULTS))
def test_comparator_rejects_faulty_computation(fault):
    c = CASES[FAULTS[fault]]
    inp = make_inputs(c)
    rep = check_case(c, inp, emulate(c, inp, fault))
    assert not all(r["ok"] for r in rep.values()), f"{fault} injected into {c.name} passed: {rep}"
    print(f"[tap_gemm] fault {fault} in {c.name}: rejected "
          + ", ".join(f"{k}: {r['n_outside']} of {r['n']} outside" for k, r in rep.items()))


def test_descriptor_layout_matches_header(tmp_path):
    from qwen3_tts_b200 import _lib
    fields = [f for f, _ in _lib.TapGemmDesc._fields_]
    src = tmp_path / "layout.cpp"
    src.write_text('#include <cstdio>\n#include <cstddef>\n#include "qwen3tts_b200.h"\nint main() {\n'
                   '  printf("size %zu\\n", sizeof(q3_tap_gemm_desc));\n'
                   + "".join(f'  printf("{f} %zu\\n", offsetof(q3_tap_gemm_desc, {f}));\n' for f in fields) + "}\n")
    exe = tmp_path / "layout"
    subprocess.run(["g++", "-std=c++17", "-I", os.path.join(ROOT, "include"), "-o", str(exe), str(src)], check=True)
    got = dict(line.split() for line in subprocess.run([str(exe)], capture_output=True, text=True, check=True).stdout.split("\n") if line)
    assert int(got.pop("size")) == ctypes.sizeof(_lib.TapGemmDesc)
    assert {f: int(v) for f, v in got.items()} == {f: getattr(_lib.TapGemmDesc, f).offset for f in fields}
