"""The tcgen05 tap-GEMM (csrc/gemm_sm100.cu) on its own, through q3_debug_tap_gemm, against the float64 reference and
comparator of tests/test_tap_gemm_reference_cpu.py: every tile width, partial tiles in T and N, K that is not a
multiple of 64, 1 to 8 taps, every epilogue the product uses, streaming history views, and the production shapes of
the codec decoder, the talker prefill and the code-predictor projection table with the production tile width.
Every case also checks that nothing outside the output rows and columns is written (sentinel canaries), that the
result does not depend on the grid (one and three CTAs walking all tiles), and that two launches agree bit for bit."""
import pytest
import torch

from oracle import codec as OC
from tests.helpers import report_parity
from tests.test_tap_gemm_reference_cpu import (ACT_GELU, ACT_NONE, ACT_SNAKE, ACT_SWIGLU_BLK8, ACT_SWIGLU_PAIR, CASES,
                                               SENTINEL, Case, _conv_shifts, check_case, launch, layouts, make_inputs,
                                               out_buffers, run)

pytestmark = pytest.mark.gpu
DEV = "cuda:0"
ACT_NAMES = {ACT_NONE: "none", ACT_SNAKE: "snake", ACT_GELU: "gelu", ACT_SWIGLU_PAIR: "swiglu_pair",
             ACT_SWIGLU_BLK8: "swiglu_blk8"}


@pytest.fixture(scope="module")
def figures():
    """Worst |out - ref| / bound and the mismatch rate per epilogue over the module, reported at its end."""
    fig = {}
    yield fig
    report_parity("tap_gemm", {f"{k}_{m}": v for k, d in sorted(fig.items()) for m, v in d.items()})


def _views(c, outs):
    _, _, lraw, lact = layouts(c)
    return {k: l.view(outs[k]) for k, l in (("out_raw", lraw), ("out_act", lact)) if outs[k] is not None}


def _canaries(c, outs):
    _, _, lraw, lact = layouts(c)
    for name, l in (("out_raw", lraw), ("out_act", lact)):
        t = outs[name]
        if t is None:
            continue
        m = l.mask(t.device)
        assert (t.view(torch.int16)[~m] == SENTINEL).all(), f"{c.name}: {name} written outside its rows / columns"
        assert torch.isfinite(t[m].float()).all(), f"{c.name}: {name} has unwritten or non-finite elements"


def _same(a, b):
    return all((x is None and y is None) or torch.equal(x.view(torch.int16), y.view(torch.int16))
               for x, y in zip(a.values(), b.values()))


def _check(c, inp, outs, figures):
    _canaries(c, outs)
    rep = check_case(c, inp, _views(c, outs))
    for k, r in rep.items():
        assert r["ok"], (c.name, k, r)
        f = figures.setdefault(ACT_NAMES[c.act], {"worst_ratio": 0.0, "mismatch_rate": 0.0, "elements": 0})
        f["worst_ratio"] = max(f["worst_ratio"], r["worst_ratio"])
        f["mismatch_rate"] = max(f["mismatch_rate"], r["mismatch_rate"])
        f["elements"] += r["n"]


@pytest.mark.parametrize("name", list(CASES))
def test_tap_gemm_sweep(name, figures):
    c = CASES[name]
    inp = make_inputs(c, DEV)
    outs = run(c, inp)
    torch.cuda.synchronize()
    _check(c, inp, outs, figures)
    assert _same(outs, run(c, inp)), f"{name}: two launches differ"
    for ctas in (1, 3):
        assert _same(outs, run(c, inp, max_ctas=ctas)), f"{name}: result depends on the grid ({ctas} CTAs)"


def production_cases():
    """The tap-GEMMs of the default codec decoder at B in {1, 8} over 3 frames, of one 1.7B talker prefill layer at
    37 and 488 tokens, and the 1.7B code-predictor projection table; all at the production tile width (bn = 0)."""
    g = OC.CodecCfg()
    cases = []
    for B in (1, 8):
        T = 3
        qkv = 3 * g.num_heads * g.head_dim
        P = lambda nm, **kw: cases.append(Case(f"codec_b{B}_{nm}", B=B, seed=len(cases), **kw))  # noqa: E731
        P("rvq_proj", T=T, K=g.codebook_dim, N=g.codebook_dim, bias=False)
        P("pre_conv", T=T, K=g.codebook_dim, N=g.latent_dim, shifts=(-2, -1, 0))
        P("tr_in", T=T, K=g.latent_dim, N=g.hidden_size)
        P("qkv", T=T, K=g.hidden_size, N=qkv, bias=False)
        P("o", T=T, K=g.num_heads * g.head_dim, N=g.hidden_size, bias=False, scale=True, resid=True)
        P("gate_up", T=T, K=g.hidden_size, N=2 * g.intermediate_size, bias=False, act=ACT_SWIGLU_PAIR, raw=False, actout=True)
        P("down", T=T, K=g.intermediate_size, N=g.hidden_size, bias=False, scale=True, resid=True)
        P("tr_out", T=T, K=g.hidden_size, N=g.latent_dim)
        Tc = T
        for i, f in enumerate(g.upsampling_ratios):
            P(f"up{i}_ct", T=Tc, K=g.latent_dim, N=f * g.latent_dim, cmod=g.latent_dim)
            Tc *= f
            P(f"up{i}_pw1", T=Tc, K=g.latent_dim, N=4 * g.latent_dim, act=ACT_GELU, raw=False, actout=True)
            P(f"up{i}_pw2", T=Tc, K=4 * g.latent_dim, N=g.latent_dim, scale=True, resid=True)
        C = g.decoder_dim
        P("dec_in", T=Tc, K=g.latent_dim, N=C, shifts=_conv_shifts(7, 1), act=ACT_SNAKE, raw=False, actout=True)
        for i, r in enumerate(g.upsample_rates):
            P(f"blk{i}_ct", T=Tc, K=C, N=r * C // 2, cmod=C // 2, shifts=(0, -1), act=ACT_SNAKE, actout=True)
            Tc, C = Tc * r, C // 2
            P(f"blk{i}_c1_dil9", T=Tc, K=C, N=C, shifts=_conv_shifts(7, 9), act=ACT_SNAKE, raw=False, actout=True)
            P(f"blk{i}_c2", T=Tc, K=C, N=C, resid=True, act=ACT_SNAKE, actout=True)
    H, QKV, I = 2048, (16 + 2 * 8) * 128, 6144
    for ntok in (37, 488):
        cases += [Case(f"prefill_{ntok}_qkv", B=1, T=ntok, K=H, N=QKV, bias=False, seed=100),
                  Case(f"prefill_{ntok}_o", B=1, T=ntok, K=16 * 128, N=H, bias=False, resid=True, inplace=True, seed=101),
                  Case(f"prefill_{ntok}_gate_up", B=1, T=ntok, K=H, N=2 * I, bias=False, act=ACT_SWIGLU_BLK8, raw=False,
                       actout=True, seed=102),
                  Case(f"prefill_{ntok}_down", B=1, T=ntok, K=I, N=H, bias=False, resid=True, inplace=True, seed=103)]
    cases.append(Case("cp_proj_table", B=1, T=15 * 2048, K=2048, N=1024, seed=104))
    return {c.name: c for c in cases}


PRODUCTION = production_cases()


@pytest.mark.parametrize("name", list(PRODUCTION))
def test_tap_gemm_production_shapes(name, figures):
    c = PRODUCTION[name]
    inp = make_inputs(c, DEV)
    outs = run(c, inp)
    torch.cuda.synchronize()
    _check(c, inp, outs, figures)
    assert _same(outs, run(c, inp)), f"{name}: two launches differ"
    if name == "codec_b8_blk1_ct":
        assert _same(outs, run(c, inp, max_ctas=3)), f"{name}: result depends on the grid"


def _refusals():
    base = dict(B=2, T=40, K=64, N=128, seed=200)
    return {"bn24": (Case("bn24", bn=24, **base), "bn must be"),
            "n40": (Case("n40", B=1, T=8, K=64, N=40, bn=16, seed=201), "N must be a multiple of 16"),
            "misaligned_bias": (Case("misaligned_bias", **base), "16-byte aligned"),
            "ntaps9": (Case("ntaps9", shifts=tuple(range(-8, 1)), **base), "ntaps out of range"),
            "swiglu_resid": (Case("swiglu_resid", act=ACT_SWIGLU_PAIR, resid=True, raw=False, actout=True, **base),
                             "gated epilogues")}


@pytest.mark.parametrize("name", list(_refusals()))
def test_hook_refuses_invalid_descriptors(name):
    c, msg = _refusals()[name]
    inp = make_inputs(c, DEV)
    if name == "misaligned_bias":
        b = torch.zeros(c.N + 1, device=DEV)
        b[1:] = inp["bias"]
        inp["bias"] = b[1:]
    outs = out_buffers(c, DEV)
    with pytest.raises(RuntimeError, match=msg):
        launch(c, inp, outs)
    torch.cuda.synchronize()
    for t in outs.values():
        if t is not None:
            assert (t.view(torch.int16) == SENTINEL).all(), f"{name}: refused, yet something was written"
