"""Row a1 (composite generate(): prefill assembly) — our PyTorch host code against the reference's own
`Qwen3TTSForConditionalGeneration.generate`, whose call into `talker.generate` (seam B) was intercepted by
oracle/make_golden.py: tests/golden/host_prefill.npz holds what it handed over (prefill rows, mask, trailing text rows,
pad row, EOS / suppression settings) for each of oracle.make_golden.host_prefill_cases().  Embedding rows are stored as
pins (oracle.make_golden.pin: sampled columns, row max and row RMS)."""
import os

import numpy as np
import pytest
import torch

from oracle.make_golden import host_prefill_cases, host_prefill_setup, pin

GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "host_prefill.npz"))


def _setup():
    from tests import helpers as Hh
    cfg, W, spk_id, lang, dial = host_prefill_setup()
    from qwen3_tts_b200.model import Qwen3TTSForConditionalGenerationB200
    ours = Qwen3TTSForConditionalGenerationB200.__new__(Qwen3TTSForConditionalGenerationB200)
    Qwen3TTSForConditionalGenerationB200.__init__(ours, Hh.to_pkg_cfg(cfg), W, device="cpu", spk_id=spk_id, spk_is_dialect=dial,
                                                  codec_language_id=lang, engine=object())
    ours.dtype = torch.float32
    for n in ("text_embedding", "fc1_w", "fc1_b", "fc2_w", "fc2_b", "codec_embedding"):
        setattr(ours, n, getattr(ours, n).float())
    ours.cp_embeddings = [e.float() for e in ours.cp_embeddings]
    # float32 copies of the exact same weights for an exact comparison
    g = lambda k: W[k].float()  # noqa: E731
    ours.text_embedding = g("talker.model.text_embedding.weight")
    ours.fc1_w, ours.fc1_b = g("talker.text_projection.linear_fc1.weight"), g("talker.text_projection.linear_fc1.bias")
    ours.fc2_w, ours.fc2_b = g("talker.text_projection.linear_fc2.weight"), g("talker.text_projection.linear_fc2.bias")
    ours.codec_embedding = g("talker.model.codec_embedding.weight")
    ours.cp_embeddings = [g(f"talker.code_predictor.model.codec_embedding.{j}.weight") for j in range(15)]
    return cfg, ours


def _case(name):
    (ns, kw), = [(ns, kw) for n, ns, kw in host_prefill_cases() if n == name]
    return ns, kw


def _pin(x, cols):
    return dict(pin(x.numpy(), cols), hidden=x.shape[-1])


def _close(p, name, part, rows, atol=1e-6, rtol=1e-5):
    """torch.allclose(got, ref, atol, rtol) over pinned rows: sampled columns directly; max and RMS, which move by at
    most max|got - ref|, within atol + rtol * max|ref| (max|ref| <= sqrt(H) * RMS)."""
    want = {k: GOLD[f"{name}.{part}.{k}"][rows] for k in ("cols", "max", "rms")}
    assert np.allclose(p["cols"], want["cols"], atol=atol, rtol=rtol), (name, part)
    tol = atol + rtol * np.sqrt(p["hidden"]) * float(want["rms"].max(initial=0.0))
    assert np.abs(p["max"] - want["max"]).max(initial=0.0) <= tol and np.abs(p["rms"] - want["rms"]).max(initial=0.0) <= tol, (name, part)


def _check(name, embeds, trailing, pad):
    cols = GOLD["cols"]
    mask = GOLD[f"{name}.mask"]
    B, L = mask.shape
    for b in range(B):
        n = int(mask[b].sum())
        assert embeds[b].shape[0] == n
        _close(_pin(embeds[b], cols), name, "embeds", (b, slice(L - n, L)))
        assert float(np.abs(GOLD[f"{name}.embeds.rms"][b, :L - n]).max(initial=0.0)) == 0.0   # left padding is zero
    T = GOLD[f"{name}.trailing.rms"].shape[1]
    for b in range(B):
        t = trailing[b]
        _close(_pin(t, cols), name, "trailing", (b, slice(0, t.shape[0])))
        if t.shape[0] < T:
            _close(_pin(pad.expand(T - t.shape[0], -1), cols), name, "trailing", (b, slice(t.shape[0], T)))
    assert torch.allclose(torch.from_numpy(GOLD[f"{name}.pad"]), pad, atol=1e-6)


@pytest.mark.parametrize("non_streaming", [True, False])
def test_custom_voice_and_voice_design_prefill(non_streaming):
    cfg, ours = _setup()
    name = f"custom_voice_ns{int(non_streaming)}"
    ns, kw = _case(name)
    e, t, pad = ours.build_prefill(kw["input_ids"], kw["instruct_ids"], None, None, kw["languages"], kw["speakers"], ns)
    _check(name, e, t, pad)
    # talker kwargs the engine must honour (:2044-2066)
    assert int(GOLD[f"{name}.min_new_tokens"]) == 2 and int(GOLD[f"{name}.eos_token_id"]) == cfg.codec_eos_token_id
    V = cfg.talker.vocab_size
    assert GOLD[f"{name}.suppress_tokens"].tolist() == [i for i in range(V - 1024, V) if i != cfg.codec_eos_token_id]
    if non_streaming:
        assert [x.shape[0] for x in e] == [3 + 6 + (6 + 1) + 1, 9 + 3 + 6 + (11 + 1) + 1, 5 + 3 + 5 + 0 + (4 + 1) + 1]  # row 1: dialect speaker => language tag present


@pytest.mark.parametrize("non_streaming", [True, False])
def test_voice_clone_icl_and_xvector_prefill(non_streaming):
    _, ours = _setup()
    name = f"voice_clone_ns{int(non_streaming)}"
    ns, kw = _case(name)
    e, t, pad = ours.build_prefill(kw["input_ids"], None, kw["ref_ids"], kw["voice_clone_prompt"], kw["languages"], None, ns)
    _check(name, e, t, pad)


def test_unknown_speaker_and_language_raise():
    _, ours = _setup()
    ids = torch.randint(0, 990, (1, 12), generator=torch.Generator().manual_seed(1))
    with pytest.raises(NotImplementedError):
        ours.build_prefill([ids], None, None, None, ["english"], ["carol"], True)
    with pytest.raises(NotImplementedError):
        ours.build_prefill([ids], None, None, None, ["klingon"], ["alice"], True)
