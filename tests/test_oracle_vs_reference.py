"""Pin the oracle against the reference's OWN modules: tests/golden/reference_pins.npz holds what those modules computed
(oracle/make_golden.py, run through oracle/ref_shims.py) on the seeded weights and inputs rebuilt here.  The reference
ships no tests or golden vectors (SURVEY §4), so this is the strongest pin available; its modules were driven by hand
with a DynamicCache (HF generate() cannot run under transformers 5.5.0).  Arrays too large to store whole are compared
through oracle.make_golden.pin (sampled columns, row max and row RMS) under the tolerance of the whole array.
"""
import os

import numpy as np
import pytest
import torch

from oracle import talker as T
from oracle.make_golden import pin

GOLD = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_pins.npz"))


def _assert_pin(a, prefix, cols, tol):
    p = pin(a, cols)
    for k in ("cols", "max", "rms"):
        want = GOLD[f"{prefix}.{k}"]
        assert p[k].shape == want.shape, (prefix, k, p[k].shape, want.shape)
        assert np.abs(p[k] - want).max() < tol, (prefix, k, float(np.abs(p[k] - want).max()))


def _params(prefix):
    """name -> shape of the reference module's state_dict, as stored."""
    ref = dict(s.split(":") for s in GOLD[f"{prefix}.params"])
    return {k: tuple(int(d) for d in v.split(",") if d) for k, v in ref.items()}


def test_talker_and_code_predictor_teacher_forced():
    cfg = T.cfg_tiny()
    cfg.talker.rope_theta = 1e6
    cfg.cp.rope_theta = 1e4
    W = T.random_weights(cfg, seed=1)
    torch.manual_seed(0)
    B, lens, H = 3, [5, 9, 7], cfg.talker.hidden_size
    embs = [torch.randn(l, H) * 0.5 for l in lens]
    trail = [torch.randn(n, H) * 0.1 for n in (2, 1, 4)]
    pad = torch.randn(H) * 0.1
    sp = T.SamplingCfg(do_sample=False, subtalker_dosample=False, max_new_tokens=6, suppress_eos=True)
    r = T.generate(W, cfg, embs, trail, pad, sp, record_logits=True)
    n_frames = r.codes[0].shape[0]
    assert n_frames == 5
    codes = torch.stack(r.codes)  # (B,N,16)
    # the reference was driven along these codes
    assert np.array_equal(codes.numpy(), GOLD["tf.codes"])
    tl = np.stack(r.record["talker_logits"])
    # prefill row within 2e-5 of the reference, decode steps within 3e-5
    p = pin(tl, GOLD["tf.talker_cols"])
    for k in ("cols", "max", "rms"):
        d = np.abs(p[k] - GOLD[f"tf.talker.{k}"])
        assert d.shape[0] == n_frames + 1 and d[0].max() < 2e-5 and d[1:].max() < 3e-5, k
    cl = np.stack(r.record["cp_logits"])
    _assert_pin(cl, "tf.cp", GOLD["tf.cp_cols"], 2e-5)
    for step in range(n_frames):
        for j in range(cfg.num_code_groups - 1):
            ol = cl[step * (cfg.num_code_groups - 1) + j]
            assert (np.argmax(ol, -1) == codes[:, step, j + 1].numpy()).all()


def test_leaf_ops_match_reference():
    x, w = torch.from_numpy(GOLD["leaf.x"]), torch.from_numpy(GOLD["leaf.w"])  # the inputs the reference was given
    assert torch.equal(torch.from_numpy(GOLD["leaf.rms"]), T.rms_norm(x, w, 1e-6))
    assert torch.equal(torch.from_numpy(GOLD["leaf.rms_bf16"]).bfloat16(), T.rms_norm(x.bfloat16(), w.bfloat16(), 1e-6))
    assert torch.equal(torch.from_numpy(GOLD["leaf.rotate_half"]), T.rotate_half(x))


def _codec_weights(cfg, prefix, seed=3):
    from oracle import codec as C
    W = C.random_weights(cfg, seed=seed)
    sd = _params(prefix)
    missing = [k for k in sd if k not in W and "rotary_emb" not in k]
    extra = [k for k in W if k not in sd]
    assert not missing and not extra, (missing[:5], extra[:5])
    for k in sd:
        if k in W:
            assert sd[k] == tuple(W[k].shape), (k, sd[k], W[k].shape)
    return W


def test_codec_decoder_tiny_matches_reference():
    from oracle import codec as C
    cfg = C.cfg_tiny_codec()
    W = _codec_weights(cfg, "codec_tiny")
    g = torch.Generator().manual_seed(5)
    codes = torch.randint(0, cfg.codebook_size, (2, 16, 13), generator=g)
    out = C.decoder_forward(W, cfg, codes)
    assert out.shape == tuple(GOLD["codec_tiny.wav_shape"]) == (2, 1, 13 * 1920)
    _assert_pin(out.reshape(2, -1, 1920).numpy(), "codec_tiny.wav", GOLD["codec_tiny.cols"], 2e-5)
    assert out.abs().max() > 0.05  # not a degenerate all-zero / all-clamped signal
    # chunked decode with several chunks + wrapper semantics (pad -1, trim)
    codes_long = torch.randint(0, cfg.codebook_size, (2, 16, 40), generator=g)
    out_c = C.chunked_decode(W, cfg, codes_long, chunk_size=16, left_context_size=5)
    assert out_c.shape == tuple(GOLD["codec_tiny.wav_chunked_shape"])
    _assert_pin(out_c.reshape(2, -1, 1920).numpy(), "codec_tiny.wav_chunked", GOLD["codec_tiny.cols"], 2e-5)


def test_codec_decoder_default_shapes_names():
    """Full default config: parameter names/shapes line up with the reference (195.08 M params)."""
    from oracle import codec as C
    cfg = C.CodecCfg()
    W = _codec_weights(cfg, "codec_default")
    assert int(GOLD["codec_default.numel"]) == sum(v.numel() for v in W.values())
    torch.manual_seed(0)
    codes = torch.randint(0, cfg.codebook_size, (1, 16, 3))
    out = C.decoder_forward(W, cfg, codes)
    assert out.shape == tuple(GOLD["codec_default.wav_shape"])
    _assert_pin(out.reshape(1, -1, 1920).numpy(), "codec_default.wav", GOLD["codec_tiny.cols"], 5e-5)


@pytest.mark.parametrize("which", ["tiny", "default"])
def test_speaker_encoder_and_mel_match_reference(which):
    """ECAPA-TDNN x-vector (modeling_qwen3_tts.py:300-393) and the log-mel front end (:396-448).  The mel FILTERBANK is
    librosa's (absent): the reference function was run with oracle.speaker_encoder's restatement patched in, so STFT,
    magnitude, projection and log are pinned; the filterbank itself stays 'parity unpinned'."""
    from oracle import speaker_encoder as S
    cfg = S.cfg_tiny_spk() if which == "tiny" else S.SpkEncCfg()
    W = S.random_weights(cfg, seed=1)
    # strict: every reference parameter has a counterpart, and no other
    assert _params(f"spk_{which}") == {k: tuple(v.shape) for k, v in W.items()}
    torch.manual_seed(0)
    mels = torch.randn(2, 57, cfg.mel_dim)
    assert (torch.from_numpy(GOLD[f"spk_{which}.emb"]) - S.speaker_encoder(W, cfg, mels)).abs().max() < 1e-5
    y = (torch.randn(2, 9000) * 0.1).clamp(-1, 1)
    mel = S.mel_spectrogram(y, num_mels=cfg.mel_dim)
    assert mel.shape == tuple(GOLD[f"spk_{which}.mel_shape"])
    _assert_pin(mel.numpy(), f"spk_{which}.mel", GOLD[f"spk_{which}.mel_cols"], 1e-5)
    fb = S.slaney_mel_filterbank(24000, 1024, 128, 0, 12000)
    assert fb.shape == (128, 513) and (fb >= 0).all() and (fb.sum(1) > 0).all()
