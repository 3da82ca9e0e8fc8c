"""`from_pretrained` plumbing (checkpoint.py): a synthetic checkpoint directory in the reference's on-disk format
(config.json + [sharded] safetensors + speech_tokenizer/ + generation_config.json) must load into exactly the config
records and state_dict the engines are built from.  CPU only (no engine is constructed here)."""
import dataclasses
import json
import os
import types

import pytest
import torch

from tests.helpers import tiny_checkpoint_configs, write_tiny_checkpoint


@pytest.mark.parametrize("sharded", [False, True])
def test_load_tts_checkpoint(tmp_path, sharded):
    from qwen3_tts_b200 import checkpoint
    cfg, W, *_ = write_tiny_checkpoint(str(tmp_path), sharded=sharded)
    tcfg, LW, meta, gen = checkpoint.load_tts_checkpoint(str(tmp_path), device="cpu")
    assert dataclasses.asdict(tcfg) == dataclasses.asdict(cfg)
    assert set(LW) == {k for k in W if k.startswith("talker.")} and "speaker_encoder.fc.weight" not in LW
    assert all(LW[k].dtype == torch.bfloat16 and torch.equal(LW[k], W[k]) for k in LW)
    assert meta["spk_id"] == {"Alice": 3000, "bob": 3001} and meta["tts_model_type"] == "custom_voice"
    assert meta["codec_language_id"]["english"] == 2050 and gen["top_k"] == 40


def test_load_speech_tokenizer_checkpoint(tmp_path):
    from qwen3_tts_b200 import checkpoint
    _, _, ccfg, DW, ecfg, EW = write_tiny_checkpoint(str(tmp_path))
    c2, dec, e2, enc, rates = checkpoint.load_speech_tokenizer_checkpoint(str(tmp_path / "speech_tokenizer"), device="cpu")
    assert dataclasses.asdict(c2) == dataclasses.asdict(ccfg)
    assert dataclasses.asdict(e2) == dataclasses.asdict(ecfg)
    assert set(dec) == set(DW) and set(enc) == set(EW)
    assert all(torch.equal(dec[k], DW[k]) for k in dec) and all(torch.equal(enc[k], EW[k]) for k in enc)
    assert rates["decode_upsample_rate"] == 1920 == c2.total_upsample


def test_config_defaults_and_errors(tmp_path):
    """Missing keys fall back to the reference constructors' defaults; the checks the reference would trip on later
    (codebook_dim absent, rate/stride mismatch, missing weights) fail early with a clear message."""
    from qwen3_tts_b200 import checkpoint
    top, tok, _ = tiny_checkpoint_configs()
    t = dict(top["talker_config"])
    for k in ("num_code_groups", "codec_bos_id"):
        t.pop(k)
    tcfg, meta = checkpoint.tts_config_from_dict(dict(top, talker_config=dict(t, codec_eos_token_id=3000)))
    assert tcfg.num_code_groups == 32 and tcfg.codec_bos_id == 4197   # configuration_qwen3_tts.py:391,400
    bad = dict(tok, decoder_config={k: v for k, v in tok["decoder_config"].items() if k != "codebook_dim"})
    with pytest.raises(ValueError):
        checkpoint.tokenizer_configs_from_dict(bad)
    with pytest.raises(ValueError):
        checkpoint.tokenizer_configs_from_dict(dict(tok, decode_upsample_rate=960))
    with pytest.raises(FileNotFoundError):
        checkpoint.read_state_dict(str(tmp_path))


def _reference_configs():
    """The reference's config classes as oracle/make_golden.py recorded them: to_dict() of the tiny checkpoint's
    configs, and the attributes of those objects and of default-constructed ones."""
    from oracle.make_golden import from_json
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_configs.json")) as f:
        return json.load(f, object_hook=from_json)


def test_config_dict_matches_reference_config_classes():
    """The reference's own config classes, serialised with to_dict(), must map to the same records as from_hf()."""
    from qwen3_tts_b200 import checkpoint
    from qwen3_tts_b200.config import TTSConfig
    R = _reference_configs()
    ref = types.SimpleNamespace(**R["tts"]["top"])
    ref.talker_config = types.SimpleNamespace(**R["tts"]["talker"])
    ref.talker_config.code_predictor_config = types.SimpleNamespace(**R["tts"]["cp"])
    via_dict, meta = checkpoint.tts_config_from_dict(R["tts_to_dict"])
    assert dataclasses.asdict(via_dict) == dataclasses.asdict(TTSConfig.from_hf(ref))
    assert meta["spk_id"] == ref.talker_config.spk_id
    # defaults table == the reference's constructor defaults
    d = R["tts_defaults"]
    # (rope_scaling is skipped: transformers 5.x rewrites None into {"rope_type": "default", ...} on construction)
    for k, v in checkpoint.TALKER_DEFAULTS.items():
        assert k == "rope_scaling" or d["talker"][k] == v, k
    for k, v in checkpoint.CODE_PREDICTOR_DEFAULTS.items():
        assert k == "rope_scaling" or d["cp"][k] == v, k
    for k, v in checkpoint.TOP_DEFAULTS.items():
        assert d["top"][k] == v, k


def test_from_pretrained_plumbing_with_stub_engines(tmp_path, monkeypatch):
    """Qwen3TTSModel.from_pretrained end to end on the CPU: the three engines are replaced by recorders, everything
    else (checkpoint reading, config mapping, speaker/language tables, speech_tokenizer/ sub-directory,
    generation_config.json -> generate_defaults, processor override) is the real code."""
    import numpy as np
    from qwen3_tts_b200 import model as M, codec_encoder as CE
    cfg, W, ccfg, DW, ecfg, EW = write_tiny_checkpoint(str(tmp_path))
    made = {}

    class _AR:
        def __init__(self, c, w, device=None, max_batch=None, max_ctx=None):
            made["ar"] = (c, set(w), str(device), max_batch, max_ctx)
            self.max_batch = max_batch

    class _Dec:
        def __init__(self, c, w, device=None, max_frames=None):
            made["dec"] = (c, set(w), max_frames)

    class _Enc:
        def __init__(self, c, w, device=None):
            made["enc"] = (c, set(w))

        def encode(self, wavs):
            return [torch.zeros(-(-int(x.shape[0]) // 1920), 16, dtype=torch.long) for x in wavs]

    monkeypatch.setattr(M, "AREngine", _AR)
    monkeypatch.setattr(M, "CodecDecoder", _Dec)
    monkeypatch.setattr(CE, "CodecEncoder", _Enc)
    proc = lambda text=None, **kw: {"input_ids": torch.tensor([[1, 2, 3, 9, 4, 5, 6, 7, 8]])}  # noqa: E731
    m = M.Qwen3TTSModel.from_pretrained(str(tmp_path), device_map="cpu", processor=proc, max_batch=4, max_ctx=128,
                                        codec_max_frames=32, dtype=torch.bfloat16, attn_implementation="flash_attention_2")
    assert dataclasses.asdict(made["ar"][0]) == dataclasses.asdict(cfg) and made["ar"][2:] == ("cpu", 4, 128)
    assert made["ar"][1] == {k for k in W if k.startswith("talker.")}
    assert dataclasses.asdict(made["dec"][0]) == dataclasses.asdict(ccfg) and made["dec"][1] == set(DW) and made["dec"][2] == 32
    assert dataclasses.asdict(made["enc"][0]) == dataclasses.asdict(ecfg) and made["enc"][1] == set(EW)
    assert m.generate_defaults["top_k"] == 40 and m.model.tts_model_type == "custom_voice" and m.model.tts_model_size == "1b7"
    assert m.get_supported_speakers() == ["alice", "bob"] and "english" in m.get_supported_languages()
    tok = m.model.speech_tokenizer
    assert tok.get_decode_upsample_rate() == 1920 and tok.get_input_sample_rate() == 24000
    out = tok.encode(np.zeros(5000, np.float32), sr=24000)
    assert tuple(out.audio_codes[0].shape) == (3, 16)
    # an fp32 decoder request is answered loudly (the decoder computes in bf16), a bf16 request is not
    import warnings
    with pytest.warns(RuntimeWarning, match="bf16"):
        M.Qwen3TTSTokenizer.from_pretrained(str(tmp_path / "speech_tokenizer"), device_map="cpu", dtype=torch.float32)
    with warnings.catch_warnings():
        warnings.simplefilter("error", RuntimeWarning)
        M.Qwen3TTSTokenizer.from_pretrained(str(tmp_path / "speech_tokenizer"), device_map="cpu", dtype=torch.bfloat16)
    # a tokenizer directory of the wrong kind is refused
    import json
    json.dump({"model_type": "qwen3_tts_tokenizer_25hz"}, open(tmp_path / "speech_tokenizer" / "config.json", "w"))
    with pytest.raises(ValueError):
        M.Qwen3TTSTokenizer.from_pretrained(str(tmp_path / "speech_tokenizer"), device_map="cpu")


def test_tokenizer_config_defaults_match_reference():
    from qwen3_tts_b200 import checkpoint
    R = _reference_configs()
    for k, v in checkpoint.DECODER_DEFAULTS.items():
        assert R["decoder_defaults"][k] == v, k
    for k, v in checkpoint.TOKENIZER_DEFAULTS.items():
        assert R["tokenizer_defaults"][k] == v, k
    _, tok, _ = tiny_checkpoint_configs()
    c1, e1, _ = checkpoint.tokenizer_configs_from_dict(R["tokenizer_to_dict"])
    c2, e2, _ = checkpoint.tokenizer_configs_from_dict(tok)
    assert dataclasses.asdict(c1) == dataclasses.asdict(c2) and dataclasses.asdict(e1) == dataclasses.asdict(e2)


def test_base_checkpoint_carries_speaker_encoder(tmp_path):
    from qwen3_tts_b200 import checkpoint, synthetic
    write_tiny_checkpoint(str(tmp_path), model_type="base")
    tcfg, W, meta, _ = checkpoint.load_tts_checkpoint(str(tmp_path), device="cpu")
    scfg = synthetic.cfg_speaker_encoder_tiny()
    assert meta["tts_model_type"] == "base" and dataclasses.asdict(meta["speaker_encoder_config"]) == dataclasses.asdict(scfg)
    want = synthetic.random_speaker_encoder_weights(scfg, seed=3)
    got = meta["speaker_encoder_weights"]
    assert set(got) == set(want) and all(got[k].dtype == torch.float32 and got[k].shape == want[k].shape for k in got)
    assert not any(k.startswith("speaker_encoder.") for k in W)
