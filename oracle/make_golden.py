"""Mint golden vectors from the REFERENCE's own modules (through oracle/ref_shims.py) and commit them under
tests/golden/.  Run in the build container only:  python -m oracle.make_golden

The reference ships no fixtures (SURVEY §4); these pin the oracle wherever /root/reference is absent (GPU box).
Shapes are deliberately micro (weights travel inside the .npz)."""
import os

import numpy as np
import torch

from . import codec as OC
from . import mimi_encoder as OM
from . import speaker_encoder as OS
from . import ref_driver as R, ref_shims
from . import talker as OT

OUT = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "tests", "golden")


def micro_tts_cfg():
    V = 1200
    return OT.TTSCfg(talker=OT.StackCfg(64, 2, 2, 1, 32, 128, V, rope_theta=1e6),
                     cp=OT.StackCfg(32, 2, 2, 1, 32, 64, 64, rope_theta=1e4), text_hidden_size=64, text_vocab_size=100,
                     codec_eos_token_id=V - 10, codec_pad_id=V - 12, codec_bos_id=V - 11, tts_bos_token_id=97,
                     tts_eos_token_id=98, tts_pad_token_id=96)


def micro_codec_cfg():
    return OC.CodecCfg(codebook_size=32, codebook_dim=16, hidden_size=32, latent_dim=32, num_heads=2, num_kv_heads=2,
                       head_dim=16, sliding_window=4, intermediate_size=48, num_layers=2, num_quantizers=16,
                       upsample_rates=(8, 5, 4, 3), upsampling_ratios=(2, 2), decoder_dim=48)


def reference_teacher_forced(m, embs, trail, pad, codes):
    """Drive the reference talker `m` by hand along `codes` (B, N, G): left-padded prefill, then per frame the code
    predictor (15 forwards) and one talker step (:1250-1312, :1682-1727).  Returns the talker logits (N+1, B, V) and
    the code-predictor logits (N*(G-1), B, Vc)."""
    from transformers.cache_utils import DynamicCache
    B, N, G = codes.shape
    H = embs[0].shape[-1]
    Lmax = max(len(e) for e in embs)
    x = torch.zeros(B, Lmax, H)
    mask = torch.zeros(B, Lmax, dtype=torch.long)
    for i, e in enumerate(embs):
        x[i, Lmax - len(e):] = e
        mask[i, Lmax - len(e):] = 1
    cache = DynamicCache()
    m.rope_deltas = None
    tl, cl = [], []
    with torch.no_grad():
        out = m(inputs_embeds=x, attention_mask=mask, past_key_values=cache, use_cache=True, cache_position=torch.arange(Lmax))
        tl.append(out.logits[:, -1].numpy().copy())
        past_hidden = out.past_hidden
        for step in range(N):
            c0 = codes[:, step, 0]
            cpc = DynamicCache()
            e0 = m.get_input_embeddings()(c0[:, None])
            o = m.code_predictor(inputs_embeds=torch.cat((past_hidden, e0), dim=1), past_key_values=cpc, use_cache=True)
            cl.append(o.logits[:, -1].numpy().copy())
            gs = o.generation_steps
            for j in range(1, G - 1):
                o = m.code_predictor(input_ids=codes[:, step, j:j + 1], past_key_values=cpc, use_cache=True, generation_steps=gs)
                gs = o.generation_steps
                cl.append(o.logits[:, -1].numpy().copy())
            hid = [e0] + [m.code_predictor.get_input_embeddings()[i](codes[:, step, i + 1:i + 2]) for i in range(G - 1)]
            xe = torch.cat(hid, dim=1).sum(1, keepdim=True)
            tr = torch.stack([t[step] if step < t.shape[0] else pad for t in trail])[:, None]
            xe = xe + tr
            mask = torch.cat((mask, torch.ones(B, 1, dtype=torch.long)), dim=1)
            cp = torch.tensor([Lmax + step])
            pos = (cp[0] + m.rope_deltas).view(1, B, 1).expand(3, -1, -1)
            mo = m.model(inputs_embeds=xe, attention_mask=mask, position_ids=pos, past_key_values=cache, use_cache=True, cache_position=cp)
            past_hidden = mo.last_hidden_state[:, -1:]
            tl.append(m.codec_head(mo.last_hidden_state)[:, -1].numpy().copy())
    return np.stack(tl), np.stack(cl)


def make_talker():
    cfg = micro_tts_cfg()
    W = OT.random_weights(cfg, seed=11, with_text=False)
    m = R.build_reference_talker(cfg, text_vocab=100)
    R.load_weights_into_reference(m, {k: v for k, v in W.items()})
    g = torch.Generator().manual_seed(5)
    H, B, lens, N, G = 64, 2, [4, 7], 4, 16
    embs = [torch.randn(l, H, generator=g) * 0.5 for l in lens]
    trail = [torch.randn(n, H, generator=g) * 0.1 for n in (2, 0)]
    pad = torch.randn(H, generator=g) * 0.1
    codes = torch.randint(0, 64, (B, N, G), generator=g)
    codes[:, :, 0] = torch.randint(0, 150, (B, N), generator=g)
    tl, cl = reference_teacher_forced(m, embs, trail, pad, codes)
    blob = {f"W::{k}": v.numpy() for k, v in W.items()}
    blob.update({f"emb{i}": e.numpy() for i, e in enumerate(embs)})
    blob.update({f"trail{i}": t.numpy() for i, t in enumerate(trail)})
    blob.update(pad=pad.numpy(), codes=codes.numpy(), talker_logits=tl, cp_logits=cl)
    np.savez_compressed(os.path.join(OUT, "talker_micro.npz"), **blob)
    print("talker_micro.npz", tl.shape, cl.shape)


def make_codec():
    cfg = micro_codec_cfg()
    W = OC.random_weights(cfg, seed=13)
    m = R.build_reference_codec_decoder(cfg)
    m.load_state_dict(W, strict=False)
    g = torch.Generator().manual_seed(2)
    codes = torch.randint(0, cfg.codebook_size, (2, 16, 9), generator=g)
    with torch.no_grad():
        wav = m(codes)
        wav_c = m.chunked_decode(codes, chunk_size=4, left_context_size=2)
    blob = {f"W::{k}": v.numpy() for k, v in W.items()}
    blob.update(codes=codes.numpy(), wav=wav.numpy(), wav_chunked=wav_c.numpy())
    np.savez_compressed(os.path.join(OUT, "codec_micro.npz"), **blob)
    print("codec_micro.npz", wav.shape, float(wav.abs().max()))


def micro_encoder_cfg():
    return OM.MimiEncCfg(num_filters=4, hidden_size=32, num_layers=2, num_heads=2, head_dim=16, intermediate_size=48,
                         sliding_window=5, codebook_size=32, codebook_dim=16, num_quantizers=32, valid_num_quantizers=16)


def make_encoder():
    """Golden codes from the third-party encoder the reference wraps: transformers MimiModel (installed 5.5.0; the
    reference pins 4.57.3) driven exactly like Qwen3TTSTokenizerV2Model.encode (…v2.py:977-983)."""
    from transformers import MimiConfig, MimiModel
    cfg = micro_encoder_cfg()
    W = OM.random_weights(cfg, seed=17)
    hf = MimiModel(MimiConfig(**cfg.to_hf_kwargs())).eval()
    missing, unexpected = hf.load_state_dict(W, strict=False)
    assert not unexpected, unexpected
    g = torch.Generator().manual_seed(4)
    wav = (torch.randn(2, 15000, generator=g) * 0.1).clamp(-1, 1)  # 16 transformer frames > window 5, 8 code frames
    with torch.no_grad():
        codes = hf.encode(wav[:, None, :], return_dict=True).audio_codes[:, : cfg.valid_num_quantizers]
    blob = {f"W::{k}": v.numpy() for k, v in W.items()}
    blob.update(wav=wav.numpy(), codes=codes.numpy())
    np.savez_compressed(os.path.join(OUT, "encoder_micro.npz"), **blob)
    print("encoder_micro.npz", tuple(codes.shape))


def make_speaker():
    """Golden x-vectors from the reference's own Qwen3TTSSpeakerEncoder (modeling_qwen3_tts.py:300-393) and log-mels from
    its mel_spectrogram (:396-448; the absent librosa filterbank is supplied by oracle.speaker_encoder)."""
    from . import ref_shims
    ref_shims.install()
    from qwen_tts.core.models import modeling_qwen3_tts as RM
    from qwen_tts.core.models.configuration_qwen3_tts import Qwen3TTSSpeakerEncoderConfig
    cfg = OS.cfg_tiny_spk()
    rc = Qwen3TTSSpeakerEncoderConfig(mel_dim=cfg.mel_dim, enc_dim=cfg.enc_dim, enc_channels=list(cfg.enc_channels),
                                      enc_kernel_sizes=list(cfg.enc_kernel_sizes), enc_dilations=list(cfg.enc_dilations),
                                      enc_attention_channels=cfg.enc_attention_channels,
                                      enc_res2net_scale=cfg.enc_res2net_scale, enc_se_channels=cfg.enc_se_channels)
    m = RM.Qwen3TTSSpeakerEncoder(rc).eval()
    W = OS.random_weights(cfg, seed=19)
    m.load_state_dict(W)
    g = torch.Generator().manual_seed(6)
    wav = (torch.randn(2, 6000, generator=g) * 0.1).clamp(-1, 1)
    RM.librosa_mel_fn = lambda sr, n_fft, n_mels, fmin, fmax: OS.slaney_mel_filterbank(sr, n_fft, n_mels, fmin, fmax)
    mel = RM.mel_spectrogram(wav, n_fft=1024, num_mels=cfg.mel_dim, sampling_rate=24000, hop_size=256, win_size=1024,
                             fmin=0, fmax=12000)
    with torch.no_grad():
        emb = m(mel.transpose(1, 2))
    blob = {f"W::{k}": v.numpy() for k, v in W.items()}
    blob.update(wav=wav.numpy(), mel=mel.numpy(), emb=emb.numpy())
    np.savez_compressed(os.path.join(OUT, "speaker_micro.npz"), **blob)
    print("speaker_micro.npz", tuple(mel.shape), tuple(emb.shape))


# ---------------------------------------------------------------------------------------------- reference pins
# What tests/test_oracle_vs_reference.py, tests/test_host_generate_vs_reference.py and the config tests of
# tests/test_checkpoint_cpu.py compare against: the reference's own outputs on seeded inputs that the tests rebuild.
# Arrays too large to commit whole are stored as a pin (see `pin`).
PIN_COLS = 32


def pin_cols(n, seed=0):
    """A fixed, seeded sample of PIN_COLS indices along an axis of length n."""
    return np.sort(np.random.default_rng(seed).choice(n, size=min(PIN_COLS, n), replace=False))


def pin(a, cols):
    """Compact pin of the last axis of `a`: the values at `cols`, and the max and the RMS of the whole axis.  Max and
    RMS move by at most max|a - b| between two arrays a and b, so a tolerance on max|a - b| carries over to all three."""
    a = np.asarray(a, dtype=np.float32)
    return {"cols": a[..., cols], "max": a.max(-1), "rms": np.sqrt(np.square(a.astype(np.float64)).mean(-1))}


def _put(blob, prefix, p):
    blob.update({f"{prefix}.{k}": v for k, v in p.items()})


def _shapes(sd):
    """state_dict names and shapes as one string array ("name:d0,d1,...")."""
    return np.array([f"{k}:{','.join(map(str, v.shape))}" for k, v in sd.items()])


def make_reference_pins():
    """tests/golden/reference_pins.npz: the reference's talker / code-predictor logits along the oracle's greedy codes,
    RMSNorm and rotate_half, the codec decoder (tiny config, full and chunked; default config) and the speaker encoder
    with its log-mel front end (tiny and default config)."""
    ref_shims.install()
    from qwen_tts.core.models import modeling_qwen3_tts as RM
    from qwen_tts.core.models.configuration_qwen3_tts import Qwen3TTSSpeakerEncoderConfig
    blob = {}
    # ---- talker + code predictor, teacher-forced along the oracle's greedy codes
    cfg = OT.cfg_tiny()
    cfg.talker.rope_theta, cfg.cp.rope_theta = 1e6, 1e4
    W = OT.random_weights(cfg, seed=1)
    m = R.build_reference_talker(cfg)
    R.load_weights_into_reference(m, W)
    torch.manual_seed(0)
    lens, H = [5, 9, 7], cfg.talker.hidden_size
    embs = [torch.randn(n, H) * 0.5 for n in lens]
    trail = [torch.randn(n, H) * 0.1 for n in (2, 1, 4)]
    pad = torch.randn(H) * 0.1
    sp = OT.SamplingCfg(do_sample=False, subtalker_dosample=False, max_new_tokens=6, suppress_eos=True)
    codes = torch.stack(OT.generate(W, cfg, embs, trail, pad, sp).codes)  # (B, N, 16)
    tl, cl = reference_teacher_forced(m, embs, trail, pad, codes)
    blob["tf.codes"] = codes.numpy()
    blob["tf.talker_cols"], blob["tf.cp_cols"] = pin_cols(cfg.talker.vocab_size), pin_cols(cfg.cp.vocab_size)
    _put(blob, "tf.talker", pin(tl, blob["tf.talker_cols"]))
    _put(blob, "tf.cp", pin(cl, blob["tf.cp_cols"]))
    # ---- leaf ops
    torch.manual_seed(0)
    x = torch.randn(2, 5, 64)
    n = RM.Qwen3TTSRMSNorm(64, eps=1e-6)
    n.weight.data = torch.randn(64)
    blob.update({"leaf.x": x.numpy(), "leaf.w": n.weight.data.numpy(), "leaf.rms": n(x).detach().numpy(),
                 "leaf.rms_bf16": n.to(torch.bfloat16)(x.bfloat16()).detach().float().numpy(),
                 "leaf.rotate_half": RM.rotate_half(x).numpy()})
    # ---- codec decoder, tiny config: one forward and a several-chunk chunked_decode
    ccfg = OC.cfg_tiny_codec()
    cd = R.build_reference_codec_decoder(ccfg)
    blob["codec_tiny.params"] = _shapes(cd.state_dict())
    cd.load_state_dict(OC.random_weights(ccfg, seed=3), strict=False)
    g = torch.Generator().manual_seed(5)
    c = torch.randint(0, ccfg.codebook_size, (2, 16, 13), generator=g)
    c_long = torch.randint(0, ccfg.codebook_size, (2, 16, 40), generator=g)
    with torch.no_grad():
        wav, wav_c = cd(c), cd.chunked_decode(c_long, chunk_size=16, left_context_size=5)
    blob["codec_tiny.cols"] = pin_cols(1920)
    _put(blob, "codec_tiny.wav", pin(wav.reshape(2, -1, 1920).numpy(), blob["codec_tiny.cols"]))
    _put(blob, "codec_tiny.wav_chunked", pin(wav_c.reshape(2, -1, 1920).numpy(), blob["codec_tiny.cols"]))
    blob["codec_tiny.wav_shape"], blob["codec_tiny.wav_chunked_shape"] = np.array(wav.shape), np.array(wav_c.shape)
    # ---- codec decoder, default config: names, shapes and parameter count, and 3 frames decoded whole
    dcfg = OC.CodecCfg()
    cd = R.build_reference_codec_decoder(dcfg)
    blob["codec_default.params"] = _shapes(cd.state_dict())
    blob["codec_default.numel"] = np.array(sum(p.numel() for p in cd.parameters()))
    cd.load_state_dict(OC.random_weights(dcfg, seed=3), strict=False)
    torch.manual_seed(0)
    c = torch.randint(0, dcfg.codebook_size, (1, 16, 3))
    with torch.no_grad():
        wav = cd(c)
    blob["codec_default.wav_shape"] = np.array(wav.shape)
    _put(blob, "codec_default.wav", pin(wav.reshape(1, -1, 1920).numpy(), blob["codec_tiny.cols"]))
    del cd
    # ---- speaker encoder + log-mel front end (the absent librosa filterbank is oracle.speaker_encoder's)
    RM.librosa_mel_fn = lambda sr, n_fft, n_mels, fmin, fmax: OS.slaney_mel_filterbank(sr, n_fft, n_mels, fmin, fmax)
    for which, scfg in (("tiny", OS.cfg_tiny_spk()), ("default", OS.SpkEncCfg())):
        rc = Qwen3TTSSpeakerEncoderConfig(mel_dim=scfg.mel_dim, enc_dim=scfg.enc_dim, enc_channels=list(scfg.enc_channels),
                                          enc_kernel_sizes=list(scfg.enc_kernel_sizes), enc_dilations=list(scfg.enc_dilations),
                                          enc_attention_channels=scfg.enc_attention_channels,
                                          enc_res2net_scale=scfg.enc_res2net_scale, enc_se_channels=scfg.enc_se_channels)
        sm = RM.Qwen3TTSSpeakerEncoder(rc).eval()
        blob[f"spk_{which}.params"] = _shapes(sm.state_dict())
        sm.load_state_dict(OS.random_weights(scfg, seed=1))
        torch.manual_seed(0)
        mels = torch.randn(2, 57, scfg.mel_dim)
        with torch.no_grad():
            blob[f"spk_{which}.emb"] = sm(mels).numpy()
        y = (torch.randn(2, 9000) * 0.1).clamp(-1, 1)
        mel = RM.mel_spectrogram(y, n_fft=1024, num_mels=scfg.mel_dim, sampling_rate=24000, hop_size=256, win_size=1024,
                                 fmin=0, fmax=12000).numpy()
        blob[f"spk_{which}.mel_shape"], blob[f"spk_{which}.mel_cols"] = np.array(mel.shape), pin_cols(mel.shape[-1])
        _put(blob, f"spk_{which}.mel", pin(mel, blob[f"spk_{which}.mel_cols"]))
    np.savez_compressed(os.path.join(OUT, "reference_pins.npz"), **blob)
    print("reference_pins.npz", len(blob), "arrays")


class _Captured(Exception):
    def __init__(self, kw):
        self.kw = kw


def host_prefill_setup():
    """Seeded config and weights of the prefill-assembly comparison, and its speaker / language tables."""
    cfg = OT.cfg_tiny()
    cfg.talker.rope_theta, cfg.cp.rope_theta = 1e6, 1e4
    W = OT.random_weights(cfg, seed=2, with_text=True, text_vocab=1000)
    spk_id = {"alice": 3000, "bob": 3001}
    lang = {"english": 2050, "chinese": 2055, "sichuan_dialect": 2060}
    dial = {"alice": False, "bob": "sichuan_dialect"}
    return cfg, W, spk_id, lang, dial


def host_prefill_cases():
    """(name, non_streaming, generate kwargs) of every prefill-assembly comparison: custom voice / voice design with
    and without instruct, dialect speaker and 'auto' language; voice clone in ICL and x-vector-only mode."""
    def ids(n, seed):
        return torch.randint(0, 990, (1, n), generator=torch.Generator().manual_seed(seed))
    H = OT.cfg_tiny().talker.hidden_size
    cases = []
    for ns in (True, False):
        cases.append((f"custom_voice_ns{int(ns)}", ns, dict(
            input_ids=[ids(3 + T + 5, 10 + T) for T in (6, 11, 4)], instruct_ids=[None, ids(9, 50), ids(5, 51)],
            languages=["english", "auto", "chinese"], speakers=["alice", "bob", None])))
    for ns in (True, False):
        g = torch.Generator().manual_seed(3)
        vcp = dict(ref_code=[torch.randint(0, 2000, (9, 16), generator=g), torch.randint(0, 2000, (5, 16), generator=g), None],
                   ref_spk_embedding=[torch.randn(H, generator=g) for _ in range(3)],
                   x_vector_only_mode=[False, False, True], icl_mode=[True, True, False])
        cases.append((f"voice_clone_ns{int(ns)}", ns, dict(
            input_ids=[ids(3 + 7 + 5, 20), ids(3 + 30 + 5, 21), ids(3 + 5 + 5, 22)],
            ref_ids=[ids(3 + 6 + 2, 30), ids(3 + 4 + 2, 31), None], voice_clone_prompt=vcp,
            languages=["english", "chinese", "auto"])))
    return cases


def make_host_prefill():
    """tests/golden/host_prefill.npz: what the reference's Qwen3TTSForConditionalGeneration.generate hands to
    talker.generate (prefill embeddings, mask, trailing text rows, pad row, EOS / suppression settings)."""
    import types
    ref_shims.install()
    from qwen_tts.core.models.modeling_qwen3_tts import Qwen3TTSForConditionalGeneration as RefTop
    cfg, W, spk_id, lang, dial = host_prefill_setup()
    talker = R.build_reference_talker(cfg, text_vocab=1000)
    R.load_weights_into_reference(talker, W)
    tc = talker.config
    tc.spk_id, tc.codec_language_id, tc.spk_is_dialect = spk_id, lang, dial
    fake = types.SimpleNamespace(
        talker=talker,
        config=types.SimpleNamespace(talker_config=tc, tts_bos_token_id=cfg.tts_bos_token_id,
                                     tts_eos_token_id=cfg.tts_eos_token_id, tts_pad_token_id=cfg.tts_pad_token_id))
    fake.generate_speaker_prompt = types.MethodType(RefTop.generate_speaker_prompt, fake)
    fake.generate_icl_prompt = types.MethodType(RefTop.generate_icl_prompt, fake)

    def cap(**kw):
        raise _Captured(kw)
    talker.generate = cap
    ref_generate = types.MethodType(getattr(RefTop.generate, "__wrapped__", RefTop.generate), fake)
    cols = pin_cols(cfg.talker.hidden_size)
    blob = {"cols": cols}
    for name, ns, kw in host_prefill_cases():
        try:
            with torch.no_grad():
                    ref_generate(non_streaming_mode=ns, **kw, **({"max_new_tokens": 7} if "speakers" in kw else {}))
            raise AssertionError("talker.generate was not reached")
        except _Captured as e:
            k = e.kw
        _put(blob, f"{name}.embeds", pin(k["inputs_embeds"].numpy(), cols))
        _put(blob, f"{name}.trailing", pin(k["trailing_text_hidden"].numpy(), cols))
        blob[f"{name}.mask"] = k["attention_mask"].numpy()
        blob[f"{name}.pad"] = k["tts_pad_embed"].reshape(-1).numpy()
        blob[f"{name}.min_new_tokens"] = np.array(k["min_new_tokens"])
        blob[f"{name}.eos_token_id"] = np.array(k["eos_token_id"])
        blob[f"{name}.suppress_tokens"] = np.array(k["suppress_tokens"])
    np.savez_compressed(os.path.join(OUT, "host_prefill.npz"), **blob)
    print("host_prefill.npz", len(blob), "arrays")


def to_json(v):
    """JSON form of a config value that keeps tuples apart from lists (the defaults tables compare them by ==)."""
    if isinstance(v, tuple):
        return {"__tuple__": [to_json(x) for x in v]}
    if isinstance(v, list):
        return [to_json(x) for x in v]
    if isinstance(v, dict):
        return {k: to_json(x) for k, x in v.items()}
    return v


def from_json(d):
    """json.load object_hook undoing to_json."""
    return tuple(d["__tuple__"]) if set(d) == {"__tuple__"} else d


def _attrs(obj):
    """The plain (JSON-representable) attributes of a reference config object."""
    import json
    out = {}
    for k, v in vars(obj).items():
        try:
            json.dumps(to_json(v))
        except TypeError:
            continue
        out[k] = to_json(v)
    return out


def make_configs():
    """tests/golden/reference_configs.json: the reference's config classes — to_dict() of the tiny checkpoint's
    configs, and the attributes of those objects and of default-constructed ones."""
    import json
    from tests.helpers import tiny_checkpoint_configs
    ref_shims.install()
    from qwen_tts.core.models.configuration_qwen3_tts import Qwen3TTSConfig
    from qwen_tts.core.tokenizer_12hz.configuration_qwen3_tts_tokenizer_v2 import (Qwen3TTSTokenizerV2Config,
                                                                                   Qwen3TTSTokenizerV2DecoderConfig)
    top, tok, _ = tiny_checkpoint_configs()
    kw = {k: v for k, v in top.items() if k != "model_type"}
    kw["talker_config"] = dict(kw["talker_config"], pad_token_id=None)
    kw["talker_config"]["code_predictor_config"] = dict(kw["talker_config"]["code_predictor_config"], pad_token_id=None)

    def tts(c):
        return {"top": _attrs(c), "talker": _attrs(c.talker_config), "cp": _attrs(c.talker_config.code_predictor_config)}
    ref = Qwen3TTSConfig(**kw)
    d = Qwen3TTSConfig(talker_config=dict(pad_token_id=None, code_predictor_config=dict(pad_token_id=None)))
    out = {"tts": tts(ref), "tts_to_dict": to_json(ref.to_dict()), "tts_defaults": tts(d),
           "decoder_defaults": _attrs(Qwen3TTSTokenizerV2DecoderConfig()),
           "tokenizer_defaults": _attrs(Qwen3TTSTokenizerV2Config()),
           "tokenizer_to_dict": to_json(Qwen3TTSTokenizerV2Config(**{k: v for k, v in tok.items() if k != "model_type"}).to_dict())}
    with open(os.path.join(OUT, "reference_configs.json"), "w") as f:
        json.dump(out, f, indent=0, sort_keys=True)
    print("reference_configs.json")


if __name__ == "__main__":
    os.makedirs(OUT, exist_ok=True)
    import sys
    which = sys.argv[1:] or ["talker", "codec", "encoder", "speaker", "pins", "prefill", "configs"]
    if "pins" in which:
        make_reference_pins()
    if "prefill" in which:
        make_host_prefill()
    if "configs" in which:
        make_configs()
    if "talker" in which:
        make_talker()
    if "codec" in which:
        make_codec()
    if "encoder" in which:
        make_encoder()
    if "speaker" in which:
        make_speaker()
