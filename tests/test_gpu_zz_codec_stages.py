"""Per-stage parity of the codec DECODER against the CPU oracle (through q3_codec_debug_capture), so an error in one
small kernel cannot hide behind the waveform SNR, and the full default config at 64 frames."""
import pytest
import torch

from oracle import codec as OC
from tests.helpers import report_parity
from tests.test_gpu_codec import DEV, _bf16_round, _pkg_cfg, _small_cfg, _snr_db

pytestmark = pytest.mark.gpu


def _reference_stages(Wf, cfg, codes):
    """name -> (B, T_stage, C_stage) fp32, the tensors q3_codec_debug_capture copies (same order as stage_shapes)."""
    taps = {}
    wav = OC.decoder_forward(Wf, cfg, codes, taps=taps)
    cl = lambda x: x.transpose(1, 2).contiguous()  # noqa: E731  (B,C,T) -> channels-last
    ref = {"pre_conv": taps["pre_conv"].contiguous(), "pre_transformer": cl(taps["pre_transformer"]), "upsample": cl(taps["upsample"]),
           "decoder0_act": cl(OC.snake_beta(taps["decoder0"], Wf["decoder.1.block.0.alpha"], Wf["decoder.1.block.0.beta"]))}
    for i in range(len(cfg.upsample_rates)):
        ref[f"block{i}"] = cl(taps[f"block{i}"])
    return wav, ref


def _run_stages(cfg, B, T, seed):
    from qwen3_tts_b200.codec import CodecDecoder
    Wb, Wf = _bf16_round(OC.random_weights(cfg, seed=seed))
    g = torch.Generator().manual_seed(seed + 1)
    codes = torch.randint(0, cfg.codebook_size, (B, cfg.num_quantizers, T), generator=g)
    ref_wav, ref = _reference_stages(Wf, cfg, codes)
    dec = CodecDecoder(_pkg_cfg(cfg), Wb, device=DEV, max_frames=max(T, 64))
    assert [n for n, _ in dec.stage_shapes(B, T)] == list(ref.keys())
    wav, got = dec.forward_with_stages(codes.to(DEV))
    plain = dec.forward(codes.to(DEV))
    dec.close()
    assert torch.equal(wav, plain), "capturing must not change the result"
    snr = {}
    for name, r in ref.items():
        o = got[name].float().cpu()
        assert o.shape == r.shape, (name, o.shape, r.shape)
        assert torch.isfinite(o).all(), name
        snr[name] = _snr_db(r, o)
    snr["wav"] = _snr_db(ref_wav, wav.cpu())
    return snr


# bf16 activations against the fp32 oracle on the same bf16 weights.  A broken stage kernel shows up as < 10 dB at its
# stage and everything after it.  Each bar is the SNR measured on an NVIDIA B200 (1000 W power limit) minus 3 dB, rounded
# down (profiles/codec_stage_snr.txt); the seeded inputs make the figures reproducible.
SMALL_BARS = {"pre_conv": 41, "pre_transformer": 39, "upsample": 38, "decoder0_act": 37, "block0": 36, "block1": 34,
              "block2": 33, "block3": 31, "wav": 32}
FULL_BARS = {"pre_conv": 42, "pre_transformer": 37, "upsample": 36, "decoder0_act": 35, "block0": 34, "block1": 33,
             "block2": 32, "block3": 30, "wav": 28}


def test_small_codec_every_stage_matches_oracle():
    snr = _run_stages(_small_cfg(), 2, 13, seed=3)
    report_parity("codec_stages_small_2x13", snr)
    assert set(snr) == set(SMALL_BARS)
    for name, v in snr.items():
        assert v > SMALL_BARS[name], f"{name}: SNR {v:.1f} dB, bar {SMALL_BARS[name]} dB ({snr})"


def test_full_config_64_frames_stagewise():
    """Reference default config (195 M parameters) at 2 x 64 frames."""
    snr = _run_stages(OC.CodecCfg(), 2, 64, seed=7)
    report_parity("codec_stages_full_2x64", snr)
    assert set(snr) == set(FULL_BARS)
    for name, v in snr.items():
        assert v > FULL_BARS[name], f"{name}: SNR {v:.1f} dB, bar {FULL_BARS[name]} dB ({snr})"
