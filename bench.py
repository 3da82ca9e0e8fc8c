#!/usr/bin/env python
"""bench.py — hot-path benchmark of the B200-native Qwen3-TTS engine (contract: see the task statement).

One "step" = one pass of the hot path over one batch of synthetic utterances of the configuration BASELINE.json
quotes the metric on (config[2]: Qwen3-TTS-12Hz-1.7B CustomVoice, batch 8, non-streaming):
    prefill (8 prompts, L_i = T_i + 11 [+12 instruct on odd rows], T_i in 16..72)  ->
    125 frame-steps of the fused AR kernel (15 code-predictor passes + 28 talker layers + sampling each)  ->
    codec decode of the 8 x 125 frames to 24 kHz waveform.
metric = speech tokens (12.5 Hz frames; x16 for individual codebook tokens) per second, whole job.

  python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference]
N > 1 is launched by torchrun (one rank per GPU, full replica each; the request list is sharded and the waveforms
gathered by qwen3_tts_b200.parallel.run_data_parallel; `value` is the weak view — B utterances per GPU — and
`strong_scaling` the fixed-global-batch-32 view).  `--impl reference` times the reference's own modules
(baseline/_ref, installed by baseline/install_reference.sh) on the host cores, driven by the restated generation
loop (its HF generate() cannot run under transformers 5.5.0, SURVEY §8c); see baseline/ref_arm.py.
"""
import argparse
import json
import os
import re
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# NCCL's communicator / topology lines are wanted (the driver reads them) but stdout must stay the single JSON line:
# NCCL logs at INFO level to file descriptor 1, so fd 1 is pointed at stderr for everything except the result line,
# which is written to a private duplicate of the real stdout.
os.environ.setdefault("NCCL_DEBUG", "INFO")
_RESULT_OUT = os.fdopen(os.dup(1), "w")
os.dup2(2, 1)


def emit(obj):
    _RESULT_OUT.write(json.dumps(obj) + "\n")
    _RESULT_OUT.flush()


import numpy as np  # noqa: E402
import torch  # noqa: E402

FRAME_SEC = 0.08
METRIC = "speech_tokens_per_s"
UNIT = "frames/s (12.5 Hz speech tokens; x16 codebook tokens)"   # ONE string for both arms: the driver divides them
CPU_BUDGET_S = 200.0   # wall-clock target of a whole `--impl reference` run


def usable_cores():
    """Cores this process may really use: affinity mask capped by the cgroup CPU quota (a 128-CPU host can
    hand a container an 8-core quota; 128 threads on that quota thrash)."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = min(n, max(1, int(float(q) / float(per))))
    except Exception:
        try:
            q = int(open("/sys/fs/cgroup/cpu/cpu.cfs_quota_us").read())
            per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
            if q > 0:
                n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, min(n, 64))


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--batch", type=int, default=8)
    ap.add_argument("--frames", type=int, default=125)
    ap.add_argument("--model", default="1.7b", choices=["1.7b", "0.6b", "tiny"])
    ap.add_argument("--greedy", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--cpu-frames", type=int, default=0, help="frame-steps per CPU sample (0 = sized from the time budget)")
    ap.add_argument("--no-extras", action="store_true", help="skip the side measurements (other batch sizes, 0.6B, encoders)")
    ap.add_argument("--no-parity-check", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy "
                    "(waveforms and codes, float32), so that two builds can be compared output for output")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


def _pin(t):
    """Pinned host memory for the GPU arm's H2D copies; the CPU reference arm also runs where no driver exists."""
    return t.pin_memory() if torch.cuda.is_available() else t


def workload(args, H):
    """Synthetic inputs of config[2]'s shape (SURVEY §8d): seeded, bf16, pinned host memory."""
    B = args.batch
    lens = []
    for i in range(B):
        T = 16 + 8 * (i % 8)
        lens.append(T + 11 + (12 if i % 2 else 0))
    embs, trail = [], []
    for i, L in enumerate(lens):
        g = torch.Generator().manual_seed(1000 + i)
        embs.append(_pin((torch.randn(L, H, generator=g) * 0.5).to(torch.bfloat16)))
        trail.append(torch.zeros(0, H, dtype=torch.bfloat16))
    g = torch.Generator().manual_seed(999)
    pad = _pin((torch.randn(H, generator=g) * 0.1).to(torch.bfloat16))
    return lens, embs, trail, pad


def model_cfg(name):
    from qwen3_tts_b200 import synthetic
    return {"1.7b": synthetic.cfg_1p7b, "0.6b": synthetic.cfg_0p6b, "tiny": synthetic.cfg_tiny}[name]()


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "100",
                                          "-i", str(self.index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.th = threading.Thread(target=self._read, daemon=True)
            self.th.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 8:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[4:8]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


# ----------------------------------------------------------------------------------------------- CPU arm
def make_reference_arm(cfg, ccfg, W_bf16_cpu, CW_cpu, ncores):
    """The reference's own modules (baseline/_ref, through the shims) or, if they cannot be imported, the oracle port."""
    import contextlib
    from baseline import ref_arm
    Wcpu = {k: v.float().cpu() for k, v in W_bf16_cpu.items()}
    Ccpu = {k: v.to(torch.bfloat16).float().cpu() for k, v in CW_cpu.items()}
    ocfg, occfg = to_oracle_cfgs(cfg, ccfg)
    with contextlib.redirect_stdout(sys.stderr):  # the reference's import-time chatter must not reach stdout
        arm = ref_arm.ReferenceArm(ocfg, occfg, Wcpu, Ccpu, ncores)
    return arm


def to_oracle_cfgs(cfg, ccfg):
    from oracle import talker as OT, codec as OC
    st = lambda s: OT.StackCfg(s.hidden_size, s.num_layers, s.num_heads, s.num_kv_heads, s.head_dim,  # noqa: E731
                               s.intermediate_size, s.vocab_size, s.rms_eps, s.rope_theta)
    o = OT.TTSCfg(talker=st(cfg.talker), cp=st(cfg.cp), num_code_groups=cfg.num_code_groups,
                  codec_eos_token_id=cfg.codec_eos_token_id)
    oc = OC.CodecCfg(**{k: getattr(ccfg, k) for k in OC.CodecCfg.__dataclass_fields__})
    return o, oc


def sampling_kwargs(args):
    if args.greedy:
        return dict(do_sample=False, subtalker_dosample=False)
    return dict(do_sample=True, top_k=50, top_p=1.0, temperature=0.9, repetition_penalty=1.05, subtalker_dosample=True,
                subtalker_top_k=50, subtalker_top_p=1.0, subtalker_temperature=0.9)


def config_block(args, lens, n_gpus):
    return {"workload": f"Qwen3-TTS-12Hz-{args.model.upper()} CustomVoice-shaped, batch {args.batch}/GPU, non-streaming, "
                        f"{args.frames} frames/utterance, prefill+AR decode+codec decode",
            "batch_per_gpu": args.batch, "global_batch": args.batch * n_gpus, "frames": args.frames, "prompt_lens": lens,
            "sampling": "greedy" if args.greedy else "do_sample top_k=50 T=0.9 rep=1.05 (reference defaults)",
            "weights": "seeded random, expected shipped shapes (no checkpoints offline)",
            "parallelism": f"dp{n_gpus} (independent replicas, no data-path collective)",
            "l2": "per-step weight stream (>=3 GB) exceeds the 126 MB L2: no flush needed"}


def codec_encoder_probe(dev):
    """3 s of 24 kHz audio -> (16, 38) codes through Qwen3TTSTokenizer.encode's engine (fp32, default Mimi shapes,
    seeded random weights), device-resident input, CUDA-event timed."""
    import qwen3_tts_b200  # noqa: F401
    from qwen3_tts_b200 import synthetic
    from qwen3_tts_b200.codec_encoder import CodecEncoder
    from qwen3_tts_b200.config import EncoderConfig
    ecfg = EncoderConfig()
    enc = CodecEncoder(ecfg, synthetic.random_encoder_weights(ecfg, seed=2), device=dev)
    res = {"what": "codec encoder, 72000 samples (3 s) per row, fp32, ms per call", "launches": None}
    for B in (1, 8):
        wav = (torch.randn(B, 72000, device=dev) * 0.1).clamp(-1, 1)
        for _ in range(2):
            codes = enc.forward(wav)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            codes = enc.forward(wav)
        e1.record()
        torch.cuda.synchronize()
        assert tuple(codes.shape) == (B, 16, 38)
        res[f"ms_batch{B}"] = e0.elapsed_time(e1) / 5
    res["launches"] = enc.last_launches()
    return res


def speaker_encoder_probe(dev):
    """3 s of 24 kHz audio -> (1024,) x-vector (log-mel + ECAPA-TDNN, fp32, default shapes, seeded random weights)."""
    import qwen3_tts_b200  # noqa: F401
    from qwen3_tts_b200 import synthetic
    from qwen3_tts_b200.config import SpeakerEncoderConfig
    from qwen3_tts_b200.speaker_encoder import SpeakerEncoder
    scfg = SpeakerEncoderConfig()
    enc = SpeakerEncoder(scfg, synthetic.random_speaker_encoder_weights(scfg, seed=1), device=dev)
    res = {"what": "speaker x-vector, 72000 samples (3 s) per row, fp32, ms per call", "launches": None}
    for B in (1, 8):
        wav = (torch.randn(B, 72000, device=dev) * 0.1).clamp(-1, 1)
        for _ in range(2):
            emb = enc.embed_waveform(wav)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize()
        e0.record()
        for _ in range(5):
            emb = enc.embed_waveform(wav)
        e1.record()
        torch.cuda.synchronize()
        assert tuple(emb.shape) == (B, scfg.enc_dim) and bool(torch.isfinite(emb).all())
        res[f"ms_batch{B}"] = e0.elapsed_time(e1) / 5
    res["launches"] = enc.last_launches()
    return res


def cpu_sample(arm, embs, trail, pad, spk, B, frames, n_first, plan_steps=0, budget_s=None):
    """Bounded sample of the workload on the host: prefill (measured once) + frame-steps + codec decode of them.
    With plan_steps > 0 the frames per step are sized so that plan_steps steps fit `budget_s`."""
    from baseline import ref_arm
    t_pre = arm.start(embs, trail, pad, spk)
    timing, _ = arm.step_frames(n_first)
    per = float(np.median(timing["frames"])) + timing["codec"] / n_first
    n = n_first
    if plan_steps > 0:
        n = int(max(1, min(16, (budget_s - t_pre - per * n_first) / max(plan_steps * per, 1e-9))))
    rate, det = ref_arm.workload_rate(timing, B, frames)
    return rate, det, timing, n


def parity_self_check(eng, cfg, W, embs, trail, pad, dev, frames=4):
    """Teacher-forced check of THIS workload on THIS engine before anything is timed: the oracle (fp32, same
    bf16-rounded weights) generates `frames` greedy frames from the bench prompts; the engine is forced along the same
    codes and every talker / code-predictor logits row must agree within the parity tolerance of tests/test_gpu_ar.py."""
    from oracle import talker as OT
    from tests import helpers as Hh
    import qwen3_tts_b200 as q
    ocfg, _ = to_oracle_cfgs(cfg, q.CodecConfig())
    Wf = {k: v.float().cpu() for k, v in W.items()}
    osp = OT.SamplingCfg(do_sample=False, subtalker_dosample=False, max_new_tokens=frames + 1, suppress_eos=True)
    t0 = time.perf_counter()
    ref = OT.generate(Wf, ocfg, [e.float() for e in embs], [t.float() for t in trail], pad.float(), osp, record_logits=True)
    forced = torch.stack(ref.codes).numpy()
    sp = q.SamplingParams(do_sample=False, subtalker_dosample=False, max_new_tokens=frames + 1, suppress_eos=True)
    codes, tl, cl, prog = Hh.run_engine_forced(eng.ar, [e.to(dev) for e in embs], [t.to(dev) for t in trail], pad.to(dev), sp, forced, dev)
    G = cfg.num_code_groups
    worst, worst_mean = 0.0, 0.0
    for f in range(frames + 1):
        r = ref.record["talker_logits"][f]
        d = np.abs(tl[f] - r) / float(np.std(r))
        worst, worst_mean = max(worst, float(d.max())), max(worst_mean, float(d.mean()))
    for f in range(frames):
        for j in range(G - 1):
            r = ref.record["cp_logits"][f * (G - 1) + j]
            d = np.abs(cl[f, j] - r) / float(np.std(r))
            worst, worst_mean = max(worst, float(d.max())), max(worst_mean, float(d.mean()))
    ok = bool(prog[0] == frames and (codes == forced).all() and worst < 0.4 and worst_mean < 0.075)
    return {"ok": ok, "frames": frames, "rows": int(len(embs)), "max_abs_err_over_std": worst, "max_mean_err_over_std": worst_mean,
            "tolerance": "max < 0.4 std, mean < 0.075 std = 1.5x PyTorch bf16's own gap to the fp32 oracle at these shapes (profiles/r02_tolerance_calibration.txt)", "oracle_s": time.perf_counter() - t0}


def decode_probe(eng, q, cfg, args, spk, B, N, dev, greedy=False):
    """Device-resident prefill + N frame-steps + codec decode at batch B on an existing engine (side measurement)."""
    class A:
        batch = B
    lens, embs, trail, pad = workload(A, cfg.talker.hidden_size)
    kw = dict(do_sample=False, subtalker_dosample=False) if greedy else spk
    sp = q.SamplingParams(max_new_tokens=N + 1, suppress_eos=True, seed=1234, **kw)
    d_embs, d_trail, d_pad = [e.to(dev) for e in embs], [t.to(dev) for t in trail], pad.to(dev)
    G = cfg.num_code_groups
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    res = []
    for i in range(3):
        e0, e1, e2, e3 = ev(), ev(), ev(), ev()
        e0.record()
        eng.ar.prefill(d_embs, d_trail, d_pad, sp)
        codes = torch.zeros(B, N, G, dtype=torch.int32, device=dev)
        e1.record()
        eng.ar.decode(N, codes)
        e2.record()
        eng.codec.chunked_decode(codes.transpose(1, 2))
        e3.record()
        torch.cuda.synchronize()
        res.append((e0.elapsed_time(e1), e1.elapsed_time(e2), e2.elapsed_time(e3)))
    pre, dec, cod = res[-1]
    tot = pre + dec + cod
    # first packet: prefill + 4 frame-steps + codec of them, host in / host out
    sp_fp = q.SamplingParams(max_new_tokens=5, suppress_eos=True, seed=1234, **kw)
    fp = None
    try:
        for _ in range(2):
            next(iter(eng.stream_synthesize(embs, trail, pad, sp_fp, packet_frames=4)))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            next(iter(eng.stream_synthesize(embs, trail, pad, sp_fp, packet_frames=4)))
        fp = (time.perf_counter() - t0) / 3 * 1000.0
    except Exception as e:
        print(f"[bench] first-packet probe (B={B}) failed: {e!r}", file=sys.stderr)
    S_mean = int(np.mean(lens) + N / 2)
    a_bytes, _ = eng.ar.algorithmic_bytes(B, S_mean)
    return {"batch": B, "frames": N, "sampling": "greedy" if greedy else "do_sample", "frames_per_s": B * N / (tot / 1000.0),
            "rtf": (tot / 1000.0) / (B * N * FRAME_SEC), "ms_prefill": pre, "ms_decode": dec, "ms_codec": cod,
            "ms_per_frame_step": dec / N, "first_packet_ms": fp, "roofline_frac_decode": a_bytes / (dec / N / 1000.0) / 1e9 / hbm_peak()[0]}


REF_FRAMES = 38   # 3 s of prompt audio at 12.5 Hz (72000 samples / 1920, rounded up)


def voice_clone_probe(eng, q, cfg, W, args, spk, B, N, dev):
    """BASELINE config[4] composed at full 1.7B-Base shape, host in / host out: 3 s of prompt audio per row ->
    codec encoder (ref codes) + speaker x-vector -> ICL prefill (role prefix, x-vector row, BOS + 38 reference frames whose
    embedding is the sum of the 16 codebook embeddings, text rows as trailing input) -> N frame-steps -> codec decode of the
    38 + N frames -> proportional cut of the reference part (inference/qwen3_tts_model.py:566-598).  Random weights:
    a timing of the composed path, stage by stage; parity of each stage is in tests/ (test_gpu_voice_clone.py et al.)."""
    from qwen3_tts_b200 import synthetic
    from qwen3_tts_b200.codec_encoder import CodecEncoder
    from qwen3_tts_b200.config import EncoderConfig, SpeakerEncoderConfig
    from qwen3_tts_b200.speaker_encoder import SpeakerEncoder
    H, G = cfg.talker.hidden_size, cfg.num_code_groups
    ecfg, scfg = EncoderConfig(), SpeakerEncoderConfig(enc_dim=H)
    cenc = CodecEncoder(ecfg, synthetic.random_encoder_weights(ecfg, seed=2), device=dev)
    senc = SpeakerEncoder(scfg, synthetic.random_speaker_encoder_weights(scfg, seed=1), device=dev)
    tabs = [W["talker.model.codec_embedding.weight"]] + [W[f"talker.code_predictor.model.codec_embedding.{j}.weight"] for j in range(G - 1)]
    tabs = [t.to(dev, torch.bfloat16) for t in tabs]
    g = torch.Generator().manual_seed(77)
    wav_h = _pin((torch.randn(B, 72000, generator=g) * 0.1).clamp(-1, 1))
    n_prefix, n_trail = 9, 24
    text_h = _pin((torch.randn(B, n_prefix + 1 + 1 + REF_FRAMES + n_trail, H, generator=g) * 0.5).to(torch.bfloat16))
    pad = (torch.randn(H, generator=g) * 0.1).to(torch.bfloat16).to(dev)
    sp = q.SamplingParams(max_new_tokens=N + 1, suppress_eos=True, seed=4321, **spk)
    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    runs = []
    for it in range(3):
        e = [ev() for _ in range(7)]
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        e[0].record()
        wav = wav_h.to(dev, non_blocking=True)
        text = text_h.to(dev, non_blocking=True)
        ref = cenc.forward(wav)                                            # (B, 16, 38) codes
        e[1].record()
        xvec = senc.embed_waveform(wav).to(torch.bfloat16)                   # (B, H)
        e[2].record()
        R = ref.shape[-1]
        icl = tabs[0][ref[:, 0, :].long()]
        for j in range(1, G):
            icl = icl + tabs[j][ref[:, j, :].long()]                       # (B, R, H): sum over the 16 codebooks
        bos = tabs[0][torch.full((B, 1), cfg.codec_bos_id, device=dev)]
        rows = torch.cat([text[:, :n_prefix], xvec[:, None, :] + text[:, n_prefix:n_prefix + 1],
                          text[:, n_prefix + 1:n_prefix + 2 + R] + torch.cat([bos, icl], dim=1)], dim=1)
        trail = text[:, n_prefix + 2 + R:n_prefix + 2 + R + n_trail]
        eng.ar.prefill([rows[b] for b in range(B)], [trail[b] for b in range(B)], pad, sp)
        codes = torch.zeros(B, N, G, dtype=torch.int32, device=dev)
        e[3].record()
        eng.ar.decode(N, codes)
        e[4].record()
        full = torch.cat([ref.to(torch.int32), codes.transpose(1, 2)], dim=2)    # (B, 16, 38 + N)
        wav_out = eng.codec.chunked_decode(full)
        cut = int(REF_FRAMES / full.shape[-1] * wav_out.shape[-1])
        e[5].record()
        out_h = wav_out[..., cut:].contiguous().cpu()
        e[6].record()
        torch.cuda.synchronize()
        wall = (time.perf_counter() - t0) * 1000.0
        runs.append(([e[i].elapsed_time(e[i + 1]) for i in range(6)], wall, tuple(out_h.shape)))
    st, wall, shape = runs[-1]
    assert shape[0] == B and abs(shape[-1] - N * 1920) <= 1920, shape
    return {"what": "config[4] voice clone, 1.7B-Base shape: 3 s prompt audio/row -> codec encode + x-vector + ICL prefill "
                    f"({n_prefix + 2 + REF_FRAMES} rows + {n_trail} trailing) + {N} frame-steps + codec decode of {REF_FRAMES}+{N} frames + cut; "
                    "host audio in, host audio out",
            "batch": B, "frames": N, "ms_total_wall": wall,
            "ms": dict(zip(("codec_encode", "x_vector", "icl_prefill", "ar_decode", "codec_decode", "d2h"), st)),
            "frames_per_s": B * N / (wall / 1000.0), "rtf": (wall / 1000.0) / (B * N * FRAME_SEC),
            "h2d_bytes": int(wav_h.numel() * 4 + text_h.numel() * 2), "d2h_bytes": int(B * shape[-1] * 4)}


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, wav, codes):
    """The last timed step's waveforms (B, N*1920) and codes (B, N, 16) as float32 .npy files (7.7 MB + 64 KB at the
    default shape).  Waveforms that would take the dump past DUMP_BYTES are cut to a fixed, seeded sample of time
    positions, the same for every row, written beside them as wav_index.npy."""
    os.makedirs(out_dir, exist_ok=True)
    codes = codes.float().cpu().numpy()
    wav = wav.float().reshape(wav.shape[0], -1).cpu().numpy()
    keep = (DUMP_BYTES - codes.nbytes - 4096) // (4 * wav.shape[0] + 8)   # a float32 per row and a float64 index per position, .npy headers
    if wav.shape[1] > keep:
        idx = np.sort(np.random.default_rng(0).choice(wav.shape[1], keep, replace=False))
        wav = wav[:, idx]
        np.save(os.path.join(out_dir, "wav_index.npy"), idx.astype(np.float64))
    np.save(os.path.join(out_dir, "wav.npy"), wav)
    np.save(os.path.join(out_dir, "codes.npy"), codes)


def hbm_peak():
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        return float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback 6.65 TB/s (B200_PROFILING.md)"


def main():
    args = parse()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.manual_seed(0)

    import qwen3_tts_b200 as q
    from qwen3_tts_b200 import synthetic
    cfg = model_cfg(args.model)
    ccfg = q.CodecConfig() if args.model != "tiny" else q.CodecConfig(
        codebook_size=2048, codebook_dim=64, hidden_size=64, latent_dim=64, num_heads=4, num_kv_heads=4, head_dim=16,
        sliding_window=6, intermediate_size=96, num_layers=2, decoder_dim=256)
    H = cfg.talker.hidden_size
    lens, embs, trail, pad = workload(args, H)
    spk = sampling_kwargs(args)
    ncores = usable_cores()

    # ------------------------------------------------------------------ reference arm (CPU)
    if args.impl == "reference":
        if rank != 0:
            return
        t_begin = time.perf_counter()
        torch.set_num_threads(ncores)
        Wg = synthetic.random_tts_weights(cfg, device="cpu", seed=0, dtype=torch.bfloat16)
        CWg = synthetic.random_codec_weights(ccfg, device="cpu", seed=0)
        arm = make_reference_arm(cfg, ccfg, Wg, CWg, ncores)
        del Wg, CWg
        t_build = time.perf_counter() - t_begin
        n_steps = args.warmup + args.steps
        # warm-up step 1 = prefill (measured once) + 1 frame-step; it sizes the frames per step for the budget
        _, _, tim0, n = cpu_sample(arm, embs, trail, pad, spk, args.batch, args.frames, 1, plan_steps=max(n_steps - 1, 1),
                                   budget_s=max(CPU_BUDGET_S - t_build, 30.0))
        if args.cpu_frames > 0:
            n = args.cpu_frames
        from baseline import ref_arm
        frame_times, codec_per_frame = [], []
        for i in range(1, args.warmup):
            arm.step_frames(n)
        t0 = time.perf_counter()
        for i in range(args.steps):
            tim, _ = arm.step_frames(n)
            frame_times += tim["frames"]
            codec_per_frame.append(tim["codec"] / n)
        elapsed = time.perf_counter() - t0
        pooled = {"prefill": arm.t_prefill, "frames": frame_times, "codec": float(np.median(codec_per_frame)) * len(frame_times)}
        val, det = ref_arm.workload_rate(pooled, args.batch, args.frames)
        sample = (f"prefill of B={args.batch} measured once ({arm.t_prefill:.2f} s); each timed step = {n} consecutive frame-steps of the "
                  f"running batch (15 code-predictor forwards + sampling + 1 talker step each) + chunked_decode of those {n} frames; "
                  f"value = B*{args.frames} / (prefill + {args.frames} x (median frame-step + codec per frame)) over "
                  f"{len(frame_times)} measured frame-steps; fp32, {ncores} threads; ms_per_step is the elapsed time of a timed step")
        out = {"impl": "reference", "metric": METRIC, "value": val, "unit": UNIT,
               "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
               "ms_per_step": 1000.0 * elapsed / max(args.steps, 1), "higher_is_better": True, "scaling": "weak",
               "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config_block(args, lens, 1),
               "rtf": 1.0 / (val * FRAME_SEC),
               "cpu_baseline": {"value": val, "unit": UNIT, "cores": ncores, "kind": arm.kind, "sample": sample,
                                "frames_per_step": n, **det},
               "e2e": {"value": val, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
               "gpu_launches": 0, "wall_s": time.perf_counter() - t_begin, "build_s": t_build}
        emit(out)
        return

    # ------------------------------------------------------------------ B200 arm
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the B200 path has no CPU fallback)")
    dev = f"cuda:{local}"
    torch.cuda.set_device(local)
    dist = None
    if world > 1:
        import torch.distributed as dist
        dist.init_process_group("nccl", device_id=torch.device(dev))
    from qwen3_tts_b200 import parallel
    from qwen3_tts_b200.pipeline import TTSEngine
    # weights are made on the CPU (seeded) and copied: the first kernels of this process are the engine's own
    W = synthetic.random_tts_weights(cfg, device="cpu", seed=0)
    CW = synthetic.random_codec_weights(ccfg, device="cpu", seed=0)
    big = (rank == 0 and world == 1 and not args.no_extras) or world > 1
    max_batch = max(args.batch, 32 if big else 1)
    max_ctx = max(lens) + args.frames + 8
    eng = TTSEngine(cfg, W, ccfg, CW, device=dev, max_batch=max_batch, max_ctx=max_ctx,
                    codec_max_frames=max(args.frames + 8 + (REF_FRAMES if big else 0), 64))
    sp = q.SamplingParams(max_new_tokens=args.frames + 1, suppress_eos=True, seed=1234, **spk)
    B, N, G = args.batch, args.frames, cfg.num_code_groups
    d_embs = [e.to(dev) for e in embs]
    d_trail = [t.to(dev) for t in trail]
    d_pad = pad.to(dev)
    stream = torch.cuda.current_stream()

    # ---- parity first: the exact engine / kernel instantiation that is timed below, against the oracle
    parity = None
    if rank == 0 and world == 1 and not args.no_parity_check:
        parity = parity_self_check(eng, cfg, W, embs, trail, pad, dev)
        if not parity["ok"]:
            raise SystemExit(f"bench.py: parity self-check failed: {json.dumps(parity)}")

    def barrier():
        torch.cuda.synchronize()
        if dist is not None:
            dist.barrier()
        torch.cuda.synchronize()

    ev = lambda: torch.cuda.Event(enable_timing=True)  # noqa: E731
    t_pre = t_dec = t_cod = 0.0

    def step_resident(timed):
        nonlocal t_pre, t_dec, t_cod
        e0, e1, e2, e3 = ev(), ev(), ev(), ev()
        e0.record(stream)
        eng.ar.prefill(d_embs, d_trail, d_pad, sp)
        codes = torch.zeros(B, N, G, dtype=torch.int32, device=dev)
        e1.record(stream)
        eng.ar.decode(N, codes)
        e2.record(stream)
        wav = eng.codec.chunked_decode(codes.transpose(1, 2))
        e3.record(stream)
        if timed:
            torch.cuda.synchronize()
            t_pre += e0.elapsed_time(e1); t_dec += e1.elapsed_time(e2); t_cod += e2.elapsed_time(e3)
        return wav, codes

    for _ in range(args.warmup):
        step_resident(False)
    clocks = ClockSampler(local)
    barrier()
    clocks.start()
    s0, s1 = ev(), ev()
    s0.record(stream)
    for _ in range(args.steps):
        wav, codes = step_resident(True)
    s1.record(stream)
    barrier()
    ms_total = s0.elapsed_time(s1)
    clk = clocks.stop()
    fd, n_valid, _ = eng.ar.progress()
    assert fd == N and all(v == N for v in n_valid), (fd, n_valid)
    assert torch.isfinite(wav).all()
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, wav, codes)

    # ---- end-to-end through the public calls: pinned host inputs, H2D + D2H inside the timed region.  The global
    # request list (B per GPU) goes through parallel.run_data_parallel: shard -> synthesize -> gather of waveforms
    requests = []
    for r in range(world):
        requests += list(zip(embs, trail))

    def serve(reqs):
        wavs, _ = eng.synthesize([e for e, _ in reqs], [t for _, t in reqs], pad, sp)
        return wavs

    for _ in range(2):
        parallel.run_data_parallel(serve, requests)
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        wavs_host = parallel.run_data_parallel(serve, requests)
    torch.cuda.synchronize()
    e2e_s = time.perf_counter() - t0
    assert len(wavs_host) == world * B and all(w.shape == (N * 1920,) for w in wavs_host)
    h2d = sum(e.numel() * 2 for e in embs) + pad.numel() * 2
    d2h = sum(w.size * 4 for w in wavs_host[:B])

    # ---- first-packet latency (config[3]): prefill + 4 frame-steps + codec decode of the 4 frames, host in / host out
    sp_fp = q.SamplingParams(max_new_tokens=5, suppress_eos=True, seed=1234, **spk)
    try:  # a side measurement: the headline line must survive a failure here
        for _ in range(2):
            next(iter(eng.stream_synthesize(embs, trail, pad, sp_fp, packet_frames=4)))
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        for _ in range(3):
            next(iter(eng.stream_synthesize(embs, trail, pad, sp_fp, packet_frames=4)))
        first_packet_ms = (time.perf_counter() - t0) / 3 * 1000.0
    except Exception as e:
        first_packet_ms = None
        print(f"[bench] first-packet probe failed: {e!r}", file=sys.stderr)

    # ---- strong-scaling view (SURVEY §8e): a FIXED global batch of 32 utterances split over the N GPUs
    strong = None
    if world > 1:
        class A32:
            batch = 32
        l32, e32, t32, _ = workload(A32, H)
        req32 = list(zip(e32, t32))
        try:
            for _ in range(2):
                parallel.run_data_parallel(serve, req32)
            barrier()
            t0 = time.perf_counter()
            reps = max(2, args.steps // 2)
            for _ in range(reps):
                w32 = parallel.run_data_parallel(serve, req32)
            torch.cuda.synchronize()
            strong_s = parallel.max_over_ranks((time.perf_counter() - t0) / reps, device=dev)
            strong = {"global_batch": 32, "per_gpu_batch": 32 // world if 32 % world == 0 else f"{32 // world}-{32 // world + 1}",
                      "value": 32 * N / strong_s, "unit": UNIT, "ms": strong_s * 1e3,
                      "what": "host inputs -> run_data_parallel(shard, synthesize, all_gather_object of waveforms) -> host outputs"}
            assert len(w32) == 32
        except Exception as e:
            strong = {"error": repr(e)[:200]}
        if 32 % world == 0:   # BASELINE config[4]: the voice-clone path at a global batch of 32 split over the N GPUs
            vc, vc_err = None, None
            try:
                vc = voice_clone_probe(eng, q, cfg, W, args, spk, 32 // world, N, dev)
            except Exception as e:
                vc_err = repr(e)[:200]
            vc_ms = parallel.max_over_ranks(vc["ms_total_wall"] if vc else 1e12, device=dev)   # every rank reaches this collective
            if strong is None or "error" in strong:
                strong = dict(strong or {})
            if vc_ms >= 1e12:
                strong["config4_voice_clone"] = {"error": vc_err or "failed on another rank"}
            else:
                strong["config4_voice_clone"] = {"global_batch": 32, "per_gpu_batch": 32 // world, "ms": vc_ms, "value": 32 * N / (vc_ms / 1e3),
                                                 "unit": UNIT, "rank0_stages_ms": vc["ms"], "what": vc["what"]}

    tms = torch.tensor([ms_total, e2e_s * 1000.0, t_dec], dtype=torch.float64, device=dev)
    if dist is not None:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms_total, e2e_ms, t_dec_max = [float(x) for x in tms.tolist()]
    frames_total = world * B * N * args.steps
    value = frames_total / (ms_total / 1000.0)
    e2e_val = frames_total / (e2e_ms / 1000.0)

    # ---- roofline of the dominant kernel (fused frame-step kernel): algorithmic bytes / measured duration
    S_mean = int(np.mean(lens) + N / 2)
    a_bytes, a_stream = eng.ar.algorithmic_bytes(B, S_mean)
    t_step = (t_dec / args.steps) / N / 1000.0  # s per frame-step (this rank)
    peak, peak_src = hbm_peak()
    achieved = a_bytes / t_step / 1e9
    # measured DRAM traffic of this kernel from the committed `ncu --set full` capture (profiles/): bytes per
    # frame-step of the B=8 capture scaled to this launch's frame count; null when no capture of this round exists
    traffic, traffic_src = None, None
    try:
        if args.batch == 8 and args.model == "1.7b":
            meta = json.load(open(os.path.join(ROOT, "profiles", "r02_decode_kernel_traffic.json")))
            traffic = float(meta["dram_bytes_per_frame_step"]) * N
            traffic_src = meta["source"]
    except Exception:
        traffic = None
    roof = {"bound": "hbm", "kernel": "q3_step_kernel (fused frame-step)", "achieved": achieved, "peak": peak, "unit": "GB/s",
            "frac": achieved / peak, "peak_source": peak_src, "traffic": traffic, "traffic_source": traffic_src,
            "algorithmic_bytes_per_launch": a_bytes * N, "algorithmic_bytes_per_frame_step": a_bytes,
            "no_residency_bytes_per_frame_step": a_stream, "ms_per_frame_step": t_step * 1e3, "mean_context": S_mean}

    out = {"metric": METRIC, "value": value, "unit": UNIT,
           "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_total / args.steps,
           "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "bf16", "data": "synthetic",
           "config": config_block(args, lens, world), "rtf": (ms_total / 1000.0) / (frames_total * FRAME_SEC),
           "breakdown_ms_per_step": {"prefill": t_pre / args.steps, "decode": t_dec / args.steps, "codec": t_cod / args.steps},
           "roofline": roof, "first_packet_ms": first_packet_ms,
           "e2e": {"value": e2e_val, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                   "rtf": (e2e_ms / 1000.0) / (frames_total * FRAME_SEC),
                   "path": "parallel.run_data_parallel(TTSEngine.synthesize): pinned host embeddings in, host waveforms out"},
           "gpu_launches": args.steps * (cfg.talker.num_layers * 8 + 4 + eng.codec.last_launches()),  # prefill (7 GEMM/row kernels + attention per layer, index + gather) + head + fused decode + codec
           "clocks": clk, "parity_check": parity, "strong_scaling": strong}

    # ---- reference CPU path beside it (rank 0, N=1 only): bounded sample on the host cores
    if rank == 0 and world == 1 and not args.no_cpu_baseline:
        arm = make_reference_arm(cfg, ccfg, W, CW, ncores)
        nfr = args.cpu_frames if args.cpu_frames > 0 else 4
        v, det, _, _ = cpu_sample(arm, embs, trail, pad, spk, B, N, nfr)
        out["cpu_baseline"] = {"value": v, "unit": UNIT, "cores": ncores, "kind": arm.kind,
                               "sample": f"prefill of B={B} + {nfr} frame-steps + chunked_decode of those {nfr} frames, fp32, {ncores} threads; "
                                         f"value = B*{N} / (prefill + {N} x (median frame-step + codec per frame))", **det}
        del arm
    # ---- side measurements, never part of `value`
    if rank == 0 and world == 1 and not args.no_extras:
        out["extras"] = {}
        for name, fn in (("batch1", lambda: decode_probe(eng, q, cfg, args, spk, 1, N, dev)),
                         ("batch32", lambda: decode_probe(eng, q, cfg, args, spk, 32, N, dev)),
                         ("batch8_first_packet", lambda: {"first_packet_ms": first_packet_ms}),
                         ("config4_voice_clone_batch4", lambda: voice_clone_probe(eng, q, cfg, W, args, spk, 4, N, dev)),
                         ("config4_voice_clone_batch32", lambda: voice_clone_probe(eng, q, cfg, W, args, spk, 32, N, dev))):
            try:
                out["extras"][name] = fn()
            except Exception as e:
                out["extras"][name] = {"error": repr(e)[:200]}
        if args.model == "1.7b":
            try:  # BASELINE config[1]: 0.6B, single utterance, greedy
                eng.close()
                del eng
                torch.cuda.empty_cache()
                c06 = model_cfg("0.6b")
                e06 = TTSEngine(c06, synthetic.random_tts_weights(c06, device="cpu", seed=0), ccfg, CW, device=dev, max_batch=8,
                                max_ctx=max_ctx, codec_max_frames=max(args.frames + 8, 64))
                out["extras"]["0.6b_greedy_batch1"] = decode_probe(e06, q, c06, args, spk, 1, N, dev, greedy=True)
                out["extras"]["0.6b_batch8"] = decode_probe(e06, q, c06, args, spk, 8, N, dev)
                e06.close()
            except Exception as e:
                out["extras"]["0.6b"] = {"error": repr(e)[:200]}
        for name, probe in (("codec_encoder", codec_encoder_probe), ("speaker_encoder", speaker_encoder_probe)):
            try:
                out["extras"][name] = probe(dev)
            except Exception as e:  # the headline line must survive whatever happens here
                out["extras"][name] = {"error": repr(e)[:200]}
    if rank == 0:
        emit(out)
    if dist is not None:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
