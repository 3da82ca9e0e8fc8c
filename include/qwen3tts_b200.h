/*
 * qwen3tts_b200.h — C ABI of the B200-native Qwen3-TTS hot-path library (libqwen3tts_b200.so).
 *
 * The reference (QwenLM/Qwen3-TTS) is pure Python with no FFI/plugin interface (SURVEY.md §8b), so the
 * boundary below is defined at the two narrowest seams of the reference and each entry point cites the
 * reference interface it replaces (paths relative to /root/reference/qwen_tts/):
 *
 *   seam B (AR)   : Qwen3TTSTalkerForConditionalGeneration.generate(inputs_embeds, attention_mask,
 *                   trailing_text_hidden, tts_pad_embed, **talker_kwargs)
 *                   as called at core/models/modeling_qwen3_tts.py:2272-2278, including the per-frame
 *                   forward :1636-1744, the nested code-predictor generate :1671-1680 / :1250-1312 and the
 *                   HF logits processors + sampling configured at :2044-2066.
 *   seam C (codec): Qwen3TTSTokenizerV2Decoder.forward / chunked_decode
 *                   core/tokenizer_12hz/modeling_qwen3_tts_tokenizer_v2.py:869-896 (called by
 *                   Qwen3TTSTokenizerV2Model.decode :993-1024).
 *
 * Conventions
 *   - every function returns 0 on success, non-zero on error; q3_last_error() gives the message
 *     (thread-local).
 *   - all `dev` pointers are CUDA device pointers on the engine's device; the caller (PyTorch) OWNS them.
 *     The engine owns only what it allocates itself (packed weights, KV cache, workspaces).
 *   - `stream` is a cudaStream_t passed as void* (torch.cuda.current_stream().cuda_stream); work is
 *     enqueued on it, calls do not synchronise unless documented.  One engine = one device, not re-entrant.
 *   - bf16 tensors are raw uint16 storage (torch.bfloat16).  No torch types cross this boundary.
 */
#ifndef QWEN3TTS_B200_H
#define QWEN3TTS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define Q3_ABI_VERSION 1
#define Q3_MAX_BATCH 32        /* sequences per engine pass (reference batches = padded batch on one GPU) */
#define Q3_NUM_GROUPS_MAX 32

typedef struct q3_engine q3_engine; /* AR engine: talker + code predictor + sampler */
typedef struct q3_codec q3_codec;   /* 12 Hz codec decoder */

/* One decoder stack.  Mirrors Qwen3TTSTalkerConfig / Qwen3TTSTalkerCodePredictorConfig
 * (core/models/configuration_qwen3_tts.py:370-404, :187-212); values come from the loaded config. */
typedef struct {
  int32_t hidden_size, num_layers, num_heads, num_kv_heads, head_dim, intermediate_size, vocab_size;
  float rms_eps;
} q3_stack_cfg;

typedef struct {
  q3_stack_cfg talker, cp;
  int32_t num_code_groups;   /* 16 */
  int32_t has_cp_projection; /* small_to_mtp_projection is a Linear (1.7B) or Identity (0.6B), :1171-1174 */
  int32_t codec_eos_token_id;
  int32_t max_batch;         /* <= Q3_MAX_BATCH */
  int32_t max_ctx;           /* talker KV capacity per sequence (prompt + frames) */
  int32_t device;            /* CUDA ordinal */
} q3_engine_cfg;

/* Generation kwargs of seam B (modeling_qwen3_tts.py:2044-2066; defaults inference/qwen3_tts_model.py:287-352). */
typedef struct {
  int32_t do_sample, top_k;
  float top_p, temperature, repetition_penalty;
  int32_t subtalker_dosample, subtalker_top_k;
  float subtalker_top_p, subtalker_temperature;
  int32_t min_new_tokens;  /* 2 */
  int32_t suppress_eos;    /* benchmark-only: fixed horizon (EOS never sampled) */
  uint64_t seed;           /* Philox key; u = philox(seed; row, frame, group) */
} q3_sampling;

int q3_abi_version(void);
const char* q3_last_error(void);

/* ---------------------------------------------------------------- AR engine (seam B) */
int q3_engine_create(const q3_engine_cfg* cfg, q3_engine** out);
void q3_engine_destroy(q3_engine* e);

/* Copy+repack one weight from device memory (bf16, row-major [rows][cols], i.e. nn.Linear/nn.Embedding
 * layout).  `name` is one of the engine tensor names documented in INTEGRATION.md, e.g.
 *   "talker.layers.<i>.qkv"  = cat(q_proj,k_proj,v_proj).weight          (:740-748)
 *   "talker.layers.<i>.gate_up" = gate/up rows interleaved in blocks of 8 (:848-849)
 *   "talker.layers.<i>.o", ".down", ".ln1", ".ln2", ".q_norm", ".k_norm"
 *   "talker.norm", "talker.codec_head", "talker.codec_embedding", "talker.rope_cos", "talker.rope_sin"
 *   "cp.layers.<i>.*", "cp.norm", "cp.proj", "cp.proj_bias", "cp.lm_head.<j>", "cp.codec_embedding.<j>",
 *   "cp.rope_cos", "cp.rope_sin".
 * The source may be freed after the call returns (the call synchronises the copy stream). */
int q3_engine_load_tensor(q3_engine* e, const char* name, const void* dev_bf16, int64_t rows, int64_t cols);
int q3_engine_finalize(q3_engine* e); /* verifies that every tensor is present */

/* Prefill = first `talker.generate` forward (modeling_qwen3_tts.py:1665-1667 -> :1457-1561).
 * embeds: bf16 [sum(lens)][H], rows of sequence 0 first (NO padding: the reference's left-pad+mask,
 * :2239-2254, is equivalent to per-sequence positions 0..len-1).  lens: host int32[B].
 * trailing: bf16 [B][trailing_stride][H] (row b valid for trailing_lens[b] steps, then tts_pad, :1689-1692);
 * tts_pad: bf16 [H].  Resets all per-request state (per request, never on a module: SURVEY F10) and samples
 * codebook-0 of frame 0. */
int q3_prefill(q3_engine* e, int32_t B, const void* embeds_dev, const int32_t* lens_host,
               const void* trailing_dev, const int32_t* trailing_lens_host, int32_t trailing_stride,
               const void* tts_pad_dev, const q3_sampling* sp, void* stream);

/* Run up to `max_frames` further frame-steps (code predictor x15 -> embed -> talker -> head -> sample),
 * stopping early once every row has sampled EOS.  No host sync per token (HF syncs every token).
 * codes_dev: int32 [B][codes_stride][num_code_groups], frame f of row b at [b][f][:]; frames accumulate
 * across calls (streaming = repeated calls with small max_frames).  Asynchronous. */
int q3_decode(q3_engine* e, int32_t max_frames, int32_t* codes_dev, int32_t codes_stride, void* stream);

/* ---- continuous batching (SURVEY §8f-4; the reference has only the static padded batch of
 * modeling_qwen3_tts.py:2239-2254 behind a Gradio queue, cli/demo.py:629).  A session owns n_slots rows; a finished or
 * never-used slot is a row that keeps stepping and is ignored (exactly what HF does with finished rows of a batch).
 * q3_admit prefills n new requests into free slots WHILE the others keep their state: their K/V, positions, sampling
 * history and Philox streams are per row, so a request admitted at any frame generates what it would generate alone
 * (keys_host[r] is the request's Philox row key).  q3_decode / q3_get_progress are shared with the static path;
 * n_valid[b] counts the row's OWN frames, and the row's codes land at codes[b][0..n_valid).  q3_admit synchronises
 * `stream` (it needs the frame counter).  embeds_dev: the n prompts packed back to back; trailing_dev: [n][stride][H]. */
int q3_session_begin(q3_engine* e, int32_t n_slots, int32_t max_trailing, const void* tts_pad_dev, const q3_sampling* sp,
                     void* stream);
int q3_admit(q3_engine* e, int32_t n, const int32_t* slots_host, const uint32_t* keys_host, const void* embeds_dev,
             const int32_t* lens_host, const void* trailing_dev, const int32_t* trailing_lens_host,
             int32_t trailing_stride, void* stream);
/* Streaming text input: append n rows [n][H] bf16 to the trailing_text_hidden of a running row (static batch or session);
 * frame t adds trailing[t] while t < the row's trailing length and tts_pad afterwards (modeling_qwen3_tts.py:1689-1692).
 * The capacity is the trailing stride given at q3_prefill / max_trailing of q3_session_begin. */
int q3_append_trailing(q3_engine* e, int32_t slot, const void* rows_dev, int32_t n, void* stream);
/* give up rows that reached their frame horizon without EOS (their slots become free) */
int q3_release_slots(q3_engine* e, int32_t n, const int32_t* slots_host, void* stream);

/* After synchronising `stream`: frames_done = frames whose 16 codes are complete (same for all rows);
 * n_valid[b] = frames of row b before its first EOS (== modeling_qwen3_tts.py:2283-2290 trim);
 * finished[b] = 1 once row b sampled EOS.  Host pointers (may be NULL). */
int q3_get_progress(q3_engine* e, int32_t* frames_done, int32_t* n_valid, int32_t* finished);

/* Per-step hidden states = the second return value of generate() (modeling_qwen3_tts.py:2281: the last layer's normed
 * output of the newest position of every step): hid_dev bf16 [B][stride][hidden] gets row b's step s at [b][s][:]
 * (s = 0 is the prefill).  NULL disables the capture.  Call before q3_prefill. */
int q3_set_hidden_capture(q3_engine* e, void* hid_dev, int32_t stride);

/* Test hooks (used by tests/ only): teacher forcing and raw-logit capture.
 * forced: int32 [B][n_frames][G] device (or NULL to disable); talker_logits: fp32 [n_frames+1][B][V];
 * cp_logits: fp32 [n_frames][G-1][B][Vc].  Pointers must stay valid until cleared. */
int q3_set_debug(q3_engine* e, const int32_t* forced_dev, int32_t n_frames, float* talker_logits_dev,
                 float* cp_logits_dev);

/* Profiling hooks (tools/critical_path.py, tools/profile_frame.py): prof_dev = uint64 [n_phases][grid][8] %globaltimer
 * ns written by thread 0 of EVERY CTA during the first frame of each q3_decode: [0] phase body end, [1] barrier passed,
 * [2..5] inner marks of the phase body, [6] phase start, [7] staging mark; q3_describe_frame_program returns -n_phases
 * and fills kinds[i] = type*100 + stack*10 + epilogue. */
int q3_set_profile(q3_engine* e, unsigned long long* prof_dev);
int q3_describe_frame_program(q3_engine* e, int32_t* kinds, int32_t capacity);
/* time `count` repetitions of frame-program phases [first, first+span) as one launch (instruction-cache probe) */
int q3_debug_set_skip(q3_engine* e, int32_t mask); /* ablation bits for tools/ablate_phase.py; 0 = normal */
int q3_debug_time_phases(q3_engine* e, int32_t first, int32_t span, int32_t count, float* ms_out, void* stream);

/* Bytes the fused frame-step kernel must stream per step for batch B at mean context S
 * (SURVEY §8d: W_talker + W_cp_unique + B*(S+1)*KV_tok), and the no-residency figure. */
int q3_algorithmic_bytes(q3_engine* e, int32_t B, int32_t S, double* a_bytes, double* a_stream_bytes);

/* ---------------------------------------------------------------- codec decoder (seam C) */
/* Mirrors Qwen3TTSTokenizerV2DecoderConfig (core/tokenizer_12hz/configuration_qwen3_tts_tokenizer_v2.py:72-93). */
typedef struct {
  int32_t codebook_size, codebook_dim, hidden_size, latent_dim;
  int32_t num_heads, num_kv_heads, head_dim, sliding_window, intermediate_size, num_layers, num_quantizers;
  int32_t n_upsample_rates;    int32_t upsample_rates[8];    /* (8,5,4,3) */
  int32_t n_upsampling_ratios; int32_t upsampling_ratios[8]; /* (2,2)     */
  int32_t decoder_dim;
  float rms_eps, rope_theta;
  int32_t max_frames;  /* per forward (chunk_size + left_context = 325 in the reference) */
  int32_t max_batch;
  int32_t device;
} q3_codec_cfg;

int q3_codec_create(const q3_codec_cfg* cfg, q3_codec** out);
void q3_codec_destroy(q3_codec* c);
/* Engine-native tensors, converted from the reference decoder's state_dict by the host
 * (qwen3-tts_b200/codec.py documents every name; INTEGRATION.md lists the mapping).  GEMM weights are bf16
 * [N][ntaps*Kp] (K-major per tap, Kp = K rounded up to 64; Conv1d taps in kernel order, ConvTranspose1d as
 * N = stride*Cout with 2 taps), biases / SnakeBeta / LayerScale / LayerNorm parameters fp32.  dtype is implied
 * by the name (".w", ".table", ".proj", ".norm", ".ln1", ".ln2", ".cos", ".sin" = bf16; the rest fp32). */
int q3_codec_load_tensor(q3_codec* c, const char* name, const void* dev, const int64_t* shape, int32_t ndim);
int q3_codec_finalize(q3_codec* c);
/* One full causal forward == Qwen3TTSTokenizerV2Decoder.forward (…v2.py:869-884).
 * codes: int32 [B][K][T] device; wav: fp32 [B][T*upsample] device.  Asynchronous. */
int q3_codec_forward(q3_codec* c, const int32_t* codes_dev, int32_t B, int32_t T, float* wav_dev, void* stream);

/* ---- stateful streaming decoder (SURVEY §8b / §8f-2).  The reference decodes whole utterances, or chunks with 25
 * re-decoded frames of left context (chunked_decode, tokenizer_12hz/modeling_qwen3_tts_tokenizer_v2.py:886-896); this
 * handle carries the decoder's causal state instead (conv tails, ConvTranspose overlap row, 71 frames of rotated K/V
 * per transformer layer), so pushing packets of any sizes yields exactly the waveform of the full causal forward
 * (…v2.py:869-884) over everything pushed, with only the NEW frames' work per packet.
 * open: B rows, packets of <= max_packet_frames frames.  step: codes_dev int32 [B][num_quantizers][n] (the next n
 * frames of every row) -> wav_dev fp32 [B][n * total_upsample]; asynchronous on `stream`.  reset: start new
 * utterances in all rows.  The position (frames pushed) must stay below the engine's max_frames (RoPE table). */
typedef struct q3_codec_stream q3_codec_stream;
int q3_codec_stream_open(q3_codec* c, int32_t B, int32_t max_packet_frames, q3_codec_stream** out);
int q3_codec_stream_step(q3_codec_stream* s, const int32_t* codes_dev, int32_t n, float* wav_dev, void* stream);
int q3_codec_stream_reset(q3_codec_stream* s, void* stream);
int q3_codec_stream_position(q3_codec_stream* s);
void q3_codec_stream_close(q3_codec_stream* s);
int q3_codec_total_upsample(q3_codec* c);
/* kernels launched by the last q3_codec_forward (bench.py's gpu_launches bookkeeping) */
int q3_codec_last_launch_count(q3_codec* c);
/* Test hook (tests/ only): per-stage capture of the DECODER, so that an error in one small kernel cannot hide behind the
 * waveform SNR.  The following q3_codec_forward calls copy the bf16 [B][T_stage][C_stage] tensor of `stage` into dst_dev
 * (at most `capacity` elements): 0 pre_conv output (…v2.py:874), 1 pre-transformer output (:875-876), 2 output of the
 * upsample stack (:878-880), 3 SnakeBeta(decoder.0 output) as fed to block 0 (:857,:646), 4+i output of decoder block i
 * (:638-658).  stage < 0 clears all captures. */
int q3_codec_debug_capture(q3_codec* c, int32_t stage, void* dst_dev, int64_t capacity);

/* Test hook (tests/ only): one launch of the tcgen05 tap-GEMM that runs every codec Conv1d / ConvTranspose1d / Linear,
 * the talker prefill GEMMs and the code-predictor projection table, planned exactly as those callers plan it:
 *   C[b][m][n] = epilogue( sum_tap sum_k A[b][m + shifts[tap] + a_row0][k] * W[n][tap*Kp + k] ),
 * rows outside [0, a_rows) reading as zero.  A: bf16 [B] rows of a_bs elements, each holding a_rows rows of K (row
 * pitch K); W: bf16 [N][ntaps*Kp].  bn = 0 takes the production tile width (gemm_pick_bn); a_rows = 0 means T; batch
 * strides of 0 mean contiguous [B][T][N] ([B][T][N/2] for the gated activations); cmod = 0 means N; max_ctas = 0 runs
 * one CTA per SM.  act: 0 none, 1 SnakeBeta, 2 GELU, 3 SwiGLU (gate, up) column pairs, 4 SwiGLU blocks of 8 gate | 8 up.
 * bias / scale / snake_ea (exp(alpha)) / snake_ib (1/(exp(beta)+1e-9)) are fp32 [cmod]; resid / out_raw / out_act
 * bf16.  An invalid descriptor is refused with a message before anything is enqueued. */
typedef struct {
  const void* a;
  int32_t B, T, K, a_rows, a_row0;
  int64_t a_bs;
  const void* w;
  int32_t N, Kp, ntaps, shifts[8];
  int32_t bn, act, cmod;
  const float *bias, *scale, *snake_ea, *snake_ib;
  const void* resid;
  int64_t resid_bs;
  void* out_raw;
  int64_t raw_bs;
  void* out_act;
  int64_t act_bs;
  int32_t max_ctas;
} q3_tap_gemm_desc;
int q3_debug_tap_gemm(const q3_tap_gemm_desc* d, void* stream);

/* ---------------------------------------------------------------- codec ENCODER (Qwen3TTSTokenizer.encode)
 * Replaces Qwen3TTSTokenizerV2Model.encode (core/tokenizer_12hz/modeling_qwen3_tts_tokenizer_v2.py:961-991), i.e.
 * transformers MimiModel._encode_frame (modeling_mimi.py:1455-1488), restricted to the first
 * `encoder_valid_num_quantizers` levels (the reference computes 32 and keeps 16, :981-983).  fp32 end to end:
 * the output is discrete (nearest-centroid indices), see csrc/codec_encoder.cu. */
typedef struct {
  int32_t num_filters, kernel_size, last_kernel_size, residual_kernel_size, compress; /* MimiConfig SEANet fields */
  int32_t n_ratios, ratios[8];        /* downsampling strides in encoder order = reversed(upsampling_ratios): 4,5,6,8 */
  int32_t hidden_size, num_layers, num_heads, head_dim, intermediate_size, sliding_window;
  float norm_eps;
  int32_t codebook_size, codebook_dim;
  int32_t num_semantic_quantizers;    /* 1 */
  int32_t num_quantizers;             /* levels to compute = encoder_valid_num_quantizers (16) */
  int32_t downsample_stride;          /* encodec_frame_rate / frame_rate = 2 */
  int32_t max_frames;                 /* rows of the RoPE tables (transformer frames, 25 Hz) */
  int32_t device;
} q3_codec_enc_cfg;
typedef struct q3_codec_enc q3_codec_enc;

int q3_codec_enc_create(const q3_codec_enc_cfg* cfg, q3_codec_enc** out);
void q3_codec_enc_destroy(q3_codec_enc* e);
/* fp32 device tensors, engine-native names (qwen3-tts_b200/codec_encoder.py::_load maps MimiModel's state_dict):
 *   "enc.conv0|enc.res<i>.a|enc.res<i>.b|enc.down<i>|enc.conv_last" + ".w" [Cout][Cin][k] / ".b" [Cout];
 *   "tr.<l>.ln1.w/.b", "tr.<l>.qkv.w" [3C][C] = cat(q,k,v), "tr.<l>.o.w", "tr.<l>.ls1", "tr.<l>.ln2.w/.b",
 *   "tr.<l>.fc1.w" [I][C], "tr.<l>.fc2.w" [C][I], "tr.<l>.ls2"; "rope.cos|sin" [max_frames][head_dim/2];
 *   "down.w" [C][C][2*stride]; "rvq.sem.proj.w|rvq.ac.proj.w" [D][C]; per level q (0 = semantic):
 *   "rvq.<q>.e" [K][D] = embed_sum / clamp(cluster_usage, 1e-5), "rvq.<q>.et" [D][K], "rvq.<q>.e2" [K] = |e|^2. */
int q3_codec_enc_load_tensor(q3_codec_enc* e, const char* name, const float* dev, const int64_t* shape, int32_t ndim);
int q3_codec_enc_finalize(q3_codec_enc* e);
/* wav: fp32 [B][T] device (rows right-padded with zeros: every layer is causal, so padding never reaches earlier
 * frames); codes: int32 [B][num_quantizers][q3_codec_enc_frames(T)] device.  Asynchronous. */
int q3_codec_enc_encode(q3_codec_enc* e, const float* wav_dev, int32_t B, int32_t T, int32_t* codes_dev, void* stream);
int q3_codec_enc_frames(q3_codec_enc* e, int32_t T);   /* ceil-chain through every stride */
int q3_codec_enc_hop(q3_codec_enc* e);                 /* samples per frame (1920) */
int q3_codec_enc_last_launch_count(q3_codec_enc* e);
/* Test hook: copy the activation [B][C][T] after stage `stage` (conv0, per ratio [res, down], conv_last, one per
 * transformer layer, downsample) of the next encode into dst; stage < 0 clears all captures. */
int q3_codec_enc_debug_capture(q3_codec_enc* e, int32_t stage, float* dst_dev, int64_t capacity);

/* ---------------------------------------------------------------- speaker x-vector (voice cloning)
 * Replaces Qwen3TTSForConditionalGeneration.extract_speaker_embedding (core/models/modeling_qwen3_tts.py:1941-1954):
 * mel_spectrogram (:396-448) + Qwen3TTSSpeakerEncoder.forward (:371-393).  fp32. */
typedef struct {
  int32_t mel_dim, enc_dim;                 /* Qwen3TTSSpeakerEncoderConfig (configuration_qwen3_tts.py:47-57) */
  int32_t n_blocks;                         /* len(enc_channels) */
  int32_t channels[8], kernel_sizes[8], dilations[8];
  int32_t attention_channels, res2net_scale, se_channels;
  int32_t n_fft, hop, win;                  /* 1024, 256, 1024 at the reference call site (:1943-1951) */
  int32_t device;
} q3_spk_cfg;
typedef struct q3_spk q3_spk;

int q3_spk_create(const q3_spk_cfg* cfg, q3_spk** out);
void q3_spk_destroy(q3_spk* e);
/* fp32 device tensors: the reference's own `speaker_encoder.` state_dict names with the prefix stripped
 * ("blocks.0.conv.weight", "blocks.<i>.tdnn1.conv.weight", "blocks.<i>.res2net_block.blocks.<j>.conv.weight",
 * "blocks.<i>.se_block.conv1.weight", "mfa.conv.weight", "asp.tdnn.conv.weight", "asp.conv.weight", "fc.weight", and
 * the matching ".bias"), plus the host-computed front-end tables "mel.window" [n_fft] (Hann), "mel.cos" / "mel.sin"
 * [n_fft] = cos/sin(2*pi*j/n_fft), "mel.fbT" [n_fft/2+1][mel_dim] (librosa-style Slaney filterbank, transposed). */
int q3_spk_load_tensor(q3_spk* e, const char* name, const float* dev, const int64_t* shape, int32_t ndim);
int q3_spk_finalize(q3_spk* e);
int q3_spk_frames(q3_spk* e, int32_t T);    /* STFT frames of a T-sample waveform */
/* wav fp32 [B][T] -> log-mel fp32 [B][mel_dim][frames] */
int q3_spk_mel(q3_spk* e, const float* wav_dev, int32_t B, int32_t T, float* mel_dev, void* stream);
/* wav fp32 [B][T] (or, when mel_dev != NULL, a ready mel [B][mel_dim][frames]) -> emb fp32 [B][enc_dim] */
int q3_spk_embed(q3_spk* e, const float* wav_dev, int32_t B, int32_t T, const float* mel_dev, int32_t frames,
                 float* emb_dev, void* stream);
int q3_spk_last_launch_count(q3_spk* e);

#ifdef __cplusplus
}
#endif
#endif /* QWEN3TTS_B200_H */
