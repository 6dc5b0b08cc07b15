/*
 * viettts_b200.h -- C ABI of the B200-native vietTTS hot path (libviettts_b200.so).
 *
 * The reference (NTT123/vietTTS) has no FFI: its seams for this path are three
 * Python callables.  Each entry point below names the reference interface it
 * replaces (file:line into the reference tree):
 *
 *   vietTTS/hifigan/mel2wave.py:20-41     mel2wave(mel)            -> vtts_mel2wave_host / vtts_hifigan_forward
 *   vietTTS/nat/text2mel.py:61-82         predict_mel(tok, dur)    -> vtts_predict_mel_host / vtts_acoustic_forward
 *   vietTTS/nat/dsp.py:104-128            MelFilter(...)(y)        -> vtts_melspec_host / vtts_melspec
 *   vietTTS/hifigan/mel2wave.py:35-36     pickle.load(hk_hifi)     -> vtts_load_hifigan
 *   vietTTS/nat/text2mel.py:62-71         pickle.load(acoustic)    -> vtts_load_acoustic
 *   vietTTS/nat/text2mel.py:22-34         predict_duration(tokens) -> vtts_predict_duration_host / vtts_duration_forward
 *   vietTTS/nat/text2mel.py:27-28         pickle.load(duration)    -> vtts_load_duration
 *   vietTTS/nat/gta.py:28-41              forward_fn(params, ...)  -> vtts_gta_host / vtts_acoustic_teacher_forward
 *
 * Conventions
 *   - plain C types only; no torch / CUDA types in signatures (`stream` is a
 *     cudaStream_t passed as void*, NULL = default stream).
 *   - every call returns 0 on success or a negative vtts_status; the message is
 *     available from vtts_last_error().  Nothing throws across the ABI.  There is
 *     NO CPU fallback: without a usable sm_100 device vtts_create fails.
 *   - one context per GPU; a context is not thread-safe; `*_forward` calls are
 *     stream-ordered and asynchronous, `*_host` calls copy H2D/D2H through pinned
 *     staging owned by the context and return after the result is in host memory.
 *   - "dev" pointers are device memory owned by the caller (e.g. torch tensors'
 *     data_ptr()), float32 unless stated, dense row-major in the documented shape.
 *   - tensors are NWC ([batch, time, channels]) exactly like the Haiku models.
 */
#ifndef VIETTTS_B200_H
#define VIETTTS_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

typedef struct vtts_ctx vtts_ctx;

typedef enum vtts_status {
  VTTS_OK = 0,
  VTTS_ERR_BAD_ARG = -1,
  VTTS_ERR_CUDA = -2,
  VTTS_ERR_NOT_LOADED = -3,   /* weights for this stage were not loaded */
  VTTS_ERR_NO_DEVICE = -4,    /* no CUDA device / not an sm_100 part */
  VTTS_ERR_OOM = -5,
  VTTS_ERR_NCCL = -6          /* NCCL missing or a collective failed (vtts_broadcast_weights) */
} vtts_status;

/* dropout handling for the prenet (vietTTS/nat/model.py:95-100: dropout is live at inference) */
typedef enum vtts_dropout_mode {
  VTTS_DROPOUT_OFF = 0,     /* deterministic parity mode: no mask, scale 1 */
  VTTS_DROPOUT_MASK = 1,    /* caller supplies uint8 keep-mask [B,N,2,256]; kept values are scaled by 2 */
  VTTS_DROPOUT_SEED = 2     /* keep bits drawn on device from threefry2x32(seed; b,t,layer,unit) */
} vtts_dropout_mode;

/* arithmetic of the dense conv contractions (97 % of the FLOPs):
 *   FP32    every product and sum in IEEE fp32 on the FMA pipe (conv1d.cu) -- the strict parity mode
 *   BF16X3  tcgen05 tensor cores, each fp32 operand split into bf16 hi+lo, three products
 *           (hi*hi + hi*lo + lo*hi) accumulated in fp32 in TMEM (tc_conv.cu); fp32-class accuracy
 *           (waveform L-inf 2e-5 vs float64), no reduced-precision storage anywhere. */
typedef enum vtts_precision { VTTS_PRECISION_FP32 = 0, VTTS_PRECISION_BF16X3 = 1 } vtts_precision;

/* ---- library / context ------------------------------------------------------------ */
int vtts_version(void);                                  /* ABI version, currently 1 */
int vtts_create(int device, vtts_ctx** out);
int vtts_destroy(vtts_ctx* ctx);
const char* vtts_last_error(vtts_ctx* ctx);              /* ctx may be NULL: last error of failed create */
int vtts_device_info(vtts_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, int64_t* hbm_bytes);
int vtts_set_precision(vtts_ctx* ctx, int mode);          /* vtts_precision; applies to later forward calls */
int vtts_get_precision(vtts_ctx* ctx);

/* ---- weights --------------------------------------------------------------------------
 * A "blob" is the float32 concatenation of the Haiku-layout tensors in the canonical order
 * listed in INTEGRATION.md (viettts_b200/weights.py builds it from the unchanged pickles).
 * `blob` may be a host or a device pointer (detected); device blobs let rank != 0 load
 * weights received by an NCCL broadcast without a host round trip. */
int64_t vtts_hifigan_blob_floats(void);                  /* 13 926 017 */
int64_t vtts_acoustic_blob_floats(void);                 /* params + BatchNorm eval statistics */
int64_t vtts_duration_blob_floats(void);                 /* TokenEncoder block of the acoustic blob + projection head */
int vtts_load_hifigan(vtts_ctx* ctx, const float* blob, int64_t n_floats);
int vtts_load_acoustic(vtts_ctx* ctx, const float* blob, int64_t n_floats);
int vtts_load_duration(vtts_ctx* ctx, const float* blob, int64_t n_floats);
/* The one collective of the path (SURVEY.md 8e): rank `root` has loaded its weights (vtts_load_*), every other rank
 * receives the same models -- whichever of hifigan / acoustic / duration the root holds -- by ONE grouped ncclBroadcast
 * of the device arenas and derives its packed tensor-core copies locally; no host round trip, nothing on the hot path
 * afterwards.  `nccl_comm` is an ncclComm_t (passed as void*) whose rank on this process's device matches ctx; `is_root`
 * != 0 on the root rank; `stream` a cudaStream_t or NULL.  Replaces the per-process pickle.load of the reference
 * (hifigan/mel2wave.py:35-36, nat/text2mel.py:62-71) on ranks != root.  NCCL is bound with dlopen at the first call
 * (libnccl.so.2 already in the process, else the loader path, else $VTTS_NCCL_LIB); VTTS_ERR_NCCL if that fails. */
int vtts_broadcast_weights(vtts_ctx* ctx, void* nccl_comm, int root, int is_root, void* stream);
/* librosa-style filterbank [80][513] (MelFilter.__init__, dsp.py:107-113) */
int vtts_load_mel_filterbank(vtts_ctx* ctx, const float* fb, int n_mels, int n_bins);

/* ---- device-pointer, stream-ordered entry points ---------------------------------------- */

/* Generator.__call__ (vietTTS/hifigan/model.py:109-125).
 * mel_dev [B,T,80]; n_frames_dev int32 [B] or NULL (= T for every row; rows are zero-padded
 * at their true end, SURVEY H4); wav_dev [B,256*T] (samples past 256*n_frames[b] are 0). */
int vtts_hifigan_forward(vtts_ctx* ctx, const float* mel_dev, const int32_t* n_frames_dev,
                         int B, int T, float* wav_dev, void* stream);

/* AcousticModel.inference (vietTTS/nat/model.py:123-144).
 * tokens_dev int32 [B,L]; lengths_dev int32 [B] or NULL (= L); dur_frames_dev [B,L] durations in
 * FRAMES (seconds*62.5); n_frames_dev int32 [B] or NULL (= N); keep_mask_dev uint8 [B,N,2,256]
 * (mode MASK) or NULL; mel_dev [B,N,80] (rows past n_frames[b] are 0).
 * Row b equals the reference run on row b alone (batch semantics the reference lacks). */
int vtts_acoustic_forward(vtts_ctx* ctx, const int32_t* tokens_dev, const int32_t* lengths_dev,
                          const float* dur_frames_dev, const int32_t* n_frames_dev,
                          const uint8_t* keep_mask_dev, int dropout_mode, uint64_t seed,
                          int B, int L, int N, float* mel_dev, void* stream);

/* AcousticModel.__call__ (vietTTS/nat/model.py:146-169) with is_training=False, the teacher-forced pass gta.py:24-25 runs:
 * mels_in_dev [B,N,80] is the ground-truth mel ALREADY shifted by one frame (gta.py:34-36).  keep_mask_dev uint8
 * [B,N,2,256] prenet keep-masks (kept values x2); zone_mask_dev uint8 [B,N,4,512] zoneout masks in state order
 * (h0, c0, h1, c1), 1 = keep the previous state (Bernoulli(0.1) in the reference, model.py:161-164); mode SEED draws
 * both on the device, OFF disables both.  mel1 = projection output (may be NULL), mel2 = mel1 + postnet(mel1). */
int vtts_acoustic_teacher_forward(vtts_ctx* ctx, const int32_t* tokens_dev, const int32_t* lengths_dev,
                                  const float* dur_frames_dev, const int32_t* n_frames_dev, const float* mels_in_dev,
                                  const uint8_t* keep_mask_dev, const uint8_t* zone_mask_dev, int dropout_mode, uint64_t seed,
                                  int B, int L, int N, float* mel1_dev_or_null, float* mel2_dev, void* stream);

/* DurationModel.__call__ (vietTTS/nat/model.py:64-70, is_training=False): TokenEncoder -> Linear(256) -> gelu(tanh
 * form, the jax default) -> Linear(1) -> softplus.  tokens_dev int32 [B,L]; lengths_dev int32 [B] or NULL (= L);
 * dur_sec_dev [B,L] predicted durations in SECONDS (0 past lengths[b]).  Row b equals the reference run on row b alone.
 * The silence clip / word-end zeroing of text2mel (text2mel.py:88-97) is host logic (viettts_b200/nat/text2mel.py). */
int vtts_duration_forward(vtts_ctx* ctx, const int32_t* tokens_dev, const int32_t* lengths_dev, int B, int L,
                          float* dur_sec_dev, void* stream);

/* MelFilter.__call__ (vietTTS/nat/dsp.py:115-128). wav_dev [B,S], S % 256 == 0, S >= 512;
 * mel_dev [B,S/256,80]. */
int vtts_melspec(vtts_ctx* ctx, const float* wav_dev, int B, int S, float* mel_dev, void* stream);

/* optional taps for tests: copy an internal activation of the LAST forward call to host.
 * name: "enc" [B,L,512] (of the last acoustic OR duration call), "cond" [B,N,512], "mel_pre" [B,N,80] (before the postnet). */
int vtts_debug_read(vtts_ctx* ctx, const char* name, float* host_out, int64_t n_floats);

/* test hook: one conv launch of the models, run the way the models run it.  `geom` is the geometry every problem
 * shares, `probs` 1..8 problems; all pointers are device memory.
 *   input   x0 (and x1, x2 for pre_mode 2) [B][T_rows][Cin]; pre_mode 0 none, 1 leaky_relu(pre_slope),
 *           2 leaky_relu(pre_slope) of (x0+x1+x2)/3
 *   weights w Haiku layout [k][Cin][Cout], bias [Cout]; bn_mean / bn_inv / bn_off [Cout] all three or none:
 *           y = (y - mean) * inv + off after the bias
 *   output  post_act 0 none, 1 tanh, 2 relu after the BatchNorm, then + resid; out / resid [B][rows_out][Cout]
 *   rows    output index tau reads input rows tau + j*dil + in_off (tap j, zero outside [0, valid_b)) and writes
 *           output row tau*out_stride + out_off, for tau < valid_b = min(len[b]*len_mul, T_rows) (len NULL: T_rows).
 *           Nothing else is written: output rows of tau >= valid_b keep their contents in both precisions.
 * precision FP32: the strict fp32 conv (conv1d.cu).  BF16X3: every w packed by the loader's packer into N tiles of
 * the width the models use, then the tensor-core dispatcher (tile width, partial last tile, epilogue form,
 * launches of at most 8 tile problems).  Malformed descriptors (nprob outside 1..8, Cin % 16, Cout % 4, a partial
 * BatchNorm triple, ...) return VTTS_ERR_BAD_ARG.  Synchronous. */
typedef struct vtts_conv_geometry {
  int32_t B, T_rows, rows_out, Cin, Cout;
  const int32_t* len;
  int32_t len_mul, pre_mode;
  float pre_slope;
  int32_t post_act;
} vtts_conv_geometry;
typedef struct vtts_conv_problem {
  const float *x0, *x1, *x2;
  const float* w;
  const float* bias;
  const float* resid;
  const float *bn_mean, *bn_inv, *bn_off;
  float* out;
  int32_t k, dil, in_off, out_stride, out_off;
} vtts_conv_problem;
int vtts_debug_conv(vtts_ctx* ctx, int precision, const vtts_conv_geometry* geom, const vtts_conv_problem* probs, int nprob);

/* test hook: one up-sampling stage of the generator, leaky_relu(0.1) -> hk.Conv1DTranspose(C/2, K, stride u, SAME)
 * (vietTTS/hifigan/model.py:112-114), through the generator's own weight preparation and launch code.
 * x0 [B][T][C]; x1, x2 NULL (stage 0: the input is x0) or both set (stages 1-3: the input is (x0+x1+x2)/3);
 * w Haiku layout [K][C/2][C]; bias [C/2]; out [B][T*u][C/2]; len int32 [B] or NULL.  Output rows t = tau*u + r are
 * written for tau < min(len[b]*len_mul, T), the others keep their contents.  (C, u, K) must be one of the generator's
 * stages: (512, 8, 16), (256, 8, 16), (128, 2, 4), (64, 2, 4).  Synchronous. */
int vtts_debug_conv_transpose(vtts_ctx* ctx, int precision, const float* x0_dev, const float* x1_dev, const float* x2_dev,
                              const float* w_dev, const float* bias_dev, const int32_t* len_dev, int len_mul, int B, int T,
                              int C, int u, int K, float* out_dev);

/* test hook: one fused ResBlock pair  out = conv2(lrelu(conv1(lrelu(x)) + b1)) + b2 + x  (vietTTS/hifigan/model.py:44-51)
 * on the tensor-core path; x/out [B,T,C] with C in {32,64}, w1/w2 Haiku layout [k,C,C], conv1 dilation `dil`. Synchronous. */
int vtts_debug_pair(vtts_ctx* ctx, const float* x_dev, const float* w1_dev, const float* b1_dev, const float* w2_dev,
                    const float* b2_dev, const int32_t* len_dev, int B, int T, int C, int k, int dil, float slope, float* out_dev);

/* profiling aid: per-CTA stall counters (SM clocks) of the LAST tensor-core conv launch.
 * Row = CTA, columns: 0 MMA-role total, 1 MMA wait accumulator-free, 2 MMA wait activations, 3 MMA wait
 * weights, 4 weight-producer wait slot, 5 converter wait slot, 6 converter fill, 7 epilogue wait
 * accumulator, 8 epilogue drain.  enable!=0 turns collection on for later launches; the call
 * synchronises, copies (if host_out != NULL) and clears the counters. */
int vtts_debug_tc_stats(vtts_ctx* ctx, int enable, int64_t* host_out_256x16);

/* profiling aid: per-kernel-group times of the LAST forward calls.  enable != 0 switches the event recording on for later
 * calls.  ms_out24 (may be NULL) receives, for every id with both marks recorded, the elapsed ms since the previous
 * id of the same group (0 otherwise); the call synchronises the device.  ids:
 *   acoustic: 1 TokenEncoder, 2 upsample, 3 hoisted cond GEMMs, 4 decoder scan, 5 output projection, 6 postnet
 *   hifigan:  9 conv_pre, 10..13 up-sampling stage 0..3 (ConvTranspose + three ResBlocks), 14 conv_post
 *   teacher-forced pass: 17 encoder + upsample, 18 prenet + hoisted GEMMs, 19 zoneout scan, 20 projection + postnet */
int vtts_debug_substages(vtts_ctx* ctx, int enable, float* ms_out24);

/* ---- host-buffer entry points (what a ctypes / cgo / JNI binding calls) ------------------ */
int vtts_mel2wave_host(vtts_ctx* ctx, const float* mel, const int32_t* n_frames, int B, int T, float* wav);
int vtts_predict_mel_host(vtts_ctx* ctx, const int32_t* tokens, const int32_t* lengths,
                          const float* dur_frames, const int32_t* n_frames,
                          const uint8_t* keep_mask, int dropout_mode, uint64_t seed,
                          int B, int L, int N, float* mel);
int vtts_predict_duration_host(vtts_ctx* ctx, const int32_t* tokens, const int32_t* lengths, int B, int L, float* dur_sec);
/* predict_mel -> mel2wave without leaving the device: tokens/durations in, waveform out */
int vtts_synthesize_host(vtts_ctx* ctx, const int32_t* tokens, const int32_t* lengths,
                         const float* dur_frames, const int32_t* n_frames,
                         const uint8_t* keep_mask, int dropout_mode, uint64_t seed,
                         int B, int L, int N, float* mel_out_or_null, float* wav);
/* text2mel (vietTTS/nat/text2mel.py:85-103) + mel2wave (synthesizer.py:36-37) for a batch of token rows in one call:
 * predicted durations -> silence tokens clipped from below at silence_duration, word-end tokens 0 s -> frames ->
 * AcousticModel.inference -> trailing-silence frames cut -> Generator.
 * tokens int32 [B,L]; lengths int32 [B] or NULL; dropout_mode OFF or SEED.  Outputs: dur_sec_out [B,L] adjusted
 * durations in seconds (may be NULL); n_frames_out int32 [B] frames of each row's waveform; *n_max_out = row pitch in
 * frames; wav = dense [B][256 * n_max] (samples past 256*n_frames_out[b] are 0), capacity B*256*max_frames floats.
 * If n_max > max_frames nothing is synthesized: the call fails with VTTS_ERR_BAD_ARG after setting *n_max_out and
 * n_frames_out, so the caller can retry with a buffer of that size. */
int vtts_tts_host(vtts_ctx* ctx, const int32_t* tokens, const int32_t* lengths, int B, int L, float silence_duration,
                  int dropout_mode, uint64_t seed, int max_frames, float* dur_sec_out, int32_t* n_frames_out,
                  int32_t* n_max_out, float* wav);
int vtts_melspec_host(vtts_ctx* ctx, const float* wav, int B, int S, float* mel);
/* forward_fn_ of vietTTS/nat/gta.py:28-41 (ground-truth-aligned mels for vocoder fine-tuning): wav_i16 int16 [B,S]
 * (S % 256 == 0) -> /2^15 -> MelFilter -> shift by one frame -> teacher-forced acoustic model -> mel2_out [B,S/256,80].
 * wav_lengths int32 [B] samples or NULL (= S): frames past wav_lengths[b]/256 are 0 (gta.py:74-75 slices them away);
 * dur_sec [B,L] aligned phoneme durations in seconds; masks as in vtts_acoustic_teacher_forward;
 * mel_gt_out_or_null [B,S/256,80] receives the MelFilter output.  Needs vtts_load_acoustic + vtts_load_mel_filterbank. */
int vtts_gta_host(vtts_ctx* ctx, const int16_t* wav_i16, const int32_t* wav_lengths, const int32_t* tokens,
                  const int32_t* lengths, const float* dur_sec, const uint8_t* keep_mask, const uint8_t* zone_mask,
                  int dropout_mode, uint64_t seed, int B, int L, int S, float* mel_gt_out_or_null, float* mel2_out);

/* ---- introspection for bench / tests ------------------------------------------------------ */
/* number of kernel launches issued by this context since creation (our kernels only) */
int64_t vtts_launch_count(vtts_ctx* ctx);
/* elapsed ms of the last forward call of the given stage, measured with CUDA events on the
 * stream the kernels were launched on: stage 0 = hifigan, 1 = acoustic, 2 = melspec, 3 = duration.
 * Synchronises the stream. */
int vtts_last_stage_ms(vtts_ctx* ctx, int stage, float* ms);

#ifdef __cplusplus
}
#endif
#endif /* VIETTTS_B200_H */
