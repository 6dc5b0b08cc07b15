// Internal declarations shared by the translation units of libviettts_b200.so.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>
#include <string.h>
#include <string>
#include <vector>

#include "../../include/viettts_b200.h"

// ---- model constants (vietTTS/nat/config.py:8-59, assets/hifigan/config.json:2-28) ----------
namespace vc {
constexpr int MEL = 80;
constexpr int HOP = 256;
constexpr int NFFT = 1024;
constexpr int NBINS = 513;
constexpr int ENC_D = 256;        // acoustic_encoder_dim
constexpr int ENC_OUT = 512;      // BiLSTM concat
constexpr int DEC_H = 512;        // acoustic_decoder_dim
constexpr int PRENET = 256;
constexpr int POSTNET = 512;
constexpr int VOCAB = 256;
constexpr int SIL_INDEX = 0;      // nat/config.py:26 special_phonemes.index("sil")
constexpr int WORD_END_INDEX = 3; // nat/config.py:28 special_phonemes.index(" ")
constexpr int HG_C0 = 512;        // upsample_initial_channel
constexpr int HG_NSTAGE = 4;
__host__ __device__ constexpr int hg_rate(int i) { return i < 2 ? 8 : 2; }
__host__ __device__ constexpr int hg_upk(int i) { return i < 2 ? 16 : 4; }
__host__ __device__ constexpr int hg_rbk(int j) { return j == 0 ? 3 : (j == 1 ? 7 : 11); }
__host__ __device__ constexpr int hg_dil(int m) { return m == 0 ? 1 : (m == 1 ? 3 : 5); }
}  // namespace vc

#define VTTS_CUDA(expr)                                                                          \
  do {                                                                                           \
    cudaError_t _e = (expr);                                                                     \
    if (_e != cudaSuccess) {                                                                     \
      return ctx->fail(VTTS_ERR_CUDA, "%s:%d %s -> %s", __FILE__, __LINE__, #expr,               \
                       cudaGetErrorString(_e));                                                  \
    }                                                                                            \
  } while (0)

// ---- generic NWC conv problem description (conv1d.cu) ----------------------------------------
struct ConvProb {
  const float* x0;       // input  [B][rows_in][Cin]
  const float* x1;       // extra inputs for pre_mode 2 (sum of three / 3), else null
  const float* x2;
  const float* w;        // [k][Cin][Cout]
  const float* bias;     // [Cout]
  const float* resid;    // [B][rows_out][Cout] or null, added after the activation
  const float* bn_mean;  // eval BatchNorm (all four or none): y = (y-mean)*inv + off
  const float* bn_inv;   //   inv = scale*rsqrt(var+1e-5) precomputed at load
  const float* bn_off;
  float* out;            // [B][rows_out][Cout]
  int k, dil, in_off;    // input row of tap j for output index tau: tau + j*dil + in_off
  int out_stride, out_off;  // output row = tau*out_stride + out_off (transposed-conv phases)
};

struct ConvLaunch {
  ConvProb p[8];
  int nprob;
  int Cin, Cout;
  int B;
  int T_rows;         // tau range per batch row (== allocated input rows)
  int rows_out;       // allocated output rows per batch row
  const int* len;     // int32 [B] or null
  int len_mul;        // valid tau < len[b]*len_mul (clamped to T_rows)
  int pre_mode;       // 0 none, 1 leaky_relu(pre_slope), 2 (x0+x1+x2)/3 then leaky_relu(pre_slope)
  float pre_slope;
  int post_act;       // 0 none, 1 tanh, 2 relu
};

// ---- tensor-core conv (tc_conv.cu) ----------------------------------------------------------------
struct TcProb {
  const float* x0;
  const float* x1;
  const float* x2;
  const void* wpk;       // packed bf16 hi/lo weights (vtts_tc_pack_weights)
  const float* bias;     // [N]
  const float* resid;    // rows_out x out_ld or null
  const float* bn_mean;  // eval BatchNorm (all three or none), applied after the bias
  const float* bn_inv;
  const float* bn_off;
  float* out;
  int k, dil, in_off, out_stride, out_off;
  // multi-phase tiles (TcLaunch::nphase > 1): phase ph of this problem uses weights wpk_ph[ph], reads input rows
  // shifted by in_off_ph[ph] and writes output rows tau*out_stride + out_off_ph[ph]; one converted activation
  // tile feeds all phases (ConvTranspose output phases share their input)
  const void* wpk_ph[4];
  int in_off_ph[4];
  int out_off_ph[4];
};

struct TcLaunch {
  TcProb p[8];
  int nprob;
  int Cin, N;            // N = output channels of this launch (32/64/128/256)
  int in_ld, out_ld;     // row strides in floats
  int B, T_rows, rows_out;
  const int* len;
  int len_mul;
  int pre_mode;
  float pre_slope;
  int nphase;            // phases per tile (1, 2 or 4); 0 means 1
  int post_act;          // 0 none, 1 tanh, 2 relu (after BN, before the residual)
  int n_valid;           // real output channels of this N tile (<= N); 0 means N
  int tiles_per_row, ntiles;  // filled by the launcher
  int problem_major;          // tile -> problem map.  0 (default): round robin (problem = tile % nprob): row tile r of every problem
                              // is in flight at the same time, so an input / residual tensor the problems SHARE (the first pair
                              // of every ResBlock stage, the ConvTranspose phases) is read from DRAM once and served from L2 to
                              // the others: generator 19.8 -> 19.1 ms.  1: problems back to back (experiments only)
  int* err;                   // device int: set before trapping on a barrier timeout
  long long* dbg;             // optional [grid][16] per-role stall counters (vtts_debug_tc_stats)
  int exp;                    // experiment bits of the CTA-pair form (VTTS_PAIR_EXP; 0 in production): 1 = the issuer polls with
                              // test_wait instead of try_wait, 4 = cluster-scope release on the weight forwarder's arrive (slow)
};

// ---- fused ResBlock pair (tc_pair.cu): out = conv2(lrelu(conv1(lrelu(x)) + b1)) + b2 + x, C = N channels ----
struct TcPairProb {
  const float* x;        // [B][T_rows][N] input and residual
  const void* w1pk;      // packed bf16 hi/lo weights of the dilated conv (vtts_tc_pack_weights)
  const void* w2pk;      // ... of the dilation-1 conv
  const float* b1;
  const float* b2;
  float* out;            // [B][T_rows][N], must differ from x
  int k, dil;
  const void* w1pc;      // the same weights in the CTA-pair layout (vtts_tc_pack_weights_pc) or null
  const void* w2pc;
};

struct TcPairLaunch {
  TcPairProb p[3];
  int nprob;
  int N;
  int B, T_rows;
  const int* len;
  int len_mul;
  float slope;
  int tile_start[3], tiles_per_row[3], ntiles;   // filled by the launcher
  int* err;
  long long* dbg;
};

struct vtts_ctx {
  int device = 0;
  int precision = 1;            // 0 = strict fp32 (FMA pipe), 1 = bf16x3 on tcgen05 tensor cores (default)
  int* d_err = nullptr;
  long long* d_tc_dbg = nullptr;   // [256][16] profiling counters of the last tensor-core conv launch
  bool tc_dbg_on = false;
  int fuse_pairs = 1;              // 1 = ResBlock pairs with C <= 64 run in a fused pair kernel (intermediate stays on chip: 8 instead of 20 B of HBM traffic per element pair)
  int pair_ts = 2;                 // fused pair kernel: 0 tc_pair.cu (one issuer, smem operand), 1 tc_pair_ts.cu (operand in TMEM), 2 tc_pair2.cu (two decoupled pipelines, smem operand),
                                   // 3 tc_pair2.cu in the CTA-pair form (cta_group::2 over clusters of two SMs)
  int tc_variant = 3;              // tile-shape variant of the tensor-core conv (see TcCfg): 3 = CTA pairs (cta_group::2) for N >= 128 (default), 1 = single-CTA form, 0 / 2 = older experiments
  void* hg_wpk = nullptr;       // packed tensor-core weights of the 72 resblock convs
  std::vector<void*> hg_wpk_t;
  std::vector<void*> hg_wpc_t;     // CTA-pair layout of the C <= 64 resblock convs (null for the others)
  std::vector<void*> hg_wpk_ups;   // [stage][phase] packed transposed-conv phase weights
  void* hg_wpk_pre[2] = {nullptr, nullptr};  // conv_pre, two N=256 output tiles
  int sm_count = 0;
  int cc_major = 0, cc_minor = 0;
  size_t hbm_bytes = 0;
  std::string err;
  int64_t launches = 0;
  cudaStream_t own_stream = nullptr;   // used by the *_host entry points

  // ---- weights (device) ----
  float* hg_blob = nullptr;     // haiku-layout tensors, each 256B aligned inside the arena
  std::vector<float*> hg_t;     // tensor pointers in canonical order
  float* hg_upsw = nullptr;     // transposed-conv weights repacked per output phase
  bool hg_loaded = false;

  float* ac_blob = nullptr;
  std::vector<float*> ac_t;
  void* ac_wpk = nullptr;       // packed tensor-core weights of the acoustic model's convs / hoisted GEMMs
  std::vector<void*> ac_wpk_t;
  float* ac_derived = nullptr;  // bn inv, repacked recurrent weights, ...
  std::vector<float*> ac_d;
  bool ac_loaded = false;

  float* du_blob = nullptr;     // duration model (TokenEncoder + projection head), same layout rules as ac_*
  std::vector<float*> du_t;
  void* du_wpk = nullptr;
  std::vector<void*> du_wpk_t;
  float* du_derived = nullptr;
  std::vector<float*> du_d;
  bool du_loaded = false;

  // mel filterbank + fft tables
  float* mel_fb = nullptr;      // dense [80][513]
  int* mel_lo = nullptr;        // [80] first non-zero bin
  int* mel_hi = nullptr;        // [80] one past last non-zero bin
  float* fft_tw = nullptr;      // [1024][2] cos/sin(-2 pi k/1024)
  float* hann = nullptr;        // [1024]
  bool mel_loaded = false;

  // ---- workspace (device), grown on demand ----
  void* ws = nullptr;
  size_t ws_bytes = 0;
  // pinned host staging + device staging for *_host calls
  void* hpin = nullptr;
  size_t hpin_bytes = 0;
  void* dstage = nullptr;
  size_t dstage_bytes = 0;

  // taps of the last acoustic forward (point into ws)
  float* tap_enc = nullptr; int64_t tap_enc_n = 0;
  float* tap_cond = nullptr; int64_t tap_cond_n = 0;
  float* tap_melpre = nullptr; int64_t tap_melpre_n = 0;

  static constexpr int NSTAGE = 4;   // 0 hifigan, 1 acoustic, 2 melspec, 3 duration
  cudaEvent_t ev0[NSTAGE] = {nullptr, nullptr, nullptr, nullptr};
  cudaEvent_t ev1[NSTAGE] = {nullptr, nullptr, nullptr, nullptr};
  cudaStream_t ev_stream[NSTAGE] = {nullptr, nullptr, nullptr, nullptr};
  bool ev_valid[NSTAGE] = {false, false, false, false};

  // optional sub-stage timers (vtts_debug_substages): CUDA events recorded between the kernels of a forward call.
  // ids: acoustic 0 start | 1 encoder | 2 upsample | 3 hoisted cond GEMMs | 4 decoder scan | 5 projection | 6 postnet
  //      hifigan  8 start | 9 conv_pre | 10..13 stage 0..3 (ConvTranspose + 3 ResBlocks) | 14 conv_post
  //      teacher  16 start | 17 encoder+upsample | 18 prenet+hoisted GEMMs | 19 zoneout scan | 20 projection+postnet
  static constexpr int NSUB = 24;
  bool sub_on = false;
  cudaEvent_t sub_ev[NSUB] = {};
  bool sub_set[NSUB] = {};
  void sub_mark(int id, cudaStream_t st) {
    if (!sub_on) return;
    if (!sub_ev[id]) cudaEventCreate(&sub_ev[id]);
    cudaEventRecord(sub_ev[id], st);
    sub_set[id] = true;
  }

  int fail(int code, const char* fmt, ...);
  int ensure_ws(size_t bytes);
  int ensure_staging(size_t host_bytes, size_t dev_bytes);
};

extern std::string g_vtts_create_error;

// bump allocator over the context workspace
struct Arena {
  char* base;
  size_t off = 0;
  size_t cap;
  bool measure;  // if true only compute the size
  Arena(void* b, size_t c, bool m) : base((char*)b), cap(c), measure(m) {}
  template <typename T>
  T* take(size_t n) {
    off = (off + 255) & ~size_t(255);
    T* p = measure ? nullptr : (T*)(base + off);
    off += n * sizeof(T);
    return p;
  }
};

// conv1d.cu
int vtts_launch_conv(vtts_ctx* ctx, const ConvLaunch& L, cudaStream_t st);
// tc_conv.cu
size_t vtts_tc_packed_elems(int k, int Cin, int N);
int vtts_tc_pack_weights(vtts_ctx* ctx, const float* w, void* dst, int k, int Cin, int Cout_total, int n0, int N);
int vtts_launch_tc_conv(vtts_ctx* ctx, TcLaunch& L, cudaStream_t st);
// tc_pair.cu
int vtts_launch_tc_pair(vtts_ctx* ctx, TcPairLaunch& L, cudaStream_t st);   // dispatches on ctx->pair_ts
// tc_pair_ts.cu: same operator with the A operand in tensor memory (TS form of tcgen05.mma)
int vtts_launch_tc_pair_ts(vtts_ctx* ctx, TcPairLaunch& L, cudaStream_t st);
// tc_pair2.cu: shared-memory operand, conv1 / conv2 as two decoupled pipelines with one issuing warp each
int vtts_launch_tc_pair2(vtts_ctx* ctx, TcPairLaunch& L, cudaStream_t st);
int vtts_launch_tc_pair2c(vtts_ctx* ctx, TcPairLaunch& L, cudaStream_t st);   // the same kernel in the CTA-pair form
// CTA-pair weight layout of a C x C conv for tc_pair2.cu: [chunk][rank][tap][k-half][1.5 C rows][8 bf16]
size_t vtts_tc_packed_pc_bytes(int k, int C);
int vtts_tc_pack_weights_pc(vtts_ctx* ctx, const float* w, void* dst, int k, int C);
// generic dispatch: runs `L` on the tensor-core path when ctx->precision == 1 and packed weights are given
// (wpk[prob * ntile + tile], ntile = ceil(Cout/256) tiles of width vtts_tc_tile_n(Cout)), else on the FP32 path
int vtts_tc_tile_n(int Cout);
int vtts_conv_dispatch(vtts_ctx* ctx, const ConvLaunch& L, void* const* wpk, cudaStream_t st);
// packs every N tile of one conv weight; returns the number of tiles, appends device pointers to `out`
int vtts_tc_pack_conv(vtts_ctx* ctx, const float* w, int k, int Cin, int Cout, char*& cursor, std::vector<void*>& out);
size_t vtts_tc_conv_packed_bytes(int k, int Cin, int Cout);
// hifigan.cu
int vtts_hifigan_prepare(vtts_ctx* ctx);   // derived weights after load
int vtts_hifigan_run(vtts_ctx* ctx, const float* mel, const int32_t* n_frames, int B, int T, float* wav, cudaStream_t st);
size_t vtts_hifigan_ws_bytes(int B, int T);
// one up-sampling stage (C -> C/2 channels, rate u, kernel K) of the generator; vtts_debug_conv_transpose runs the same two.
// prepare: Haiku w[K][C/2][C] -> per output phase r the two-tap conv weight upsw[r] = [2][C][C/2] (fp32 path, u*2*C*C/2
//          floats) and its packed tensor-core copy wpk[r] (vtts_tc_packed_elems(2, C, C/2) bf16 each)
// run:     lrelu(0.1)(x0), or lrelu(0.1)((x0+x1+x2)/3) when x1 != null, -> ConvTranspose as u phases: x [B][T][C] ->
//          out [B][T*u][C/2], rows tau*u + r written for tau < min(len[b]*len_mul, T); tc selects the tensor-core path
int vtts_hg_ups_prepare(vtts_ctx* ctx, const float* w, int C, int u, int K, float* upsw, void* const* wpk);
int vtts_hg_ups_run(vtts_ctx* ctx, bool tc, const float* x0, const float* x1, const float* x2, const float* upsw,
                    void* const* wpk, const float* bias, const int32_t* len, int len_mul, int B, int T, int C, int u, int K,
                    float* out, cudaStream_t st);
// nat.cu
int vtts_acoustic_prepare(vtts_ctx* ctx);
int vtts_acoustic_run(vtts_ctx* ctx, const int32_t* tokens, const int32_t* lengths, const float* dur,
                      const int32_t* n_frames, const uint8_t* keep, int mode, uint64_t seed, int B, int L, int N,
                      float* mel, cudaStream_t st, void* ws_base, size_t ws_cap, size_t* ws_need);
// melspec.cu
int vtts_melspec_prepare(vtts_ctx* ctx);
int vtts_acoustic_teacher_run(vtts_ctx* ctx, const int32_t* tokens, const int32_t* lengths, const float* dur,
                              const int32_t* n_frames, const float* mels_in, const uint8_t* keep, const uint8_t* zone, int mode,
                              uint64_t seed, int B, int L, int N, float* mel1, float* mel2, cudaStream_t st, void* ws_base,
                              size_t ws_cap, size_t* ws_need);
int vtts_duration_prepare(vtts_ctx* ctx);
// DurationModel.__call__ (model.py:64-70); dur_sec [B][L] seconds, 0 past lengths[b]
int vtts_duration_run(vtts_ctx* ctx, const int32_t* tokens, const int32_t* lengths, int B, int L, float* dur_sec,
                      cudaStream_t st, void* ws_base, size_t ws_cap, size_t* ws_need);
int vtts_melspec_run(vtts_ctx* ctx, const float* wav, int B, int S, float* mel, cudaStream_t st);

// canonical blob layouts (weights.cu)
struct TensorSpec { const char* name; int64_t n; };
const std::vector<TensorSpec>& vtts_hifigan_specs();
const std::vector<TensorSpec>& vtts_acoustic_specs();
const std::vector<TensorSpec>& vtts_duration_specs();

// indices into ctx->hg_t  (canonical order: pre, ups 0..3, resblocks 0..11 x (c1_0,c1_1,c1_2,c2_0,c2_1,c2_2), post)
namespace hgi {
constexpr int PRE_W = 0, PRE_B = 1;
__host__ __device__ constexpr int UPS_W(int i) { return 2 + 2 * i; }
__host__ __device__ constexpr int UPS_B(int i) { return 3 + 2 * i; }
// resblock n (0..11), which: 0 = convs1, 1 = convs2, m = 0..2
__host__ __device__ constexpr int RB_W(int n, int which, int m) { return 10 + n * 12 + (which * 3 + m) * 2; }
__host__ __device__ constexpr int RB_B(int n, int which, int m) { return RB_W(n, which, m) + 1; }
constexpr int POST_W = 10 + 12 * 12, POST_B = POST_W + 1;
constexpr int COUNT = POST_B + 1;
}  // namespace hgi

// indices into ctx->ac_t
namespace aci {
constexpr int EMBED = 0;
// encoder conv i: w, b, bn_scale, bn_offset, bn_mean, bn_var
__host__ __device__ constexpr int ENC_CONV(int i, int f) { return 1 + i * 6 + f; }
constexpr int ENC_LSTM_F_W = 19, ENC_LSTM_F_B = 20, ENC_LSTM_B_W = 21, ENC_LSTM_B_B = 22;
constexpr int DEC_L0_W = 23, DEC_L0_B = 24, DEC_L1_W = 25, DEC_L1_B = 26;
constexpr int PROJ_W = 27, PROJ_B = 28, PRE1_W = 29, PRE2_W = 30;
// postnet conv i (0..4): w, b [, bn_scale, bn_offset, bn_mean, bn_var for i<4]
__host__ __device__ constexpr int POST_CONV(int i, int f) { return 31 + i * 6 + f; }
constexpr int COUNT = 31 + 4 * 6 + 2;
}  // namespace aci

// indices into ctx->du_t (duration model): the TokenEncoder block has the acoustic model's layout (aci::EMBED ..
// aci::ENC_LSTM_B_B), followed by the projection head hk.Sequential([Linear(256), gelu, Linear(1)]) (model.py:60-62)
namespace dui {
constexpr int FC1_W = 23, FC1_B = 24, FC2_W = 25, FC2_B = 26;
constexpr int COUNT = 27;
}  // namespace dui
