// C ABI of libviettts_b200.so (see include/viettts_b200.h for the contract and the reference
// interfaces each entry point replaces).
#include <stdarg.h>

#include <algorithm>

#include <dlfcn.h>

#include "vtts_internal.cuh"

std::string g_vtts_create_error;

int vtts_ctx::fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  err = buf;
  return code;
}

int vtts_ctx::ensure_ws(size_t bytes) {
  vtts_ctx* ctx = this;
  if (bytes <= ws_bytes) return VTTS_OK;
  if (ws) {
    VTTS_CUDA(cudaDeviceSynchronize());
    cudaFree(ws);
    ws = nullptr;
    ws_bytes = 0;
  }
  size_t want = bytes + bytes / 8;
  cudaError_t e = cudaMalloc(&ws, want);
  if (e != cudaSuccess) {
    cudaGetLastError();
    want = bytes;
    e = cudaMalloc(&ws, want);
  }
  if (e != cudaSuccess) {
    cudaGetLastError();
    ws = nullptr;
    return fail(VTTS_ERR_OOM, "workspace of %zu bytes: %s", bytes, cudaGetErrorString(e));
  }
  ws_bytes = want;
  return VTTS_OK;
}

int vtts_ctx::ensure_staging(size_t host_bytes, size_t dev_bytes) {
  vtts_ctx* ctx = this;
  if (host_bytes > hpin_bytes) {
    if (hpin) cudaFreeHost(hpin);
    hpin = nullptr;
    hpin_bytes = 0;
    VTTS_CUDA(cudaMallocHost(&hpin, host_bytes));
    hpin_bytes = host_bytes;
  }
  if (dev_bytes > dstage_bytes) {
    if (dstage) {
      VTTS_CUDA(cudaDeviceSynchronize());
      cudaFree(dstage);
    }
    dstage = nullptr;
    dstage_bytes = 0;
    cudaError_t e = cudaMalloc(&dstage, dev_bytes);
    if (e != cudaSuccess) {
      cudaGetLastError();
      return fail(VTTS_ERR_OOM, "device staging of %zu bytes: %s", dev_bytes, cudaGetErrorString(e));
    }
    dstage_bytes = dev_bytes;
  }
  return VTTS_OK;
}

// ---- canonical blob layouts ------------------------------------------------------------------------
const std::vector<TensorSpec>& vtts_hifigan_specs() {
  static std::vector<TensorSpec> s;
  if (!s.empty()) return s;
  s.push_back({"conv_pre.w[7,80,512]", 7 * 80 * 512});
  s.push_back({"conv_pre.b", 512});
  int C = 512;
  for (int i = 0; i < 4; ++i) {
    s.push_back({"ups.w[K,C/2,C]", (int64_t)vc::hg_upk(i) * (C / 2) * C});
    s.push_back({"ups.b", C / 2});
    C /= 2;
  }
  C = 256;
  for (int n = 0; n < 12; ++n) {
    const int k = vc::hg_rbk(n % 3);
    const int ch = 256 >> (n / 3);
    for (int which = 0; which < 2; ++which)
      for (int m = 0; m < 3; ++m) {
        s.push_back({"resblock.conv.w[k,C,C]", (int64_t)k * ch * ch});
        s.push_back({"resblock.conv.b", ch});
      }
  }
  s.push_back({"conv_post.w[7,32,1]", 7 * 32});
  s.push_back({"conv_post.b", 1});
  return s;
}

const std::vector<TensorSpec>& vtts_acoustic_specs() {
  static std::vector<TensorSpec> s;
  if (!s.empty()) return s;
  s.push_back({"embed[256,256]", 256 * 256});
  for (int i = 0; i < 3; ++i) {
    s.push_back({"enc.conv.w[3,256,256]", 3 * 256 * 256});
    s.push_back({"enc.conv.b", 256});
    s.push_back({"enc.bn.scale", 256});
    s.push_back({"enc.bn.offset", 256});
    s.push_back({"enc.bn.mean", 256});
    s.push_back({"enc.bn.var", 256});
  }
  for (int d = 0; d < 2; ++d) {
    s.push_back({"enc.lstm.w[512,1024]", 512 * 1024});
    s.push_back({"enc.lstm.b", 1024});
  }
  s.push_back({"dec.lstm0.w[1280,2048]", 1280 * 2048});
  s.push_back({"dec.lstm0.b", 2048});
  s.push_back({"dec.lstm1.w[1792,2048]", 1792 * 2048});
  s.push_back({"dec.lstm1.b", 2048});
  s.push_back({"proj.w[1024,80]", 1024 * 80});
  s.push_back({"proj.b", 80});
  s.push_back({"prenet.fc1.w[80,256]", 80 * 256});
  s.push_back({"prenet.fc2.w[256,256]", 256 * 256});
  const int dims[6] = {80, 512, 512, 512, 512, 80};
  for (int i = 0; i < 5; ++i) {
    s.push_back({"postnet.conv.w[5,cin,cout]", (int64_t)5 * dims[i] * dims[i + 1]});
    s.push_back({"postnet.conv.b", dims[i + 1]});
    if (i < 4) {
      s.push_back({"postnet.bn.scale", 512});
      s.push_back({"postnet.bn.offset", 512});
      s.push_back({"postnet.bn.mean", 512});
      s.push_back({"postnet.bn.var", 512});
    }
  }
  return s;
}

// duration checkpoint: the TokenEncoder tensors in the acoustic blob's order, then the projection head
const std::vector<TensorSpec>& vtts_duration_specs() {
  static std::vector<TensorSpec> s;
  if (!s.empty()) return s;
  const std::vector<TensorSpec>& a = vtts_acoustic_specs();
  for (int i = 0; i <= aci::ENC_LSTM_B_B; ++i) s.push_back(a[i]);
  s.push_back({"proj.fc1.w[512,256]", 512 * 256});
  s.push_back({"proj.fc1.b", 256});
  s.push_back({"proj.fc2.w[256,1]", 256});
  s.push_back({"proj.fc2.b", 1});
  return s;
}

static int64_t total_floats(const std::vector<TensorSpec>& s) {
  int64_t t = 0;
  for (auto& e : s) t += e.n;
  return t;
}

// copy a contiguous blob (host or device) into per-tensor 256B-aligned device slots
// device arena of one model: every tensor of `specs` 256 B aligned; returns the arena size in floats
static size_t arena_floats(const std::vector<TensorSpec>& specs) {
  size_t total = 0;
  for (size_t i = 0; i < specs.size(); ++i) total += ((size_t)specs[i].n + 63) & ~size_t(63);
  return total;
}
static int alloc_arena(vtts_ctx* ctx, const std::vector<TensorSpec>& specs, float** store, std::vector<float*>& ptrs) {
  const size_t total = arena_floats(specs);
  if (*store) {
    VTTS_CUDA(cudaDeviceSynchronize());
    cudaFree(*store);
    *store = nullptr;
  }
  VTTS_CUDA(cudaMalloc(store, total * sizeof(float)));
  VTTS_CUDA(cudaMemset(*store, 0, total * sizeof(float)));
  ptrs.resize(specs.size());
  size_t off = 0;
  for (size_t i = 0; i < specs.size(); ++i) {
    ptrs[i] = *store + off;
    off += ((size_t)specs[i].n + 63) & ~size_t(63);
  }
  return VTTS_OK;
}
static int load_blob(vtts_ctx* ctx, const std::vector<TensorSpec>& specs, const float* blob, int64_t n_floats, float** store,
                     std::vector<float*>& ptrs) {
  if (!blob) return ctx->fail(VTTS_ERR_BAD_ARG, "load: null blob");
  if (n_floats != total_floats(specs))
    return ctx->fail(VTTS_ERR_BAD_ARG, "load: blob has %lld floats, expected %lld", (long long)n_floats, (long long)total_floats(specs));
  int rc = alloc_arena(ctx, specs, store, ptrs);
  if (rc) return rc;
  int64_t src = 0;
  for (size_t i = 0; i < specs.size(); ++i) {
    VTTS_CUDA(cudaMemcpy(ptrs[i], blob + src, (size_t)specs[i].n * sizeof(float), cudaMemcpyDefault));
    src += specs[i].n;
  }
  return VTTS_OK;
}

// ---- NCCL, bound at run time (the library has no link-time dependency on it: single-GPU users never load it) ----
namespace {
struct NcclApi {
  void* h = nullptr;
  int (*Broadcast)(const void*, void*, size_t, int, int, void*, cudaStream_t) = nullptr;
  int (*GroupStart)() = nullptr;
  int (*GroupEnd)() = nullptr;
  const char* (*GetErrorString)(int) = nullptr;
};
NcclApi g_nccl;
const char* nccl_bind() {
  if (g_nccl.Broadcast) return nullptr;
  const char* env = getenv("VTTS_NCCL_LIB");
  void* h = nullptr;
  if (env) h = dlopen(env, RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);        // the copy the host process (e.g. torch) already loaded
  if (!h) h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_GLOBAL);
  if (!h) h = dlopen("libnccl.so", RTLD_NOW | RTLD_GLOBAL);
  if (!h) return "libnccl.so.2 not found (set VTTS_NCCL_LIB to its path)";
  g_nccl.h = h;
  g_nccl.Broadcast = (decltype(g_nccl.Broadcast))dlsym(h, "ncclBroadcast");
  g_nccl.GroupStart = (decltype(g_nccl.GroupStart))dlsym(h, "ncclGroupStart");
  g_nccl.GroupEnd = (decltype(g_nccl.GroupEnd))dlsym(h, "ncclGroupEnd");
  g_nccl.GetErrorString = (decltype(g_nccl.GetErrorString))dlsym(h, "ncclGetErrorString");
  if (!g_nccl.Broadcast || !g_nccl.GroupStart || !g_nccl.GroupEnd) {
    g_nccl.Broadcast = nullptr;
    return "libnccl.so.2 lacks ncclBroadcast / ncclGroupStart / ncclGroupEnd";
  }
  return nullptr;
}
}  // namespace

extern "C" {

int vtts_version(void) { return 1; }

int vtts_create(int device, vtts_ctx** out) {
  if (!out) {
    g_vtts_create_error = "vtts_create: out is NULL";
    return VTTS_ERR_BAD_ARG;
  }
  *out = nullptr;
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess || n == 0) {
    g_vtts_create_error = std::string("vtts_create: no CUDA device (") + cudaGetErrorString(e) + "); there is no CPU fallback";
    cudaGetLastError();
    return VTTS_ERR_NO_DEVICE;
  }
  if (device < 0 || device >= n) {
    g_vtts_create_error = "vtts_create: device index out of range";
    return VTTS_ERR_BAD_ARG;
  }
  cudaDeviceProp prop;
  if ((e = cudaSetDevice(device)) != cudaSuccess || (e = cudaGetDeviceProperties(&prop, device)) != cudaSuccess) {
    g_vtts_create_error = std::string("vtts_create: ") + cudaGetErrorString(e);
    return VTTS_ERR_CUDA;
  }
  if (prop.major != 10) {
    char buf[256];
    snprintf(buf, sizeof(buf), "vtts_create: device %d is sm_%d%d; this library contains sm_100a code only", device, prop.major, prop.minor);
    g_vtts_create_error = buf;
    return VTTS_ERR_NO_DEVICE;
  }
  vtts_ctx* ctx = new vtts_ctx();
  ctx->device = device;
  ctx->sm_count = prop.multiProcessorCount;
  ctx->cc_major = prop.major;
  ctx->cc_minor = prop.minor;
  ctx->hbm_bytes = prop.totalGlobalMem;
  if (const char* v = getenv("VTTS_TC_VARIANT")) ctx->tc_variant = atoi(v);   // tuning aid (same values as vtts_debug_tc_stats bits 4..7)
  if ((e = cudaStreamCreateWithFlags(&ctx->own_stream, cudaStreamNonBlocking)) != cudaSuccess) {
    g_vtts_create_error = std::string("vtts_create: ") + cudaGetErrorString(e);
    delete ctx;
    return VTTS_ERR_CUDA;
  }
  for (int i = 0; i < vtts_ctx::NSTAGE; ++i) {
    cudaEventCreate(&ctx->ev0[i]);
    cudaEventCreate(&ctx->ev1[i]);
  }
  if (cudaMalloc(&ctx->d_err, sizeof(int)) != cudaSuccess || cudaMemset(ctx->d_err, 0, sizeof(int)) != cudaSuccess) {
    g_vtts_create_error = "vtts_create: cannot allocate the error flag";
    delete ctx;
    return VTTS_ERR_CUDA;
  }
  if (cudaMalloc(&ctx->d_tc_dbg, 256 * 16 * sizeof(long long)) != cudaSuccess) {
    g_vtts_create_error = "vtts_create: cannot allocate the profiling counters";
    delete ctx;
    return VTTS_ERR_CUDA;
  }
  cudaMemset(ctx->d_tc_dbg, 0, 256 * 16 * sizeof(long long));
  *out = ctx;
  return VTTS_OK;
}

int vtts_destroy(vtts_ctx* ctx) {
  if (!ctx) return VTTS_OK;
  cudaSetDevice(ctx->device);
  cudaDeviceSynchronize();
  cudaFree(ctx->hg_blob); cudaFree(ctx->hg_upsw); cudaFree(ctx->ac_blob); cudaFree(ctx->ac_derived);
  cudaFree(ctx->du_blob); cudaFree(ctx->du_derived); cudaFree(ctx->du_wpk);
  cudaFree(ctx->mel_fb); cudaFree(ctx->mel_lo); cudaFree(ctx->mel_hi); cudaFree(ctx->fft_tw); cudaFree(ctx->hann);
  cudaFree(ctx->ws); cudaFree(ctx->dstage); cudaFree(ctx->d_err); cudaFree(ctx->hg_wpk); cudaFree(ctx->ac_wpk); cudaFree(ctx->d_tc_dbg);
  if (ctx->hpin) cudaFreeHost(ctx->hpin);
  for (int i = 0; i < vtts_ctx::NSTAGE; ++i) {
    cudaEventDestroy(ctx->ev0[i]);
    cudaEventDestroy(ctx->ev1[i]);
  }
  if (ctx->own_stream) cudaStreamDestroy(ctx->own_stream);
  delete ctx;
  return VTTS_OK;
}

const char* vtts_last_error(vtts_ctx* ctx) { return ctx ? ctx->err.c_str() : g_vtts_create_error.c_str(); }

int vtts_device_info(vtts_ctx* ctx, int* sm_count, int* cc_major, int* cc_minor, int64_t* hbm_bytes) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (sm_count) *sm_count = ctx->sm_count;
  if (cc_major) *cc_major = ctx->cc_major;
  if (cc_minor) *cc_minor = ctx->cc_minor;
  if (hbm_bytes) *hbm_bytes = (int64_t)ctx->hbm_bytes;
  return VTTS_OK;
}

int vtts_set_precision(vtts_ctx* ctx, int mode) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (mode != VTTS_PRECISION_FP32 && mode != VTTS_PRECISION_BF16X3) return ctx->fail(VTTS_ERR_BAD_ARG, "set_precision: mode %d", mode);
  ctx->precision = mode;
  return VTTS_OK;
}

int vtts_get_precision(vtts_ctx* ctx) { return ctx ? ctx->precision : VTTS_ERR_BAD_ARG; }

int vtts_debug_substages(vtts_ctx* ctx, int enable, float* ms_out24) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  VTTS_CUDA(cudaDeviceSynchronize());
  if (ms_out24) {
    for (int i = 0; i < vtts_ctx::NSUB; ++i) {
      ms_out24[i] = 0.f;
      if ((i % 8) == 0 || !ctx->sub_set[i] || !ctx->sub_set[i - 1]) continue;
      float ms = 0.f;
      if (cudaEventElapsedTime(&ms, ctx->sub_ev[i - 1], ctx->sub_ev[i]) == cudaSuccess) ms_out24[i] = ms;
    }
  }
  for (int i = 0; i < vtts_ctx::NSUB; ++i) ctx->sub_set[i] = false;
  ctx->sub_on = enable != 0;
  return VTTS_OK;
}

int vtts_debug_tc_stats(vtts_ctx* ctx, int enable, int64_t* host_out_256x16) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  VTTS_CUDA(cudaSetDevice(ctx->device));
  VTTS_CUDA(cudaDeviceSynchronize());
  if (host_out_256x16) VTTS_CUDA(cudaMemcpy(host_out_256x16, ctx->d_tc_dbg, 256 * 16 * sizeof(long long), cudaMemcpyDeviceToHost));
  VTTS_CUDA(cudaMemset(ctx->d_tc_dbg, 0, 256 * 16 * sizeof(long long)));
  ctx->tc_dbg_on = (enable & 1) != 0;
  if (enable & 0x200) ctx->fuse_pairs = (enable >> 10) & 1;        // bit 9 set: bit 10 selects fused ResBlock pairs (tuning aid)
  if (enable & 0x800) ctx->pair_ts = (enable >> 12) & 3;           // bit 11 set: bits 12..13 select the pair kernel (vtts_ctx::pair_ts)
  if (enable & 0x100) ctx->tc_variant = (enable >> 4) & 0xF;   // bit 8 set: bits 4..7 select the tile-shape variant (tuning aid)
  return VTTS_OK;
}

int vtts_debug_conv(vtts_ctx* ctx, int precision, const vtts_conv_geometry* geom, const vtts_conv_problem* probs, int nprob) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (precision != VTTS_PRECISION_FP32 && precision != VTTS_PRECISION_BF16X3) return ctx->fail(VTTS_ERR_BAD_ARG, "debug_conv: precision %d", precision);
  if (!geom || !probs || nprob < 1 || nprob > 8) return ctx->fail(VTTS_ERR_BAD_ARG, "debug_conv: nprob %d", nprob);
  const vtts_conv_geometry& g = *geom;
  if (g.Cin < 16 || g.Cin % 16 != 0 || g.Cout < 4 || g.Cout % 4 != 0) return ctx->fail(VTTS_ERR_BAD_ARG, "debug_conv: Cin %d / Cout %d", g.Cin, g.Cout);
  if (g.B < 1 || g.T_rows < 1 || g.rows_out < 1 || g.len_mul < 1 || g.pre_mode < 0 || g.pre_mode > 2 || g.post_act < 0 || g.post_act > 2)
    return ctx->fail(VTTS_ERR_BAD_ARG, "debug_conv: B %d T_rows %d rows_out %d len_mul %d pre_mode %d post_act %d", g.B, g.T_rows,
                     g.rows_out, g.len_mul, g.pre_mode, g.post_act);
  ConvLaunch L;
  memset(&L, 0, sizeof(L));
  L.nprob = nprob; L.Cin = g.Cin; L.Cout = g.Cout; L.B = g.B; L.T_rows = g.T_rows; L.rows_out = g.rows_out;
  L.len = g.len; L.len_mul = g.len_mul; L.pre_mode = g.pre_mode; L.pre_slope = g.pre_slope; L.post_act = g.post_act;
  for (int i = 0; i < nprob; ++i) {
    const vtts_conv_problem& q = probs[i];
    const int nbn = (q.bn_mean != nullptr) + (q.bn_inv != nullptr) + (q.bn_off != nullptr);
    // x1 and x2 go together, and exactly with pre_mode 2 (as in vtts_debug_conv_transpose)
    if (!q.x0 || !q.w || !q.bias || !q.out || (nbn != 0 && nbn != 3) || (q.x1 == nullptr) != (q.x2 == nullptr) ||
        (q.x1 != nullptr) != (g.pre_mode == 2))
      return ctx->fail(VTTS_ERR_BAD_ARG, "debug_conv: problem %d: missing pointer, partial BatchNorm, or x1/x2 not both set with pre_mode 2", i);
    if (q.k < 1 || q.dil < 1 || q.out_stride < 1 || q.out_off < 0 || (int64_t)(g.T_rows - 1) * q.out_stride + q.out_off >= g.rows_out)
      return ctx->fail(VTTS_ERR_BAD_ARG, "debug_conv: problem %d: k %d dil %d out_stride %d out_off %d", i, q.k, q.dil, q.out_stride, q.out_off);
    L.p[i] = ConvProb{q.x0, q.x1, q.x2, q.w, q.bias, q.resid, q.bn_mean, q.bn_inv, q.bn_off, q.out, q.k, q.dil, q.in_off, q.out_stride, q.out_off};
  }
  VTTS_CUDA(cudaSetDevice(ctx->device));
  if (precision == VTTS_PRECISION_FP32) {
    int rc = vtts_launch_conv(ctx, L, nullptr);
    if (rc) return rc;
    VTTS_CUDA(cudaDeviceSynchronize());
    return VTTS_OK;
  }
  size_t bytes = 0;
  for (int i = 0; i < nprob; ++i) bytes += vtts_tc_conv_packed_bytes(L.p[i].k, g.Cin, g.Cout);
  void* pk = nullptr;
  VTTS_CUDA(cudaMalloc(&pk, bytes));
  std::vector<void*> wpk;   // wpk[prob * ntile + tile], the order vtts_conv_dispatch reads
  char* cur = (char*)pk;
  int rc = VTTS_OK;
  for (int i = 0; i < nprob && !rc; ++i) rc = vtts_tc_pack_conv(ctx, L.p[i].w, L.p[i].k, g.Cin, g.Cout, cur, wpk);
  const int saved = ctx->precision;
  ctx->precision = VTTS_PRECISION_BF16X3;     // the dispatcher takes the tensor-core path in this mode only; restored below
  if (!rc) rc = vtts_conv_dispatch(ctx, L, wpk.data(), nullptr);
  ctx->precision = saved;
  cudaError_t e = cudaDeviceSynchronize();
  cudaFree(pk);
  if (rc) return rc;
  if (e != cudaSuccess) return ctx->fail(VTTS_ERR_CUDA, "debug_conv (tensor path): %s", cudaGetErrorString(e));
  return VTTS_OK;
}

int vtts_debug_conv_transpose(vtts_ctx* ctx, int precision, const float* x0_dev, const float* x1_dev, const float* x2_dev,
                              const float* w_dev, const float* bias_dev, const int32_t* len_dev, int len_mul, int B, int T,
                              int C, int u, int K, float* out_dev) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (precision != VTTS_PRECISION_FP32 && precision != VTTS_PRECISION_BF16X3) return ctx->fail(VTTS_ERR_BAD_ARG, "debug_conv_transpose: precision %d", precision);
  bool stage = false;
  for (int i = 0, c = vc::HG_C0; i < vc::HG_NSTAGE; ++i, c /= 2) stage |= C == c && u == vc::hg_rate(i) && K == vc::hg_upk(i);
  if (!stage) return ctx->fail(VTTS_ERR_BAD_ARG, "debug_conv_transpose: (C %d, u %d, K %d) is not a generator stage", C, u, K);
  if (!x0_dev || !w_dev || !bias_dev || !out_dev || (x1_dev == nullptr) != (x2_dev == nullptr))
    return ctx->fail(VTTS_ERR_BAD_ARG, "debug_conv_transpose: missing pointer (x1 and x2 go together)");
  if (B < 1 || T < 1 || len_mul < 1 || (int64_t)T * u > INT32_MAX / 64) return ctx->fail(VTTS_ERR_BAD_ARG, "debug_conv_transpose: B %d T %d len_mul %d", B, T, len_mul);
  VTTS_CUDA(cudaSetDevice(ctx->device));
  const size_t upsw_bytes = ((size_t)u * 2 * C * (C / 2) * sizeof(float) + 255) & ~size_t(255);
  const size_t ph_bytes = (vtts_tc_packed_elems(2, C, C / 2) * 2 + 255) & ~size_t(255);
  char* buf = nullptr;
  VTTS_CUDA(cudaMalloc(&buf, upsw_bytes + u * ph_bytes));
  void* wpk[8];
  for (int r = 0; r < u; ++r) wpk[r] = buf + upsw_bytes + r * ph_bytes;
  int rc = vtts_hg_ups_prepare(ctx, w_dev, C, u, K, (float*)buf, wpk);
  if (!rc) rc = vtts_hg_ups_run(ctx, precision == VTTS_PRECISION_BF16X3, x0_dev, x1_dev, x2_dev, (const float*)buf, wpk, bias_dev,
                                len_dev, len_mul, B, T, C, u, K, out_dev, nullptr);
  cudaError_t e = cudaDeviceSynchronize();
  cudaFree(buf);
  if (rc) return rc;
  if (e != cudaSuccess) return ctx->fail(VTTS_ERR_CUDA, "debug_conv_transpose: %s", cudaGetErrorString(e));
  return VTTS_OK;
}

int vtts_debug_pair(vtts_ctx* ctx, const float* x_dev, const float* w1_dev, const float* b1_dev, const float* w2_dev,
                    const float* b2_dev, const int32_t* len_dev, int B, int T, int C, int k, int dil, float slope, float* out_dev) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  VTTS_CUDA(cudaSetDevice(ctx->device));
  void* wpk = nullptr;
  const size_t bytes = vtts_tc_packed_elems(k, C, C) * 2;
  const size_t cb = (vtts_tc_packed_pc_bytes(k, C) + 255) & ~size_t(255);
  VTTS_CUDA(cudaMalloc(&wpk, 2 * bytes + 2 * cb));
  int rc = vtts_tc_pack_weights(ctx, w1_dev, wpk, k, C, C, 0, C);
  if (!rc) rc = vtts_tc_pack_weights(ctx, w2_dev, (char*)wpk + bytes, k, C, C, 0, C);
  if (!rc) rc = vtts_tc_pack_weights_pc(ctx, w1_dev, (char*)wpk + 2 * bytes, k, C);
  if (!rc) rc = vtts_tc_pack_weights_pc(ctx, w2_dev, (char*)wpk + 2 * bytes + cb, k, C);
  if (rc) { cudaFree(wpk); return rc; }
  TcPairLaunch PL;
  memset(&PL, 0, sizeof(PL));
  PL.nprob = 1; PL.N = C; PL.B = B; PL.T_rows = T; PL.len = len_dev; PL.len_mul = 1; PL.slope = slope;
  PL.p[0] = TcPairProb{x_dev, wpk, (char*)wpk + bytes, b1_dev, b2_dev, out_dev, k, dil, (char*)wpk + 2 * bytes, (char*)wpk + 2 * bytes + cb};
  rc = vtts_launch_tc_pair(ctx, PL, nullptr);
  cudaError_t e = cudaDeviceSynchronize();
  cudaFree(wpk);
  if (rc) return rc;
  if (e != cudaSuccess) return ctx->fail(VTTS_ERR_CUDA, "debug_pair: %s", cudaGetErrorString(e));
  return VTTS_OK;
}

int64_t vtts_hifigan_blob_floats(void) { return total_floats(vtts_hifigan_specs()); }
int64_t vtts_acoustic_blob_floats(void) { return total_floats(vtts_acoustic_specs()); }
int64_t vtts_duration_blob_floats(void) { return total_floats(vtts_duration_specs()); }

int vtts_load_hifigan(vtts_ctx* ctx, const float* blob, int64_t n_floats) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  VTTS_CUDA(cudaSetDevice(ctx->device));
  ctx->hg_loaded = false;
  int rc = load_blob(ctx, vtts_hifigan_specs(), blob, n_floats, &ctx->hg_blob, ctx->hg_t);
  if (rc) return rc;
  rc = vtts_hifigan_prepare(ctx);
  if (rc) return rc;
  ctx->hg_loaded = true;
  return VTTS_OK;
}

int vtts_load_acoustic(vtts_ctx* ctx, const float* blob, int64_t n_floats) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  VTTS_CUDA(cudaSetDevice(ctx->device));
  ctx->ac_loaded = false;
  int rc = load_blob(ctx, vtts_acoustic_specs(), blob, n_floats, &ctx->ac_blob, ctx->ac_t);
  if (rc) return rc;
  rc = vtts_acoustic_prepare(ctx);
  if (rc) return rc;
  ctx->ac_loaded = true;
  return VTTS_OK;
}

int vtts_load_duration(vtts_ctx* ctx, const float* blob, int64_t n_floats) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  VTTS_CUDA(cudaSetDevice(ctx->device));
  ctx->du_loaded = false;
  int rc = load_blob(ctx, vtts_duration_specs(), blob, n_floats, &ctx->du_blob, ctx->du_t);
  if (rc) return rc;
  rc = vtts_duration_prepare(ctx);
  if (rc) return rc;
  ctx->du_loaded = true;
  return VTTS_OK;
}

// One start-up broadcast of the packed weights from `root` (SURVEY.md 8e: the only collective of the path).
int vtts_broadcast_weights(vtts_ctx* ctx, void* nccl_comm, int root, int is_root, void* stream) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (!nccl_comm) return ctx->fail(VTTS_ERR_BAD_ARG, "broadcast_weights: null communicator");
  VTTS_CUDA(cudaSetDevice(ctx->device));
  if (const char* e = nccl_bind()) return ctx->fail(VTTS_ERR_NCCL, "broadcast_weights: %s", e);
  cudaStream_t st = (cudaStream_t)stream;
  auto nccl_ck = [&](int r, const char* what) -> int {
    if (r == 0) return VTTS_OK;
    return ctx->fail(VTTS_ERR_NCCL, "broadcast_weights: %s -> %s", what, g_nccl.GetErrorString ? g_nccl.GetErrorString(r) : "nccl error");
  };
  // which models travel: bit 0 hifigan, 1 acoustic, 2 duration (decided by the root's loaded state)
  int32_t* d_flags = nullptr;
  VTTS_CUDA(cudaMalloc(&d_flags, sizeof(int32_t)));
  int32_t flags = is_root ? ((ctx->hg_loaded ? 1 : 0) | (ctx->ac_loaded ? 2 : 0) | (ctx->du_loaded ? 4 : 0)) : 0;
  VTTS_CUDA(cudaMemcpyAsync(d_flags, &flags, sizeof(flags), cudaMemcpyHostToDevice, st));
  int rc = nccl_ck(g_nccl.Broadcast(d_flags, d_flags, 1, /*ncclInt32*/ 2, root, nccl_comm, st), "ncclBroadcast(flags)");
  if (rc) { cudaFree(d_flags); return rc; }
  VTTS_CUDA(cudaMemcpyAsync(&flags, d_flags, sizeof(flags), cudaMemcpyDeviceToHost, st));
  VTTS_CUDA(cudaStreamSynchronize(st));
  cudaFree(d_flags);
  if (is_root && flags == 0) return ctx->fail(VTTS_ERR_NOT_LOADED, "broadcast_weights: the root context has no weights loaded");
  struct M { int bit; const std::vector<TensorSpec>* specs; float** store; std::vector<float*>* ptrs; bool* loaded; };
  M models[3] = {{1, &vtts_hifigan_specs(), &ctx->hg_blob, &ctx->hg_t, &ctx->hg_loaded},
                 {2, &vtts_acoustic_specs(), &ctx->ac_blob, &ctx->ac_t, &ctx->ac_loaded},
                 {4, &vtts_duration_specs(), &ctx->du_blob, &ctx->du_t, &ctx->du_loaded}};
  if (!is_root)
    for (auto& m : models)
      if (flags & m.bit) {
        *m.loaded = false;
        rc = alloc_arena(ctx, *m.specs, m.store, *m.ptrs);
        if (rc) return rc;
      }
  // the arenas have the same layout on every rank (it only depends on the tensor specs): ONE grouped broadcast
  rc = nccl_ck(g_nccl.GroupStart(), "ncclGroupStart");
  if (rc) return rc;
  for (auto& m : models)
    if (flags & m.bit) {
      rc = nccl_ck(g_nccl.Broadcast(*m.store, *m.store, arena_floats(*m.specs), /*ncclFloat32*/ 7, root, nccl_comm, st), "ncclBroadcast(weights)");
      if (rc) { g_nccl.GroupEnd(); return rc; }
    }
  rc = nccl_ck(g_nccl.GroupEnd(), "ncclGroupEnd");
  if (rc) return rc;
  VTTS_CUDA(cudaStreamSynchronize(st));
  if (!is_root) {
    if (flags & 1) { rc = vtts_hifigan_prepare(ctx); if (rc) return rc; ctx->hg_loaded = true; }
    if (flags & 2) { rc = vtts_acoustic_prepare(ctx); if (rc) return rc; ctx->ac_loaded = true; }
    if (flags & 4) { rc = vtts_duration_prepare(ctx); if (rc) return rc; ctx->du_loaded = true; }
  }
  return VTTS_OK;
}

int vtts_load_mel_filterbank(vtts_ctx* ctx, const float* fb, int n_mels, int n_bins) {
  if (!ctx || !fb) return VTTS_ERR_BAD_ARG;
  if (n_mels != vc::MEL || n_bins != vc::NBINS) return ctx->fail(VTTS_ERR_BAD_ARG, "mel filterbank must be [80][513], got [%d][%d]", n_mels, n_bins);
  VTTS_CUDA(cudaSetDevice(ctx->device));
  ctx->mel_loaded = false;
  if (!ctx->mel_fb) VTTS_CUDA(cudaMalloc(&ctx->mel_fb, (size_t)vc::MEL * vc::NBINS * sizeof(float)));
  VTTS_CUDA(cudaMemcpy(ctx->mel_fb, fb, (size_t)vc::MEL * vc::NBINS * sizeof(float), cudaMemcpyDefault));
  int rc = vtts_melspec_prepare(ctx);
  if (rc) return rc;
  ctx->mel_loaded = true;
  return VTTS_OK;
}

static void stage_begin(vtts_ctx* ctx, int stage, cudaStream_t st) {
  cudaEventRecord(ctx->ev0[stage], st);
  ctx->ev_stream[stage] = st;
}
static void stage_end(vtts_ctx* ctx, int stage, cudaStream_t st) {
  cudaEventRecord(ctx->ev1[stage], st);
  ctx->ev_valid[stage] = true;
}

int vtts_hifigan_forward(vtts_ctx* ctx, const float* mel_dev, const int32_t* n_frames_dev, int B, int T, float* wav_dev, void* stream) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (!mel_dev || !wav_dev) return ctx->fail(VTTS_ERR_BAD_ARG, "hifigan_forward: null pointer");
  VTTS_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  stage_begin(ctx, 0, st);
  int rc = vtts_hifigan_run(ctx, mel_dev, n_frames_dev, B, T, wav_dev, st);
  stage_end(ctx, 0, st);
  return rc;
}

int vtts_acoustic_forward(vtts_ctx* ctx, const int32_t* tokens_dev, const int32_t* lengths_dev, const float* dur_frames_dev,
                          const int32_t* n_frames_dev, const uint8_t* keep_mask_dev, int dropout_mode, uint64_t seed, int B, int L,
                          int N, float* mel_dev, void* stream) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (!tokens_dev || !dur_frames_dev || !mel_dev) return ctx->fail(VTTS_ERR_BAD_ARG, "acoustic_forward: null pointer");
  VTTS_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  size_t need = 0;
  int rc = vtts_acoustic_run(ctx, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0, B, L, N, nullptr, st, nullptr, 0, &need);
  if (rc) return rc;
  // the acoustic workspace lives after the hifigan one is released: both share ctx->ws, so a
  // synthesize call sizes it for the larger of the two (see vtts_synthesize_host)
  rc = ctx->ensure_ws(need);
  if (rc) return rc;
  stage_begin(ctx, 1, st);
  rc = vtts_acoustic_run(ctx, tokens_dev, lengths_dev, dur_frames_dev, n_frames_dev, keep_mask_dev, dropout_mode, seed, B, L, N,
                         mel_dev, st, ctx->ws, ctx->ws_bytes, nullptr);
  stage_end(ctx, 1, st);
  return rc;
}

int vtts_acoustic_teacher_forward(vtts_ctx* ctx, const int32_t* tokens_dev, const int32_t* lengths_dev, const float* dur_frames_dev,
                                  const int32_t* n_frames_dev, const float* mels_in_dev, const uint8_t* keep_mask_dev,
                                  const uint8_t* zone_mask_dev, int dropout_mode, uint64_t seed, int B, int L, int N,
                                  float* mel1_dev_or_null, float* mel2_dev, void* stream) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (!tokens_dev || !dur_frames_dev || !mels_in_dev || !mel2_dev) return ctx->fail(VTTS_ERR_BAD_ARG, "acoustic_teacher_forward: null pointer");
  VTTS_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  size_t need = 0;
  int rc = vtts_acoustic_teacher_run(ctx, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, 0, 0, B, L, N, nullptr, nullptr, st,
                                     nullptr, 0, &need);
  if (rc) return rc;
  rc = ctx->ensure_ws(need);
  if (rc) return rc;
  stage_begin(ctx, 1, st);
  rc = vtts_acoustic_teacher_run(ctx, tokens_dev, lengths_dev, dur_frames_dev, n_frames_dev, mels_in_dev, keep_mask_dev, zone_mask_dev,
                                 dropout_mode, seed, B, L, N, mel1_dev_or_null, mel2_dev, st, ctx->ws, ctx->ws_bytes, nullptr);
  stage_end(ctx, 1, st);
  return rc;
}

int vtts_duration_forward(vtts_ctx* ctx, const int32_t* tokens_dev, const int32_t* lengths_dev, int B, int L, float* dur_sec_dev,
                          void* stream) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (!tokens_dev || !dur_sec_dev) return ctx->fail(VTTS_ERR_BAD_ARG, "duration_forward: null pointer");
  VTTS_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  size_t need = 0;
  int rc = vtts_duration_run(ctx, nullptr, nullptr, B, L, nullptr, st, nullptr, 0, &need);
  if (rc) return rc;
  rc = ctx->ensure_ws(need);
  if (rc) return rc;
  stage_begin(ctx, 3, st);
  rc = vtts_duration_run(ctx, tokens_dev, lengths_dev, B, L, dur_sec_dev, st, ctx->ws, ctx->ws_bytes, nullptr);
  stage_end(ctx, 3, st);
  return rc;
}

int vtts_melspec(vtts_ctx* ctx, const float* wav_dev, int B, int S, float* mel_dev, void* stream) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (!wav_dev || !mel_dev) return ctx->fail(VTTS_ERR_BAD_ARG, "melspec: null pointer");
  VTTS_CUDA(cudaSetDevice(ctx->device));
  cudaStream_t st = (cudaStream_t)stream;
  stage_begin(ctx, 2, st);
  int rc = vtts_melspec_run(ctx, wav_dev, B, S, mel_dev, st);
  stage_end(ctx, 2, st);
  return rc;
}

int vtts_debug_read(vtts_ctx* ctx, const char* name, float* host_out, int64_t n_floats) {
  if (!ctx || !name || !host_out) return VTTS_ERR_BAD_ARG;
  const float* src = nullptr;
  int64_t n = 0;
  if (!strcmp(name, "enc")) { src = ctx->tap_enc; n = ctx->tap_enc_n; }
  else if (!strcmp(name, "cond")) { src = ctx->tap_cond; n = ctx->tap_cond_n; }
  else if (!strcmp(name, "mel_pre")) { src = ctx->tap_melpre; n = ctx->tap_melpre_n; }
  else return ctx->fail(VTTS_ERR_BAD_ARG, "debug_read: unknown tap %s", name);
  if (!src || n_floats != n) return ctx->fail(VTTS_ERR_BAD_ARG, "debug_read: tap %s has %lld floats, asked %lld", name, (long long)n, (long long)n_floats);
  VTTS_CUDA(cudaSetDevice(ctx->device));
  VTTS_CUDA(cudaDeviceSynchronize());
  VTTS_CUDA(cudaMemcpy(host_out, src, (size_t)n * sizeof(float), cudaMemcpyDeviceToHost));
  return VTTS_OK;
}

// ---- host-buffer entry points -------------------------------------------------------------------
// Layout of the staging areas: inputs first, outputs after, every block 256B aligned; the same
// offsets are used in the pinned host buffer and in the device staging buffer.
namespace {
// true if `p` is page-locked host memory known to CUDA (cudaHostAlloc / cudaHostRegister / torch pin_memory):
// results can then be copied D2H straight into the caller's buffer instead of through the context's staging area
bool is_pinned_host(const void* p) {
  cudaPointerAttributes at;
  if (cudaPointerGetAttributes(&at, p) != cudaSuccess) {
    cudaGetLastError();
    return false;
  }
  return at.type == cudaMemoryTypeHost;
}

struct Stager {
  size_t off = 0;
  size_t take(size_t bytes) {
    off = (off + 255) & ~size_t(255);
    size_t o = off;
    off += bytes;
    return o;
  }
};
}  // namespace

int vtts_mel2wave_host(vtts_ctx* ctx, const float* mel, const int32_t* n_frames, int B, int T, float* wav) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (!mel || !wav || B < 1 || T < 1) return ctx->fail(VTTS_ERR_BAD_ARG, "mel2wave_host: bad argument");
  VTTS_CUDA(cudaSetDevice(ctx->device));
  Stager s;
  const size_t mel_b = (size_t)B * T * vc::MEL * 4, nf_b = (size_t)B * 4, wav_b = (size_t)B * T * vc::HOP * 4;
  const size_t o_mel = s.take(mel_b), o_nf = s.take(nf_b), o_wav = s.take(wav_b);
  int rc = ctx->ensure_staging(s.off, s.off);
  if (rc) return rc;
  char* hp = (char*)ctx->hpin;
  char* dp = (char*)ctx->dstage;
  cudaStream_t st = ctx->own_stream;
  memcpy(hp + o_mel, mel, mel_b);
  if (n_frames) memcpy(hp + o_nf, n_frames, nf_b);
  VTTS_CUDA(cudaMemcpyAsync(dp + o_mel, hp + o_mel, (n_frames ? o_nf + nf_b : mel_b) - o_mel, cudaMemcpyHostToDevice, st));
  rc = vtts_hifigan_forward(ctx, (const float*)(dp + o_mel), n_frames ? (const int32_t*)(dp + o_nf) : nullptr, B, T, (float*)(dp + o_wav), st);
  if (rc) return rc;
  const bool direct = is_pinned_host(wav);
  VTTS_CUDA(cudaMemcpyAsync(direct ? (void*)wav : (void*)(hp + o_wav), dp + o_wav, wav_b, cudaMemcpyDeviceToHost, st));
  VTTS_CUDA(cudaStreamSynchronize(st));
  if (!direct) memcpy(wav, hp + o_wav, wav_b);
  return VTTS_OK;
}

static int synth_common(vtts_ctx* ctx, const int32_t* tokens, const int32_t* lengths, const float* dur, const int32_t* n_frames,
                        const uint8_t* keep, int mode, uint64_t seed, int B, int L, int N, float* mel_out, float* wav_out,
                        const int32_t* n_frames_voc = nullptr) {
  // n_frames_voc: optional per-row frame counts for the generator only (text2mel trims the trailing silence from the
  // mel AFTER the postnet, text2mel.py:99-102); default = n_frames
  if (!tokens || !dur || B < 1 || L < 1 || N < 1) return ctx->fail(VTTS_ERR_BAD_ARG, "predict_mel/synthesize_host: bad argument");
  if (mode == VTTS_DROPOUT_MASK && !keep) return ctx->fail(VTTS_ERR_BAD_ARG, "dropout_mode MASK needs keep_mask");
  VTTS_CUDA(cudaSetDevice(ctx->device));
  Stager s;
  const size_t tok_b = (size_t)B * L * 4, len_b = (size_t)B * 4, dur_b = (size_t)B * L * 4, nf_b = (size_t)B * 4;
  const size_t keep_b = mode == VTTS_DROPOUT_MASK ? (size_t)B * N * 2 * vc::PRENET : 0;
  const size_t mel_b = (size_t)B * N * vc::MEL * 4, wav_b = wav_out ? (size_t)B * N * vc::HOP * 4 : 0;
  const size_t o_tok = s.take(tok_b), o_len = s.take(len_b), o_dur = s.take(dur_b), o_nf = s.take(nf_b), o_keep = s.take(keep_b);
  const size_t o_nfv = s.take(n_frames_voc ? nf_b : 0);
  const size_t in_end = s.off;
  const size_t o_mel = s.take(mel_b), o_wav = s.take(wav_b);
  int rc = ctx->ensure_staging(s.off, s.off);
  if (rc) return rc;
  char* hp = (char*)ctx->hpin;
  char* dp = (char*)ctx->dstage;
  cudaStream_t st = ctx->own_stream;
  memcpy(hp + o_tok, tokens, tok_b);
  if (lengths) memcpy(hp + o_len, lengths, len_b);
  memcpy(hp + o_dur, dur, dur_b);
  if (n_frames) memcpy(hp + o_nf, n_frames, nf_b);
  if (keep_b) memcpy(hp + o_keep, keep, keep_b);
  if (n_frames_voc) memcpy(hp + o_nfv, n_frames_voc, nf_b);
  VTTS_CUDA(cudaMemcpyAsync(dp, hp, in_end, cudaMemcpyHostToDevice, st));
  const int32_t* d_len = lengths ? (const int32_t*)(dp + o_len) : nullptr;
  const int32_t* d_nf = n_frames ? (const int32_t*)(dp + o_nf) : nullptr;
  rc = vtts_acoustic_forward(ctx, (const int32_t*)(dp + o_tok), d_len, (const float*)(dp + o_dur), d_nf,
                             keep_b ? (const uint8_t*)(dp + o_keep) : nullptr, mode, seed, B, L, N, (float*)(dp + o_mel), st);
  if (rc) return rc;
  const bool mel_direct = mel_out && is_pinned_host(mel_out);
  const bool wav_direct = wav_out && is_pinned_host(wav_out);
  if (mel_out) VTTS_CUDA(cudaMemcpyAsync(mel_direct ? (void*)mel_out : (void*)(hp + o_mel), dp + o_mel, mel_b, cudaMemcpyDeviceToHost, st));
  if (wav_out) {
    // the hifigan workspace replaces the acoustic one: its kernels are stream-ordered after the acoustic ones,
    // but growing the workspace frees memory -> make sure `mel` (in dstage) is complete first
    size_t need = vtts_hifigan_ws_bytes(B, N);
    if (need > ctx->ws_bytes) VTTS_CUDA(cudaStreamSynchronize(st));
    rc = vtts_hifigan_forward(ctx, (const float*)(dp + o_mel), n_frames_voc ? (const int32_t*)(dp + o_nfv) : d_nf, B, N,
                              (float*)(dp + o_wav), st);
    if (rc) return rc;
    VTTS_CUDA(cudaMemcpyAsync(wav_direct ? (void*)wav_out : (void*)(hp + o_wav), dp + o_wav, wav_b, cudaMemcpyDeviceToHost, st));
  }
  VTTS_CUDA(cudaStreamSynchronize(st));
  if (mel_out && !mel_direct) memcpy(mel_out, hp + o_mel, mel_b);
  if (wav_out && !wav_direct) memcpy(wav_out, hp + o_wav, wav_b);
  return VTTS_OK;
}

int vtts_predict_mel_host(vtts_ctx* ctx, const int32_t* tokens, const int32_t* lengths, const float* dur_frames,
                          const int32_t* n_frames, const uint8_t* keep_mask, int dropout_mode, uint64_t seed, int B, int L, int N,
                          float* mel) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (!mel) return ctx->fail(VTTS_ERR_BAD_ARG, "predict_mel_host: null output");
  return synth_common(ctx, tokens, lengths, dur_frames, n_frames, keep_mask, dropout_mode, seed, B, L, N, mel, nullptr);
}

int vtts_synthesize_host(vtts_ctx* ctx, const int32_t* tokens, const int32_t* lengths, const float* dur_frames,
                         const int32_t* n_frames, const uint8_t* keep_mask, int dropout_mode, uint64_t seed, int B, int L, int N,
                         float* mel_out_or_null, float* wav) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (!wav) return ctx->fail(VTTS_ERR_BAD_ARG, "synthesize_host: null output");
  return synth_common(ctx, tokens, lengths, dur_frames, n_frames, keep_mask, dropout_mode, seed, B, L, N, mel_out_or_null, wav);
}

int vtts_predict_duration_host(vtts_ctx* ctx, const int32_t* tokens, const int32_t* lengths, int B, int L, float* dur_sec) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (!tokens || !dur_sec || B < 1 || L < 1) return ctx->fail(VTTS_ERR_BAD_ARG, "predict_duration_host: bad argument");
  VTTS_CUDA(cudaSetDevice(ctx->device));
  Stager s;
  const size_t tok_b = (size_t)B * L * 4, len_b = (size_t)B * 4, dur_b = (size_t)B * L * 4;
  const size_t o_tok = s.take(tok_b), o_len = s.take(len_b), o_dur = s.take(dur_b);
  int rc = ctx->ensure_staging(s.off, s.off);
  if (rc) return rc;
  char* hp = (char*)ctx->hpin;
  char* dp = (char*)ctx->dstage;
  cudaStream_t st = ctx->own_stream;
  memcpy(hp + o_tok, tokens, tok_b);
  if (lengths) memcpy(hp + o_len, lengths, len_b);
  VTTS_CUDA(cudaMemcpyAsync(dp + o_tok, hp + o_tok, tok_b, cudaMemcpyHostToDevice, st));
  if (lengths) VTTS_CUDA(cudaMemcpyAsync(dp + o_len, hp + o_len, len_b, cudaMemcpyHostToDevice, st));
  rc = vtts_duration_forward(ctx, (const int32_t*)(dp + o_tok), lengths ? (const int32_t*)(dp + o_len) : nullptr, B, L,
                             (float*)(dp + o_dur), st);
  if (rc) return rc;
  VTTS_CUDA(cudaMemcpyAsync(hp + o_dur, dp + o_dur, dur_b, cudaMemcpyDeviceToHost, st));
  VTTS_CUDA(cudaStreamSynchronize(st));
  memcpy(dur_sec, hp + o_dur, dur_b);
  return VTTS_OK;
}

namespace {
__global__ void pcm16_to_float_kernel(const int16_t* __restrict__ in, float* __restrict__ out, size_t n) {
  for (size_t i = blockIdx.x * (size_t)blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    out[i] = (float)in[i] * (1.0f / 32768.0f);                      // gta.py:32  wavs.astype(float32) / 2**15
}
}  // namespace

// forward_fn_ of vietTTS/nat/gta.py:28-41: int16 waveform -> MelFilter -> ground-truth mel shifted by one frame ->
// AcousticModel.__call__ (teacher forced, zoneout) -> mel2_hat.
int vtts_gta_host(vtts_ctx* ctx, const int16_t* wav_i16, const int32_t* wav_lengths, const int32_t* tokens, const int32_t* lengths,
                  const float* dur_sec, const uint8_t* keep_mask, const uint8_t* zone_mask, int dropout_mode, uint64_t seed, int B,
                  int L, int S, float* mel_gt_out_or_null, float* mel2_out) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (!wav_i16 || !tokens || !dur_sec || !mel2_out || B < 1 || L < 1 || S < 512 || S % vc::HOP)
    return ctx->fail(VTTS_ERR_BAD_ARG, "gta_host: bad argument (S must be a multiple of %d, >= 512)", vc::HOP);
  if (dropout_mode == VTTS_DROPOUT_MASK && (!keep_mask || !zone_mask)) return ctx->fail(VTTS_ERR_BAD_ARG, "gta_host: MASK mode needs both masks");
  if (!ctx->mel_loaded) return ctx->fail(VTTS_ERR_NOT_LOADED, "gta_host: mel filterbank not loaded");
  VTTS_CUDA(cudaSetDevice(ctx->device));
  const int N = S / vc::HOP;
  Stager s;
  const size_t wav_b = (size_t)B * S * 2, tok_b = (size_t)B * L * 4, len_b = (size_t)B * 4, dur_b = (size_t)B * L * 4, nf_b = (size_t)B * 4;
  const size_t keep_b = dropout_mode == VTTS_DROPOUT_MASK ? (size_t)B * N * 2 * vc::PRENET : 0;
  const size_t zone_b = dropout_mode == VTTS_DROPOUT_MASK ? (size_t)B * N * 4 * vc::DEC_H : 0;
  const size_t mel_b = (size_t)B * N * vc::MEL * 4;
  const size_t o_wav = s.take(wav_b), o_tok = s.take(tok_b), o_len = s.take(len_b), o_dur = s.take(dur_b), o_nf = s.take(nf_b);
  const size_t o_keep = s.take(keep_b), o_zone = s.take(zone_b);
  const size_t in_end = s.off;
  const size_t o_gt = s.take(mel_b), o_out = s.take(mel_b);
  const size_t host_end = s.off;
  const size_t o_wavf = s.take((size_t)B * S * 4), o_in = s.take(mel_b);      // device-only scratch
  int rc = ctx->ensure_staging(host_end, s.off);
  if (rc) return rc;
  char* hp = (char*)ctx->hpin;
  char* dp = (char*)ctx->dstage;
  cudaStream_t st = ctx->own_stream;
  memcpy(hp + o_wav, wav_i16, wav_b);
  memcpy(hp + o_tok, tokens, tok_b);
  if (lengths) memcpy(hp + o_len, lengths, len_b);
  {
    float* d = (float*)(hp + o_dur);                                  // gta.py:37  durations * sample_rate / (n_fft // 4), float32
    for (size_t i = 0; i < (size_t)B * L; ++i) d[i] = (dur_sec[i] * 16000.0f) / 256.0f;
    int32_t* nf = (int32_t*)(hp + o_nf);                              // gta.py:74  l = wav_length // hop
    for (int b = 0; b < B; ++b) {
      int n = wav_lengths ? wav_lengths[b] / vc::HOP : N;
      nf[b] = n < 1 ? 1 : (n > N ? N : n);
    }
  }
  if (keep_b) memcpy(hp + o_keep, keep_mask, keep_b);
  if (zone_b) memcpy(hp + o_zone, zone_mask, zone_b);
  VTTS_CUDA(cudaMemcpyAsync(dp, hp, in_end, cudaMemcpyHostToDevice, st));
  pcm16_to_float_kernel<<<148 * 4, 256, 0, st>>>((const int16_t*)(dp + o_wav), (float*)(dp + o_wavf), (size_t)B * S);
  ctx->launches++;
  VTTS_CUDA(cudaGetLastError());
  rc = vtts_melspec(ctx, (const float*)(dp + o_wavf), B, S, (float*)(dp + o_gt), st);
  if (rc) return rc;
  // inp_mels = concat(zeros[B,1,D], mels[:, :-1]) (gta.py:34-36)
  VTTS_CUDA(cudaMemsetAsync(dp + o_in, 0, mel_b, st));
  if (N > 1)
    VTTS_CUDA(cudaMemcpy2DAsync(dp + o_in + vc::MEL * 4, (size_t)N * vc::MEL * 4, dp + o_gt, (size_t)N * vc::MEL * 4,
                                (size_t)(N - 1) * vc::MEL * 4, B, cudaMemcpyDeviceToDevice, st));
  rc = vtts_acoustic_teacher_forward(ctx, (const int32_t*)(dp + o_tok), lengths ? (const int32_t*)(dp + o_len) : nullptr,
                                     (const float*)(dp + o_dur), (const int32_t*)(dp + o_nf), (const float*)(dp + o_in),
                                     keep_b ? (const uint8_t*)(dp + o_keep) : nullptr, zone_b ? (const uint8_t*)(dp + o_zone) : nullptr,
                                     dropout_mode, seed, B, L, N, nullptr, (float*)(dp + o_out), st);
  if (rc) return rc;
  VTTS_CUDA(cudaMemcpyAsync(hp + o_gt, dp + o_gt, 2 * mel_b + (o_out - o_gt - mel_b), cudaMemcpyDeviceToHost, st));
  VTTS_CUDA(cudaStreamSynchronize(st));
  if (mel_gt_out_or_null) memcpy(mel_gt_out_or_null, hp + o_gt, mel_b);
  memcpy(mel2_out, hp + o_out, mel_b);
  return VTTS_OK;
}

// text2mel (vietTTS/nat/text2mel.py:85-103) + mel2wave for a batch of token rows, in one call:
//   predict_duration -> [host: silence clip, word-end zeroing, seconds -> frames, n_frames, trailing-silence trim]
//   -> AcousticModel.inference -> Generator.  The one unavoidable host round trip is the [B,L] duration matrix:
//   the frame count N (every later grid size) depends on it.
int vtts_tts_host(vtts_ctx* ctx, const int32_t* tokens, const int32_t* lengths, int B, int L, float silence_duration,
                  int dropout_mode, uint64_t seed, int max_frames, float* dur_sec_out, int32_t* n_frames_out,
                  int32_t* n_max_out, float* wav) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (!tokens || !n_frames_out || !n_max_out || !wav || B < 1 || L < 1 || max_frames < 1)
    return ctx->fail(VTTS_ERR_BAD_ARG, "tts_host: bad argument");
  if (dropout_mode != VTTS_DROPOUT_OFF && dropout_mode != VTTS_DROPOUT_SEED)
    return ctx->fail(VTTS_ERR_BAD_ARG, "tts_host: dropout_mode must be OFF or SEED (the frame count is not known to the caller)");
  VTTS_CUDA(cudaSetDevice(ctx->device));
  std::vector<float> sec((size_t)B * L), frames((size_t)B * L);
  int rc = vtts_predict_duration_host(ctx, tokens, lengths, B, L, sec.data());
  if (rc) return rc;
  std::vector<int32_t> nf_ac(B), nf_voc(B);
  int n_max = 0;
  for (int b = 0; b < B; ++b) {
    const int len = lengths ? lengths[b] : L;
    if (len < 1 || len > L) return ctx->fail(VTTS_ERR_BAD_ARG, "tts_host: lengths[%d]=%d outside [1,%d]", b, len, L);
    double total = 0.0;
    for (int l = 0; l < L; ++l) {
      float d = l < len ? sec[(size_t)b * L + l] : 0.f;
      const int tok = tokens[(size_t)b * L + l];
      if (l < len && tok == vc::SIL_INDEX && d < silence_duration) d = silence_duration;   // text2mel.py:88-94
      if (tok == vc::WORD_END_INDEX) d = 0.f;                                              // text2mel.py:95-97
      sec[(size_t)b * L + l] = d;
      const float f = (d * 16000.0f) / 256.0f;                                             // text2mel.py:78 (float32)
      frames[(size_t)b * L + l] = f;
      total += f;
    }
    const int n = (int)(float)total;                                                       // text2mel.py:79
    int trim = 0;
    if (tokens[(size_t)b * L + len - 1] == vc::SIL_INDEX)                                  // text2mel.py:99-102
      trim = (int)((double)sec[(size_t)b * L + len - 1] * 16000.0 / 256.0);
    nf_ac[b] = n;
    nf_voc[b] = n - trim > 0 ? n - trim : 0;
    if (n > n_max) n_max = n;
  }
  if (dur_sec_out) memcpy(dur_sec_out, sec.data(), sec.size() * sizeof(float));
  memcpy(n_frames_out, nf_voc.data(), (size_t)B * sizeof(int32_t));
  *n_max_out = n_max;
  if (n_max < 1) return ctx->fail(VTTS_ERR_BAD_ARG, "tts_host: predicted durations sum to less than one frame");
  if (n_max > max_frames)
    return ctx->fail(VTTS_ERR_BAD_ARG, "tts_host: needs %d frames, caller buffer holds %d (n_max_out is set: retry with that size)", n_max, max_frames);
  return synth_common(ctx, tokens, lengths, frames.data(), nf_ac.data(), nullptr, dropout_mode, seed, B, L, n_max, nullptr, wav,
                      nf_voc.data());
}

int vtts_melspec_host(vtts_ctx* ctx, const float* wav, int B, int S, float* mel) {
  if (!ctx) return VTTS_ERR_BAD_ARG;
  if (!wav || !mel || B < 1 || S < 512 || S % vc::HOP) return ctx->fail(VTTS_ERR_BAD_ARG, "melspec_host: bad argument");
  VTTS_CUDA(cudaSetDevice(ctx->device));
  Stager s;
  const size_t wav_b = (size_t)B * S * 4, mel_b = (size_t)B * (S / vc::HOP) * vc::MEL * 4;
  const size_t o_wav = s.take(wav_b), o_mel = s.take(mel_b);
  int rc = ctx->ensure_staging(s.off, s.off);
  if (rc) return rc;
  char* hp = (char*)ctx->hpin;
  char* dp = (char*)ctx->dstage;
  cudaStream_t st = ctx->own_stream;
  memcpy(hp + o_wav, wav, wav_b);
  VTTS_CUDA(cudaMemcpyAsync(dp + o_wav, hp + o_wav, wav_b, cudaMemcpyHostToDevice, st));
  rc = vtts_melspec(ctx, (const float*)(dp + o_wav), B, S, (float*)(dp + o_mel), st);
  if (rc) return rc;
  VTTS_CUDA(cudaMemcpyAsync(hp + o_mel, dp + o_mel, mel_b, cudaMemcpyDeviceToHost, st));
  VTTS_CUDA(cudaStreamSynchronize(st));
  memcpy(mel, hp + o_mel, mel_b);
  return VTTS_OK;
}

int64_t vtts_launch_count(vtts_ctx* ctx) { return ctx ? ctx->launches : 0; }

int vtts_last_stage_ms(vtts_ctx* ctx, int stage, float* ms) {
  if (!ctx || !ms || stage < 0 || stage >= vtts_ctx::NSTAGE) return VTTS_ERR_BAD_ARG;
  if (!ctx->ev_valid[stage]) return ctx->fail(VTTS_ERR_BAD_ARG, "last_stage_ms: stage %d has not run", stage);
  VTTS_CUDA(cudaSetDevice(ctx->device));
  VTTS_CUDA(cudaEventSynchronize(ctx->ev1[stage]));
  VTTS_CUDA(cudaEventElapsedTime(ms, ctx->ev0[stage], ctx->ev1[stage]));
  return VTTS_OK;
}

}  // extern "C"
