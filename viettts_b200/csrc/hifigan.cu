// HiFiGAN generator forward (strict fp32 path) -- restates Generator.__call__
// (vietTTS/hifigan/model.py:109-125) on top of the generic conv kernel.
//
//   conv_pre                              model.py:110
//   per stage: lrelu(0.1) -> ups[i]       model.py:112-114   (u output phases, 2 taps each)
//              3 x ResBlock1, mean        model.py:115-121   (mean fused into the next consumer)
//   lrelu(0.01) -> conv_post -> tanh      model.py:122-124   (conv_post_kernel below)
#include "vtts_internal.cuh"

namespace {

// ---- ConvTranspose weight repack: Haiku w[K][Cout][Cin] -> per phase r: [2][Cin][Cout] ----------
// hk.Conv1DTranspose("SAME"): y[t,o] = b[o] + sum_j sum_i xdpad[t+j, i] w[j,o,i] with the input
// zero-dilated by `u` and padded by a = ceil((K+u-2)/2) on the left.  For t = tau*u + r only taps
// j = j0 + q*u (q = 0,1; j0 = (a - r) mod u) hit a non-zero sample, x[tau + e + q], e = (r + j0 - a)/u.
__global__ void repack_ups_kernel(const float* __restrict__ w, float* __restrict__ out, int u, int K, int Cin, int Cout, int a) {
  const size_t total = (size_t)u * 2 * Cin * Cout;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    int o = idx % Cout;
    int i = (idx / Cout) % Cin;
    int q = (idx / ((size_t)Cout * Cin)) % 2;
    int r = idx / ((size_t)Cout * Cin * 2);
    int j0 = ((a - r) % u + u) % u;
    int j = j0 + q * u;
    out[idx] = w[((size_t)j * Cout + o) * Cin + i];
  }
}

// conv_post: out[b,t] = tanh(bias + sum_{j<7} sum_{i<32} lrelu_0.01(mean3(x)[t+j-3, i]) w[j,i])
__global__ void __launch_bounds__(256) conv_post_kernel(const float* __restrict__ a0, const float* __restrict__ a1,
                                                        const float* __restrict__ a2, const float* __restrict__ w,
                                                        const float* __restrict__ bias, const int* __restrict__ len,
                                                        int len_mul, int R, float* __restrict__ wav) {
  constexpr int C = 32, KW = 7, TT = 256, ST = 33;
  __shared__ float xs[(TT + KW - 1) * ST];
  __shared__ float wsm[KW * C];
  const int b = blockIdx.y, t0 = blockIdx.x * TT, tid = threadIdx.x;
  int valid = R;
  if (len) {
    int v = len[b] * len_mul;
    valid = v < valid ? v : valid;
  }
  if (tid < KW * C) wsm[tid] = w[tid];
  const size_t base = (size_t)b * R * C;
  if (t0 < valid) {
    for (int e = tid; e < (TT + KW - 1) * (C / 4); e += 256) {
      int rr = e / (C / 4), q = e % (C / 4);
      int r = t0 - 3 + rr;
      float4 v = make_float4(0, 0, 0, 0);
      if (r >= 0 && r < valid) {
        size_t off = base + (size_t)r * C + q * 4;
        float4 x = __ldg(reinterpret_cast<const float4*>(a0 + off));
        float4 y = __ldg(reinterpret_cast<const float4*>(a1 + off));
        float4 z = __ldg(reinterpret_cast<const float4*>(a2 + off));
        v.x = ((x.x + y.x) + z.x) / 3.0f;
        v.y = ((x.y + y.y) + z.y) / 3.0f;
        v.z = ((x.z + y.z) + z.z) / 3.0f;
        v.w = ((x.w + y.w) + z.w) / 3.0f;
        v.x = v.x >= 0.f ? v.x : 0.01f * v.x;
        v.y = v.y >= 0.f ? v.y : 0.01f * v.y;
        v.z = v.z >= 0.f ? v.z : 0.01f * v.z;
        v.w = v.w >= 0.f ? v.w : 0.01f * v.w;
      }
      float* d = xs + rr * ST + q * 4;
      d[0] = v.x; d[1] = v.y; d[2] = v.z; d[3] = v.w;
    }
  }
  __syncthreads();
  const int t = t0 + tid;
  if (t >= R) return;
  float out = 0.f;
  if (t < valid) {
    float acc = 0.f;
#pragma unroll
    for (int j = 0; j < KW; ++j)
#pragma unroll
      for (int i = 0; i < C; ++i) acc = fmaf(xs[(tid + j) * ST + i], wsm[j * C + i], acc);
    out = tanhf(acc + bias[0]);
  }
  wav[(size_t)b * R + t] = out;
}

struct HgBufs {
  float* P0;        // conv_pre out [B][T][512]
  float* A[2][3];   // resblock outputs (alternate by stage parity)
  float* X;         // ups out
  float* Tb[3];     // conv1 out
  float* Bb[3];     // ping-pong
};

void carve(Arena& ar, int B, int T, HgBufs& hb) {
  const size_t frames = (size_t)B * T;
  hb.P0 = ar.take<float>(frames * 512);
  const size_t big = frames * 8192;
  for (int p = 0; p < 2; ++p)
    for (int j = 0; j < 3; ++j) hb.A[p][j] = ar.take<float>(big);
  hb.X = ar.take<float>(big);
  for (int j = 0; j < 3; ++j) hb.Tb[j] = ar.take<float>(big);
  for (int j = 0; j < 3; ++j) hb.Bb[j] = ar.take<float>(big);
}

}  // namespace

size_t vtts_hifigan_ws_bytes(int B, int T) {
  Arena ar(nullptr, 0, true);
  HgBufs hb;
  carve(ar, B, T, hb);
  return ar.off + 256;
}

int vtts_hg_ups_prepare(vtts_ctx* ctx, const float* w, int C, int u, int K, float* upsw, void* const* wpk) {
  const int Co = C / 2, a = (K + u - 2 + 1) / 2;
  repack_ups_kernel<<<256, 256>>>(w, upsw, u, K, C, Co, a);
  VTTS_CUDA(cudaGetLastError());
  // (same stream as the repack: the phase weights are packed from upsw after it is complete)
  for (int r = 0; r < u; ++r) {
    int rc = vtts_tc_pack_weights(ctx, upsw + (size_t)r * 2 * C * Co, wpk[r], 2, C, Co, 0, Co);
    if (rc) return rc;
  }
  return VTTS_OK;
}

int vtts_hg_ups_run(vtts_ctx* ctx, bool tc, const float* x0, const float* x1, const float* x2, const float* upsw,
                    void* const* wpk, const float* bias, const int32_t* len, int len_mul, int B, int T, int C, int u, int K,
                    float* out, cudaStream_t st) {
  const int Co = C / 2;
  const int a = (K + u - 2 + 1) / 2;
  ConvLaunch L;
  memset(&L, 0, sizeof(L));
  L.B = B; L.len = len; L.len_mul = len_mul;
  L.nprob = u; L.Cin = C; L.Cout = Co;
  L.T_rows = T; L.rows_out = T * u;
  L.pre_mode = x1 ? 2 : 1; L.pre_slope = 0.1f; L.post_act = 0;
  for (int r = 0; r < u; ++r) {
    int j0 = ((a - r) % u + u) % u;
    int e = (r + j0 - a) / u;  // exact division, <= 0
    ConvProb p;
    memset(&p, 0, sizeof(p));
    p.x0 = x0; p.x1 = x1; p.x2 = x2;
    p.w = upsw + (size_t)r * 2 * C * Co;
    p.bias = bias;
    p.out = out;
    p.k = 2; p.dil = 1; p.in_off = e; p.out_stride = u; p.out_off = r;
    L.p[r] = p;
  }
  if (!tc) return vtts_launch_conv(ctx, L, st);
  // ConvTranspose phases share their input: for N <= 128 one converted activation tile feeds NPH phases
  // (multi-phase tiles of tc_conv.cu); N = 256 keeps one problem per phase.
  const int nph = Co == 256 ? 1 : (Co == 128 ? 4 : 2);
  TcLaunch TL;
  memset(&TL, 0, sizeof(TL));
  TL.nprob = u / nph; TL.nphase = nph; TL.Cin = C; TL.N = Co; TL.in_ld = C; TL.out_ld = Co;
  TL.B = B; TL.T_rows = T; TL.rows_out = T * u; TL.len = len; TL.len_mul = len_mul;
  TL.pre_mode = L.pre_mode; TL.pre_slope = 0.1f;
  for (int g = 0; g < u / nph; ++g) {
    const ConvProb& c0 = L.p[g * nph];
    TcProb q;
    memset(&q, 0, sizeof(q));
    q.x0 = c0.x0; q.x1 = c0.x1; q.x2 = c0.x2; q.bias = c0.bias; q.out = c0.out;
    q.k = 2; q.dil = 1; q.out_stride = u;
    q.wpk = wpk[g * nph]; q.in_off = c0.in_off; q.out_off = g * nph;
    for (int ph = 0; ph < nph; ++ph) {
      const int r = g * nph + ph;
      q.wpk_ph[ph] = wpk[r];
      q.in_off_ph[ph] = L.p[r].in_off;
      q.out_off_ph[ph] = r;
    }
    TL.p[g] = q;
  }
  return vtts_launch_tc_conv(ctx, TL, st);
}

int vtts_hifigan_prepare(vtts_ctx* ctx) {
  // repacked transposed-conv weights
  size_t total = 0;
  size_t offs[4];
  int C = vc::HG_C0;
  for (int i = 0; i < 4; ++i) {
    offs[i] = total;
    total += (size_t)vc::hg_rate(i) * 2 * C * (C / 2);
    C /= 2;
  }
  if (ctx->hg_upsw) cudaFree(ctx->hg_upsw);
  VTTS_CUDA(cudaMalloc(&ctx->hg_upsw, total * sizeof(float)));
  // ---- tensor-core path: bf16 hi/lo split + canonical K-major packing of every dense conv ----
  {
    size_t elems = 0;
    std::vector<size_t> eoff(72), uoff(32), poff(2);
    for (int n = 0; n < 12; ++n) {
      const int ch = 256 >> (n / 3), kk = vc::hg_rbk(n % 3);
      for (int q = 0; q < 6; ++q) {
        eoff[n * 6 + q] = elems;
        elems += vtts_tc_packed_elems(kk, ch, ch);
      }
    }
    int Cc = vc::HG_C0;
    for (int i = 0; i < 4; ++i) {
      for (int r = 0; r < vc::hg_rate(i); ++r) {
        uoff[i * 8 + r] = elems;
        elems += vtts_tc_packed_elems(2, Cc, Cc / 2);
      }
      Cc /= 2;
    }
    for (int t = 0; t < 2; ++t) {
      poff[t] = elems;
      elems += vtts_tc_packed_elems(7, vc::MEL, 256);
    }
    // CTA-pair layout of the convs the fused pair kernel runs (C <= 64), appended to the same allocation
    std::vector<size_t> coff(72, 0);
    size_t cbytes = 0;
    for (int n = 6; n < 12; ++n) {
      const int ch = 256 >> (n / 3), kk = vc::hg_rbk(n % 3);
      for (int q = 0; q < 6; ++q) {
        coff[n * 6 + q] = cbytes;
        cbytes += (vtts_tc_packed_pc_bytes(kk, ch) + 255) & ~size_t(255);
      }
    }
    const size_t base_bytes = (elems * 2 + 255) & ~size_t(255);
    if (ctx->hg_wpk) cudaFree(ctx->hg_wpk);
    VTTS_CUDA(cudaMalloc(&ctx->hg_wpk, base_bytes + cbytes));
    ctx->hg_wpc_t.assign(72, nullptr);
    for (int n = 6; n < 12; ++n) {
      const int ch = 256 >> (n / 3), kk = vc::hg_rbk(n % 3);
      for (int which = 0; which < 2; ++which)
        for (int m = 0; m < 3; ++m) {
          const int q = which * 3 + m;
          ctx->hg_wpc_t[n * 6 + q] = (char*)ctx->hg_wpk + base_bytes + coff[n * 6 + q];
          int rc = vtts_tc_pack_weights_pc(ctx, ctx->hg_t[hgi::RB_W(n, which, m)], ctx->hg_wpc_t[n * 6 + q], kk, ch);
          if (rc) return rc;
        }
    }
    ctx->hg_wpk_t.resize(72);
    ctx->hg_wpk_ups.assign(32, nullptr);
    for (int n = 0; n < 12; ++n) {
      const int ch = 256 >> (n / 3), kk = vc::hg_rbk(n % 3);
      for (int which = 0; which < 2; ++which)
        for (int m = 0; m < 3; ++m) {
          const int q = which * 3 + m;
          ctx->hg_wpk_t[n * 6 + q] = (char*)ctx->hg_wpk + eoff[n * 6 + q] * 2;
          int rc = vtts_tc_pack_weights(ctx, ctx->hg_t[hgi::RB_W(n, which, m)], ctx->hg_wpk_t[n * 6 + q], kk, ch, ch, 0, ch);
          if (rc) return rc;
        }
    }
    Cc = vc::HG_C0;
    for (int i = 0; i < 4; ++i) {
      for (int r = 0; r < vc::hg_rate(i); ++r) ctx->hg_wpk_ups[i * 8 + r] = (char*)ctx->hg_wpk + uoff[i * 8 + r] * 2;
      int rc = vtts_hg_ups_prepare(ctx, ctx->hg_t[hgi::UPS_W(i)], Cc, vc::hg_rate(i), vc::hg_upk(i), ctx->hg_upsw + offs[i],
                                   &ctx->hg_wpk_ups[i * 8]);
      if (rc) return rc;
      Cc /= 2;
    }
    for (int t = 0; t < 2; ++t) {
      ctx->hg_wpk_pre[t] = (char*)ctx->hg_wpk + poff[t] * 2;
      int rc = vtts_tc_pack_weights(ctx, ctx->hg_t[hgi::PRE_W], ctx->hg_wpk_pre[t], 7, vc::MEL, vc::HG_C0, 256 * t, 256);
      if (rc) return rc;
    }
  }
  VTTS_CUDA(cudaDeviceSynchronize());
  return VTTS_OK;
}

int vtts_hifigan_run(vtts_ctx* ctx, const float* mel, const int32_t* n_frames, int B, int T, float* wav, cudaStream_t st) {
  if (!ctx->hg_loaded) return ctx->fail(VTTS_ERR_NOT_LOADED, "hifigan weights not loaded");
  if (B < 1 || T < 1 || B > 65535) return ctx->fail(VTTS_ERR_BAD_ARG, "hifigan: B=%d T=%d", B, T);
  if ((int64_t)T * 256 > (int64_t)INT32_MAX / 64) return ctx->fail(VTTS_ERR_BAD_ARG, "hifigan: T=%d too long", T);
  size_t need = vtts_hifigan_ws_bytes(B, T);
  int rc = ctx->ensure_ws(need);
  if (rc) return rc;
  Arena ar(ctx->ws, ctx->ws_bytes, false);
  HgBufs hb;
  carve(ar, B, T, hb);
  auto& W = ctx->hg_t;

  ConvLaunch L;
  memset(&L, 0, sizeof(L));
  L.B = B;
  L.len = n_frames;

  ctx->sub_mark(8, st);
  // conv_pre: 80 -> 512, k7 pad 3
  L.nprob = 1;
  L.Cin = vc::MEL; L.Cout = vc::HG_C0;
  L.T_rows = T; L.rows_out = T; L.len_mul = 1;
  L.pre_mode = 0; L.pre_slope = 1.f; L.post_act = 0;
  L.p[0] = ConvProb{mel, nullptr, nullptr, W[hgi::PRE_W], W[hgi::PRE_B], nullptr, nullptr, nullptr, nullptr, hb.P0, 7, 1, -3, 1, 0};
  const bool tc = ctx->precision == 1;
  if (tc) {
    TcLaunch TL;
    memset(&TL, 0, sizeof(TL));
    TL.nprob = 2; TL.Cin = vc::MEL; TL.N = 256; TL.in_ld = vc::MEL; TL.out_ld = vc::HG_C0;
    TL.B = B; TL.T_rows = T; TL.rows_out = T; TL.len = n_frames; TL.len_mul = 1; TL.pre_mode = 0; TL.pre_slope = 1.f;
    for (int t = 0; t < 2; ++t)
      TL.p[t] = TcProb{mel, nullptr, nullptr, ctx->hg_wpk_pre[t], W[hgi::PRE_B] + 256 * t, nullptr, nullptr, nullptr, nullptr, hb.P0 + 256 * t, 7, 1, -3, 1, 0};
    rc = vtts_launch_tc_conv(ctx, TL, st);
  } else {
    rc = vtts_launch_conv(ctx, L, st);
  }
  if (rc) return rc;
  ctx->sub_mark(9, st);

  int C = vc::HG_C0;      // input channels of the stage
  int rows_in = T;        // rows per batch item entering the stage
  int scale_in = 1;       // rows_in = T*scale_in
  size_t ups_off = 0;     // offset of the stage's phase weights in ctx->hg_upsw
  for (int i = 0; i < 4; ++i) {
    const int u = vc::hg_rate(i), K = vc::hg_upk(i), Co = C / 2;
    const int par = i & 1;
    // ---- lrelu(0.1) [of the 3-way mean for i>0] -> ConvTranspose as u two-tap phases ----
    if (i == 0)
      rc = vtts_hg_ups_run(ctx, tc, hb.P0, nullptr, nullptr, ctx->hg_upsw + ups_off, &ctx->hg_wpk_ups[i * 8], W[hgi::UPS_B(i)],
                           n_frames, scale_in, B, rows_in, C, u, K, hb.X, st);
    else
      rc = vtts_hg_ups_run(ctx, tc, hb.A[par ^ 1][0], hb.A[par ^ 1][1], hb.A[par ^ 1][2], ctx->hg_upsw + ups_off,
                           &ctx->hg_wpk_ups[i * 8], W[hgi::UPS_B(i)], n_frames, scale_in, B, rows_in, C, u, K, hb.X, st);
    if (rc) return rc;
    ups_off += (size_t)u * 2 * C * Co;

    // ---- three ResBlock1 (k = 3,7,11), each 3 x [lrelu, conv(d), lrelu, conv(1), +x] ----
    const int rows = rows_in * u;
    const int scale = scale_in * u;
    for (int m = 0; m < 3; ++m) {
      const int d = vc::hg_dil(m);
      const float* src[3];
      for (int j = 0; j < 3; ++j) src[j] = (m == 0) ? hb.X : (m == 1 ? hb.A[par][j] : hb.Bb[j]);
      if (tc && ctx->fuse_pairs && Co <= 64) {
        // ---- fused pair: conv(d) -> lrelu -> conv(1) -> + x, intermediate kept on chip (tc_pair.cu) ----
        TcPairLaunch PL;
        memset(&PL, 0, sizeof(PL));
        PL.nprob = 3; PL.N = Co; PL.B = B; PL.T_rows = rows; PL.len = n_frames; PL.len_mul = scale; PL.slope = 0.1f;
        for (int j = 0; j < 3; ++j) {
          const int kk = vc::hg_rbk(j), n = i * 3 + j;
          PL.p[j] = TcPairProb{src[j], ctx->hg_wpk_t[n * 6 + m], ctx->hg_wpk_t[n * 6 + 3 + m], W[hgi::RB_B(n, 0, m)], W[hgi::RB_B(n, 1, m)],
                               (m == 1) ? hb.Bb[j] : hb.A[par][j], kk, d, ctx->hg_wpc_t[n * 6 + m], ctx->hg_wpc_t[n * 6 + 3 + m]};
        }
        rc = vtts_launch_tc_pair(ctx, PL, st);
        if (rc) return rc;
        continue;
      }
      if (tc) {
        // ---- bf16x3 tensor-core path (tc_conv.cu) ----
        TcLaunch TL;
        for (int which = 0; which < 2; ++which) {
          memset(&TL, 0, sizeof(TL));
          TL.nprob = 3; TL.Cin = Co; TL.N = Co; TL.in_ld = Co; TL.out_ld = Co;
          TL.B = B; TL.T_rows = rows; TL.rows_out = rows; TL.len = n_frames; TL.len_mul = scale;
          TL.pre_mode = 1; TL.pre_slope = 0.1f;
          for (int j = 0; j < 3; ++j) {
            const int kk = vc::hg_rbk(j), n = i * 3 + j;
            const int dd = which == 0 ? d : 1;
            TcProb p;
            memset(&p, 0, sizeof(p));
            p.x0 = which == 0 ? src[j] : hb.Tb[j];
            p.wpk = ctx->hg_wpk_t[n * 6 + which * 3 + m];
            p.bias = W[hgi::RB_B(n, which, m)];
            p.resid = which == 0 ? nullptr : src[j];
            p.out = which == 0 ? hb.Tb[j] : ((m == 1) ? hb.Bb[j] : hb.A[par][j]);
            p.k = kk; p.dil = dd; p.in_off = -((kk - 1) * dd) / 2; p.out_stride = 1; p.out_off = 0;
            TL.p[j] = p;
          }
          rc = vtts_launch_tc_conv(ctx, TL, st);
          if (rc) return rc;
        }
        continue;
      }
      // conv1 (dilated)
      memset(&L, 0, sizeof(L));
      L.B = B; L.len = n_frames; L.len_mul = scale;
      L.nprob = 3; L.Cin = Co; L.Cout = Co; L.T_rows = rows; L.rows_out = rows;
      L.pre_mode = 1; L.pre_slope = 0.1f; L.post_act = 0;
      for (int j = 0; j < 3; ++j) {
        const int kk = vc::hg_rbk(j), n = i * 3 + j;
        ConvProb p;
        memset(&p, 0, sizeof(p));
        p.x0 = src[j];
        p.w = W[hgi::RB_W(n, 0, m)]; p.bias = W[hgi::RB_B(n, 0, m)];
        p.out = hb.Tb[j];
        p.k = kk; p.dil = d; p.in_off = -((kk - 1) * d) / 2; p.out_stride = 1; p.out_off = 0;
        L.p[j] = p;
      }
      rc = vtts_launch_conv(ctx, L, st);
      if (rc) return rc;
      // conv2 (dilation 1) + residual
      for (int j = 0; j < 3; ++j) {
        const int kk = vc::hg_rbk(j), n = i * 3 + j;
        ConvProb p;
        memset(&p, 0, sizeof(p));
        p.x0 = hb.Tb[j];
        p.w = W[hgi::RB_W(n, 1, m)]; p.bias = W[hgi::RB_B(n, 1, m)];
        p.resid = src[j];
        p.out = (m == 1) ? hb.Bb[j] : hb.A[par][j];
        p.k = kk; p.dil = 1; p.in_off = -(kk - 1) / 2; p.out_stride = 1; p.out_off = 0;
        L.p[j] = p;
      }
      rc = vtts_launch_conv(ctx, L, st);
      if (rc) return rc;
    }
    C = Co;
    rows_in = rows;
    scale_in = scale;
    ctx->sub_mark(10 + i, st);
  }
  // ---- mean of 3, lrelu(0.01), conv_post (32 -> 1, k7), tanh ----
  {
    const int R = rows_in;  // 256*T
    dim3 grid((R + 255) / 256, B);
    conv_post_kernel<<<grid, 256, 0, st>>>(hb.A[1][0], hb.A[1][1], hb.A[1][2], W[hgi::POST_W], W[hgi::POST_B], n_frames, 256, R, wav);
    ctx->launches++;
    VTTS_CUDA(cudaGetLastError());
  }
  ctx->sub_mark(14, st);
  return VTTS_OK;
}
