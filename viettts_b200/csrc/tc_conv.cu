// Tensor-core NWC conv1d for sm_100a: implicit GEMM on tcgen05.mma with TMEM accumulators.
//
// Same operator as conv1d.cu (hk.Conv1D of vietTTS/hifigan/model.py:21-41 with the leaky_relu /
// 3-way-mean / bias / residual fusions), but the contraction runs on the 5th-gen tensor cores in
// "bf16x3" arithmetic:  every fp32 operand v is split into hi = bf16(v), lo = bf16(v - hi) and the
// product is accumulated in fp32 as  a_hi*w_hi + a_hi*w_lo + a_lo*w_hi  (the dropped a_lo*w_lo
// term and the split truncation are ~2^-17 relative; measured end-to-end waveform error of the
// whole generator vs float64: L-inf 1.7e-5, RMS 3.7e-6 -- see DESIGN.md).
//
// GEMM view per tap j:  D[time, cout] += A_j[time, cin] * W_j[cin, cout]
//   M = 128 time rows per MMA (TMEM lane = row), N = Cout (<= 256 TMEM columns), K = 16 channels.
//   A operand: activations in shared memory, K-major, NO swizzle, rows 16 B apart:
//       [plane hi|lo][k-half (8 ch)][row][8 x bf16]
//     so tap j / dilation d is just a start-address offset of j*d*16 bytes in the descriptor.
//   B operand: weights pre-split and pre-packed at load time into the same canonical layout,
//     streamed with cp.async.bulk (TMA bulk copy) through a 4-stage mbarrier ring.
//
// One persistent CTA per SM, 18 warps:
//   warps 0-3, 14-17  epilogue (two groups, alternate 32-column chunks): tcgen05.ld TMEM -> regs -> smem slab ->
//              coalesced + bias (+ BN/act) (+ residual) fp32 NWC store
//   warp  4    MMA issue  (one lane) + TMEM alloc/dealloc
//   warp  5    weight producer (one lane, cp.async.bulk + expect_tx)
//   warps 6-13 activation converters: fp32 global -> [mean3] -> leaky_relu -> hi/lo bf16 -> smem
// A "super tile" is MT = min(4, 512/N) M-tiles (128*MT rows) that share every weight stage, so a
// weight block fetched from L2 feeds MT MMAs.
//
// N >= 128 runs in the CTA-PAIR form by default (template parameter PAIR, tc_variant 3): the grid is 74 clusters of two
// CTAs, a tile is 2 x 128*MT rows, and rank 0 issues `tcgen05.mma.cta_group::2` (M = 256) for both SMs: each CTA
// converts its own rows and fetches only ITS HALF of every weight block, so the shared-memory operand bytes per MMA drop
// from 8 KB to 6 KB (N = 128) and the instruction runs at the math rate (66 instead of 97 clk, scripts/umma_probe3.cu).
//   * barriers the issuer waits on (a_full, w_full, tmem_empty) live in rank 0 and count the arrivals of both CTAs;
//     rank 1's threads arrive through `mapa` + `mbarrier.arrive.shared::cluster` (release at CTA scope -- a cluster-
//     scope release costs ~1000 clk per arrive), rank 1's otherwise idle warp 4 forwards its weight-stage completions;
//   * `tcgen05.commit ... multicast::cluster` frees the stages / publishes the accumulators in both CTAs at once;
//   * weight stages are grouped four taps per barrier so that the issuing warp spends one wait + one elected region
//     per 24 MMAs (its loop otherwise costs about as much as the MMAs of one tap take at the math rate).
#include <cuda_bf16.h>

#include <algorithm>

#include "tc_common.cuh"
#include "vtts_internal.cuh"

namespace {

using namespace tcx;

constexpr int NA_DEFAULT = 4;       // activation stages (single-CTA form)
constexpr int NW_MAX = 8;            // weight stages: 6 x 16 KB for N = 256, 8 smaller ones otherwise (covers the L2 latency)
constexpr int COLL = 1;          // A-operand collector reuse between the a_hi x W_hi and a_hi x W_lo MMAs
constexpr int NTHREADS = 576;     // 4 epilogue + MMA + weight producer + 8 converter + 4 more epilogue warps
constexpr int NEPI = 256;         // epilogue threads (two groups of 4 warps; warp % 4 = TMEM lane quadrant)
constexpr int NCONV = 256;        // converter threads
constexpr int NGRP = 2;           // independent converter groups (alternate chunks -> two chunks in flight)
constexpr int GRP_THREADS = NCONV / NGRP;

// MT  = M-tiles (128 rows) per super tile, NPH = output phases accumulated per tile (ConvTranspose), the
// accumulator set of a tile is NPH*MT*N TMEM columns; two sets (epilogue overlaps the next tile's MMAs) when
// they fit in the 512 columns.
// PAIR = 1: two CTAs of a cluster work as one (tcgen05 cta_group::2, M = 256): each CTA converts the activations of its
// own 128*MT rows and fetches HALF of every weight block (the output columns [N/2 r, N/2 r + N/2) of rank r), the MMAs
// are issued by rank 0 for both SMs -- the shared-memory operand traffic per FLOP drops by the weight half, which is
// what bounds the single-CTA form (scripts/umma_probe3.cu: 66 instead of 97 clk per N=128 MMA).
template <int N, int MT_, int NPH_, int STK_ = 0, int PAIR_ = 0>
struct TcCfg {
  static constexpr int MT = MT_;
  static constexpr int NPH = NPH_;
  static constexpr int STK = STK_;            // 1: A_hi x [W_hi | W_lo] as ONE MMA of width 2N (main | aux accumulator columns)
  static constexpr int PAIR = PAIR_;
  static constexpr int CPP = PAIR ? 2 : 1;    // CTAs per tile
  static constexpr int NB = N / CPP;          // weight rows (output columns) held by one CTA
  static_assert(!(PAIR && STK), "the pair form keeps three MMAs per product");
  static constexpr int DW = STK ? 2 * N : N;  // accumulator columns per (phase, M tile)
  // weight ring: NW groups of G taps behind ONE barrier pair each.  The pair form's MMAs run at the math rate (6 MMAs of
  // a tap = 384 clk), which is about what one wait + one elected issue region + one commit cost the issuing warp, so
  // it handles G = 4 taps per region; the single-CTA form (>= 510 clk of MMAs per tap) keeps G = 1.
  static constexpr int G = PAIR_ ? 4 : 1;
  static constexpr int NW = PAIR_ ? (N == 256 ? 3 : 4) : (N == 256 ? 6 : ((N == 128 && MT_ == 4) ? 4 : NW_MAX));
  static constexpr int NA = NA_DEFAULT;   // (6 stages in the pair form measured slower: the converters then crowd out the epilogue's loads)
  static constexpr int R = 128 * MT;          // output rows per super tile
  static constexpr int RA = R + 64;           // allocated activation rows per stage (halo <= 50)
  static constexpr int A_STAGE = RA * 64;     // bytes: 2 planes x 2 k-halves x RA rows x 16 B
  static constexpr int W_STAGE = NB * 64;     // bytes: 2 planes x 2 k-halves x NB rows x 16 B
  static constexpr int W_BLOCK = N * 64;      // bytes of one packed (chunk, tap) block in global memory
  static constexpr int W_GROUP = G * W_STAGE; // bytes of one ring slot
  static constexpr int ACC_COLS = NPH * MT * DW;
  static_assert(ACC_COLS <= 512, "accumulators exceed TMEM");
  static constexpr int NACC = (2 * ACC_COLS <= 512) ? 2 : 1;
  static constexpr int TMEM_RAW = NACC * ACC_COLS;
  static constexpr int TMEM_COLS = TMEM_RAW <= 32 ? 32 : (TMEM_RAW <= 64 ? 64 : (TMEM_RAW <= 128 ? 128 : (TMEM_RAW <= 256 ? 256 : 512)));
  static constexpr int NBAR = 2 * NA + 2 * NW + 2 * NACC;
  static constexpr int EPI_PITCH = 144;                      // bytes per staged row: 32 floats + 16 B pad (conflict-free)
  static constexpr int EPI_STAGE = 8 * 32 * EPI_PITCH;       // one 32-row slab per epilogue warp
  static constexpr int SMEM_BYTES = NA * A_STAGE + NW * W_GROUP + EPI_STAGE + NBAR * 8 + 16 + 1024;
};

// EPI = 0: bias (+ residual) only -- the HiFiGAN generator's hot path.  EPI = 1: bias, eval BatchNorm,
// tanh / relu, residual, partial N tile (acoustic model convs and GEMMs).
template <int N, int EPI, int MT_, int NPH_, int STK_, int PAIR_>
__global__ void __launch_bounds__(NTHREADS, 1) tc_conv_kernel(const __grid_constant__ TcLaunch L) {
  using Cfg = TcCfg<N, MT_, NPH_, STK_, PAIR_>;
  constexpr int MT = Cfg::MT, R = Cfg::R, RA = Cfg::RA, NPH = Cfg::NPH, STK = Cfg::STK, DW = Cfg::DW, NW = Cfg::NW;
  constexpr int PAIR = Cfg::PAIR, CPP = Cfg::CPP, NB = Cfg::NB, G = Cfg::G, NA = Cfg::NA;
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = (uint8_t*)(((uintptr_t)smem_raw + 1023) & ~(uintptr_t)1023);
  uint8_t* a_st = smem;
  constexpr int NACC = Cfg::NACC;
  uint8_t* w_st = smem + NA * Cfg::A_STAGE;
  uint8_t* epi_st = w_st + NW * Cfg::W_GROUP;
  uint64_t* bars = reinterpret_cast<uint64_t*>(epi_st + Cfg::EPI_STAGE);
  uint64_t* a_full = bars;
  uint64_t* a_empty = bars + NA;
  uint64_t* w_full = bars + 2 * NA;
  uint64_t* w_empty = bars + 2 * NA + NW;
  uint64_t* tmem_full = bars + 2 * NA + 2 * NW;          // [NACC]
  uint64_t* tmem_empty = tmem_full + NACC;               // [NACC]
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tmem_empty + NACC);

  const int tid = threadIdx.x, lane = tid & 31;
  // warp index broadcast from lane 0: provably warp-uniform, so role code can live on the uniform datapath
  const int warp = __shfl_sync(0xffffffffu, tid >> 5, 0);
  // pair form: the barriers the issuer (rank 0) waits on collect the arrivals of BOTH CTAs (the peer arrives through
  // the cluster address space); a_empty / w_empty / tmem_full are signalled in both CTAs by the multicast commit
  const uint32_t prank = PAIR ? cluster_rank() : 0u;

  if (warp == 5 && lane == 0) {
    for (int i = 0; i < NA; ++i) { mbar_init(&a_full[i], CPP * GRP_THREADS); mbar_init(&a_empty[i], 1); }
    for (int i = 0; i < NW; ++i) { mbar_init(&w_full[i], (PAIR && prank == 0) ? 2 : 1); mbar_init(&w_empty[i], 1); }
    for (int i = 0; i < NACC; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], CPP * NEPI); }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 4) {
    if constexpr (PAIR) {
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) cluster_sync_all();     // the peer's barriers exist before anything is signalled across
  tc_fence_after();
  const uint32_t tmem_base = __shfl_sync(0xffffffffu, *tmem_slot, 0);

  const int Cin = L.Cin;
  const int nch = Cin / 16;
  const int tiles_per_row = L.tiles_per_row;
  const int ntiles = L.ntiles;
  const int tiles_per_prob = tiles_per_row * L.B;

  // every role walks the same tile sequence
#define TILE_LOOP_BEGIN                                                        \
  for (int tile = blockIdx.x / CPP; tile < ntiles; tile += gridDim.x / CPP) {  \
    const int pi = L.problem_major ? tile / tiles_per_prob : tile % L.nprob;    \
    const int rest = L.problem_major ? tile - pi * tiles_per_prob : tile / L.nprob; \
    const int tt = rest % tiles_per_row;                                       \
    const int b = rest / tiles_per_row;                                        \
    const int tau0 = (tt * CPP + (int)prank) * R;                              \
    int valid = L.T_rows;                                                      \
    if (L.len) {                                                               \
      const int v = L.len[b] * L.len_mul;                                      \
      valid = v < valid ? v : valid;                                           \
    }                                                                          \
    if (tt * CPP * R >= valid) continue;     /* the same decision in both CTAs of a pair */ \
    const TcProb& P = L.p[pi];                                                 \
    int sh_min = P.in_off_ph[0], sh_max = P.in_off_ph[0];                      \
    _Pragma("unroll") for (int ph_ = 1; ph_ < NPH; ++ph_) {                    \
      sh_min = P.in_off_ph[ph_] < sh_min ? P.in_off_ph[ph_] : sh_min;          \
      sh_max = P.in_off_ph[ph_] > sh_max ? P.in_off_ph[ph_] : sh_max;          \
    }
#define TILE_LOOP_END }

  if (warp == 4 && PAIR && prank != 0) {
    // ============================ pair form, rank 1: weight-stage forwarder ============================
    // this CTA's half of a weight block lands on its own w_full (bulk-copy complete_tx); tell the issuer in rank 0
    uint32_t sw = 0, pw = 0;
    long long w_w = 0;
    TILE_LOOP_BEGIN
      (void)b; (void)tau0; (void)sh_max;
      const int k = P.k;
      const int nst = nch * NPH * ((k + G - 1) / G);
      for (int s = 0; s < nst; ++s) {
        mbar_wait_t(&w_full[sw], pw, L.err, 3, w_w);
        // (release at CTA scope: the data was written by the bulk copy, not by this thread.  A release at CLUSTER scope
        //  costs ~1000 clk per arrive and made this hop the bottleneck of the whole kernel: VTTS_PAIR_EXP=4 shows it)
        if (elect_one()) { if (L.exp & 4) mbar_arrive_rank<1>(&w_full[sw], 0); else mbar_arrive_rank<0>(&w_full[sw], 0); }
        __syncwarp();
        if (++sw == NW) { sw = 0; pw ^= 1; }
      }
    TILE_LOOP_END
    if (L.dbg && lane == 0) L.dbg[(size_t)blockIdx.x * 16 + 3] = w_w;
  } else if (warp == 4) {
    // ============================ MMA issuer ============================
    // The whole warp walks the pipeline (uniform control flow, operands in uniform registers); only the
    // tcgen05.mma / tcgen05.commit instructions themselves are predicated on one elected lane.
    {
      constexpr uint32_t idesc = PAIR ? make_idesc2(N) : make_idesc(N);
      uint32_t sa = 0, pa = 0, sw = 0, pw = 0, acc = 0, tph = 0;
      long long w_tmem = 0, w_a = 0, w_w = 0;
      const long long t_begin = clock64();
      const uint32_t a_st_u32 = smem_u32(a_st), w_st_u32 = smem_u32(w_st);
      // descriptor templates: start address added per use (row stride 16 B == 1 descriptor address unit)
      const uint64_t a_tmpl = make_desc(0, RA * 16, 128);
      const uint64_t b_tmpl = make_desc(0, 2 * NB * 16, 128);    // k-half blocks are 2 NB rows apart ([hi rows | lo rows])
      constexpr uint32_t idesc2 = make_idesc(2 * N <= 256 ? 2 * N : N);
      TILE_LOOP_BEGIN
        (void)b; (void)tau0;
        const int k = P.k, dil = P.dil;
        if constexpr (PAIR) { if (L.exp & 1) mbar_wait_tc<1>(&tmem_empty[acc], tph ^ 1, L.err, 1, w_tmem); else mbar_wait_tc(&tmem_empty[acc], tph ^ 1, L.err, 1, w_tmem); }
        else mbar_wait_t(&tmem_empty[acc], tph ^ 1, L.err, 1, w_tmem);
        tc_fence_after();
        const uint32_t d0 = tmem_base + acc * Cfg::ACC_COLS;
        for (int c = 0; c < nch; ++c) {
          if constexpr (PAIR) { if (L.exp & 1) mbar_wait_tc<1>(&a_full[sa], pa, L.err, 2, w_a); else mbar_wait_tc(&a_full[sa], pa, L.err, 2, w_a); }
          else mbar_wait_t(&a_full[sa], pa, L.err, 2, w_a);
          tc_fence_after();
          const uint32_t a_base16 = (a_st_u32 + sa * Cfg::A_STAGE) >> 4;
#pragma unroll 1
          for (int ph = 0; ph < NPH; ++ph) {
            const int shift = P.in_off_ph[ph] - sh_min;
            for (int j0 = 0; j0 < k; j0 += G) {
              if constexpr (PAIR) { if (L.exp & 1) mbar_wait_tc<1>(&w_full[sw], pw, L.err, 3, w_w); else mbar_wait_tc(&w_full[sw], pw, L.err, 3, w_w); }
              else mbar_wait_t(&w_full[sw], pw, L.err, 3, w_w);
              tc_fence_after();
              const int gn = (G == 1 || k - j0 >= G) ? G : k - j0;     // taps in this group
              if (elect_one()) {
               for (int jj = 0; jj < gn; ++jj) {
                const int j = j0 + jj;
                const uint32_t w_base16 = (w_st_u32 + sw * Cfg::W_GROUP + jj * Cfg::W_STAGE) >> 4;
                const uint64_t b_hi = b_tmpl | (uint64_t)w_base16;
                const uint64_t b_lo = b_tmpl | (uint64_t)(w_base16 + NB);
                const uint32_t first = (c | j) != 0 ? 1u : 0u;
#pragma unroll
                for (int mt = 0; mt < MT; ++mt) {
                  const uint32_t row = a_base16 + mt * 128 + shift + j * dil;
                  const uint64_t a_hi = a_tmpl | (uint64_t)row;
                  const uint64_t a_lo = a_tmpl | (uint64_t)(row + 2 * RA);
                  const uint32_t d = d0 + (ph * MT + mt) * DW;
                  if constexpr (PAIR) {
                    umma2<1>(d, a_hi, b_hi, idesc, first);
                    umma2<2>(d, a_hi, b_lo, idesc, 1u);
                    umma2<0>(d, a_lo, b_hi, idesc, 1u);
                  } else if constexpr (STK) {
                    umma(d, a_hi, b_hi, idesc2, first);     // [main | aux] (+)= A_hi . [W_hi | W_lo]
                    umma(d, a_lo, b_hi, idesc, 1u);         // main += A_lo . W_hi
                  } else {
                    umma<COLL ? 1 : 0>(d, a_hi, b_hi, idesc, first);
                    umma<COLL ? 2 : 0>(d, a_hi, b_lo, idesc, 1u);
                    umma(d, a_lo, b_hi, idesc, 1u);
                  }
                }
               }
                if constexpr (PAIR) umma_commit2(&w_empty[sw]); else umma_commit(&w_empty[sw]);
              }
              if (++sw == NW) { sw = 0; pw ^= 1; }
            }
          }
          if (elect_one()) { if constexpr (PAIR) umma_commit2(&a_empty[sa]); else umma_commit(&a_empty[sa]); }
          if (++sa == NA) { sa = 0; pa ^= 1; }
        }
        if (elect_one()) { if constexpr (PAIR) umma_commit2(&tmem_full[acc]); else umma_commit(&tmem_full[acc]); }
        if (++acc == NACC) { acc = 0; tph ^= 1; }
      TILE_LOOP_END
      if (L.dbg && lane == 0) {
        long long* d = L.dbg + (size_t)blockIdx.x * 16;
        d[0] = clock64() - t_begin; d[1] = w_tmem; d[2] = w_a; d[3] = w_w;
      }
    }
    __syncwarp();
  } else if (warp == 5) {
    // ============================ weight producer ============================
    if (PAIR || lane == 0) {
      // (pair form: the whole warp walks the loop and one elected lane issues, so the four bulk copies of a stage
      //  come from uniform code)
      uint32_t sw = 0, pw = 0;
      long long w_e = 0;
      TILE_LOOP_BEGIN
        const int k = P.k;
        (void)b; (void)tau0;
        for (int c = 0; c < nch; ++c)
          for (int ph = 0; ph < NPH; ++ph) {
            const uint8_t* wsrc = reinterpret_cast<const uint8_t*>(P.wpk_ph[ph]) + (size_t)c * k * Cfg::W_BLOCK;
            for (int j = 0; j < k; j += G) {
              mbar_wait_t(&w_empty[sw], pw ^ 1, L.err, 4, w_e);
              if constexpr (PAIR) {
                // the packed block is [k-half][plane][N rows][16 B]: this CTA's NB rows of each of the four sub-blocks
                const int gn = k - j >= G ? G : k - j;
                if (elect_one()) {
                  mbar_expect_tx(&w_full[sw], gn * Cfg::W_STAGE);
                  for (int jj = 0; jj < gn; ++jj) {
#pragma unroll
                    for (int sb = 0; sb < 4; ++sb)
                      bulk_g2s(w_st + sw * Cfg::W_GROUP + jj * Cfg::W_STAGE + sb * NB * 16,
                               wsrc + (size_t)(j + jj) * Cfg::W_BLOCK + (size_t)(sb * N + prank * NB) * 16, NB * 16, &w_full[sw]);
                  }
                }
                __syncwarp();
              } else {
                mbar_expect_tx(&w_full[sw], Cfg::W_STAGE);
                bulk_g2s(w_st + sw * Cfg::W_STAGE, wsrc + (size_t)j * Cfg::W_BLOCK, Cfg::W_STAGE, &w_full[sw]);
              }
              if (++sw == NW) { sw = 0; pw ^= 1; }
            }
          }
      TILE_LOOP_END
      if (L.dbg && lane == 0) L.dbg[(size_t)blockIdx.x * 16 + 4] = w_e;
    }
    __syncwarp();
  } else if (warp >= 6 && warp < 14) {
    // ============================ activation converters ============================
    // Two groups of 4 warps; group g fills the chunks with (global chunk counter) % 2 == g, so one group's
    // memory round trip overlaps the other's convert+store phase.
    const int ct = tid - 192;                 // 0..255
    const int grp = ct / GRP_THREADS;         // 0..1
    const int gt = ct - grp * GRP_THREADS;    // 0..127 inside the group
    const int q = gt & 3;                     // 4-channel group inside the 16-channel chunk
    const int r0 = gt >> 2;                   // 0..31
    const int pre_mode = L.pre_mode;
    const float slope = L.pre_slope;
    const int ld = L.in_ld;
    uint32_t item = 0;                        // global chunk counter (same sequence in both groups and the MMA warp)
    long long w_ae = 0, t_fill = 0;
    TILE_LOOP_BEGIN
      const int k = P.k, dil = P.dil;
      const int rows = R + (k - 1) * dil + (sh_max - sh_min);
      const size_t in_base = (size_t)b * L.T_rows * ld;
      const float* x0 = P.x0 + in_base;
      const float* x1 = pre_mode == 2 ? P.x1 + in_base : nullptr;
      const float* x2 = pre_mode == 2 ? P.x2 + in_base : nullptr;
      const int row_base = tau0 + sh_min;
      for (int c = 0; c < nch; ++c, ++item) {
        if ((int)(item % NGRP) != grp) continue;
        const uint32_t sa = item % NA, pa = (item / NA) & 1;
        mbar_wait_t(&a_empty[sa], pa ^ 1, L.err, 5, w_ae);
        const long long tf0 = clock64();
        uint8_t* st = a_st + sa * Cfg::A_STAGE + ((q >> 1) * RA) * 16 + (q & 1) * 8;
        const int coff = c * 16 + q * 4;
        constexpr int U = 10;          // loads in flight per thread (memory-level parallelism)
        for (int rr0 = r0; rr0 < rows; rr0 += 32 * U) {
          float4 v[U];
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int rr = rr0 + u * 32;
            const int t = row_base + rr;
            v[u] = make_float4(0.f, 0.f, 0.f, 0.f);
            if (rr < rows && t >= 0 && t < valid) {
              const size_t off = (size_t)t * ld + coff;
              v[u] = ldg_pf256(x0 + off);
              if (pre_mode == 2) {
                const float4 a = ldg_pf256(x1 + off);
                const float4 bb = ldg_pf256(x2 + off);
                v[u].x = ((v[u].x + a.x) + bb.x) / 3.0f;
                v[u].y = ((v[u].y + a.y) + bb.y) / 3.0f;
                v[u].z = ((v[u].z + a.z) + bb.z) / 3.0f;
                v[u].w = ((v[u].w + a.w) + bb.w) / 3.0f;
              }
            }
          }
#pragma unroll
          for (int u = 0; u < U; ++u) {
            const int rr = rr0 + u * 32;
            if (rr < rows) {
              float4 x = v[u];
              if (pre_mode >= 1) {
                x.x = lrelu(x.x, slope); x.y = lrelu(x.y, slope); x.z = lrelu(x.z, slope); x.w = lrelu(x.w, slope);
              }
              uint2 hi, lo;
              split4(x, hi, lo);
              *reinterpret_cast<uint2*>(st + (size_t)rr * 16) = hi;
              *reinterpret_cast<uint2*>(st + (size_t)(2 * RA + rr) * 16) = lo;
            }
          }
        }
        fence_proxy_async();
        if constexpr (PAIR) mbar_arrive_rank<0>(&a_full[sa], 0); else mbar_arrive(&a_full[sa]);
        t_fill += clock64() - tf0;
      }
    TILE_LOOP_END
    if (L.dbg && gt == 0) { L.dbg[(size_t)blockIdx.x * 16 + 5 + 4 * grp] = w_ae; L.dbg[(size_t)blockIdx.x * 16 + 6 + 4 * grp] = t_fill; }
  } else {
    // ============================ epilogue (warps 0-3 and 14-17) ============================
    // TMEM -> registers (thread = row) -> per-warp padded smem slab -> registers (8 lanes = one 128 B row
    // segment) so that the residual loads and the stores are fully coalesced.  Two groups of four warps take
    // alternate 32-column chunks; each group prefetches the residuals of its next chunk.
    const int eg = warp >= 14 ? 1 : 0;      // epilogue group
    const int quad = warp & 3;              // TMEM lane quadrant of this warp
    uint32_t acc = 0, tph = 0;
    const int out_ld = L.out_ld;
    long long w_tf = 0, t_epi = 0;
    uint8_t* slab = epi_st + (eg * 4 + quad) * (32 * Cfg::EPI_PITCH);
    const int trow = lane >> 3;          // 0..3   row inside a group of 4
    const int tch = lane & 7;            // 16 B chunk inside the 128 B row segment
    constexpr int NCHUNK = N / 32;
    constexpr int NIT = NPH * MT * NCHUNK;
    const int n_valid = (EPI && L.n_valid > 0) ? L.n_valid : N;
    const int post_act = EPI ? L.post_act : 0;
    TILE_LOOP_BEGIN
      const size_t out_base = (size_t)b * L.rows_out * out_ld;
      const int ostride = P.out_stride;
      const float* __restrict__ resid = P.resid;
      const int row_w = tau0 + quad * 32;          // first row of this warp inside M-tile 0
      // residual registers rotate: rs[s8] of this group's NEXT chunk is requested right after rs[s8] of the current
      // chunk has been consumed, so one set of 8 float4 covers a whole chunk iteration of load latency
      float4 rs[8];
      auto load_resid_row = [&](int it, int s8) -> float4 {
        const int pm = it / NCHUNK, c0 = (it - pm * NCHUNK) * 32;
        const int mt = pm % MT, ooff = P.out_off_ph[pm / MT];
        const int tau = row_w + mt * 128 + s8 * 4 + trow;
        float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
        if (resid && tau < valid && c0 + tch * 4 < n_valid)
          v = __ldg(reinterpret_cast<const float4*>(resid + out_base + (size_t)(tau * ostride + ooff) * out_ld + c0 + tch * 4));
        return v;
      };
      if (eg < NIT) {
#pragma unroll
        for (int s8 = 0; s8 < 8; ++s8) rs[s8] = load_resid_row(eg, s8);
      }
      mbar_wait_t(&tmem_full[acc], tph, L.err, 6, w_tf);
      const long long te0 = clock64();
      tc_fence_after();
      const uint32_t taddr0 = tmem_base + ((uint32_t)(quad * 32) << 16) + acc * Cfg::ACC_COLS;
#pragma unroll 1
      for (int it = eg; it < NIT; it += 2) {
        const int pm = it / NCHUNK, c0 = (it - pm * NCHUNK) * 32;
        const int mt = pm % MT, ooff = P.out_off_ph[pm / MT];
        {
          uint32_t r[32];
          tmem_ld16(taddr0 + pm * DW + c0, r);
          tmem_ld16(taddr0 + pm * DW + c0 + 16, r + 16);
          if constexpr (STK) {
            uint32_t r2[32];
            tmem_ld16(taddr0 + pm * DW + N + c0, r2);
            tmem_ld16(taddr0 + pm * DW + N + c0 + 16, r2 + 16);
            tmem_ld_wait();
#pragma unroll
            for (int q = 0; q < 32; ++q) r[q] = __float_as_uint(__uint_as_float(r[q]) + __uint_as_float(r2[q]));
          } else {
            tmem_ld_wait();
          }
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<uint4*>(slab + lane * Cfg::EPI_PITCH + q * 16) = make_uint4(r[q * 4], r[q * 4 + 1], r[q * 4 + 2], r[q * 4 + 3]);
        }
        __syncwarp();
        const bool col_ok = !EPI || (c0 + tch * 4 < n_valid);
        float4 bi = make_float4(0.f, 0.f, 0.f, 0.f), mu = bi, iv = make_float4(1.f, 1.f, 1.f, 1.f), of = bi;
        if (col_ok) {
          bi = __ldg(reinterpret_cast<const float4*>(P.bias + c0 + tch * 4));
          if (EPI && P.bn_mean) {
            mu = __ldg(reinterpret_cast<const float4*>(P.bn_mean + c0 + tch * 4));
            iv = __ldg(reinterpret_cast<const float4*>(P.bn_inv + c0 + tch * 4));
            of = __ldg(reinterpret_cast<const float4*>(P.bn_off + c0 + tch * 4));
          }
        }
#pragma unroll
        for (int s8 = 0; s8 < 8; ++s8) {
          const int rl = s8 * 4 + trow;
          const int tau = row_w + mt * 128 + rl;
          const float4 a = *reinterpret_cast<const float4*>(slab + rl * Cfg::EPI_PITCH + tch * 16);
          float4 o;
          o.x = a.x + bi.x; o.y = a.y + bi.y; o.z = a.z + bi.z; o.w = a.w + bi.w;
          if (EPI && P.bn_mean) {
            o.x = (o.x - mu.x) * iv.x + of.x; o.y = (o.y - mu.y) * iv.y + of.y;
            o.z = (o.z - mu.z) * iv.z + of.z; o.w = (o.w - mu.w) * iv.w + of.w;
          }
          if (EPI && post_act == 1) { o.x = tanhf(o.x); o.y = tanhf(o.y); o.z = tanhf(o.z); o.w = tanhf(o.w); }
          else if (EPI && post_act == 2) { o.x = fmaxf(o.x, 0.f); o.y = fmaxf(o.y, 0.f); o.z = fmaxf(o.z, 0.f); o.w = fmaxf(o.w, 0.f); }
          o.x += rs[s8].x; o.y += rs[s8].y; o.z += rs[s8].z; o.w += rs[s8].w;
          if (tau < valid && col_ok)
            *reinterpret_cast<float4*>(P.out + out_base + (size_t)(tau * ostride + ooff) * out_ld + c0 + tch * 4) = o;
          if (it + 2 < NIT) rs[s8] = load_resid_row(it + 2, s8);
        }
        __syncwarp();
      }
      tc_fence_before();
      if constexpr (PAIR) mbar_arrive_rank<0>(&tmem_empty[acc], 0); else mbar_arrive(&tmem_empty[acc]);
      t_epi += clock64() - te0;
      if (++acc == NACC) { acc = 0; tph ^= 1; }
    TILE_LOOP_END
    if (L.dbg && tid == 0) { L.dbg[(size_t)blockIdx.x * 16 + 7] = w_tf; L.dbg[(size_t)blockIdx.x * 16 + 8] = t_epi; }
  }
#undef TILE_LOOP_BEGIN
#undef TILE_LOOP_END

  tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) cluster_sync_all();     // nobody leaves while the peer may still signal into this CTA's shared memory
  if (warp == 4) {
    tc_fence_after();
    if constexpr (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"((uint32_t)Cfg::TMEM_COLS) : "memory");
  }
}

// fp32 Haiku conv weight w[k][Cin][Cout_total] -> packed bf16 blocks for output columns [n0, n0+N):
//   [chunk c = Cin/16][tap j][k-half][plane hi|lo][n][8]
__global__ void pack_w_kernel(const float* __restrict__ w, __nv_bfloat16* __restrict__ dst, int k, int Cin, int Cout_total, int n0, int N) {
  const size_t total = (size_t)k * Cin * N;
  for (size_t idx = blockIdx.x * (size_t)blockDim.x + threadIdx.x; idx < total; idx += (size_t)gridDim.x * blockDim.x) {
    const int n = idx % N;
    const int i = (idx / N) % Cin;
    const int j = idx / ((size_t)N * Cin);
    const float v = (n0 + n) < Cout_total ? w[((size_t)j * Cin + i) * Cout_total + n0 + n] : 0.f;
    const __nv_bfloat16 hi = __float2bfloat16_rn(v);
    const __nv_bfloat16 lo = __float2bfloat16_rn(v - __bfloat162float(hi));
    const int c = i / 16, kh = (i % 16) / 8, e = i % 8;
    const size_t blk = ((size_t)c * k + j) * (size_t)(4 * N * 8);
    dst[blk + ((size_t)(kh * 2 + 0) * N + n) * 8 + e] = hi;   // [k-half][plane hi|lo][n][8]: hi and lo rows of a k-half are
    dst[blk + ((size_t)(kh * 2 + 1) * N + n) * 8 + e] = lo;   // adjacent, so [W_hi | W_lo] is also one 2N-row operand
  }
}

template <int N, int EPI, int MT, int NPH, int STK = 0, int PAIR = 0>
int launch_cfg(vtts_ctx* ctx, TcLaunch& L, cudaStream_t st) {
  using Cfg = TcCfg<N, MT, NPH, STK, PAIR>;
  // function attributes and cluster occupancy are per device (a process may hold contexts on several GPUs)
  static bool attr_done_dev[64] = {};
  static int max_pairs_dev[64] = {};
  bool& attr_done = attr_done_dev[ctx->device & 63];
  int& max_pairs = max_pairs_dev[ctx->device & 63];
  if (!attr_done) {
    VTTS_CUDA(cudaFuncSetAttribute(tc_conv_kernel<N, EPI, MT, NPH, STK, PAIR>, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg::SMEM_BYTES));
    if (PAIR) {
      cudaLaunchConfig_t qc = {};
      cudaLaunchAttribute qa[1];
      qa[0].id = cudaLaunchAttributeClusterDimension;
      qa[0].val.clusterDim.x = 2; qa[0].val.clusterDim.y = 1; qa[0].val.clusterDim.z = 1;
      qc.gridDim = dim3(ctx->sm_count & ~1); qc.blockDim = dim3(NTHREADS); qc.dynamicSmemBytes = Cfg::SMEM_BYTES; qc.attrs = qa; qc.numAttrs = 1;
      VTTS_CUDA(cudaOccupancyMaxActiveClusters(&max_pairs, tc_conv_kernel<N, EPI, MT, NPH, STK, PAIR>, &qc));
      if (max_pairs < 1) return ctx->fail(VTTS_ERR_CUDA, "tc_conv: no CTA pair fits on this device");
      if (max_pairs > ctx->sm_count / 2) max_pairs = ctx->sm_count / 2;
    }
    attr_done = true;
  }
  for (int i = 0; i < L.nprob; ++i) {
    if (NPH == 1) {   // single-phase problems describe themselves with the scalar fields
      L.p[i].wpk_ph[0] = L.p[i].wpk;
      L.p[i].in_off_ph[0] = L.p[i].in_off;
      L.p[i].out_off_ph[0] = L.p[i].out_off;
    }
    int mn = L.p[i].in_off_ph[0], mx = mn;
    for (int ph = 1; ph < NPH; ++ph) { mn = std::min(mn, L.p[i].in_off_ph[ph]); mx = std::max(mx, L.p[i].in_off_ph[ph]); }
    if ((L.p[i].k - 1) * L.p[i].dil + (mx - mn) > 50) return ctx->fail(VTTS_ERR_BAD_ARG, "tc_conv: halo too large");
  }
  // static round-robin tile assignment: put the expensive problems (large k) first so that the last, partial
  // wave of tiles consists of cheap ones
  std::stable_sort(L.p, L.p + L.nprob, [](const TcProb& a, const TcProb& b) { return a.k > b.k; });
  L.tiles_per_row = (L.T_rows + Cfg::CPP * Cfg::R - 1) / (Cfg::CPP * Cfg::R);
  L.ntiles = L.nprob * L.tiles_per_row * L.B;
  if (PAIR) {
    // persistent CTA pairs: clusters of two CTAs (same TPC), one pair per tile
    cudaLaunchConfig_t lc = {};
    cudaLaunchAttribute la[1];
    la[0].id = cudaLaunchAttributeClusterDimension;
    la[0].val.clusterDim.x = 2; la[0].val.clusterDim.y = 1; la[0].val.clusterDim.z = 1;
    const int pairs = L.ntiles < max_pairs ? L.ntiles : max_pairs;
    lc.gridDim = dim3(2 * pairs); lc.blockDim = dim3(NTHREADS); lc.dynamicSmemBytes = Cfg::SMEM_BYTES; lc.stream = st; lc.attrs = la; lc.numAttrs = 1;
    VTTS_CUDA(cudaLaunchKernelEx(&lc, tc_conv_kernel<N, EPI, MT, NPH, STK, PAIR>, L));
  } else {
    const int grid = L.ntiles < ctx->sm_count ? L.ntiles : ctx->sm_count;
    tc_conv_kernel<N, EPI, MT, NPH, STK, PAIR><<<grid, NTHREADS, Cfg::SMEM_BYTES, st>>>(L);
  }
  ctx->launches++;
  VTTS_CUDA(cudaGetLastError());
  return VTTS_OK;
}

// tile shapes: single-phase: N=256 -> MT 1, N=128 -> MT 2 (two accumulator sets), N<=64 -> MT 4
//              multi-phase (ConvTranspose): N=128 x 4 phases x MT 1, N=64 x 2 x MT 2, N=32 x 2 x MT 4
// (tests/test_gpu_conv_configs.py _tile_rows restates the default-variant shapes to place its rows on tile edges: keep
//  the two in step)
template <int N, int EPI>
int launch_ne(vtts_ctx* ctx, TcLaunch& L, cudaStream_t st) {
  const int nph = L.nphase > 1 ? L.nphase : 1;
  if constexpr (N == 256) {
    if (nph != 1) return ctx->fail(VTTS_ERR_BAD_ARG, "tc_conv: N=256 supports single-phase tiles only");
    if (ctx->tc_variant == 0) return launch_cfg<256, EPI, 2, 1>(ctx, L, st);   // single accumulator set (slower, kept for A/B runs)
    if (ctx->tc_variant == 3) return launch_cfg<256, EPI, 1, 1, 0, 1>(ctx, L, st);   // CTA pairs
    return launch_cfg<256, EPI, 1, 1>(ctx, L, st);
  } else if constexpr (N == 128) {
    if (nph == 4 && ctx->tc_variant == 3) return launch_cfg<128, EPI, 1, 4, 0, 1>(ctx, L, st);
    if (nph == 4) return launch_cfg<128, EPI, 1, 4>(ctx, L, st);
    if (nph != 1) return ctx->fail(VTTS_ERR_BAD_ARG, "tc_conv: N=128 supports 1 or 4 phases");
    if (ctx->tc_variant == 0) return launch_cfg<128, EPI, 4, 1>(ctx, L, st);
    // stacked [W_hi | W_lo]: two MMAs (N' = 256, then N' = 128) instead of three of N' = 128 per (chunk, tap, M tile)
    if (ctx->tc_variant == 2) return launch_cfg<128, EPI, 1, 1, 1>(ctx, L, st);
    if (ctx->tc_variant == 3) return launch_cfg<128, EPI, 2, 1, 0, 1>(ctx, L, st);   // CTA pairs
    return launch_cfg<128, EPI, 2, 1>(ctx, L, st);
  } else if constexpr (N == 64) {
    if (nph == 2) return launch_cfg<64, EPI, 2, 2>(ctx, L, st);
    if (nph != 1) return ctx->fail(VTTS_ERR_BAD_ARG, "tc_conv: N=64 supports 1 or 2 phases");
    if (ctx->tc_variant == 2) return launch_cfg<64, EPI, 2, 1, 1>(ctx, L, st);   // experimental: stacked [W_hi|W_lo] (measured slower: 298 vs 355 TFLOP/s)
    return launch_cfg<64, EPI, 4, 1>(ctx, L, st);
  } else {
    if (nph == 2) return launch_cfg<32, EPI, 4, 2>(ctx, L, st);
    if (nph != 1) return ctx->fail(VTTS_ERR_BAD_ARG, "tc_conv: N=32 supports 1 or 2 phases");
    if (ctx->tc_variant == 2) return launch_cfg<32, EPI, 4, 1, 1>(ctx, L, st);   // experimental: stacked [W_hi|W_lo] (no gain measured)
    return launch_cfg<32, EPI, 4, 1>(ctx, L, st);
  }
}

template <int N>
int launch_n(vtts_ctx* ctx, TcLaunch& L, cudaStream_t st) {
  bool generic = L.post_act != 0 || (L.n_valid > 0 && L.n_valid < N);
  for (int i = 0; i < L.nprob; ++i) generic |= L.p[i].bn_mean != nullptr;
  if (L.nphase > 1 && !generic) return launch_ne<N, 0>(ctx, L, st);
  if (L.nphase > 1) return ctx->fail(VTTS_ERR_BAD_ARG, "tc_conv: multi-phase tiles use the plain epilogue");
  return generic ? launch_ne<N, 1>(ctx, L, st) : launch_ne<N, 0>(ctx, L, st);
}

}  // namespace

size_t vtts_tc_packed_elems(int k, int Cin, int N) { return (size_t)k * Cin * N * 2; }

int vtts_tc_pack_weights(vtts_ctx* ctx, const float* w, void* dst, int k, int Cin, int Cout_total, int n0, int N) {
  pack_w_kernel<<<256, 256>>>(w, reinterpret_cast<__nv_bfloat16*>(dst), k, Cin, Cout_total, n0, N);
  VTTS_CUDA(cudaGetLastError());
  return VTTS_OK;
}

int vtts_tc_tile_n(int Cout) { return Cout <= 32 ? 32 : (Cout <= 64 ? 64 : (Cout <= 128 ? 128 : 256)); }

size_t vtts_tc_conv_packed_bytes(int k, int Cin, int Cout) {
  const int N = vtts_tc_tile_n(Cout), nt = (Cout + N - 1) / N;
  return ((vtts_tc_packed_elems(k, Cin, N) * 2 + 255) & ~size_t(255)) * nt;
}

int vtts_tc_pack_conv(vtts_ctx* ctx, const float* w, int k, int Cin, int Cout, char*& cursor, std::vector<void*>& out) {
  const int N = vtts_tc_tile_n(Cout), nt = (Cout + N - 1) / N;
  for (int t = 0; t < nt; ++t) {
    int rc = vtts_tc_pack_weights(ctx, w, cursor, k, Cin, Cout, t * N, N);
    if (rc) return rc;
    out.push_back(cursor);
    cursor += (vtts_tc_packed_elems(k, Cin, N) * 2 + 255) & ~size_t(255);
  }
  return VTTS_OK;
}

int vtts_conv_dispatch(vtts_ctx* ctx, const ConvLaunch& L, void* const* wpk, cudaStream_t st) {
  if (ctx->precision != 1 || wpk == nullptr) return vtts_launch_conv(ctx, L, st);
  const int N = vtts_tc_tile_n(L.Cout), nt = (L.Cout + N - 1) / N;
  TcLaunch TL;
  auto reset = [&]() {
    memset(&TL, 0, sizeof(TL));
    TL.Cin = L.Cin; TL.N = N; TL.in_ld = L.Cin; TL.out_ld = L.Cout; TL.B = L.B; TL.T_rows = L.T_rows; TL.rows_out = L.rows_out;
    TL.len = L.len; TL.len_mul = L.len_mul; TL.pre_mode = L.pre_mode; TL.pre_slope = L.pre_slope; TL.post_act = L.post_act;
    TL.n_valid = (L.Cout % N) ? (L.Cout % N) : N;   // only meaningful when nt == 1 or for the last tile (handled below)
  };
  reset();
  // tiles that are completely valid and a partial last tile need different n_valid -> separate launches
  for (int pass = 0; pass < 2; ++pass) {
    const bool partial = pass == 1;
    if (partial && (L.Cout % N) == 0) break;
    reset();
    TL.n_valid = partial ? (L.Cout % N) : N;
    for (int pi = 0; pi < L.nprob; ++pi) {
      const ConvProb& cp = L.p[pi];
      for (int t = 0; t < nt; ++t) {
        const bool is_partial = (t == nt - 1) && (L.Cout % N) != 0;
        if (is_partial != partial) continue;
        const int n0 = t * N;
        TcProb q;
        memset(&q, 0, sizeof(q));
        q.x0 = cp.x0; q.x1 = cp.x1; q.x2 = cp.x2;
        q.wpk = wpk[pi * nt + t];
        q.bias = cp.bias + n0;
        q.resid = cp.resid ? cp.resid + n0 : nullptr;
        if (cp.bn_mean) { q.bn_mean = cp.bn_mean + n0; q.bn_inv = cp.bn_inv + n0; q.bn_off = cp.bn_off + n0; }
        q.out = cp.out + n0;
        q.k = cp.k; q.dil = cp.dil; q.in_off = cp.in_off; q.out_stride = cp.out_stride; q.out_off = cp.out_off;
        TL.p[TL.nprob++] = q;
        if (TL.nprob == 8) {
          int rc = vtts_launch_tc_conv(ctx, TL, st);
          if (rc) return rc;
          TL.nprob = 0;
        }
      }
    }
    if (TL.nprob > 0) {
      int rc = vtts_launch_tc_conv(ctx, TL, st);
      if (rc) return rc;
    }
  }
  return VTTS_OK;
}

int vtts_launch_tc_conv(vtts_ctx* ctx, TcLaunch& L, cudaStream_t st) {
  if (L.nprob < 1 || L.nprob > 8) return ctx->fail(VTTS_ERR_BAD_ARG, "tc_conv: nprob %d", L.nprob);
  if (L.Cin % 16 != 0) return ctx->fail(VTTS_ERR_BAD_ARG, "tc_conv: Cin %d", L.Cin);
  for (int i = 0; i < L.nprob; ++i)
    if (L.p[i].k < 1) return ctx->fail(VTTS_ERR_BAD_ARG, "tc_conv: k");
  L.err = ctx->d_err;
  L.dbg = ctx->tc_dbg_on ? ctx->d_tc_dbg : nullptr;
  {
    static int pm_env = -1;    // experiment switch: VTTS_TC_PROBLEM_MAJOR=0/1 forces the tile map of every launch
    if (pm_env < 0) { const char* e = getenv("VTTS_TC_PROBLEM_MAJOR"); pm_env = e ? atoi(e) + 1 : 0; }
    if (pm_env > 0) L.problem_major = pm_env - 1;
    static int exp_env = -1;
    if (exp_env < 0) { const char* e = getenv("VTTS_PAIR_EXP"); exp_env = e ? atoi(e) : 0; }
    L.exp = exp_env;
  }
  switch (L.N) {
    case 256: return launch_n<256>(ctx, L, st);
    case 128: return launch_n<128>(ctx, L, st);
    case 64: return launch_n<64>(ctx, L, st);
    case 32: return launch_n<32>(ctx, L, st);
    default: return ctx->fail(VTTS_ERR_BAD_ARG, "tc_conv: N %d unsupported", L.N);
  }
}
