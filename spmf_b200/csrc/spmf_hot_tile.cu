// Fused dense-tile kernel of the hybrid ADVI step (sm_100a, tcgen05): everything the Poisson
// likelihood needs per (row, hot column, draw) -- rate, x log rate, dL/drate = x/rate, and both
// gradient contractions -- for the dense "hot column" block of a minibatch, without ever writing the
// (S,B,D) rate tensor of the reference (poisson.py:174-184) or its gradient.
//
// One CTA = 128 rows x one Monte-Carlo draw; it walks the hot columns in chunks of 64.  Per chunk:
//   P1  S[128x64]   = Z_s . EV_s^T                 tcgen05.mma, accumulator in tensor memory
//   E   lambda = S + phi ; w = x / lambda (x > 0) ; sum x log lambda      CUDA cores, TMEM -> registers,
//       w written to shared memory as two bf16 terms
//   P2  dZ[128xK]  += W . EV_s                     (poisson.py:177 backward to z)
//   P3  GEV[64xK]   = W^T . Z_s , Gphi = W^T . 1   (backward to the decoder / intercept rows)
// fp32 operands are split into two bf16 terms (hi + lo, 16 mantissa bits); each product is three MMAs
// (hi.hi + hi.lo + lo.hi) accumulated in fp32.  The same shared-memory tiles serve as K-major and as
// MN-major operands (a K-major core matrix of T is an MN-major core matrix of T^T), so nothing is
// transposed in software.  Chunk inputs (the bf16 count tile written by spmf_hot_split and a
// pre-split EV/phi block) arrive by TMA bulk copies, double buffered.
#include <cuda_bf16.h>
#include <cuda_runtime.h>
#include <stdint.h>
#include <stdlib.h>

#include "../../include/spmf_b200.h"
#include "spmf_record.cuh"
#include "spmf_umma_layout.cuh"
#include "spmf_umma_ptx.cuh"

namespace spmf {

// 16-byte chunk (row r, chunk kc) of a core-matrix tile with `cpr` chunks per row
__host__ __device__ __forceinline__ uint32_t core_off_g(int r, int kc, int cpr) {
  return (uint32_t)((((r >> 3) * cpr + kc) << 7) + ((r & 7) << 4));
}

template <int KP>
struct HotTile {
  static constexpr int KK = KP < 16 ? 16 : KP;          // MMA k extent of the latent dimension
  static constexpr int CPR = KK / 8;                    // chunks per row of an EV tile
  static constexpr int ZCPR = CPR + 1;                  // Z rows carry one more chunk: the ones column
  static constexpr int NZ = KK + 8;                     // N of P3: latent dims | 1 | 7 zeros
  static constexpr int EV_TILE = 64 * KK * 2;           // bytes of one bf16 term
  // EV block = one [64 columns][hi latent | lo latent] core-matrix tile (2*CPR chunks per row) + phi[64]:
  // hi and lo side by side so that [hi | lo] is ONE MN-major operand of width 2*KK (term merging)
  static constexpr int EV_BLOCK = 2 * EV_TILE + 256;
  static constexpr int X_TILE = kTileABytes;            // 128 x 64 bf16 counts
  static constexpr int STAGE = X_TILE + EV_BLOCK;
  static constexpr int Z_TILE = 128 * ZCPR * 16;        // per term; the two terms share rows: [hi | 1 | lo | 0]
  static constexpr int ZCPR2 = 2 * ZCPR;                // chunks per row of the combined Z tile
  static constexpr int W_TILE = 128 * 64 * 2;
  // 128 latent dims do not fit the fully pipelined plan (shared memory: 227 KB, tensor memory: 512
  // columns): two input stages instead of three, one W buffer instead of two (the element-wise phase of
  // chunk i+1 then waits for the MMAs of chunk i -- at K = 128 the kernel is MMA-bound anyway), the GEV
  // flush staged in two halves, and no merged [hi | lo] MMAs (their "b" accumulator halves would need
  // 864 tensor-memory columns): three MMAs per product into one accumulator instead.
  static constexpr bool WIDE = KK > 64;
  static constexpr bool MERGED = !WIDE;
  static constexpr int NSTAGE = WIDE ? 2 : 3;           // chunk inputs in flight
  static constexpr int WBUF = WIDE ? 1 : 2;             // W (hi, lo) buffers
  static constexpr int GHALF = WIDE ? 2 : 1;            // GEV flush: staged 64 / GHALF columns at a time
  static constexpr int G_STRIDE = KK + 4;               // floats per staged GEV row (latent | 1 | pad): conflict-free
  static constexpr int G_BYTES = (64 / GHALF) * G_STRIDE * 4;
  static constexpr int SMEM = NSTAGE * STAGE + 2 * Z_TILE + 2 * WBUF * W_TILE + G_BYTES + 128;
  // tensor-memory columns: S | dZ (a | b) | GEV buffer 0 (a | b) | GEV buffer 1 (a | b); the "b" halves
  // (MERGED only) receive the hi.lo products of the merged MMAs and are added at read-out
  static constexpr int ACC = MERGED ? 2 : 1;
  static constexpr int TM_S = 0, TM_DZ = 64, TM_GEV = 64 + ACC * KK, TM_GEV_STRIDE = ACC * NZ;
  static constexpr int TM_COLS = 512;                   // power of two >= 64 + ACC (KK + 2 NZ)  (<= 480)
  static_assert(TM_GEV + 2 * TM_GEV_STRIDE <= 512, "tensor memory");
  static_assert(SMEM <= 227 * 1024, "shared memory");
};

__device__ __forceinline__ uint32_t pack_bf16(float a, float b) {     // a -> low half
  __nv_bfloat162 v = __floats2bfloat162_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&v);
}
__device__ __forceinline__ float bf16_lo(uint32_t p) { return __uint_as_float(p << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t p) { return __uint_as_float(p & 0xffff0000u); }

template <int NC>
__device__ __forceinline__ void tmem_ld(uint32_t taddr, float* v) {
  static_assert(NC == 8 || NC == 16 || NC == 32, "tmem_ld width");
  uint32_t r[NC];
  if constexpr (NC == 32) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr));
  } else if constexpr (NC == 16) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x16.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
        : "r"(taddr));
  } else {
    asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
                 : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
                 : "r"(taddr));
  }
  asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
  for (int i = 0; i < NC; ++i) v[i] = __uint_as_float(r[i]);
}

__device__ __forceinline__ bool rate_ok_t(float lam) { return lam > 0.f && lam <= 3.402823466e38f; }

// ---- per-step operand prep: EV / phi of the hot columns -> per (draw, chunk) TMA blocks -------------
// block = [hi tile | lo tile | phi[64]], tiles are [64 columns][KK latent] bf16 core-matrix tiles.
template <int KP, int SV>
__global__ void __launch_bounds__(256)
hot_ev_tiles_kernel(const float* __restrict__ EV, const float* __restrict__ PH, int D, int H,
                    unsigned char* __restrict__ EVt) {
  using T = HotTile<KP>;
  const int kc = blockIdx.x, s = blockIdx.y, nch = gridDim.x;
  const int q = s / SV, sv = s - q * SV;
  unsigned char* blk = EVt + ((size_t)s * nch + kc) * T::EV_BLOCK;
  for (int t = threadIdx.x; t < 64 * T::CPR; t += blockDim.x) {
    const int c = t / T::CPR, j = t - c * T::CPR;
    const int d = kc * 64 + c;
    float x[8];
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      const int k = 8 * j + 4 * h;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (d < H && k < KP)
        v = __ldg(reinterpret_cast<const float4*>(EV + ((size_t)q * D + d) * (SV * KP) + rec_pos(KP, SV, sv, k)));
      x[4 * h + 0] = v.x; x[4 * h + 1] = v.y; x[4 * h + 2] = v.z; x[4 * h + 3] = v.w;
    }
    uint32_t hi[4], lo[4];
#pragma unroll
    for (int p = 0; p < 4; ++p) {
      hi[p] = pack_bf16(x[2 * p], x[2 * p + 1]);
      lo[p] = pack_bf16(x[2 * p] - bf16_lo(hi[p]), x[2 * p + 1] - bf16_hi(hi[p]));
    }
    *reinterpret_cast<uint4*>(blk + core_off_g(c, j, 2 * T::CPR)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
    *reinterpret_cast<uint4*>(blk + core_off_g(c, T::CPR + j, 2 * T::CPR)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    if (j == 0)     // padding columns get rate 1 (their counts are 0, so they contribute nothing)
      reinterpret_cast<float*>(blk + 2 * T::EV_TILE)[c] = d < H ? __ldg(PH + ((size_t)q * D + d) * SV + sv) : 1.f;
  }
}

// ---- the fused tile kernel --------------------------------------------------------------------------
// One CTA per SM.  Work thread t (< 512) handles row (t & 127) of the tile -- its tensor-memory lane;
// warp w can only touch lanes 32*(w&3).. -- and column quarter (t >> 7) of the chunk.  Two more warps
// only issue: MMAs must come from warp-convergent code (see spmf_umma_ptx.cuh), and an issuing warp
// that also did element-wise work would arrive late at every barrier.
// Software pipeline over the chunks of this CTA's column range (W and the GEV accumulator are
// double buffered, chunk inputs triple buffered):
//   iteration i:  wait S(i) ; E(i) -> W[i&1] ; sync ;
//                 issue P1(i+1) then P3(i) (one thread), P2(i) (another) ;
//                 flush GEV(i-1) -> atomics ; TMA for chunk i+2
// so the tensor core works on chunk i (and produces S(i+1) first) while the CUDA cores flush chunk
// i-1 and then run E(i+1).
constexpr int kTileWorkThreads = 512;               // 16 warps: element-wise phases, flushes
constexpr int kTileThreads = kTileWorkThreads + 64;  // + warp 16: P1/P3 issue, warp 17: P2 issue and TMA

template <int KP, int SV>
__global__ void __launch_bounds__(kTileThreads, 1)
hot_tile_kernel(const unsigned char* __restrict__ xhot, const unsigned char* __restrict__ EVt,
                const float* __restrict__ z, int nrows, int D, int H, int nch, int chunks_per_cta,
                float* __restrict__ dzacc, float* __restrict__ rowacc, float* __restrict__ GEV,
                float* __restrict__ Gphi, int* __restrict__ gflag) {
  using T = HotTile<KP>;
  constexpr int KK = T::KK, REC = SV * KP;
  extern __shared__ __align__(128) unsigned char smem_raw[];
  const uint32_t sbase = (smem_u32(smem_raw) + 127u) & ~127u;
  unsigned char* sp = smem_raw + (sbase - smem_u32(smem_raw));
  __shared__ __align__(8) unsigned long long mbar_store[T::NSTAGE + 3];
  __shared__ uint32_t tmem_slot;

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int rt = tid & 127;                 // row of the tile = tensor-memory lane
  const int hq = tid >> 7;                  // column quarter of the chunk this thread works on
  const uint32_t lane_base = (uint32_t)((warp & 3) * 32) << 16;
  const int mt = blockIdx.x, s = blockIdx.y;
  const int q = s / SV, sv = s - q * SV;
  const int row = mt * 128 + rt;
  const int c_begin = blockIdx.z * chunks_per_cta;
  const int n = min(nch, c_begin + chunks_per_cta) - c_begin;       // chunks of this CTA
  if (n <= 0) return;

  // shared-memory map: [stage 0..2 | Z hi | Z lo | W0 hi | W0 lo | W1 hi | W1 lo]
  const uint32_t sStage0 = sbase;
  const uint32_t sZ0 = sbase + (uint32_t)(T::NSTAGE * T::STAGE);      // combined Z tile, 2*Z_TILE bytes
  const uint32_t sWb = sZ0 + 2u * (uint32_t)T::Z_TILE;               // W buffer b: hi at sWb + b*2*W_TILE, lo + W_TILE
  unsigned char* const pZ0 = sp + T::NSTAGE * T::STAGE;
  unsigned char* const pWb = pZ0 + 2 * T::Z_TILE;

  uint32_t full[T::NSTAGE];
#pragma unroll
  for (int i = 0; i < T::NSTAGE; ++i) full[i] = smem_u32(&mbar_store[i]);
  const uint32_t bar_s = smem_u32(&mbar_store[T::NSTAGE]);
  const uint32_t bar_g[2] = {smem_u32(&mbar_store[T::NSTAGE + 1]), smem_u32(&mbar_store[T::NSTAGE + 2])};
  if (tid == 0) {
#pragma unroll
    for (int i = 0; i < T::NSTAGE; ++i) mbar_init(full[i], 1);
    mbar_init(bar_s, 1);
    mbar_init(bar_g[0], 2);       // P2 and P3 are issued (and committed) by two different threads
    mbar_init(bar_g[1], 2);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 3) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(&tmem_slot)),
                 "r"((uint32_t)T::TM_COLS)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }

  const bool worker = tid < kTileWorkThreads;
  // ---- Z_s tile: this draw's z of the 128 rows as two bf16 terms + the ones column; the four thread
  // quarters write alternate 16-byte chunks of the row
  if (worker) {
    const float* zp = z + ((size_t)q * nrows + (row < nrows ? row : 0)) * REC;
#pragma unroll
    for (int j = 0; j < T::ZCPR; ++j) {
      if ((j & 3) != hq) continue;
      float zr[8];
#pragma unroll
      for (int e = 0; e < 8; ++e) zr[e] = 0.f;
      if (8 * j < KP && row < nrows) {
#pragma unroll
        for (int h = 0; h < 2; ++h) {
          if (8 * j + 4 * h < KP) {
            const float4 v = __ldg(reinterpret_cast<const float4*>(zp + rec_pos(KP, SV, sv, 8 * j + 4 * h)));
            zr[4 * h] = v.x; zr[4 * h + 1] = v.y; zr[4 * h + 2] = v.z; zr[4 * h + 3] = v.w;
          }
        }
      }
      if (8 * j == KK) zr[0] = 1.f;               // W^T . 1 = column sums of w  (Gphi)
      uint32_t hi[4], lo[4];
#pragma unroll
      for (int p = 0; p < 4; ++p) {
        const float a = zr[2 * p], b = zr[2 * p + 1];
        hi[p] = pack_bf16(a, b);
        lo[p] = pack_bf16(a - bf16_lo(hi[p]), b - bf16_hi(hi[p]));
      }
      *reinterpret_cast<uint4*>(pZ0 + core_off_g(rt, j, T::ZCPR2)) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
      *reinterpret_cast<uint4*>(pZ0 + core_off_g(rt, T::ZCPR + j, T::ZCPR2)) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
    }
  }
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
  const uint32_t tm = tmem_slot;

  const unsigned char* xsrc = xhot + ((size_t)mt * nch + c_begin) * T::X_TILE;
  const unsigned char* esrc = EVt + ((size_t)s * nch + c_begin) * T::EV_BLOCK;
  auto issue_load = [&](int i) {              // local chunk i -> stage i % NSTAGE
    const int st = i % T::NSTAGE;
    const uint32_t dst = sStage0 + (uint32_t)(st * T::STAGE);
    mbar_expect_tx(full[st], (uint32_t)T::STAGE);
    tma_bulk_g2s(dst, xsrc + (size_t)i * T::X_TILE, T::X_TILE, full[st]);
    tma_bulk_g2s(dst + T::X_TILE, esrc + (size_t)i * T::EV_BLOCK, T::EV_BLOCK, full[st]);
  };
  auto wait_full = [&](int i) { mbar_wait(full[i % T::NSTAGE], (uint32_t)((i / T::NSTAGE) & 1)); };
  constexpr uint64_t kStageStep = (uint64_t)(T::STAGE >> 4);
  constexpr uint64_t kWStep = (uint64_t)((2 * T::W_TILE) >> 4);
  // P1: S = Z . EV^T   (both K-major), terms hi.hi, hi.lo, lo.hi
  auto issue_p1 = [&](int i) {
    constexpr uint32_t ID = umma_idesc_bf16(128, 64, 0, 0);
    const uint64_t so = (uint64_t)(i % T::NSTAGE) * kStageStep;
    const uint64_t dZk[2] = {umma_desc(sZ0, 128, T::ZCPR2 * 128), umma_desc(sZ0 + T::ZCPR * 128, 128, T::ZCPR2 * 128)};
    const uint64_t dEk[2] = {umma_desc(sStage0 + T::X_TILE, 128, 2 * T::CPR * 128),
                             umma_desc(sStage0 + T::X_TILE + T::CPR * 128, 128, 2 * T::CPR * 128)};
#pragma unroll
    for (int t = 0; t < 3; ++t) {
      const uint64_t a = dZk[t == 2 ? 1 : 0], b = dEk[t == 1 ? 1 : 0] + so;
#pragma unroll
      for (int j = 0; j < KK / 16; ++j)
        umma_bf16_elect(tm + T::TM_S, a + (uint64_t)(j * 16), b + (uint64_t)(j * 16), ID, (t | j) ? 1u : 0u);
    }
    umma_commit_elect(bar_s);
  };
  // flush GEV / Gphi of local chunk i.  Accumulator row m (a column of the chunk) sits in tensor-memory
  // lane (m/16)*32 + m%16, so a lane-owner store would scatter 16 lanes over 16 different records;
  // instead the tile is staged through shared memory and written out by all 512 workers, 8
  // consecutive threads per column (coalesced vector reductions).
  float* const gst = reinterpret_cast<float*>(pWb + 2 * T::WBUF * T::W_TILE);
  auto flush_gev = [&](int i) {
    mbar_wait(bar_g[i & 1], (uint32_t)((i >> 1) & 1));
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    const uint32_t ta = tm + lane_base + T::TM_GEV + (uint32_t)((i & 1) * T::TM_GEV_STRIDE);
    const int m = (warp & 3) * 16 + lane;          // column of the chunk held by this lane (lane < 16)
    // NQD thread quarters read HK latent dims each; the ones column (Gphi) goes to one of them
    constexpr int NQD = KK >= 64 ? 4 : 2;
    constexpr int HK = KK / NQD;                    // 8, 16 or 32
    constexpr int ONES_Q = NQD == 4 ? 0 : 2;
    float g[HK], g1 = 0.f;
    if (hq < NQD) {
      tmem_ld<HK>(ta + HK * hq, g);
      if constexpr (T::MERGED) {                    // + the hi.lo half of the merged MMA
        float gb[HK];
        tmem_ld<HK>(ta + T::NZ + HK * hq, gb);
#pragma unroll
        for (int k = 0; k < HK; ++k) g[k] += gb[k];
      }
    }
    if (hq == ONES_Q) {
      float t8[8];
      tmem_ld<8>(ta + KK, t8);
      g1 = t8[0];
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    // staged through shared memory 64 / GHALF columns at a time: tensor-memory lanes 0-15 of warps with
    // (warp & 3) = w hold columns 16 w .. 16 w + 15
    constexpr int CPH = 64 / T::GHALF;              // columns per half
#pragma unroll
    for (int half = 0; half < T::GHALF; ++half) {
      if (half > 0) asm volatile("bar.sync 1, %0;" ::"n"(kTileWorkThreads) : "memory");   // staging free again
      const int ml = m - half * CPH;
      if (lane < 16 && ml >= 0 && ml < CPH) {
        if (hq < NQD) {
#pragma unroll
          for (int k = 0; k < HK; k += 4)
            *reinterpret_cast<float4*>(gst + ml * T::G_STRIDE + HK * hq + k) = make_float4(g[k], g[k + 1], g[k + 2], g[k + 3]);
        }
        if (hq == ONES_Q) gst[ml * T::G_STRIDE + KK] = g1;
      }
      asm volatile("bar.sync 1, %0;" ::"n"(kTileWorkThreads) : "memory");
      constexpr int TPC = KK / 4;                          // threads per column, 4 latent dims each
      constexpr int PASSES = (CPH * TPC + kTileWorkThreads - 1) / kTileWorkThreads;
#pragma unroll
      for (int ps = 0; ps < PASSES; ++ps) {
        const int idx = ps * kTileWorkThreads + tid;
        const int cl = idx / TPC, k = (idx % TPC) * 4;
        const int c = (c_begin + i) * 64 + half * CPH + cl;
        if (cl < CPH && c < H) {
          if (k < KP) {
            const float4 v = *reinterpret_cast<const float4*>(gst + cl * T::G_STRIDE + k);
            atomicAdd(reinterpret_cast<float4*>(GEV + ((size_t)q * D + c) * REC + rec_pos(KP, SV, sv, k)), v);
          }
          if ((idx % TPC) == TPC - 1) atomicAdd(Gphi + ((size_t)q * D + c) * SV + sv, gst[cl * T::G_STRIDE + KK]);
        }
      }
    }
  };

  if (warp == 17) {
    if (elect_one()) {
      issue_load(0);
      if (n > 1) issue_load(1);
      if (T::NSTAGE > 2 && n > 2) issue_load(2);
    }
    __syncwarp();
  }
  if (warp == 16) {
    wait_full(0);
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    issue_p1(0);
  }

  float xlog2 = 0.f, wmax = 0.f;
  for (int i = 0; i < n; ++i) {
    const int st = i % T::NSTAGE, wb = T::WBUF == 1 ? 0 : (i & 1), gb_ = i & 1;
    if (worker) {
    wait_full(i);                                           // TMA data visible to this thread
    mbar_wait(bar_s, (uint32_t)(i & 1));                    // S(i) ready in tensor memory
    if (T::WBUF == 1 && i >= 1)                             // one W buffer: chunk i-1's MMAs must have read it
      mbar_wait(bar_g[(i - 1) & 1], (uint32_t)(((i - 1) >> 1) & 1));
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");

    // ---- E: lambda, w = x / lambda, x log lambda for 16 columns of this thread's row; W -> shared
    //      memory as two bf16 terms.  The rate is floored at 1e-30 instead of branching on it
    //      (poisson.py:606-616 guards non-finite rates; here they are sums of positive terms).
    {
      const unsigned char* xt = sp + st * T::STAGE;
      const float* ph = reinterpret_cast<const float*>(xt + T::X_TILE + 2 * T::EV_TILE) + 16 * hq;
      unsigned char* w0 = pWb + wb * 2 * T::W_TILE;
      float lam[16];
      tmem_ld<16>(tm + lane_base + T::TM_S + 16 * hq, lam);
#pragma unroll
      for (int j = 0; j < 2; ++j) {          // 2 chunks of 8 columns
        const uint32_t o = core_off(rt, 2 * hq + j);
        const uint4 xp = *reinterpret_cast<const uint4*>(xt + o);
        const uint32_t xw[4] = {xp.x, xp.y, xp.z, xp.w};
        const float4 p0 = *reinterpret_cast<const float4*>(ph + 8 * j);
        const float4 p1 = *reinterpret_cast<const float4*>(ph + 8 * j + 4);
        const float phv[8] = {p0.x, p0.y, p0.z, p0.w, p1.x, p1.y, p1.z, p1.w};
        float w[8];
#pragma unroll
        for (int e = 0; e < 8; ++e) {
          const float x = (e & 1) ? bf16_hi(xw[e >> 1]) : bf16_lo(xw[e >> 1]);
          const float l = fmaxf(lam[8 * j + e] + phv[e], 1e-30f);       // poisson.py:177
          float lg, rc;
          asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(lg) : "f"(l));
          asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(rc) : "f"(l));
          w[e] = x * rc;
          wmax = fmaxf(wmax, w[e]);                 // a floored (zero / NaN) rate at a nonzero shows up as x * 1e30
          xlog2 = fmaf(x, lg, xlog2);
        }
        uint32_t hi[4], lo[4];
#pragma unroll
        for (int p = 0; p < 4; ++p) {
          hi[p] = pack_bf16(w[2 * p], w[2 * p + 1]);
          lo[p] = pack_bf16(w[2 * p] - bf16_lo(hi[p]), w[2 * p + 1] - bf16_hi(hi[p]));
        }
        *reinterpret_cast<uint4*>(w0 + o) = make_uint4(hi[0], hi[1], hi[2], hi[3]);
        *reinterpret_cast<uint4*>(w0 + T::W_TILE + o) = make_uint4(lo[0], lo[1], lo[2], lo[3]);
      }
    }
    }   // worker
    asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();

    if (warp == 17) {
      // P2: dZ += W . EV      A = W K-major [128 x 64], B = EV MN-major (N = latent, K = 64 columns)
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      const uint64_t wo = (uint64_t)wb * kWStep, so = (uint64_t)st * kStageStep;
      const uint64_t dWh = umma_desc(sWb, 128, 1024) + wo, dWl = umma_desc(sWb + T::W_TILE, 128, 1024) + wo;
      const uint64_t dEn = umma_desc(sStage0 + T::X_TILE, 2 * T::CPR * 128, 128) + so;     // MN-major, k-group = 8 columns
      constexpr uint64_t kEStep = (uint64_t)(2 * 2 * T::CPR * 128 / 16);                   // 16 columns
      if constexpr (T::MERGED) {
        // two MMAs per k-step instead of three: W_hi . [EV_hi | EV_lo] (N = 2 KK, second half -> dZ_b)
        // and W_lo . EV_hi (N = KK, into dZ_a): the W operand is fetched twice, not three times
        constexpr uint32_t IDa = umma_idesc_bf16(128, 2 * KK, 0, 1), IDb = umma_idesc_bf16(128, KK, 0, 1);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          umma_bf16_elect(tm + T::TM_DZ, dWh + (uint64_t)(j * 16), dEn + j * kEStep, IDa, (i | j) ? 1u : 0u);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          umma_bf16_elect(tm + T::TM_DZ, dWl + (uint64_t)(j * 16), dEn + j * kEStep, IDb, 1u);
      } else {
        // 128 latent dims: hi.hi, hi.lo, lo.hi as three MMAs of N = KK into ONE accumulator
        constexpr uint32_t ID = umma_idesc_bf16(128, KK, 0, 1);
        const uint64_t dEl = umma_desc(sStage0 + T::X_TILE + T::CPR * 128, 2 * T::CPR * 128, 128) + so;   // lo latent chunks
#pragma unroll
        for (int j = 0; j < 4; ++j)
          umma_bf16_elect(tm + T::TM_DZ, dWh + (uint64_t)(j * 16), dEn + j * kEStep, ID, (i | j) ? 1u : 0u);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          umma_bf16_elect(tm + T::TM_DZ, dWh + (uint64_t)(j * 16), dEl + j * kEStep, ID, 1u);
#pragma unroll
        for (int j = 0; j < 4; ++j)
          umma_bf16_elect(tm + T::TM_DZ, dWl + (uint64_t)(j * 16), dEn + j * kEStep, ID, 1u);
      }
      umma_commit_elect(bar_g[gb_]);
      // chunk i-1 is fully consumed once its MMAs are done: refill its stage with chunk i + NSTAGE - 1
      if (i >= 1 && i + T::NSTAGE - 1 < n) {
        mbar_wait(bar_g[(i - 1) & 1], (uint32_t)(((i - 1) >> 1) & 1));
        if (elect_one()) issue_load(i + T::NSTAGE - 1);
        __syncwarp();
      }
    } else if (warp == 16) {
      asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
      // P1 of the next chunk first: its result gates the next element-wise phase
      if (i + 1 < n) {
        wait_full(i + 1);
        asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
        issue_p1(i + 1);
      }
      // P3: GEV = W^T . [Z | 1]   A = W MN-major (M = 64 columns, K = 128 rows), B = Z MN-major (N = NZ)
      const uint64_t wo = (uint64_t)wb * kWStep;
      const uint64_t dWh = umma_desc(sWb, 1024, 128) + wo, dWl = umma_desc(sWb + T::W_TILE, 1024, 128) + wo;
      const uint64_t dZn = umma_desc(sZ0, T::ZCPR2 * 128, 128);
      constexpr uint64_t kZStep = (uint64_t)(2 * T::ZCPR2 * 128 / 16);                      // 16 rows
      const uint32_t tg = tm + T::TM_GEV + (uint32_t)(gb_ * T::TM_GEV_STRIDE);
      if constexpr (T::MERGED) {
        // merged the same way: W_hi^T . [Z_hi | 1 | Z_lo | 0] (N = 2 NZ) and W_lo^T . [Z_hi | 1] (N = NZ)
        constexpr uint32_t IDa = umma_idesc_bf16(64, 2 * T::NZ, 1, 1), IDb = umma_idesc_bf16(64, T::NZ, 1, 1);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          umma_bf16_elect(tg, dWh + (uint64_t)(j * (2048 / 16)), dZn + j * kZStep, IDa, j ? 1u : 0u);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          umma_bf16_elect(tg, dWl + (uint64_t)(j * (2048 / 16)), dZn + j * kZStep, IDb, 1u);
      } else {
        // three MMAs of N = NZ into one accumulator: W_hi^T.[Z_hi | 1], W_hi^T.[Z_lo | 0], W_lo^T.[Z_hi | 1]
        constexpr uint32_t ID = umma_idesc_bf16(64, T::NZ, 1, 1);
        const uint64_t dZl = umma_desc(sZ0 + T::ZCPR * 128, T::ZCPR2 * 128, 128);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          umma_bf16_elect(tg, dWh + (uint64_t)(j * (2048 / 16)), dZn + j * kZStep, ID, j ? 1u : 0u);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          umma_bf16_elect(tg, dWh + (uint64_t)(j * (2048 / 16)), dZl + j * kZStep, ID, 1u);
#pragma unroll
        for (int j = 0; j < 8; ++j)
          umma_bf16_elect(tg, dWl + (uint64_t)(j * (2048 / 16)), dZn + j * kZStep, ID, 1u);
      }
      umma_commit_elect(bar_g[gb_]);
    } else if (i >= 1) {
      // workers: the previous chunk's MMAs have had a whole element-wise phase to finish
      flush_gev(i - 1);
    }
  }
  if (worker) {
  asm volatile("bar.sync 1, %0;" ::"n"(kTileWorkThreads) : "memory");   // staging tile free (previous flush read out)
  flush_gev(n - 1);

  // ---- dZ of the 128 rows (several CTAs share a (rows, draw) slice when the column range is split:
  //      atomics) and the row scalars; thread quarter hq owns a quarter of the latent range
  {
    constexpr int QK = KK / 4;                 // latent dims per thread quarter: 4, 8, 16 or 32
    constexpr int LD = QK < 8 ? 8 : QK;        // tensor-memory columns read per quarter (>= 8 per load)
    float dzv[LD];
    const int col0 = QK >= 8 ? QK * hq : 8 * (hq >> 1);
    tmem_ld<LD>(tm + lane_base + T::TM_DZ + col0, dzv);
    if constexpr (T::MERGED) {
      float dzb[LD];
      tmem_ld<LD>(tm + lane_base + T::TM_DZ + KK + col0, dzb);
#pragma unroll
      for (int k = 0; k < LD; ++k) dzv[k] += dzb[k];
    }
    if (row < nrows) {
      float* dp = dzacc + ((size_t)q * nrows + row) * REC;
#pragma unroll
      for (int k = 0; k < QK; k += 4) {
        const int kk = QK * hq + k;
        const int src = (QK >= 8) ? k : 4 * (hq & 1) + k;
        if (kk < KP)
          atomicAdd(reinterpret_cast<float4*>(dp + rec_pos(KP, SV, sv, kk)),
                    make_float4(dzv[src], dzv[src + 1], dzv[src + 2], dzv[src + 3]));
      }
      atomicAdd(rowacc + ((size_t)q * nrows + row) * 4 * SV + sv, xlog2 * 0.6931471805599453f);
    }
    // non-finite log-likelihood somewhere in this thread's entries (rate 0 / NaN at a nonzero, or an
    // infinite rate): the exact guard of poisson.py:606-616 re-evaluates the step (spmf_dense.cu)
    if (gflag && (!(wmax < 1e25f) || !(fabsf(xlog2) <= 3.402823466e38f))) atomicOr(gflag, 1);
  }
  }   // worker
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
  __syncthreads();
  if (warp == 3) {
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tm), "r"((uint32_t)T::TM_COLS) : "memory");
  }
}

// ---- row finalisation after the cold row pass and the hot tile kernel have both added into dzr / rowacc
// One warp per (row, draw group): lane l owns the 4 consecutive record floats [4l, 4l+4) -- one k-vector
// of one draw (spmf_record.cuh) -- so the record is read and written with coalesced 16-byte accesses.
template <int KP, int SV>
__global__ void __launch_bounds__(128)
rows_finish_kernel(const float* __restrict__ rowsum, const float* __restrict__ lgam, float inv_xi, int scale_rows,
                   int nrows, const double* __restrict__ vsum, const float* __restrict__ z,
                   float* __restrict__ dzr, float* __restrict__ rowacc, int* __restrict__ gflag) {
  constexpr int REC = SV * KP;
  static_assert(KP >= 4, "rows_finish: float4 k-vectors");
  constexpr int NCH = (REC + 127) / 128;               // a warp covers 128 record floats per pass
  const RecMap rm = rec_map(KP);
  const int row = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31, q = blockIdx.y;
  if (row >= nrows) return;
  const float r = scale_rows ? rowsum[row] * inv_xi : 1.f;
  // the row scalars' read-modify-write is issued up front (lane s owns draw s) so that its latency
  // overlaps the record traffic instead of trailing it as four dependent round trips of lane 0
  float* ra = rowacc + ((size_t)q * nrows + row) * 4 * SV;
  const float lg = lgam[row];
  const float ra0 = lane < SV ? ra[lane] : 0.f;
  float zv[SV], z2[SV];
#pragma unroll
  for (int s = 0; s < SV; ++s) { zv[s] = 0.f; z2[s] = 0.f; }
#pragma unroll
  for (int ch = 0; ch < NCH; ++ch) {
    const int p = ch * 128 + lane * 4;                 // first record float of this lane's k-vector
    if (p < REC) {
      const int sv = (p / (4 * rm.RG)) % SV;            // draw of the k-vector (spmf_record.cuh)
      const size_t o = ((size_t)q * nrows + row) * REC + p;
      const float4 zz = *reinterpret_cast<const float4*>(z + o);
      float4 d = *reinterpret_cast<float4*>(dzr + o);
      const double* vs = vsum + (size_t)q * REC + p;
      const float v0 = (float)vs[0], v1 = (float)vs[1], v2 = (float)vs[2], v3 = (float)vs[3];
      const float a = zz.x * v0 + zz.y * v1 + zz.z * v2 + zz.w * v3;
      const float b = zz.x * zz.x + zz.y * zz.y + zz.z * zz.z + zz.w * zz.w;
#pragma unroll
      for (int s = 0; s < SV; ++s) {
        zv[s] += sv == s ? a : 0.f;
        z2[s] += sv == s ? b : 0.f;
      }
      d.x = r * (d.x - v0 - zz.x);           // dL/dz incl. the HalfNormal(1) z prior (poisson.py:599-604)
      d.y = r * (d.y - v1 - zz.y);
      d.z = r * (d.z - v2 - zz.z);
      d.w = r * (d.w - v3 - zz.w);
      *reinterpret_cast<float4*>(dzr + o) = d;
    }
  }
  float am = 0.f, bm = 0.f;                  // this lane's draw (lane < SV)
#pragma unroll
  for (int s = 0; s < SV; ++s) {
    float a = zv[s], b = z2[s];
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) {
      a += __shfl_xor_sync(0xffffffffu, a, o);
      b += __shfl_xor_sync(0xffffffffu, b, o);
    }
    if (lane == s) { am = a; bm = b; }
  }
  if (lane < SV) {
    ra[0 * SV + lane] = ra0 - lg;
    ra[1 * SV + lane] = am;
    ra[2 * SV + lane] = bm;
    // closed-form sum_d rate of this row is not finite: some entry's rate is not (poisson.py:606-616)
    if (gflag && !(fabsf(am) <= 3.402823466e38f)) atomicOr(gflag, 1);
  }
}

}  // namespace spmf

using namespace spmf;

#define HT_DISPATCH(KP, SV, CALL)                                   \
  do {                                                              \
    if (KP == 32 && SV == 4) { CALL(32, 4); }                       \
    else if (KP == 32 && SV == 2) { CALL(32, 2); }                  \
    else if (KP == 32 && SV == 1) { CALL(32, 1); }                  \
    else if (KP == 16 && SV == 4) { CALL(16, 4); }                  \
    else if (KP == 16 && SV == 2) { CALL(16, 2); }                  \
    else if (KP == 8 && SV == 4) { CALL(8, 4); }                    \
    else if (KP == 64 && SV == 4) { CALL(64, 4); }                  \
    else if (KP == 64 && SV == 2) { CALL(64, 2); }                  \
    else if (KP == 64 && SV == 1) { CALL(64, 1); }                  \
    else if (KP == 128 && SV == 4) { CALL(128, 4); }                \
    else if (KP == 128 && SV == 2) { CALL(128, 2); }                \
    else if (KP == 128 && SV == 1) { CALL(128, 1); }                \
    else return SPMF_ERR_UNSUPPORTED;                               \
  } while (0)

template <int KP, int SV>
static int launch_hot_tile(const void* xhot, const void* EVt, const float* z, int nrows, int D, int H, int S,
                           float* dzacc, float* rowacc, float* GEV, float* Gphi, int* gflag, cudaStream_t st) {
  using T = HotTile<KP>;
  static bool attr = false;
  if (!attr) {
    cudaError_t e = cudaFuncSetAttribute(hot_tile_kernel<KP, SV>, cudaFuncAttributeMaxDynamicSharedMemorySize, T::SMEM);
    if (e != cudaSuccess) return (int)e;
    attr = true;
  }
  // one CTA per SM: cut the hot columns into ranges so that the grid is several waves of 148 CTAs
  const int nch = (H + 63) / 64, items = ((nrows + 127) / 128) * S;
  constexpr int waves = 6;
  int splits = (waves * 148 + items - 1) / items;
  if (splits > nch) splits = nch;
  if (splits < 1) splits = 1;
  const int per = (nch + splits - 1) / splits;
  splits = (nch + per - 1) / per;
  dim3 grid((nrows + 127) / 128, S, splits);
  hot_tile_kernel<KP, SV><<<grid, kTileThreads, T::SMEM, st>>>((const unsigned char*)xhot, (const unsigned char*)EVt, z, nrows, D,
                                                              H, nch, per, dzacc, rowacc, GEV, Gphi, gflag);
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? SPMF_OK : (int)e;
}

extern "C" {

long long spmf_hot_tile_scratch_bytes(int H, int K, int S) {
  if (H <= 0 || K <= 0 || S <= 0) return 0;
  const int KP = spmf_kpad(K), KK = KP < 16 ? 16 : KP;
  const long long nch = (H + 63) / 64;
  return (long long)S * nch * (2LL * 64 * KK * 2 + 256);
}

int spmf_hot_ev_tiles(const float* EV, const float* PH, int D, int H, int K, int S, void* EVt, void* stream) {
  if (!EV || !PH || !EVt || D <= 0 || H <= 0 || H > D || K <= 0 || K > SPMF_MAX_TILE_K || S <= 0) return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S);
  dim3 grid((H + 63) / 64, S);
  cudaStream_t st = (cudaStream_t)stream;
#define CALL_EVT(KPC, SVC) hot_ev_tiles_kernel<KPC, SVC><<<grid, 256, 0, st>>>(EV, PH, D, H, (unsigned char*)EVt)
  HT_DISPATCH(KP, SV, CALL_EVT);
#undef CALL_EVT
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? SPMF_OK : (int)e;
}

int spmf_hot_tile(const void* xhot, const void* EVt, const float* z, int nrows, int D, int H, int K, int S,
                  float* dzacc, float* rowacc, float* GEVnz, float* Gphinz, void* gs, void* stream) {
  if (!xhot || !EVt || !z || !dzacc || !rowacc || !GEVnz || !Gphinz) return SPMF_ERR_BAD_ARG;
  if (nrows <= 0 || D <= 0 || H <= 0 || H > D || K <= 0 || K > SPMF_MAX_TILE_K || S <= 0) return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S);
  cudaStream_t st = (cudaStream_t)stream;
  int rc = SPMF_OK;
#define CALL_HT(KPC, SVC) rc = launch_hot_tile<KPC, SVC>(xhot, EVt, z, nrows, D, H, S, dzacc, rowacc, GEVnz, Gphinz, (int*)gs, st)
  HT_DISPATCH(KP, SV, CALL_HT);
#undef CALL_HT
  return rc;
}

int spmf_rows_finish(const float* rowsum, const float* lgam, float inv_xi, int scale_rows, int nrows, int K, int S,
                     const double* vsum, const float* z, float* dzr, float* rowacc, void* gs, void* stream) {
  if (!rowsum || !lgam || !vsum || !z || !dzr || !rowacc || nrows <= 0 || K <= 0 || K > SPMF_MAX_TILE_K || S <= 0)
    return SPMF_ERR_BAD_ARG;
  const int KP = spmf_kpad(K), SV = spmf_draw_vec_k(K, S), NQ = S / SV;
  dim3 grid((unsigned)((nrows + 3) / 4), NQ);
  cudaStream_t st = (cudaStream_t)stream;
#define CALL_RF(KPC, SVC) rows_finish_kernel<KPC, SVC><<<grid, 128, 0, st>>>(rowsum, lgam, inv_xi, scale_rows, nrows, vsum, z, dzr, rowacc, (int*)gs)
  HT_DISPATCH(KP, SV, CALL_RF);
#undef CALL_RF
  cudaError_t e = cudaGetLastError();
  return e == cudaSuccess ? SPMF_OK : (int)e;
}

}  // extern "C"
