// il_stream.cuh — the 1x1-kind ILBlock as ONE persistent, streaming kernel on the Blackwell data path
// (reference: ILBlock.forward, CSNet/model/csnet.py:72-76 = gOctaveCBR :778-792 over gOctaveConv.forward :664-726,
// then two SimplifiedGOctConvBR.forward :838-851).
//
// A CTA walks a contiguous range of the batch's (image, 4-row chunk) sequence top to bottom, full image width:
//
//   TMA        x_h rows [4c, 4c+4) and x_l rows [2c, 2c+2) arrive by cp.async.bulk.tensor.5d straight in the
//              tensor-core operand layout  [row][8-pixel group][channel slot][8 px]  (a core matrix of the MN-major
//              A operand = 8 channel slots x 16 bytes); the map splits W into (W/8, 8), channel slots past the
//              tensor's C are zero-filled by the TMA unit = the K padding of the GEMM.  2 hi / 3 lo stages.
//   resample   bilinear x2 of x_l -> slots [Chi, Chi+Cli) of the hi chunk (lo -> hi path, csnet.py:702-707; the
//              up-sample commutes with the 1x1 conv), max-pool 2x2 of x_h -> slots [Cli, Cli+Chi) of the lo chunk
//              (hi -> lo path, :709-712).
//   GEMM       one elected thread issues tcgen05.mma (kind::f16, M = 128 pixels, N = ru16(Cout), K = 16 per
//              instruction) per 16 pixel groups; fp32 accumulators of the whole chunk live in TMEM.
//   epilogue   tcgen05.ld (a thread = a pixel), + bias, PReLU, 16-bit, written IN PLACE over the chunk (T1).
//   dw tail    a thread owns (channel, 8-pixel column) for the whole walk and keeps the 3-row windows of T1 and T2
//              in registers: dw3x3+BN+PReLU twice with no halo recomputation in y, no shared-memory round trip for
//              T2, 16-byte coalesced stores of the block output.  (mixed-precision FMA: fp16 x fp16 + fp32.)
//
// Stem form (kStem; the first block, csnet.py:60-71: both branches are 3x3 convs of the fp32 image, the lo one of its 2x2
// max-pool): the TMA ring holds 4-row blocks of the fp32 image (4-D map, zero fill outside the image = the conv padding);
// instead of the resample pass the threads build the im2col operand (27 slots: ci, ky, kx) of the hi chunk and of the
// lo chunk (pooling on the fly) in the same [row][group][slot][8 px] layout; GEMM, epilogue and depthwise tail are shared.
//
// An image is cut into `ns` column strips of gsn 8-pixel groups (gsn even); a CTA's tile of a strip carries one halo
// group on each side when ns > 1 (hl = 1: the TMA box starts one group early, out-of-image groups arrive as zeros).
// Narrow strips let two CTAs share an SM (<= 113 KB shared memory, <= 256 TMEM columns each), so one CTA's waits
// (TMA, MMA, barriers) are filled by the other's depthwise phase.  No row halo is ever re-read from HBM (except one
// warm-up chunk where a CTA's range starts inside an image); the work split is a flat division of the
// N * ns * H/4 chunks over the CTAs.  Needs W % 16 == 0, H % 4 == 0, K = Chi + Cli <= 64.  Other shapes: il_block.cuh.
#pragma once
#include <cuda.h>

#include "il_block.cuh"

namespace csnet {

constexpr int kIlsMaxThreads = 768;
constexpr int kIlsMaxC = 64;          // output channels per branch (epilogue parameter tables in the kernel arguments)
constexpr int kIlsHiStages = 2, kIlsLoStages = 3;

struct IlsArgs {
  void* yh;
  void* yl;                           // nullptr when Clo == 0
  const uint32_t* wh;                 // packed 16-bit [NH][K8]  columns [x_h | up(x_l)]
  const uint32_t* wl;                 // packed 16-bit [NL][K8]  columns [x_l | pool(x_h)]
  DwParams dw1h, dw1l, dw2h, dw2l;
  float bias_h[kIlsMaxC], sm1_h[kIlsMaxC], bias_l[kIlsMaxC], sm1_l[kIlsMaxC];   // conv bias, PReLU slope - 1
  int32_t N, H, W;
  int32_t Chi, Cli, Cho, Clo;
  int32_t K8, K16, NH, NL;            // NH / NL = ru16(Cho / Clo): the N of the MMAs (NL = 0 without a lo output)
  int32_t SH, SL, ST;                 // channel slots per pixel group: hi chunk, lo chunk, T1L buffer (all odd)
  int32_t GH, GL;                     // pixel groups per image row: W/8, W/16
  int32_t ns, gsn, hl;                // column strips per image, hi groups per strip (even), halo groups per side (0 / 1)
  int32_t GR, GLR;                    // groups per row of a CTA's tile: gsn + 2 hl, gsn/2 + 2 hl
  int32_t tmem_cols;                  // TMEM columns to allocate (power of two >= the chunk's accumulators)
  int32_t Ci, BW;                     // stem form: image channels; width in floats of an image block in shared memory (8 GR + 8)
  int32_t off_xlo;                    // stem form: the lo chunk's GEMM operand buffer
  int32_t cpi, total_chunks;          // chunks per image strip (H/4), N * ns * cpi
  int32_t dw_warps;                   // warps of the CTA = warps of the depthwise tail (tasks packed: hi columns, then lo)
  int32_t hi_stage_bytes, lo_stage_bytes;
  unsigned long long* dbg;             // optional: per-CTA phase cycle counters [grid][8] (CSNET_ILS_DBG=1)
  int32_t off_xl, off_xh, off_t1l, off_wbh, off_wbl, off_bar, off_zero, off_epi, smem_bytes;
};

__device__ __forceinline__ void tma_load_5d(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3, int c4) {
  asm volatile("cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];\n"
               ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4) : "memory");
}
__device__ __forceinline__ void tma_load_4d_a(uint32_t dst, const CUtensorMap* tm, uint32_t bar, int c0, int c1, int c2, int c3) {
  asm volatile("cp.async.bulk.tensor.4d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6}], [%2];\n"
               ::"r"(dst), "l"(tm), "r"(bar), "r"(c0), "r"(c1), "r"(c2), "r"(c3) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx_a(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;\n" ::"r"(bar), "r"(bytes) : "memory");
}
// parity wait with a wall-clock bound: a lost TMA / MMA must trap, not hang the GPU
__device__ __forceinline__ void mbar_wait_a(uint32_t bar, uint32_t parity) {
  uint32_t ok = 0;
  const long long t0 = clock64();
  while (true) {
    asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}\n"
                 : "=r"(ok) : "r"(bar), "r"(parity) : "memory");
    if (ok) break;
    if (clock64() - t0 > 4000000000LL) __trap();
  }
}
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
  // shared-memory matrix descriptor, no swizzle, version 1 (sm_100): start / LBO / SBO in 16-byte units
  return (uint64_t)((saddr & 0x3FFFF) >> 4) | ((uint64_t)((lbo_bytes >> 4) & 0x3FFF) << 16) |
         ((uint64_t)((sbo_bytes >> 4) & 0x3FFF) << 32) | ((uint64_t)1 << 46);
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t da, uint64_t db, uint32_t idesc, uint32_t accumulate) {
  asm volatile("{\n\t.reg .pred p;\n\tsetp.ne.b32 p, %4, 0;\n\ttcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}\n"
               ::"r"(tmem_d), "l"(da), "l"(db), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t taddr, uint32_t (&r)[16]) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];\n"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
        "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
}
__device__ __forceinline__ uint32_t lds32(uint32_t a) { uint32_t v; asm volatile("ld.shared.b32 %0, [%1];\n" : "=r"(v) : "r"(a)); return v; }
__device__ __forceinline__ uint2 lds64(uint32_t a) { uint2 v; asm volatile("ld.shared.v2.b32 {%0, %1}, [%2];\n" : "=r"(v.x), "=r"(v.y) : "r"(a)); return v; }
__device__ __forceinline__ uint4 lds128(uint32_t a) {
  uint4 v;
  asm volatile("ld.shared.v4.b32 {%0, %1, %2, %3}, [%4];\n" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(a));
  return v;
}
__device__ __forceinline__ uint16_t lds16(uint32_t a) { uint16_t v; asm volatile("ld.shared.u16 %0, [%1];\n" : "=h"(v) : "r"(a)); return v; }
__device__ __forceinline__ void sts128(uint32_t a, uint4 v) {
  asm volatile("st.shared.v4.b32 [%0], {%1, %2, %3, %4};\n" ::"r"(a), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void sts16(uint32_t a, uint16_t v) { asm volatile("st.shared.u16 [%0], %1;\n" ::"r"(a), "h"(v) : "memory"); }

// element j of a row of packed 16-bit pairs
__device__ __forceinline__ uint16_t h16(const uint32_t* row, int j) { return (j & 1) ? (uint16_t)(row[j >> 1] >> 16) : (uint16_t)row[j >> 1]; }

// One step of the depthwise tail: T1 row r arrives (n1: pixels x0-2 .. x0+9 of this thread's channel), T2 row r-1 is
// made from T1 rows r-2, r-1, r (10 pixels: x0-1 .. x0+8), the block output row r-2 from T2 rows r-3, r-2, r-1.
template <typename T>
__device__ __forceinline__ void ils_dw_push(uint32_t (&t1)[2][6], uint32_t (&t2)[2][5], const uint32_t (&n1)[6],
                                            const uint32_t (&w1)[5], float b1, float s1, const uint32_t (&w2)[5], float b2, float s2,
                                            bool make_t2, float mL, float mR, bool make_out, uint16_t* out) {
  uint32_t q[5];
  if (make_t2) {
#pragma unroll
    for (int i = 0; i < 10; i += 2) {
      float v0 = b1, v1 = b1;
#pragma unroll
      for (int dy = 0; dy < 3; ++dy) {
        const uint32_t* row = dy == 0 ? t1[0] : (dy == 1 ? t1[1] : n1);
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          const uint16_t w = h16(w1, dy * 3 + dx);
          v0 = Pack<T>::fma16(h16(row, i + dx), w, v0);
          v1 = Pack<T>::fma16(h16(row, i + 1 + dx), w, v1);
        }
      }
      v0 = prelu_m1(v0, s1);
      v1 = prelu_m1(v1, s1);
      if (i == 0) v0 *= mL;          // T2 at x0-1 is conv padding when the column is the image's first
      if (i == 8) v1 *= mR;          // T2 at x0+8 likewise on the right
      q[i >> 1] = Pack<T>::from_f2(v0, v1);
    }
  } else {
#pragma unroll
    for (int i = 0; i < 5; ++i) q[i] = 0u;
  }
  if (make_out) {
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 8; k += 2) {
      float v0 = b2, v1 = b2;
#pragma unroll
      for (int dy = 0; dy < 3; ++dy) {
        const uint32_t* row = dy == 0 ? t2[0] : (dy == 1 ? t2[1] : q);
#pragma unroll
        for (int dx = 0; dx < 3; ++dx) {
          const uint16_t w = h16(w2, dy * 3 + dx);
          v0 = Pack<T>::fma16(h16(row, k + dx), w, v0);
          v1 = Pack<T>::fma16(h16(row, k + 1 + dx), w, v1);
        }
      }
      o[k >> 1] = Pack<T>::from_f2(prelu_m1(v0, s2), prelu_m1(v1, s2));
    }
    *reinterpret_cast<uint4*>(out) = make_uint4(o[0], o[1], o[2], o[3]);
  }
#pragma unroll
  for (int i = 0; i < 6; ++i) { t1[0][i] = t1[1][i]; t1[1][i] = n1[i]; }
#pragma unroll
  for (int i = 0; i < 5; ++i) { t2[0][i] = t2[1][i]; t2[1][i] = q[i]; }
}

__device__ __forceinline__ void tmem_ld_16x256b_x2(uint32_t taddr, uint32_t (&r)[8]) {
  asm volatile("tcgen05.ld.sync.aligned.16x256b.x2.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]) : "r"(taddr));
  asm volatile("tcgen05.wait::ld.sync.aligned;\n" ::: "memory");
}
__device__ __forceinline__ void stsm_x4_trans(uint32_t addr, uint32_t a, uint32_t b, uint32_t c, uint32_t d) {
  asm volatile("stmatrix.sync.aligned.m8n8.x4.trans.shared.b16 [%0], {%1, %2, %3, %4};\n" ::"r"(addr), "r"(a), "r"(b), "r"(c), "r"(d) : "memory");
}

// Epilogue of one warp's 32 accumulator rows (= 32 pixels = 4 pixel groups, TMEM lanes [32 q, 32 q + 32)) of a 128-pixel
// block: tcgen05.ld in the 16x256b shape hands a thread the mma-style fragment (row lane/4 and lane/4 + 8, columns
// 2 (lane % 4) + {0, 1} of every 8-column slab) = pixel rows x channel pairs; + bias, PReLU, pack to 16 bits, then
// stmatrix.trans writes each 8 px x 8 channel fragment as 8 channel rows of 8 contiguous pixels — exactly the
// [group][slot][8 px] tile.  16 channels x 16 pixels per round trip.  g0: first pixel group of the warp's 4,
// ngroups: groups of the chunk (later ones are MMA padding: stored to `dummy`), gstride = slots * 16 bytes.
// eb / es: shared-memory tables of bias and (slope - 1) per channel.
template <typename T>
__device__ __forceinline__ void ils_epilogue_warp(uint32_t taddr, uint32_t tile, uint32_t gstride, int g0, int ngroups, int C,
                                                  uint32_t eb, uint32_t es, uint32_t dummy, int lane) {
  const int q = lane & 3, mrow = lane & 7, mat = lane >> 3;
#pragma unroll 1
  for (int cc = 0; cc * 16 < C; ++cc) {
    const uint32_t co = (uint32_t)(cc * 16 + 2 * q) * 4u;
    const uint2 bA = lds64(eb + co), bB = lds64(eb + co + 32u), sA = lds64(es + co), sB = lds64(es + co + 32u);
    const float b0 = __uint_as_float(bA.x), b1 = __uint_as_float(bA.y), b2 = __uint_as_float(bB.x), b3 = __uint_as_float(bB.y);
    const float s0 = __uint_as_float(sA.x), s1 = __uint_as_float(sA.y), s2 = __uint_as_float(sB.x), s3 = __uint_as_float(sB.y);
#pragma unroll
    for (int h = 0; h < 2; ++h) {
      uint32_t r[8];
      tmem_ld_16x256b_x2(taddr + ((uint32_t)(16 * h) << 16) + (uint32_t)(cc * 16), r);
      const uint32_t m0 = Pack<T>::from_f2(prelu_m1(__uint_as_float(r[0]) + b0, s0), prelu_m1(__uint_as_float(r[1]) + b1, s1));
      const uint32_t m1 = Pack<T>::from_f2(prelu_m1(__uint_as_float(r[2]) + b0, s0), prelu_m1(__uint_as_float(r[3]) + b1, s1));
      const uint32_t m2 = Pack<T>::from_f2(prelu_m1(__uint_as_float(r[4]) + b2, s2), prelu_m1(__uint_as_float(r[5]) + b3, s3));
      const uint32_t m3 = Pack<T>::from_f2(prelu_m1(__uint_as_float(r[6]) + b2, s2), prelu_m1(__uint_as_float(r[7]) + b3, s3));
      // matrix `mat` of the x4 store: pixel group g0 + 2h + (mat & 1), channels 16 cc + 8 (mat >> 1) ..; this lane addresses row mrow
      const int pg = g0 + 2 * h + (mat & 1);
      const uint32_t addr = pg < ngroups ? tile + (uint32_t)pg * gstride + (uint32_t)(cc * 16 + 8 * (mat >> 1) + mrow) * 16u
                                         : dummy + (uint32_t)(mat * 8 + mrow) * 16u;
      stsm_x4_trans(addr, m0, m1, m2, m3);
    }
  }
}

template <typename T, bool kTiming = false, bool kStem = false>
__global__ void __launch_bounds__(kIlsMaxThreads, 1)
il_stream_kernel(const __grid_constant__ IlsArgs A, const __grid_constant__ CUtensorMap tmH, const __grid_constant__ CUtensorMap tmL) {
  extern __shared__ uint8_t smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nthreads = blockDim.x, nwarps = nthreads >> 5;
  const uint32_t sbase = (smem_u32(smem_raw) + 127u) & ~127u;
  const uint32_t XL = sbase + A.off_xl, XH = sbase + A.off_xh, T1L = sbase + A.off_t1l, WBH = sbase + A.off_wbh,
                 WBL = sbase + A.off_wbl, BAR = sbase + A.off_bar, ZERO = sbase + A.off_zero;
  uint8_t* gbase = smem_raw + (sbase - smem_u32(smem_raw));      // generic pointer to the same place
  // barriers: [0,2) hi stage full, [2,5) lo stage full; +64 the TMEM base slot; +128: one per accumulator block (16)
  const uint32_t bar_h = BAR, bar_l = BAR + 16, bar_m = BAR + 128;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(gbase + A.off_bar + 64);
  const uint32_t EPI = sbase + A.off_epi, DUMMY = EPI + 1024;     // bias_h, sm1_h, bias_l, sm1_l (64 floats each); scratch rows

  const int H = A.H, W = A.W, Hl = H >> 1, Wl = W >> 1;
  const int Chi = A.Chi, Cli = A.Cli, Cho = A.Cho, Clo = A.Clo;
  const int GH = A.GH, GL = A.GL, SH = A.SH, SL = A.SL, ST = A.ST, NH = A.NH, NL = A.NL, K16 = A.K16;
  const int GR = A.GR, GLR = A.GLR, hl = A.hl, gsn = A.gsn;
  const int cpi = A.cpi;

  // ---- one-time setup -----------------------------------------------------------------------------------
  if (tid == 0) {
    for (int i = 0; i < 6; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(BAR + 8 * i) : "memory");
    for (int i = 0; i < 16; ++i) asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;\n" ::"r"(bar_m + 8 * i) : "memory");
    asm volatile("fence.mbarrier_init.release.cluster;\n" ::: "memory");
  }
  if (warp == 0) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;\n" ::"r"(BAR + 64), "r"(A.tmem_cols) : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;\n" ::: "memory");
  }
  // weights -> K-major B operand: core matrices [n group][k group][8 n][8 k]
  {
    uint16_t* wb = reinterpret_cast<uint16_t*>(gbase + A.off_wbh);
    const uint16_t* src = reinterpret_cast<const uint16_t*>(A.wh);
    for (int i = tid; i < NH * K16; i += nthreads) {
      const int n = i / K16, k = i - n * K16;
      wb[(((n >> 3) * (K16 >> 3) + (k >> 3)) * 8 + (n & 7)) * 8 + (k & 7)] = k < A.K8 ? src[n * A.K8 + k] : (uint16_t)0;
    }
    if (NL > 0) {
      wb = reinterpret_cast<uint16_t*>(gbase + A.off_wbl);
      src = reinterpret_cast<const uint16_t*>(A.wl);
      for (int i = tid; i < NL * K16; i += nthreads) {
        const int n = i / K16, k = i - n * K16;
        wb[(((n >> 3) * (K16 >> 3) + (k >> 3)) * 8 + (n & 7)) * 8 + (k & 7)] = k < A.K8 ? src[n * A.K8 + k] : (uint16_t)0;
      }
    }
    if (tid < 16) reinterpret_cast<uint32_t*>(gbase + A.off_zero)[tid] = 0u;
    if (kStem) {
      // K-padding slots [Chi, K16) of both operand buffers: zero once (the im2col build never touches them, the in-place
      // epilogue only writes slots < NH <= Chi)
      // (both hi buffers: the build alternates between them so that it never overwrites the T1 the depthwise tail still reads)
      const int per = K16 - Chi, padh = per * 4 * GR, padl = per * 2 * GLR;
      for (int i = tid; i < 2 * padh + padl; i += nthreads) {
        const bool hb = i < 2 * padh;
        const int st = hb ? i / padh : 0, j = hb ? i - st * padh : i - 2 * padh, g_ = j / per, k_ = Chi + (j - g_ * per);
        sts128((hb ? XH + (uint32_t)st * (uint32_t)A.hi_stage_bytes + (uint32_t)(g_ * SH + k_) * 16u
                   : sbase + A.off_xlo + (uint32_t)(g_ * SL + k_) * 16u), make_uint4(0u, 0u, 0u, 0u));
      }
    }
    if (tid < kIlsMaxC) {
      float* ep = reinterpret_cast<float*>(gbase + A.off_epi);
      ep[tid] = A.bias_h[tid]; ep[kIlsMaxC + tid] = A.sm1_h[tid]; ep[2 * kIlsMaxC + tid] = A.bias_l[tid]; ep[3 * kIlsMaxC + tid] = A.sm1_l[tid];
    }
  }
  asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
  const uint32_t tmem = *tmem_slot;

  // depthwise-tail role of this thread (fixed for the whole kernel): a channel and an 8-pixel column
  // tail tasks are packed: threads [0, Cho * gsn) own a hi (channel, column), the next Clo * gsn / 2 a lo one
  const int n_hi_tasks = Cho * gsn;
  const bool dw_hi = tid < n_hi_tasks;
  const int dwt = dw_hi ? tid : tid - n_hi_tasks;
  const int Gd = dw_hi ? gsn : gsn >> 1, Cd = dw_hi ? Cho : Clo, Sd = dw_hi ? SH : ST;   // Gd: this role's groups per strip row
  const bool dw_live = dwt < Cd * Gd;
  const int dc = dw_live ? dwt / Gd : 0, dg = dw_live ? dwt - dc * Gd : 0;
  uint32_t w1[5], w2[5];
  float b1, s1, b2, s2;
  {
    const DwParams& P1 = dw_hi ? A.dw1h : A.dw1l;
    const DwParams& P2 = dw_hi ? A.dw2h : A.dw2l;
    float f1[10], f2[10];
#pragma unroll
    for (int i = 0; i < 9; ++i) {
      f1[i] = dw_live ? __ldg(P1.w + dc * 9 + i) : 0.f;
      f2[i] = dw_live ? __ldg(P2.w + dc * 9 + i) : 0.f;
    }
    f1[9] = f2[9] = 0.f;
#pragma unroll
    for (int i = 0; i < 5; ++i) { w1[i] = Pack<T>::from_f2(f1[2 * i], f1[2 * i + 1]); w2[i] = Pack<T>::from_f2(f2[2 * i], f2[2 * i + 1]); }
    b1 = dw_live ? __ldg(P1.b + dc) : 0.f; s1 = dw_live ? __ldg(P1.s + dc) - 1.f : 0.f;
    b2 = dw_live ? __ldg(P2.b + dc) : 0.f; s2 = dw_live ? __ldg(P2.s + dc) - 1.f : 0.f;
  }
  const int dw_rows = dw_hi ? 4 : 2;                      // T1 rows per chunk of this role
  const int dHd = dw_hi ? H : Hl, dWd = dw_hi ? W : Wl;
  // byte offsets inside a T1 chunk of this thread's 16-byte row (row 0) and of its two halo pairs
  const uint32_t dw_off = (uint32_t)((dg + hl) * Sd + dc) * 16u, dw_rowstep = (uint32_t)((dw_hi ? GR : GLR) * Sd) * 16u;
  const int Gimg = dw_hi ? GH : GL;                       // groups per image row of this role

  const uint32_t idesc_h = (1u << 4) | (1u << 15) | ((uint32_t)(NH >> 3) << 17) | (8u << 24);   // f16 x f16 -> f32, A MN-major, M = 128
  const uint32_t idesc_l = (1u << 4) | (1u << 15) | ((uint32_t)(NL >> 3) << 17) | (8u << 24);
  const int nbh = (4 * GR + 15) >> 4, nbl = NL > 0 ? (2 * GLR + 15) >> 4 : 0;
  const uint32_t hi_tx = (uint32_t)(64 * SH * GR), lo_tx = kStem ? (uint32_t)(A.BW * 4 * A.Ci * 4) : (uint32_t)(32 * SL * GLR);
  const uint32_t XLO = sbase + A.off_xlo;

  // ---- the CTA's range of the (image, chunk) sequence ------------------------------------------------
  int ra = (int)((long long)blockIdx.x * A.total_chunks / gridDim.x);
  const int rb = (int)((long long)(blockIdx.x + 1) * A.total_chunks / gridDim.x);
  uint32_t hq = 0, lq = 0, mq = 0;                       // running counts: hi loads, lo loads, MMA commits
  long long tph[8] = {0, 0, 0, 0, 0, 0, 0, 0}, tlast = clock64();
  const bool timing = kTiming && A.dbg != nullptr && tid == 0;
#define ILS_MARK(i) do { if (kTiming && timing) { const long long t_ = clock64(); tph[i] += t_ - tlast; tlast = t_; } } while (0)

  while (ra < rb) {
    const int item = ra / cpi, ca = ra - item * cpi;
    const int n = item / A.ns, gs0 = (item - n * A.ns) * gsn;                      // image, first hi group of the column strip
    const int cb = (ca + (rb - ra)) < cpi ? (ca + (rb - ra)) : cpi;
    ra += cb - ca;
    const int c0 = ca > 0 ? ca - 1 : 0, c1 = cb < cpi ? cb : cpi - 1;              // hi chunks walked (warm-up / look-ahead)
    const int cl0 = c0 > 0 ? c0 - 1 : 0, cl1 = c1 + 1 < cpi ? c1 + 1 : cpi - 1;    // lo chunks loaded
    const int out_lo = dw_hi ? 4 * ca : 2 * ca, out_hi = dw_hi ? 4 * cb : 2 * cb;  // rows this role stores
    const uint32_t hq0 = hq, lq0 = lq;
    hq += (uint32_t)(c1 - c0 + 1);
    lq += (uint32_t)(cl1 - cl0 + 1);
    auto hi_stage = [&](int c) { return XH + ((hq0 + (uint32_t)(c - c0)) & 1u) * (uint32_t)A.hi_stage_bytes; };
    auto lo_stage = [&](int cl) { return XL + ((lq0 + (uint32_t)(cl - cl0)) % 3u) * (uint32_t)A.lo_stage_bytes; };
    auto issue_hi = [&](int c) {
      const uint32_t q = hq0 + (uint32_t)(c - c0), bar = bar_h + 8 * (q & 1u);
      mbar_expect_tx_a(bar, hi_tx);
      tma_load_5d(hi_stage(c), &tmH, bar, 0, 0, gs0 - hl, 4 * c, n);
    };
    auto issue_lo = [&](int cl) {
      const uint32_t q = lq0 + (uint32_t)(cl - cl0), bar = bar_l + 8 * (q % 3u);
      mbar_expect_tx_a(bar, lo_tx);
      if (kStem) tma_load_4d_a(lo_stage(cl), &tmL, bar, 8 * (gs0 - hl) - 4, 4 * cl, 0, n);     // image block: rows [4 cl, 4 cl + 4), all channels
      else tma_load_5d(lo_stage(cl), &tmL, bar, 0, 0, (gs0 >> 1) - hl, 2 * cl, n);
    };
    if (tid == 0) {
      asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
      if (!kStem) {
        issue_hi(c0);
        if (c0 + 1 <= c1) issue_hi(c0 + 1);
      }
      for (int cl = cl0; cl <= cl1 && cl <= c0 + 1; ++cl) issue_lo(cl);
    }
    int lo_waited = 0;
    uint32_t t1w[2][6], t2w[2][5];
#pragma unroll
    for (int i = 0; i < 6; ++i) t1w[0][i] = t1w[1][i] = 0u;
#pragma unroll
    for (int i = 0; i < 5; ++i) t2w[0][i] = t2w[1][i] = 0u;
    const int gimg = (dw_hi ? gs0 : gs0 >> 1) + dg;                                // this thread's group in the image row
    const bool edgeL = gimg == 0, edgeR = gimg == Gimg - 1;
    const float mL = edgeL ? 0.f : 1.f, mR = edgeR ? 0.f : 1.f;
    uint16_t* ybase = reinterpret_cast<uint16_t*>(dw_hi ? A.yh : A.yl) + ((size_t)n * Cd + dc) * dHd * dWd + 8 * gimg;

    for (int c = c0; c <= c1; ++c) {
      // ---- 1. the chunk's inputs have landed -----------------------------------------------------------
      {
        const uint32_t q = hq0 + (uint32_t)(c - c0);
        if (!kStem) mbar_wait_a(bar_h + 8 * (q & 1u), (q >> 1) & 1u);
        const int need = (c + 1 < cpi ? c + 1 : cpi - 1) - cl0 + 1;
        while (lo_waited < need) {
          const uint32_t ql = lq0 + (uint32_t)lo_waited;
          mbar_wait_a(bar_l + 8 * (ql % 3u), (ql / 3u) & 1u);
          ++lo_waited;
        }
      }
      ILS_MARK(0);
      const uint32_t xh = hi_stage(c), xl = kStem ? XLO : lo_stage(c);
      if (kStem) {
        // ---- 2s. im2col of the image chunk (hi) and of its 2x2 max-pool (lo): a task = one (row, group, ci, ky) and makes
        //          the three kx slots from one 10-pixel window -----------------------------------------------------------
        const int Ci = A.Ci, BW = A.BW;
        const int n_hi = 4 * GR * Ci * 3, n_lo = Clo > 0 ? 2 * GLR * Ci * 3 : 0;
        for (int task = tid; task < n_hi + n_lo; task += nthreads) {
          const bool hb = task < n_hi;
          const int t = hb ? task : task - n_hi, Gt = hb ? GR : GLR;
          const int ck = t % (Ci * 3), rg = t / (Ci * 3);               // ck = ci * 3 + ky; rg = row * Gt + group
          const int ci = ck / 3, ky = ck - ci * 3, r = rg / Gt, g = rg - r * Gt;
          float f[10];
          if (hb) {
            const int yy = 4 * c + r + ky - 1;                           // image row of this tap row
            if (yy >= 0 && yy < H) {
              const uint32_t a = lo_stage(yy >> 2) + (uint32_t)(((ci * 4 + (yy & 3)) * BW + 8 * g + 3) * 4);
              const uint4 m0 = lds128(a + 4u), m1 = lds128(a + 20u);
              f[0] = __uint_as_float(lds32(a)); f[9] = __uint_as_float(lds32(a + 36u));
              f[1] = __uint_as_float(m0.x); f[2] = __uint_as_float(m0.y); f[3] = __uint_as_float(m0.z); f[4] = __uint_as_float(m0.w);
              f[5] = __uint_as_float(m1.x); f[6] = __uint_as_float(m1.y); f[7] = __uint_as_float(m1.z); f[8] = __uint_as_float(m1.w);
            } else {
#pragma unroll
              for (int j = 0; j < 10; ++j) f[j] = 0.f;
            }
          } else {
            const int yl = 2 * c + r + ky - 1;                           // lo row of this tap row: max of image rows 2 yl, 2 yl + 1
            const int col0 = 16 * g - 8 * hl + 2;                        // block column of image x = 2 (xl0 - 1)
            if (yl >= 0 && yl < Hl) {
              const uint32_t a = lo_stage(yl >> 1) + (uint32_t)(((ci * 4 + ((2 * yl) & 3)) * BW) * 4);
#pragma unroll
              for (int j = 0; j < 10; ++j) {
                const int col = col0 + 2 * j;
                float v = 0.f;
                if (col >= 0 && col + 1 < BW) {                          // outside: the never-read outer half of a halo group
                  const uint2 u0 = lds64(a + (uint32_t)col * 4u), u1 = lds64(a + (uint32_t)(col + BW) * 4u);
                  v = fmaxf(fmaxf(__uint_as_float(u0.x), __uint_as_float(u0.y)), fmaxf(__uint_as_float(u1.x), __uint_as_float(u1.y)));
                }
                f[j] = v;
              }
            } else {
#pragma unroll
              for (int j = 0; j < 10; ++j) f[j] = 0.f;
            }
          }
          const uint32_t e0 = Pack<T>::from_f2(f[0], f[1]), e1 = Pack<T>::from_f2(f[2], f[3]), e2 = Pack<T>::from_f2(f[4], f[5]),
                         e3 = Pack<T>::from_f2(f[6], f[7]), e4 = Pack<T>::from_f2(f[8], f[9]);
          const uint32_t o0 = Pack<T>::from_f2(f[1], f[2]), o1 = Pack<T>::from_f2(f[3], f[4]), o2 = Pack<T>::from_f2(f[5], f[6]),
                         o3 = Pack<T>::from_f2(f[7], f[8]);
          const uint32_t dst = (hb ? xh + (uint32_t)(rg * SH) * 16u : xl + (uint32_t)(rg * SL) * 16u) + (uint32_t)(ck * 3) * 16u;
          sts128(dst, make_uint4(e0, e1, e2, e3));                       // kx = 0: pixels x-1 .. x+6
          sts128(dst + 16u, make_uint4(o0, o1, o2, o3));                 // kx = 1: x .. x+7
          sts128(dst + 32u, make_uint4(e1, e2, e3, e4));                 // kx = 2: x+1 .. x+8
        }
      } else {
      // ---- 2. resample both ways ------------------------------------------------------------------------
        const int n_up = Cli * GR, n_pool = Clo > 0 ? Chi * GLR : 0;
        for (int task = tid; task < n_up + n_pool; task += nthreads) {
          if (task < n_up) {
            // bilinear x2 (align_corners=False): hi pixel 2j = 1/4 lo[j-1] + 3/4 lo[j], 2j+1 = 3/4 lo[j] + 1/4 lo[j+1], clamped
            const int cl_ = task / GR, gr = task - cl_ * GR;                    // gr: group in the tile row; g: in the image row
            const int g = gs0 - hl + gr;
            if (g < 0 || g >= GH) continue;                                       // halo group outside the image: stays zero, never read
            const int glr = (g >> 1) - (gs0 >> 1) + hl, hf = g & 1;               // lo group in the lo tile row
            const uint32_t offM = (uint32_t)(glr * SL + cl_) * 16u + 8u * hf;
            const uint32_t offL = hf ? offM - 2u : (g == 0 ? offM : offM - (uint32_t)SL * 16u + 14u);
            const uint32_t offR = hf ? (g == GH - 1 ? offM + 6u : offM + (uint32_t)SL * 16u - 8u) : offM + 8u;
            float hrow[4][8];
            const uint16_t w25 = Pack<T>::bits(0.25f), w75 = Pack<T>::bits(0.75f);
#pragma unroll
            for (int k = 0; k < 4; ++k) {
              int R = 2 * c - 1 + k;
              R = R < 0 ? 0 : (R > Hl - 1 ? Hl - 1 : R);
              const uint32_t rowb = lo_stage(R >> 1) + (uint32_t)((R & 1) * GLR * SL) * 16u;
              const uint2 m = lds64(rowb + offM);
              const uint16_t vl = lds16(rowb + offL), vr = lds16(rowb + offR);
              const uint16_t v0 = (uint16_t)m.x, v1 = (uint16_t)(m.x >> 16), v2 = (uint16_t)m.y, v3 = (uint16_t)(m.y >> 16);
              hrow[k][0] = Pack<T>::fma16(v0, w75, Pack<T>::fma16(vl, w25, 0.f));
              hrow[k][1] = Pack<T>::fma16(v0, w75, Pack<T>::fma16(v1, w25, 0.f));
              hrow[k][2] = Pack<T>::fma16(v1, w75, Pack<T>::fma16(v0, w25, 0.f));
              hrow[k][3] = Pack<T>::fma16(v1, w75, Pack<T>::fma16(v2, w25, 0.f));
              hrow[k][4] = Pack<T>::fma16(v2, w75, Pack<T>::fma16(v1, w25, 0.f));
              hrow[k][5] = Pack<T>::fma16(v2, w75, Pack<T>::fma16(v3, w25, 0.f));
              hrow[k][6] = Pack<T>::fma16(v3, w75, Pack<T>::fma16(v2, w25, 0.f));
              hrow[k][7] = Pack<T>::fma16(v3, w75, Pack<T>::fma16(vr, w25, 0.f));
            }
            const uint32_t dst = xh + (uint32_t)(gr * SH + Chi + cl_) * 16u;
#pragma unroll
            for (int rr = 0; rr < 4; ++rr) {
              // hi row 4c+rr: rr 0: (k0 1/4, k1 3/4); 1: (k1 3/4, k2 1/4); 2: (k1 1/4, k2 3/4); 3: (k2 3/4, k3 1/4)
              const int km = rr < 2 ? 1 : 2, ko = rr == 0 ? 0 : (rr == 3 ? 3 : (rr == 1 ? 2 : 1));
              uint4 o;
              o.x = Pack<T>::from_f2(0.75f * hrow[km][0] + 0.25f * hrow[ko][0], 0.75f * hrow[km][1] + 0.25f * hrow[ko][1]);
              o.y = Pack<T>::from_f2(0.75f * hrow[km][2] + 0.25f * hrow[ko][2], 0.75f * hrow[km][3] + 0.25f * hrow[ko][3]);
              o.z = Pack<T>::from_f2(0.75f * hrow[km][4] + 0.25f * hrow[ko][4], 0.75f * hrow[km][5] + 0.25f * hrow[ko][5]);
              o.w = Pack<T>::from_f2(0.75f * hrow[km][6] + 0.25f * hrow[ko][6], 0.75f * hrow[km][7] + 0.25f * hrow[ko][7]);
              sts128(dst + (uint32_t)(rr * GR * SH) * 16u, o);
            }
          } else {
            // max_pool2d 2x2: lo group glr of lo rows 2c, 2c+1 from the two hi groups under it, 4 hi rows.  With a halo the
            // outer hi group of the tile's first / last lo group is not in the tile: that half is never read downstream.
            const int t = task - n_up, ch = t / GLR, glr = t - ch * GLR;
            const int ga = 2 * glr - hl;                                          // tile index of the left hi group
            const bool okA = ga >= 0, okB = ga + 1 < GR;
            const uint32_t src = xh + (uint32_t)(ga * SH + ch) * 16u;
            const uint32_t dst = xl + (uint32_t)(glr * SL + Cli + ch) * 16u;
#pragma unroll
            for (int lr = 0; lr < 2; ++lr) {
              const uint32_t r0 = src + (uint32_t)(2 * lr * GR * SH) * 16u, r1 = r0 + (uint32_t)(GR * SH) * 16u;
              const uint4 a0 = lds128(okA ? r0 : ZERO), a1 = lds128(okB ? r0 + (uint32_t)SH * 16u : ZERO), c0_ = lds128(okA ? r1 : ZERO),
                          c1_ = lds128(okB ? r1 + (uint32_t)SH * 16u : ZERO);
              auto hmax = [](uint32_t u, uint32_t v) {       // two lo pixels from the vertical maxima of 4 hi pixels
                return __byte_perm(Pack<T>::max2(u, __byte_perm(u, 0u, 0x1032)), Pack<T>::max2(v, __byte_perm(v, 0u, 0x1032)), 0x5410);
              };
              uint4 o;
              o.x = hmax(Pack<T>::max2(a0.x, c0_.x), Pack<T>::max2(a0.y, c0_.y));
              o.y = hmax(Pack<T>::max2(a0.z, c0_.z), Pack<T>::max2(a0.w, c0_.w));
              o.z = hmax(Pack<T>::max2(a1.x, c1_.x), Pack<T>::max2(a1.y, c1_.y));
              o.w = hmax(Pack<T>::max2(a1.z, c1_.z), Pack<T>::max2(a1.w, c1_.w));
              sts128(dst + (uint32_t)(lr * GLR * SL) * 16u, o);
            }
          }
        }
      }
      ILS_MARK(1);
      asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");    // generic writes -> visible to the tensor core / TMA
      __syncthreads();                                                    // (A)
      ILS_MARK(2);
      // ---- 3. next loads (one thread of the last warp); the chunk's MMAs: warp b's elected lane issues block b ----
      if (warp == nwarps - 1 && lane == 0) {
        asm volatile("fence.proxy.async.shared::cta;\n" ::: "memory");
        if (!kStem && c >= c0 + 1 && c + 1 <= c1) issue_hi(c + 1);       // stage of chunk c-1: its T1 was consumed
        if (c + 2 <= cl1) issue_lo(c + 2);                               // stage of lo chunk c-1: last read by this chunk's up-sample
      }
      if (lane == 0) {
        for (int b = warp; b < nbh + nbl; b += nwarps) {
          asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
          const bool hb = b < nbh;
          const int lb = hb ? b : b - nbh, S_ = hb ? SH : SL;
          const uint64_t da = umma_desc((hb ? xh : xl) + (uint32_t)(lb * 16 * S_) * 16u, 128u, (uint32_t)S_ * 16u);
          const uint64_t db = umma_desc(hb ? WBH : WBL, 128u, (uint32_t)(K16 >> 3) * 128u);
          const uint32_t tm = tmem + (uint32_t)(hb ? lb * NH : nbh * NH + lb * NL), idesc = hb ? idesc_h : idesc_l;
          for (int ks = 0; ks < (K16 >> 4); ++ks) umma_f16(tm, da + (uint64_t)(16 * ks), db + (uint64_t)(16 * ks), idesc, ks > 0);
          asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];\n" ::"r"(bar_m + 8u * b) : "memory");
        }
      }
      __syncwarp();
      ILS_MARK(3);
      // ---- 4. epilogue: TMEM -> bias, PReLU, 16-bit -> T1 (hi: in place over the chunk; lo: its own buffer) ----
      if (warp < (nwarps & ~3)) {
        const int qd = warp & 3, wstep = nwarps >> 2;
        for (int b = warp >> 2; b < nbh + nbl; b += wstep) {
          mbar_wait_a(bar_m + 8u * b, mq & 1u);                      // the block's MMAs (and all earlier ones) have completed
          asm volatile("tcgen05.fence::after_thread_sync;\n" ::: "memory");
          if (b < nbh)
            ils_epilogue_warp<T>(tmem + ((uint32_t)(qd * 32) << 16) + (uint32_t)(b * NH), xh, (uint32_t)SH * 16u, b * 16 + qd * 4, 4 * GR, Cho,
                                 EPI, EPI + 256u, DUMMY, lane);
          else
            ils_epilogue_warp<T>(tmem + ((uint32_t)(qd * 32) << 16) + (uint32_t)(nbh * NH + (b - nbh) * NL), T1L, (uint32_t)ST * 16u,
                                 (b - nbh) * 16 + qd * 4, 2 * GLR, Clo, EPI + 512u, EPI + 768u, DUMMY, lane);
        }
      }
      ++mq;
      ILS_MARK(4);
      asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
      __syncthreads();                                                    // (B)
      ILS_MARK(5);
      // ---- 5. depthwise tail over the chunk's rows --------------------------------------------------------
      if (dw_live) {
        const uint32_t t1b = (dw_hi ? xh : T1L) + dw_off;
        for (int rr = 0; rr < dw_rows; ++rr) {
          const int r = dw_rows * c + rr;                                // T1 row arriving; T2 row r-1; output row r-2
          const uint32_t p = t1b + (uint32_t)rr * dw_rowstep;
          uint32_t n1[6];
          const uint4 m = lds128(p);
          n1[0] = lds32(edgeL ? ZERO : p - (uint32_t)Sd * 16u + 12u);
          n1[1] = m.x; n1[2] = m.y; n1[3] = m.z; n1[4] = m.w;
          n1[5] = lds32(edgeR ? ZERO : p + (uint32_t)Sd * 16u);
          const int tr = r - 1, orow = r - 2;
          const bool make_t2 = tr >= 0 && tr >= out_lo - 1 && tr <= out_hi;
          const bool make_out = orow >= out_lo && orow < out_hi;
          ils_dw_push<T>(t1w, t2w, n1, w1, b1, s1, w2, b2, s2, make_t2, mL, mR, make_out, ybase + (size_t)orow * dWd);
        }
      }
      ILS_MARK(6);
    }
    // ---- image bottom: two rows of zero padding flush the last two output rows ----------------------------
    if (cb == cpi && dw_live) {
      const uint32_t z[6] = {0u, 0u, 0u, 0u, 0u, 0u};
      for (int rr = 0; rr < 2; ++rr) {
        const int r = dHd + rr, tr = r - 1, orow = r - 2;
        ils_dw_push<T>(t1w, t2w, z, w1, b1, s1, w2, b2, s2, tr < dHd, mL, mR, orow >= out_lo, ybase + (size_t)orow * dWd);
      }
    }
    __syncthreads();          // every shared-memory read of this piece is done before the next piece's loads overwrite it
  }

  if (timing) {
    ILS_MARK(7);
    for (int i = 0; i < 8; ++i) A.dbg[(size_t)blockIdx.x * 8 + i] = (unsigned long long)tph[i];
  }
#undef ILS_MARK
  asm volatile("tcgen05.fence::before_thread_sync;\n" ::: "memory");
  __syncthreads();
  if (warp == 0) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;\n" ::"r"(tmem), "r"(A.tmem_cols) : "memory");
}

}  // namespace csnet
