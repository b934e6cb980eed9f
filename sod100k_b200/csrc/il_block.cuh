// il_block.cuh — one kernel per ILBlock (1x1 kind): gOctaveCBR(1x1, 2 in-branches -> 1|2 out-branches)
// + depthwise 3x3 BN PReLU + depthwise 3x3 BN PReLU; everything between the block's input and output
// tensors stays in shared memory (reference: ILBlock.forward, CSNet/model/csnet.py:72-76, calling
// gOctaveConv.forward :664-726 and SimplifiedGOctConvBR.forward :838-851).
//
// One CTA owns a TH x TW tile of the high-resolution output branch and the co-located (TH/2 x TW/2) tile of
// the low-resolution branch; 16-bit activations (fp16 or bf16), fp32 accumulation.
//
//   load      AH[0..Chi)   = x_h over the hi region (halo 4)       cp.async, zero fill outside the image
//             AL[0..Cli)   = x_l over the lo region
//   resample  AL[Cli..)    = maxpool2x2(AH[0..Chi))                 hi -> lo path reads the pooled input (:709-712)
//             AH[Chi..)    = bilinear_x2(AL[0..Cli))                lo -> hi path; upsampling the conv INPUT is the
//                                                                   same linear map as upsampling its output (:702-707)
//   GEMMs     T1H = PReLU(WH . AH + b)   T1L = PReLU(WL . AL + b)   tensor cores (mma.sync m16n8k8), pixels are the
//                                                                   N dimension, written IN PLACE over AH / AL
//   dw1       T2  = PReLU(dw3x3(T1) + b)                            CUDA cores, fp32 accumulate, both branches
//   dw2       out = PReLU(dw3x3(T2) + b)  ->  global (tile interior only)
//
// T1/T2 are forced to 0 outside the image so the depthwise convs see the reference's zero padding.
// Region geometry (R = region-local coordinates):
//   hi region origin (hy0-4, hx0-4), size RHh x RWh = (TH+8 [+1]) x (TW+8)    halo 4 = 2 (two dw layers) x 2 (pooling)
//   lo region origin (ly0-2, lx0-4), size RHl x RWl = (TH/2+4 [+1]) x (TW/2+8) x origin kept a multiple of 4 (8-byte I/O)
//   lo R(ry, rx)  <->  hi R(2ry, 2rx-4);  the optional +1 row only makes RH*RW/8 odd (conflict-free ldmatrix).
#pragma once
#include <type_traits>
#include <cuda_bf16.h>
#include <cuda_fp16.h>
#include <stdint.h>

namespace csnet {

constexpr int kIlThreads = 512;
constexpr int kIlMaxK8 = 8;         // K (input channels hi + lo) <= 64: all B fragments of 4 pixel tiles stay in registers

struct DwParams {
  const float* w;      // [C][9]
  const float* b;      // [C]
  const float* s;      // [C] PReLU slope
};

struct IlArgs {
  const void* xh;
  const void* xl;
  void* yh;
  void* yl;                    // nullptr when Clo == 0
  const uint32_t* wh;          // packed 16-bit [MH16][K8]   columns: [x_h (Chi) | up(x_l) (Cli)]
  const uint32_t* wl;          // packed 16-bit [ML16][K8]   columns: [x_l (Cli) | pool(x_h) (Chi)]   (Clo > 0 only)
  const float *bias_h, *slope_h, *bias_l, *slope_l;
  DwParams dw1h, dw1l, dw2h, dw2l;
  int32_t H, W;                // hi resolution (lo = H/2 x W/2)
  int32_t Chi, Cli, Cho, Clo;
  int32_t TH, TW, tiles_x;     // tile (one of the instantiated geometries) and tiles per image row
  int32_t K8, MH16, ML16;
  int32_t rowsAh, rowsAl;
  int32_t first;               // 1: stem form — xh is the fp32 image [N][Chi/9][H][W], both branches are 3x3 convs of it
                               //    (lo: of its 2x2 max-pool), lowered to the same GEMMs through im2col planes built in smem
  int32_t t2h;                 // channels of the hi T2 buffer: Cho (whole layer resident) or 8 (channel-chunked dw tail)
};

// Region geometry of a TH x TW tile (compile-time: every divisor / stride below is a constant).
template <int TH_, int TW_>
struct IlGeom {
  static constexpr int TH = TH_, TW = TW_;
  static constexpr int RWh = TW + 8, RHh = (TH + 8) | 1;       // odd row count: RH * RW / 8 is odd when RW / 8 is odd
  static constexpr int RWl = TW / 2 + 8, RHl = (TH / 2 + 4) | 1;
  static constexpr int NPH = RHh * RWh, NPL = RHl * RWl;
  static_assert(TW % 16 == 0 && TH % 2 == 0, "tile shape");
};

// ---- 16-bit helpers -----------------------------------------------------------------------------------
template <typename T> struct Pack;
template <> struct Pack<__half> {
  static __device__ __forceinline__ float2 to_f2(uint32_t v) { return __half22float2(*reinterpret_cast<__half2*>(&v)); }
  static __device__ __forceinline__ float to_f(uint16_t v) { return __half2float(*reinterpret_cast<__half*>(&v)); }
  static __device__ __forceinline__ uint32_t from_f2(float a, float b) {
    __half2 h = __floats2half2_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  static __device__ __forceinline__ uint32_t max2(uint32_t a, uint32_t b) {
    __half2 r = __hmax2(*reinterpret_cast<__half2*>(&a), *reinterpret_cast<__half2*>(&b));
    return *reinterpret_cast<uint32_t*>(&r);
  }
  static __device__ __forceinline__ void mma(float* c, const uint32_t* a, uint32_t b) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};\n"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(b));
  }
  // acc += x * w with 16-bit x, w and fp32 accumulation in ONE instruction (sm_100 FHFMA): no operand conversions
  static __device__ __forceinline__ float fma16(uint16_t x, uint16_t w, float acc) {
    asm("fma.rn.f32.f16 %0, %1, %2, %0;" : "+f"(acc) : "h"(x), "h"(w));
    return acc;
  }
  static __device__ __forceinline__ uint16_t bits(float v) { return __half_as_ushort(__float2half_rn(v)); }
};
template <> struct Pack<__nv_bfloat16> {
  static __device__ __forceinline__ float2 to_f2(uint32_t v) { return __bfloat1622float2(*reinterpret_cast<__nv_bfloat162*>(&v)); }
  static __device__ __forceinline__ float to_f(uint16_t v) { return __bfloat162float(*reinterpret_cast<__nv_bfloat16*>(&v)); }
  static __device__ __forceinline__ uint32_t from_f2(float a, float b) {
    __nv_bfloat162 h = __floats2bfloat162_rn(a, b);
    return *reinterpret_cast<uint32_t*>(&h);
  }
  static __device__ __forceinline__ uint32_t max2(uint32_t a, uint32_t b) {
    __nv_bfloat162 r = __hmax2(*reinterpret_cast<__nv_bfloat162*>(&a), *reinterpret_cast<__nv_bfloat162*>(&b));
    return *reinterpret_cast<uint32_t*>(&r);
  }
  static __device__ __forceinline__ void mma(float* c, const uint32_t* a, uint32_t b) {
    asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.bf16.bf16.f32 {%0,%1,%2,%3}, {%4,%5}, {%6}, {%0,%1,%2,%3};\n"
                 : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3]) : "r"(a[0]), "r"(a[1]), "r"(b));
  }
  static __device__ __forceinline__ float fma16(uint16_t x, uint16_t w, float acc) {
    asm("fma.rn.f32.bf16 %0, %1, %2, %0;" : "+f"(acc) : "h"(x), "h"(w));
    return acc;
  }
  static __device__ __forceinline__ uint16_t bits(float v) { return __bfloat16_as_ushort(__float2bfloat16_rn(v)); }
};

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void ldmatrix_x4_trans(uint32_t* r, const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];\n"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ void ldmatrix_x2(uint32_t* r, const void* p) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x2.shared.b16 {%0,%1}, [%2];\n" : "=r"(r[0]), "=r"(r[1]) : "r"(smem_u32(p)));
}
__device__ __forceinline__ float prelu(float v, float s) { return v > 0.f ? v : s * v; }
// the same with m = slope - 1 precomputed: v + m * min(v, 0) — two instructions instead of three
__device__ __forceinline__ float prelu_m1(float v, float m) { return fmaf(fminf(v, 0.f), m, v); }

// ---- cp.async ----------------------------------------------------------------------------------------
__device__ __forceinline__ void cp_async8(void* dst, const void* src, bool valid) {
  const int sz = valid ? 8 : 0;       // src-size 0: the 8 destination bytes are zero-filled
  asm volatile("cp.async.ca.shared.global [%0], [%1], 8, %2;\n" ::"r"(smem_u32(dst)), "l"(src), "r"(sz) : "memory");
}
__device__ __forceinline__ void cp_async16(void* dst, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(smem_u32(dst)), "l"(src) : "memory");
}
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_all;\n" ::: "memory"); }

// X[m][p] <- 16-bit(prelu(bias[m] + sum_k Ws[m][k] X[k][p])) for the pixels inside the image, 0 outside: D[M16 x NP] =
// Ws[M16 x K8] . X[K8 x NP] IN PLACE — each warp owns its pixel columns and holds all their B fragments in registers
// before it overwrites them.  coord(p) tells whether the pixel pair (p, p+1) is inside the image (rows are even-sized and
// p is even, so a pair is all in or all out); rowp(m, bias, slope) whether output row m exists.
template <typename T, typename Coord, typename RowP>
__device__ __forceinline__ void gemm_pixels_inplace(const uint16_t* Ws, int M16, int K8, uint16_t* X, int NP, int warp,
                                                    int nwarps, int lane, Coord coord, RowP rowp) {
  const int ntiles = NP >> 3, ksteps = K8 >> 3;
  const int g = lane >> 2, t = lane & 3;
  for (int nt0 = warp * 4; nt0 < ntiles; nt0 += nwarps * 4) {
    int ntl = nt0 + (lane >> 3);
    ntl = ntl < ntiles ? ntl : ntiles - 1;            // clamp: the result of a clamped tile is discarded
    uint32_t bf[kIlMaxK8][4];
#pragma unroll
    for (int ks = 0; ks < kIlMaxK8; ++ks)
      if (ks < ksteps) ldmatrix_x4_trans(bf[ks], X + (size_t)(ks * 8 + (lane & 7)) * NP + ntl * 8);
    __syncwarp();
    bool inb[4];                                        // is the pixel pair (p, p+1) of n tile j inside the image?
#pragma unroll
    for (int j = 0; j < 4; ++j) inb[j] = coord((nt0 + j) * 8 + 2 * t);
    for (int mt = 0; mt < (M16 >> 4); ++mt) {
      float b0, s0, b1, s1;                               // per-row epilogue parameters, loaded once per m tile
      const bool live0 = rowp(mt * 16 + g, b0, s0), live1 = rowp(mt * 16 + g + 8, b1, s1);
      float acc[4][4];                                    // the bias is the accumulator's initial value
#pragma unroll
      for (int b = 0; b < 4; ++b) { acc[b][0] = acc[b][1] = live0 ? b0 : 0.f; acc[b][2] = acc[b][3] = live1 ? b1 : 0.f; }
#pragma unroll
      for (int ks = 0; ks < kIlMaxK8; ++ks) {
        if (ks < ksteps) {
          uint32_t af[2];
          ldmatrix_x2(af, Ws + (size_t)(mt * 16 + (lane & 7) + 8 * ((lane >> 3) & 1)) * K8 + ks * 8);
#pragma unroll
          for (int j = 0; j < 4; ++j) Pack<T>::mma(acc[j], af, bf[ks][j]);
        }
      }
      const float m0 = s0 - 1.f, m1 = s1 - 1.f;           // prelu(v) = v + (slope - 1) * min(v, 0): two instructions
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (nt0 + j < ntiles) {
          const int p = (nt0 + j) * 8 + 2 * t;
          if (live0) {
            const uint32_t v = Pack<T>::from_f2(fmaf(fminf(acc[j][0], 0.f), m0, acc[j][0]), fmaf(fminf(acc[j][1], 0.f), m0, acc[j][1]));
            *reinterpret_cast<uint32_t*>(X + (size_t)(mt * 16 + g) * NP + p) = inb[j] ? v : 0u;
          }
          if (live1) {
            const uint32_t v = Pack<T>::from_f2(fmaf(fminf(acc[j][2], 0.f), m1, acc[j][2]), fmaf(fminf(acc[j][3], 0.f), m1, acc[j][3]));
            *reinterpret_cast<uint32_t*>(X + (size_t)(mt * 16 + g + 8) * NP + p) = inb[j] ? v : 0u;
          }
        }
      }
    }
  }
}

// Depthwise 3x3 + bias + PReLU of one plane set: region rows [R0, R1), 4-pixel column groups [G0, G1) of every
// channel.  in/out: [C][NP] flat region planes with row stride RW (all compile-time).  Output pixels outside the
// image are written as 0 (smem destination) or skipped (global destination).  A task = one channel, one 4-pixel
// column group, RUN rows.
template <int RW_, int NP_, int R0_, int R1_, int G0_, int G1_>
struct DwGeom {
  static constexpr int RW = RW_, NP = NP_, R0 = R0_, R1 = R1_, G0 = G0_, G1 = G1_;
};

template <typename T, bool kToGlobal, int RUN, typename GEO>
__device__ __forceinline__ void dw_task(int task, const uint16_t* in, uint16_t* out, const DwParams& P, int oy0, int ox0,
                                        int imgH, int imgW) {
  constexpr int G = GEO::G1 - GEO::G0, NR = (GEO::R1 - GEO::R0 + RUN - 1) / RUN, RW = GEO::RW, NP = GEO::NP, r1 = GEO::R1;
  const int gi = task % G, rest = task / G;
  const int run = rest % NR, c = rest / NR;
  const int x = 4 * (GEO::G0 + gi), ra = GEO::R0 + run * RUN;
  // fp16 planes: the 9 taps run as the mixed-precision FMA (Pack<T>::fma16: 16-bit x 16-bit + fp32 in one instruction), so
  // no operand is converted; the weights are rounded to fp16 for it (measured: no change of the fp16 error figures).
  // bf16 planes keep fp32 weights and converted operands — 8-bit-mantissa weights cost accuracy there.
  constexpr bool kMixed = std::is_same<T, __half>::value;
  float wf[9];
  uint16_t wh[9];
#pragma unroll
  for (int i = 0; i < 9; ++i) {
    wf[i] = __ldg(P.w + c * 9 + i);
    wh[i] = Pack<T>::bits(wf[i]);
  }
  const float bias = __ldg(P.b + c), slope_m1 = __ldg(P.s + c) - 1.f;
  const uint16_t* plane = in + c * NP + x;
  const int gx = ox0 + x;
  const bool col_in = gx >= 0 && gx < imgW;            // imgW % 4 == 0 and gx % 4 == 0: a group is all in or all out
  uint16_t rows[RUN + 2][6];                           // pixels x-1 .. x+4 of every input row
#pragma unroll
  for (int i = 0; i < RUN + 2; ++i) {
    const int r = ra - 1 + i;
    uint32_t lft = 0u, rgt = 0u;
    uint2 mid = make_uint2(0u, 0u);
    if (r <= r1) {                                      // row R1 exists (R1 <= RH - 1)
      mid = *reinterpret_cast<const uint2*>(plane + r * RW);            // x .. x+3 (8-byte aligned)
      lft = *reinterpret_cast<const uint32_t*>(plane + r * RW - 2);     // x-2, x-1
      rgt = *reinterpret_cast<const uint32_t*>(plane + r * RW + 4);     // x+4, x+5
    }
    rows[i][0] = (uint16_t)(lft >> 16); rows[i][1] = (uint16_t)mid.x; rows[i][2] = (uint16_t)(mid.x >> 16);
    rows[i][3] = (uint16_t)mid.y; rows[i][4] = (uint16_t)(mid.y >> 16); rows[i][5] = (uint16_t)rgt;
  }
#pragma unroll
  for (int i = 0; i < RUN; ++i) {
    const int r = ra + i;
    if (r < r1) {
      float o[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        float v = bias;
#pragma unroll
        for (int dy = 0; dy < 3; ++dy)
#pragma unroll
          for (int dx = 0; dx < 3; ++dx) {
            if constexpr (kMixed) v = Pack<T>::fma16(rows[i + dy][k + dx], wh[dy * 3 + dx], v);
            else v = fmaf(Pack<T>::to_f(rows[i + dy][k + dx]), wf[dy * 3 + dx], v);
          }
        o[k] = prelu_m1(v, slope_m1);
      }
      const int gy = oy0 + r;
      const bool in_img = col_in && gy >= 0 && gy < imgH;
      uint2 v;
      v.x = Pack<T>::from_f2(o[0], o[1]);
      v.y = Pack<T>::from_f2(o[2], o[3]);
      if (kToGlobal) {
        if (in_img) *reinterpret_cast<uint2*>(out + ((size_t)c * imgH + gy) * imgW + gx) = v;
      } else {
        if (!in_img) v = make_uint2(0u, 0u);
        *reinterpret_cast<uint2*>(out + c * NP + r * RW + x) = v;
      }
    }
  }
}

// hi and lo plane sets share one task index space so the 512 threads stay evenly loaded
template <typename T, bool kToGlobal, int RUN, typename GH, typename GL, int NT>
__device__ __forceinline__ void dw_pass(const uint16_t* inH, uint16_t* outH, const DwParams& PH, int Ch, int hy, int hx, int H,
                                        int W, const uint16_t* inL, uint16_t* outL, const DwParams& PL, int Cl, int ly, int lx,
                                        int tid) {
  constexpr int perH = ((GH::R1 - GH::R0 + RUN - 1) / RUN) * (GH::G1 - GH::G0);
  constexpr int perL = ((GL::R1 - GL::R0 + RUN - 1) / RUN) * (GL::G1 - GL::G0);
  const int nA = Ch * perH, nB = Cl * perL;
  for (int task = tid; task < nA + nB; task += NT) {
    if (task < nA) dw_task<T, kToGlobal, RUN, GH>(task, inH, outH, PH, hy, hx, H, W);
    else dw_task<T, kToGlobal, RUN, GL>(task - nA, inL, outL, PL, ly, lx, H >> 1, W >> 1);
  }
}

inline size_t il_smem_bytes(const IlArgs& A, int NPH, int NPL) {
  size_t halves = (size_t)A.rowsAh * NPH + (size_t)A.t2h * NPH + (size_t)A.rowsAl * NPL + (size_t)A.Clo * NPL +
                  (size_t)A.MH16 * A.K8 + (size_t)A.ML16 * A.K8;
  return halves * 2 + 128 /*base alignment*/ + 128 /*front guard*/ + 128 /*bufAh size round-up*/ + 128 /*tail guard*/;
}

// NT threads per CTA (512, one CTA per SM; 256 x 2 CTAs, 768 and 1024 were measured and are no faster, profiles/r01_f).
template <typename T, int TH, int TW, int NT = kIlThreads>
__global__ void __launch_bounds__(NT, NT <= 256 ? 2 : 1)
il_block_kernel(const __grid_constant__ IlArgs A) {
  using GEO = IlGeom<TH, TW>;
  extern __shared__ uint8_t smem_raw[];
  const int tid = threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = NT >> 5;
  const int n = blockIdx.z;
  const int tile_y = blockIdx.x / A.tiles_x, tile_x = blockIdx.x % A.tiles_x;
  const int hy0 = tile_y * TH, hx0 = tile_x * TW, ly0 = hy0 >> 1, lx0 = hx0 >> 1;
  const int H = A.H, W = A.W, Hl = A.H >> 1, Wl = A.W >> 1;
  constexpr int RHh = GEO::RHh, RWh = GEO::RWh, RHl = GEO::RHl, RWl = GEO::RWl, NPH = GEO::NPH, NPL = GEO::NPL;
  const int Chi = A.Chi, Cli = A.Cli, Cho = A.Cho, Clo = A.Clo;

  // carve (all sizes are multiples of 16 bytes; bufAh / bufAl are 128-byte aligned)
  uint8_t* base = smem_raw + ((128 - (smem_u32(smem_raw) & 127)) & 127);   // bytes 16..127 = zero guard in front of bufAh
  uint16_t* bufAh = reinterpret_cast<uint16_t*>(base + 128);        // [x_h | up(x_l)] -> T1H (in place)
  size_t off = (size_t)A.rowsAh * NPH * 2;
  off = (off + 127) & ~(size_t)127;
  uint16_t* bufAl = bufAh + off / 2;                                // [x_l | pool(x_h)] -> T1L (in place)
  uint16_t* bufBh = bufAl + (size_t)A.rowsAl * NPL;                 // T2H
  uint16_t* bufBl = bufBh + (size_t)A.t2h * NPH;                    // T2L
  uint16_t* wsH = bufBl + (size_t)Clo * NPL;
  uint16_t* wsL = wsH + A.MH16 * A.K8;
  uint16_t* tail = wsL + A.ML16 * A.K8;

  // ---- phase 0: guards, weights, zero rows -------------------------------------------------------------
  if (tid >= 32 && tid < 32 + 28) reinterpret_cast<uint32_t*>(base + 16)[tid - 32] = 0u;   // guard in front of bufAh
  if (tid >= 64 && tid < 64 + 8) reinterpret_cast<uint32_t*>(tail)[tid - 64] = 0u;          // tail guard
  __syncthreads();

  // weights (tiny, L2-resident) and the zero K-padding rows
  for (int i = tid; i < (A.MH16 * A.K8) >> 1; i += NT) reinterpret_cast<uint32_t*>(wsH)[i] = __ldg(A.wh + i);
  if (Clo > 0)
    for (int i = tid; i < (A.ML16 * A.K8) >> 1; i += NT) reinterpret_cast<uint32_t*>(wsL)[i] = __ldg(A.wl + i);
  {
    const int z0 = (Chi + Cli) * (NPH >> 1), z1 = A.rowsAh * (NPH >> 1);
    for (int i = z0 + tid; i < z1; i += NT) reinterpret_cast<uint32_t*>(bufAh)[i] = 0u;
    const int kl = Clo > 0 ? (Chi + Cli) : Cli;
    const int y0 = kl * (NPL >> 1), y1 = A.rowsAl * (NPL >> 1);
    for (int i = y0 + tid; i < y1; i += NT) reinterpret_cast<uint32_t*>(bufAl)[i] = 0u;
  }
  // cp.async loaders (8-byte chunks, zero fill outside the image).  A thread owns one 4-pixel position of the region and
  // walks the channels: validity, source offset and destination are computed once, a copy then costs a pointer bump.
  // The lo positions are taken from the top thread indices, so the warps the hi loop leaves idle start with them.
  if (!A.first) {
    const uint16_t* xh = reinterpret_cast<const uint16_t*>(A.xh) + (size_t)n * Chi * H * W;
    constexpr int quads_row = RWh >> 2, quads_plane = NPH >> 2;
    for (int pq = tid; pq < quads_plane; pq += NT) {
      const int ry = pq / quads_row, rx = (pq - ry * quads_row) * 4;
      const int gy = hy0 - 4 + ry, gx = hx0 - 4 + rx;
      const bool ok = ry < RHh && gy >= 0 && gy < H && gx >= 0 && gx < W;
      const uint16_t* src = ok ? xh + (size_t)gy * W + gx : xh;
      const size_t sstep = ok ? (size_t)H * W : 0;
      uint16_t* dst = bufAh + pq * 4;
      for (int c = 0; c < Chi; ++c, src += sstep, dst += NPH) cp_async8(dst, src, ok);
    }
  }
  if (!A.first) {
    const uint16_t* xl = reinterpret_cast<const uint16_t*>(A.xl) + (size_t)n * Cli * Hl * Wl;
    constexpr int quads_row = RWl >> 2, quads_plane = NPL >> 2;
    for (int pq = NT - 1 - tid; pq < quads_plane; pq += NT) {
      const int ry = pq / quads_row, rx = (pq - ry * quads_row) * 4;
      const int gy = ly0 - 2 + ry, gx = lx0 - 4 + rx;
      const bool ok = ry < RHl && gy >= 0 && gy < Hl && gx >= 0 && gx < Wl;
      const uint16_t* src = ok ? xl + (size_t)gy * Wl + gx : xl;
      const size_t sstep = ok ? (size_t)Hl * Wl : 0;
      uint16_t* dst = bufAl + pq * 4;
      for (int c = 0; c < Cli; ++c, src += sstep, dst += NPL) cp_async8(dst, src, ok);
    }
  }
  cp_async_wait_all();
  __syncthreads();

  if (A.first) {
    // ---- stem form: fp32 image tile -> smem scratch (the T2 buffers, free until dw1), then the im2col planes ----
    // scratch tile: image rows [hy0-6, hy0+TH+6), cols [hx0-12, hx0+TW+12), zero outside the image; covers the hi
    // region +-1 pixel and the pooled lo region +-1 lo pixel
    constexpr int IH = TH + 12, IW = TW + 24;
    const int Ci = Chi / 9;
    float* img = reinterpret_cast<float*>(bufBh);
    const float* x = reinterpret_cast<const float*>(A.xh) + (size_t)n * Ci * H * W;
    for (int i = tid; i < Ci * IH * (IW / 4); i += NT) {
      const int c = i / (IH * (IW / 4)), r = i - c * (IH * (IW / 4));
      const int iy = r / (IW / 4), ix = (r - iy * (IW / 4)) * 4;
      const int gy = hy0 - 6 + iy, gx = hx0 - 12 + ix;          // gx % 4 == 0 and W % 4 == 0: a quad is all in or all out
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (gy >= 0 && gy < H && gx >= 0 && gx < W) v = __ldg(reinterpret_cast<const float4*>(x + ((size_t)c * H + gy) * W + gx));
      *reinterpret_cast<float4*>(img + (c * IH + iy) * IW + ix) = v;
    }
    __syncthreads();
    // hi planes: row k = (ci, ky, kx) holds the image shifted by (ky-1, kx-1); region (ry, rx) = image (hy0-4+ry, hx0-4+rx).
    // A thread owns pixel-pair positions and walks the 9 * Ci planes with compile-time tap offsets.
    const int Cin = Chi / 9;
    for (int pp = tid; pp < NPH / 2; pp += NT) {
      const int ry = (2 * pp) / RWh, rx = 2 * pp - ry * RWh;
      const float* base = img + (ry + 1) * IW + rx + 7;
      uint32_t* dst = reinterpret_cast<uint32_t*>(bufAh) + pp;
      for (int ci = 0; ci < Cin; ++ci, base += IH * IW) {
#pragma unroll
        for (int ky = 0; ky < 3; ++ky)
#pragma unroll
          for (int kx = 0; kx < 3; ++kx, dst += NPH / 2) {
            const float* src = base + ky * IW + kx;
            *dst = Pack<T>::from_f2(src[0], src[1]);
          }
      }
    }
    // lo planes: 2x2 max-pool of the image, shifted by (ky-1, kx-1) lo pixels, zero outside the lo image (conv padding).
    // A thread owns lo pixels: the 3 x 3 pooled neighbourhood is computed once per input channel and fans out to 9 planes.
    if (Clo > 0) {
      constexpr int rl_ = TH / 2 + 4;
      for (int p = NT - 1 - tid; p < NPL; p += NT) {
        const int ry = p / RWl, rx = p - ry * RWl;
        const float* base = img + (2 * ry) * IW + 2 * rx + 2;
        uint16_t* dst = bufAl + p;
        for (int ci = 0; ci < Cin; ++ci, base += IH * IW) {
#pragma unroll
          for (int ky = 0; ky < 3; ++ky)
#pragma unroll
            for (int kx = 0; kx < 3; ++kx, dst += NPL) {
              const int gy = ly0 - 3 + ry + ky, gx = lx0 - 5 + rx + kx;
              float v = 0.f;
              if (ry < rl_ && gy >= 0 && gy < Hl && gx >= 0 && gx < Wl) {
                const float* src = base + 2 * ky * IW + 2 * kx;
                v = fmaxf(fmaxf(src[0], src[1]), fmaxf(src[IW], src[IW + 1]));
              }
              *dst = (uint16_t)(Pack<T>::from_f2(v, 0.f) & 0xffffu);
            }
        }
      }
    }
  } else {
  // ---- phase 1: resample both ways --------------------------------------------------------------------
  // (a) max_pool2d 2x2 of x_h -> AL rows [Cli, Cli+Chi): two lo pixels per step from 2 hi rows x 4 hi pixels.  A thread
  //     owns one lo pixel-pair position and a residue class of the channels: index arithmetic once per thread.
  if (Clo > 0) {
    constexpr int pairs_row = RWl >> 1, pairs_plane = NPL >> 1;
    constexpr int umax = RWh >> 2;
    constexpr int groups = NT / pairs_plane > 0 ? NT / pairs_plane : 1;        // channel residue classes
    const int pp = tid % pairs_plane, cg = tid / pairs_plane;
    if (cg < groups) {
      const int ry = pp / pairs_row, u = pp - ry * pairs_row;
      const bool ok = ry < RHl && 2 * ry + 1 < RHh && u >= 1 && u <= umax;
      const uint16_t* r0 = bufAh + (size_t)cg * NPH + (ok ? (2 * ry) * RWh + 4 * u - 4 : 0);
      uint32_t* dst = reinterpret_cast<uint32_t*>(bufAl + (size_t)(Cli + cg) * NPL) + pp;
      for (int c = cg; c < Chi; c += groups, r0 += (size_t)groups * NPH, dst += (size_t)groups * (NPL >> 1)) {
        uint32_t v = 0u;
        if (ok) {
          const uint2 a = *reinterpret_cast<const uint2*>(r0), b = *reinterpret_cast<const uint2*>(r0 + RWh);
          const uint32_t m0 = Pack<T>::max2(a.x, b.x), m1 = Pack<T>::max2(a.y, b.y);
          // horizontal maximum of each 16-bit pair: max2 against the pair with its halves swapped
          v = __byte_perm(Pack<T>::max2(m0, __byte_perm(m0, 0u, 0x1032)), Pack<T>::max2(m1, __byte_perm(m1, 0u, 0x1032)), 0x5410);
        }
        *dst = v;
      }
    }
    static_assert(pairs_plane <= NT, "one pass over the lo pixel pairs");
  }
  // (b) bilinear x2 of x_l -> AH rows [Chi, Chi+Cli): F.interpolate(scale_factor=2, align_corners=False) has the
  //     fixed taps dst 2j: (1/4, 3/4) of src (j-1, j); dst 2j+1: (3/4, 1/4) of src (j, j+1), indices clamped to the
  //     image.  A task = 4 hi rows x 4 hi columns of one channel (lo rows a-1 .. a+2, lo columns j0-1 .. j0+2): the 16
  //     horizontal blends are shared by the 4 output rows; the 16-bit values go straight into the mixed-precision FMA
  //     (weights 0.25 / 0.75 are exact in both 16-bit types, so the result equals the fp32 expression).
  {
    constexpr int quads_row = RWh >> 2;
    constexpr int row_quads = RHh >> 2;               // hi rows 4b .. 4b+3; RHh = 4k + 1: the odd last row stays zero-filled
    static_assert((RHh & 3) == 1, "hi region rows = 4k + 1");
    constexpr int per_plane = row_quads * quads_row;
    const uint16_t w25 = Pack<T>::bits(0.25f), w75 = Pack<T>::bits(0.75f);
    // a thread owns one (row quad, column quad) position and a residue class of the channels: the clamped source
    // offsets are computed once
    constexpr int groups = NT / per_plane > 0 ? NT / per_plane : 1;
    static_assert(per_plane <= NT, "one pass over the bilinear positions");
    const int pos = tid % per_plane, cg = tid / per_plane;
    if (cg < groups) {
      const int b4 = pos / quads_row, q = pos - b4 * quads_row;
      // hi rows 4b..4b+3 <-> image rows hy0-4+4b ..; lo image rows li = ly0-2+2b and li+1
      const int li = ly0 - 2 + 2 * b4;
      auto clampy = [&](int y) { y = y < 0 ? 0 : (y > Hl - 1 ? Hl - 1 : y); int r = y - (ly0 - 2); return r < 0 ? 0 : (r > RHl - 1 ? RHl - 1 : r); };
      // hi cols 4q..4q+3 <-> image cols gx0 = hx0-4+4q = 2*j0; lo image cols j0-1 .. j0+2
      const int j0 = ((hx0 - 4) >> 1) + 2 * q;
      auto clampx = [&](int xx) { xx = xx < 0 ? 0 : (xx > Wl - 1 ? Wl - 1 : xx); int r = xx - (lx0 - 4); return r < 0 ? 0 : (r > RWl - 1 ? RWl - 1 : r); };
      const int c0 = clampx(j0 - 1), c1 = clampx(j0), c2 = clampx(j0 + 1), c3 = clampx(j0 + 2);
      int ro[4];
#pragma unroll
      for (int k = 0; k < 4; ++k) ro[k] = clampy(li - 1 + k) * RWl;
      const uint16_t* src = bufAl + (size_t)cg * NPL;
      uint16_t* dst = bufAh + (size_t)(Chi + cg) * NPH + (4 * b4) * RWh + 4 * q;
      for (int c = cg; c < Cli; c += groups, src += (size_t)groups * NPL, dst += (size_t)groups * NPH) {
        float h[4][4];                                // horizontally blended lo rows li-1 .. li+2 at the 4 hi columns
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const uint16_t* r = src + ro[k];
          const uint16_t v0 = r[c0], v1 = r[c1], v2 = r[c2], v3 = r[c3];
          h[k][0] = Pack<T>::fma16(v1, w75, Pack<T>::fma16(v0, w25, 0.f));   // col 2*j0    : (1/4, 3/4) of (j0-1, j0)
          h[k][1] = Pack<T>::fma16(v1, w75, Pack<T>::fma16(v2, w25, 0.f));   // col 2*j0 + 1: (3/4, 1/4) of (j0, j0+1)
          h[k][2] = Pack<T>::fma16(v2, w75, Pack<T>::fma16(v1, w25, 0.f));   // col 2*j0 + 2
          h[k][3] = Pack<T>::fma16(v2, w75, Pack<T>::fma16(v3, w25, 0.f));   // col 2*j0 + 3
        }
        // hi row 4b: lo rows (li-1, li) w (.25, .75); 4b+1: (li, li+1) w (.75, .25); 4b+2: (li, li+1) w (.25, .75); 4b+3: (li+1, li+2) w (.75, .25)
#pragma unroll
        for (int rr = 0; rr < 4; ++rr) {
          const int km = rr < 2 ? 1 : 2, ko = rr == 0 ? 0 : (rr == 3 ? 3 : (rr == 1 ? 2 : 1));   // main (3/4) and other (1/4) row
          uint2 o;
          o.x = Pack<T>::from_f2(0.75f * h[km][0] + 0.25f * h[ko][0], 0.75f * h[km][1] + 0.25f * h[ko][1]);
          o.y = Pack<T>::from_f2(0.75f * h[km][2] + 0.25f * h[ko][2], 0.75f * h[km][3] + 0.25f * h[ko][3]);
          *reinterpret_cast<uint2*>(dst + rr * RWh) = o;
        }
      }
    }
    // rows of the hi planes not covered above (odd last row, padded tail): zero
    constexpr int covered = (RHh >> 2) * 4 * RWh;
    constexpr int tailh = (NPH - covered) >> 1;
    for (int i = tid; i < Cli * tailh; i += NT) {
      const int c = i / tailh, k = i - c * tailh;
      reinterpret_cast<uint32_t*>(bufAh + (size_t)(Chi + c) * NPH + covered)[k] = 0u;
    }
  }
  }
  __syncthreads();

  // ---- phase 2: the two 1x1 convolutions on tensor cores, in place ------------------------------------
  if (Clo > 0) {
    const float* bl = A.bias_l;
    const float* sl = A.slope_l;
    auto coord = [&](int p) {                           // lo region pixel p (even): is the pair inside the lo image?
      const int ry = p / RWl;
      const int cy = ly0 - 2 + ry, cx = lx0 - 4 + (p - ry * RWl);
      return ry < RHl && cy >= 0 && cy < Hl && cx >= 0 && cx < Wl;   // Wl and cx are even: cx + 1 is inside too
    };
    auto rowp = [&](int m, float& b, float& s) {
      if (m >= Clo) return false;
      b = __ldg(bl + m); s = __ldg(sl + m);
      return true;
    };
    gemm_pixels_inplace<T>(wsL, A.ML16, A.K8, bufAl, NPL, warp, nwarps, lane, coord, rowp);
  }
  {
    const float* bh = A.bias_h;
    const float* sh = A.slope_h;
    auto coord = [&](int p) {
      const int ry = p / RWh;
      const int cy = hy0 - 4 + ry, cx = hx0 - 4 + (p - ry * RWh);
      return ry < RHh && cy >= 0 && cy < H && cx >= 0 && cx < W;     // W even, cx even: cx + 1 is inside too
    };
    auto rowp = [&](int m, float& b, float& s) {
      if (m >= Cho) return false;
      b = __ldg(bh + m); s = __ldg(sh + m);
      return true;
    };
    gemm_pixels_inplace<T>(wsH, A.MH16, A.K8, bufAh, NPH, warp, nwarps, lane, coord, rowp);
  }
  __syncthreads();

  // ---- phase 3/4: the two depthwise layers ---------------------------------------------------------------
  constexpr int rh = TH + 8, rl = TH / 2 + 4;         // region rows that matter (without the padding row)
  using GH1 = DwGeom<RWh, NPH, 3, rh - 3, 0, RWh / 4>;
  using GL1 = DwGeom<RWl, NPL, 1, rl - 1, 0, RWl / 4>;
  using GH2 = DwGeom<RWh, NPH, 4, rh - 4, 1, RWh / 4 - 1>;
  using GL2 = DwGeom<RWl, NPL, 2, rl - 2, 1, RWl / 4 - 1>;
  uint16_t* outH = reinterpret_cast<uint16_t*>(A.yh) + (size_t)n * Cho * H * W;
  uint16_t* outL = Clo > 0 ? reinterpret_cast<uint16_t*>(A.yl) + (size_t)n * Clo * Hl * Wl : nullptr;
  if (A.t2h >= Cho) {
    // whole layers resident: dw1 (T1 -> T2, smem) then dw2 (T2 -> global)
    dw_pass<T, false, 6, GH1, GL1, NT>(bufAh, bufBh, A.dw1h, Cho, hy0 - 4, hx0 - 4, H, W, bufAl, bufBl, A.dw1l, Clo, ly0 - 2, lx0 - 4, tid);
    __syncthreads();
    dw_pass<T, true, 4, GH2, GL2, NT>(bufBh, outH, A.dw2h, Cho, hy0 - 4, hx0 - 4, H, W, bufBl, outL, A.dw2l, Clo, ly0 - 2, lx0 - 4, tid);
  } else {
    // wide blocks: the hi branch goes through the two layers 8 channels at a time (T2 buffer of 8 planes), the lo
    // branch rides along with the first chunk
    for (int c0 = 0; c0 < Cho; c0 += A.t2h) {
      const int cc = (Cho - c0) < A.t2h ? (Cho - c0) : A.t2h;
      const DwParams p1{A.dw1h.w + c0 * 9, A.dw1h.b + c0, A.dw1h.s + c0}, p2{A.dw2h.w + c0 * 9, A.dw2h.b + c0, A.dw2h.s + c0};
      if (c0 > 0) __syncthreads();                      // the previous chunk's dw2 finished reading the T2 buffer
      dw_pass<T, false, 3, GH1, GL1, NT>(bufAh + (size_t)c0 * NPH, bufBh, p1, cc, hy0 - 4, hx0 - 4, H, W, bufAl, bufBl, A.dw1l,
                                     c0 == 0 ? Clo : 0, ly0 - 2, lx0 - 4, tid);
      __syncthreads();
      dw_pass<T, true, 2, GH2, GL2, NT>(bufBh, outH + (size_t)c0 * H * W, p2, cc, hy0 - 4, hx0 - 4, H, W, bufBl, outL, A.dw2l,
                                    c0 == 0 ? Clo : 0, ly0 - 2, lx0 - 4, tid);
    }
  }
}

}  // namespace csnet
