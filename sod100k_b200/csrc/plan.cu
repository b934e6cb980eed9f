// plan.cu — C ABI (include/csnet_b200.h) and the program executor of libcsnet_b200.so.
//
// A plan holds: the validated program, the device copy of the parameter blob, and one activation arena.
// csnet_plan_run() walks the op list and launches one fused kernel per op on the caller's stream.
#include <cuda.h>
#include <cuda_runtime.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <new>
#include <string>
#include <vector>

#include "../../include/csnet_b200.h"
#include "generic_ops.cuh"
#include "il_block.cuh"
#include "il_stream.cuh"
#include "mix_stream.cuh"
#include "ms_direct.cuh"
#include "mix_tc.cuh"
#include "dw_fast.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) {
  g_err = msg;
  return code;
}

#define CU_CHECK(expr)                                                                         \
  do {                                                                                         \
    cudaError_t e_ = (expr);                                                                   \
    if (e_ != cudaSuccess)                                                                     \
      return fail(CSNET_E_CUDA, std::string(#expr) + ": " + cudaGetErrorString(e_));           \
  } while (0)

size_t dtype_size(int dt) { return dt == CSNET_F32 ? 4 : 2; }

// The entry points select the plan's device for their CUDA calls and put the caller's current device back on return:
// torch (the host side's plumbing) keeps its own notion of the current device.
struct DeviceGuard {
  int prev = -1;
  explicit DeviceGuard(int dev) {
    if (cudaGetDevice(&prev) != cudaSuccess) prev = -1;
    if (prev != dev) cudaSetDevice(dev);
    else prev = -1;
  }
  ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// ------------------------------------------------------------------------------------------------
// kernels
// ------------------------------------------------------------------------------------------------
constexpr int kThreads = 256;

__global__ void __launch_bounds__(kThreads, 2) mix_generic_kernel(const __grid_constant__ csnet::MixArgs A) {
  __shared__ float ws[csnet::kMixStageFloats];
  const int co_base = blockIdx.y * csnet::kMixCT, n = blockIdx.z;
  const int pix = blockIdx.x * kThreads + threadIdx.x;
  const bool live = pix < A.H * A.W;
  const int oy = live ? pix / A.W : 0, ox = live ? pix % A.W : 0;
  float acc[csnet::kMixCT];
#pragma unroll
  for (int t = 0; t < csnet::kMixCT; ++t) acc[t] = 0.f;
  for (int p = 0; p < A.n_paths; ++p) {
    const csnet::MixPath& P = A.p[p];
    if (P.ksize == 0 || !csnet::mix_path_live(P, co_base)) continue;      // block-uniform
    const int chunk = csnet::mix_chunk_channels(P.ksize);
    for (int ci0 = 0; ci0 < P.cin; ci0 += chunk) {
      const int ci1 = ci0 + chunk < P.cin ? ci0 + chunk : P.cin;
      __syncthreads();
      csnet::mix_stage_chunk(P, co_base, ci0, ci1, ws, threadIdx.x, kThreads);
      __syncthreads();
      if (live) csnet::mix_acc_chunk(P, ws, ci0, ci1, n, oy, ox, acc);
    }
  }
  if (live) csnet::mix_finish(A, n, oy, ox, co_base, acc);
}

__global__ void __launch_bounds__(kThreads) dw_generic_kernel(const __grid_constant__ csnet::DwArgs A) {
  const int item = blockIdx.x * kThreads + threadIdx.x;
  const int strips = (A.H + csnet::kDwRows - 1) / csnet::kDwRows;
  if (item >= strips * A.W) return;
  csnet::dw_thread(A, blockIdx.z, blockIdx.y, (item / A.W) * csnet::kDwRows, item % A.W);
}

// GroupNorm statistics: one CTA per (group, image)
__global__ void __launch_bounds__(kThreads) gn_stats_kernel(const __grid_constant__ csnet::GnArgs A) {
  const int g = blockIdx.x, n = blockIdx.y, cpg = A.C / A.groups;
  const int64_t base = ((int64_t)n * A.C + (int64_t)g * cpg) * A.HW, cnt = (int64_t)cpg * A.HW;
  __shared__ float sh[2][kThreads / 32];
  __shared__ float mu_s;
  float s = 0.f;
  for (int64_t i = threadIdx.x; i < cnt; i += kThreads) s += csnet::ld_elem(A.src, A.src_dtype, base + i);
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) sh[0][threadIdx.x >> 5] = s;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < kThreads / 32; ++i) t += sh[0][i];
    mu_s = t / (float)cnt;
  }
  __syncthreads();
  const float mu = mu_s;
  float q = 0.f;
  for (int64_t i = threadIdx.x; i < cnt; i += kThreads) {
    const float d = csnet::ld_elem(A.src, A.src_dtype, base + i) - mu;
    q += d * d;
  }
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  if ((threadIdx.x & 31) == 0) sh[1][threadIdx.x >> 5] = q;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int i = 0; i < kThreads / 32; ++i) t += sh[1][i];
    A.stats[((int64_t)n * A.groups + g) * 2] = mu;
    A.stats[((int64_t)n * A.groups + g) * 2 + 1] = rsqrtf(t / (float)cnt + 1e-5f);
  }
}

__global__ void __launch_bounds__(kThreads) gn_apply_kernel(const __grid_constant__ csnet::GnArgs A) {
  const int c = blockIdx.y, n = blockIdx.z, g = c / (A.C / A.groups);
  const float mu = A.stats[((int64_t)n * A.groups + g) * 2], r = A.stats[((int64_t)n * A.groups + g) * 2 + 1];
  const float ga = A.gamma[c] * r, be = A.beta[c] - mu * ga;
  const bool has_slope = A.slope != nullptr;
  const float sl = has_slope ? A.slope[c] : 1.f;
  const int64_t base = ((int64_t)n * A.C + c) * A.HW;
  for (int i = blockIdx.x * kThreads + threadIdx.x; i < A.HW; i += gridDim.x * kThreads) {
    float v = csnet::ld_elem(A.src, A.src_dtype, base + i) * ga + be;
    if (has_slope) v = v > 0.f ? v : sl * v;
    csnet::st_elem(A.dst, A.dst_dtype, base + i, v);
  }
}

// Device-side pre / post-processing of CSNet/test.py:68-69,86-96 (SURVEY §8 f3): uint8 HWC image -> (x / 255 - mean) / std as the
// fp32 NCHW network input (the reference computes it in float64 on the host and rounds to fp32: same here), and
// sigmoid(logit) * 255 -> uint8 (astype truncation) of the saliency map.
struct PreArgs { double mean[3], std[3]; };
__global__ void __launch_bounds__(kThreads) pre_u8_kernel(const uint8_t* __restrict__ x, float* __restrict__ y, int64_t npix, int64_t hw, const __grid_constant__ PreArgs A) {
  const int64_t i = (int64_t)blockIdx.x * kThreads + threadIdx.x;          // pixel over (n, h, w)
  if (i >= npix) return;
  const int64_t n = i / hw, p = i - n * hw;
#pragma unroll
  for (int c = 0; c < 3; ++c) y[(n * 3 + c) * hw + p] = (float)(((double)x[i * 3 + c] / 255.0 - A.mean[c]) / A.std[c]);
}
__global__ void __launch_bounds__(kThreads) post_u8_kernel(const float* __restrict__ z, uint8_t* __restrict__ y, int64_t n) {
  const int64_t i = ((int64_t)blockIdx.x * kThreads + threadIdx.x) * 4;
  if (i >= n) return;
  uchar4 o;
  const float4 v = *reinterpret_cast<const float4*>(z + i);                // n % 4 == 0 (W % 16 == 0)
  o.x = (unsigned char)((1.f / (1.f + expf(-v.x))) * 255.f); o.y = (unsigned char)((1.f / (1.f + expf(-v.y))) * 255.f);
  o.z = (unsigned char)((1.f / (1.f + expf(-v.z))) * 255.f); o.w = (unsigned char)((1.f / (1.f + expf(-v.w))) * 255.f);
  *reinterpret_cast<uchar4*>(y + i) = o;
}

}  // namespace

// ------------------------------------------------------------------------------------------------
// plan
// ------------------------------------------------------------------------------------------------
struct TcChoice {
  int mt = 0;            // 0: generic kernel; else number of m16 tiles of the tensor-core kernel
  int dtype = 0;         // CSNET_F16 / CSNET_BF16 operand type
  int xs_halves = 0;
  int rows = 1;          // output rows per warp of mix_tc (tile height 8 * rows)
  int kc = 8;            // input channels per staged chunk
  int kk = 1;            // largest tap count among the conv paths
};

size_t tc_smem_bytes(const TcChoice& c) {
  return ((size_t)c.kc * c.xs_halves + (size_t)c.kk * c.mt * 16 * (c.kc + 8)) * 2;
}

// The kernel that runs an op, fixed once per op at plan creation (route_op).  It depends on the plan's max_batch, never on a
// run's N, so every sub-batch of a plan runs the same kernels, bit for bit.
enum class Route { MSD, MIX_STREAM, MIX_TC, POOL2, UPSAMPLE, RESAMPLE, MIX_GENERIC, GN, IL_STREAM, IL_BLOCK, DW_FAST, DW_GENERIC };
constexpr int kRoutes = (int)Route::DW_GENERIC + 1;

// csnet_plan_op_kernel's name of each route's kernel (family); bench.py groups per-op times by these strings
const char* const kRouteKernel[] = {
    "msd_kernel (ms_direct.cuh, FP32 pipe)", "mix_stream_kernel (TMA + tcgen05)", "mix_tc_kernel (mma.sync)",
    "pool2 / upsample / resample kernels", "pool2 / upsample / resample kernels", "pool2 / upsample / resample kernels",
    "mix_generic_kernel", "gn kernels", "il_stream_kernel (TMA + tcgen05 + TMEM)", "il_block_kernel (mma.sync, tiled)",
    "dw kernels", "dw kernels"};
static_assert(sizeof kRouteKernel / sizeof *kRouteKernel == kRoutes, "one name per route");

// An op's route and what the route needs that does not depend on a run: the launch's dynamic shared memory and the kernel
// arguments fixed at plan creation (geometry, parameter pointers; the epilogue tables are filled by csnet_plan_set_blob).
struct OpRoute {
  Route route = Route::MIX_GENERIC;
  size_t smem = 0;
  TcChoice tc;                        // MIX_TC
  std::vector<uint16_t*> w16;         // MIX_TC, per path: packed 16-bit weights (device; null for resample paths)
  csnet::IlArgs il{};                 // IL_BLOCK
  csnet::IlsArgs ils{};               // IL_STREAM
  csnet::MsArgs ms{};                 // MIX_STREAM
};

struct csnet_plan {
  int device = 0;
  int max_batch = 0;
  std::vector<csnet_tensor_desc> tensors;
  std::vector<csnet_op_desc> ops;
  int64_t blob_floats = 0;
  float* blob = nullptr;
  char* arena = nullptr;
  int64_t arena_per_image = 0;   // bytes
  int n_ext = 0;
  std::vector<OpRoute> routes;                    // per op
  // small-batch replay: the whole op list captured once per batch size into a CUDA graph over plan-owned input / output staging
  // (CSNet/test.py calls the model one image at a time: ~80 launches per forward are launch-bound there)
  struct GraphSlot { cudaGraphExec_t exec = nullptr; void* in = nullptr; void* out = nullptr; size_t in_bytes = 0, out_bytes = 0; };
  std::vector<GraphSlot> graphs;                  // index = batch size
  cudaStream_t cap_stream = nullptr;
  int graph_max_n = 8;                            // CSNET_GRAPH_MAX_N (0 disables)
  int num_sms = 148;
  // host-buffer pipeline (csnet_plan_run_host): copy streams, ping-pong staging, ordering events
  cudaStream_t s_h2d = nullptr, s_d2h = nullptr;
  void* h_in8[2] = {nullptr, nullptr};             // uint8 staging of csnet_plan_run_host_u8
  void* h_out8[2] = {nullptr, nullptr};
  size_t h_in8_bytes = 0;
  void* h_in[2] = {nullptr, nullptr};
  void* h_out[2] = {nullptr, nullptr};
  size_t h_in_bytes = 0, h_out_bytes = 0;
  cudaEvent_t ev_h2d[2] = {nullptr, nullptr}, ev_comp[2] = {nullptr, nullptr}, ev_d2h[2] = {nullptr, nullptr};
  float* gn_stats = nullptr;      // [max_batch][max groups][2] scratch of the GroupNorm ops
  int gn_groups_max = 0;

  void* tensor_ptr(int t, int N, const void* const* ext) const {
    const csnet_tensor_desc& d = tensors[t];
    if (d.external >= 0) return ext ? const_cast<void*>(ext[d.external]) : nullptr;
    return arena + (int64_t)N * d.arena_offset;
  }
};

namespace {

// Channels of a MIX-kind op's result: the destination's, or ext_off[2] when a projection consumes it in the epilogue.
static inline int mix_channels(const csnet_plan& P, const csnet_op_desc& op) {
  return op.kind == CSNET_OP_MIXPROJ ? (int)op.ext_off[2] : P.tensors[op.dst].C;
}

int validate(const csnet_plan& P) {
  const int nt = (int)P.tensors.size();
  char buf[256];
  for (int t = 0; t < nt; ++t) {
    const csnet_tensor_desc& d = P.tensors[t];
    if (d.C <= 0 || d.H <= 0 || d.W <= 0 || d.dtype < 0 || d.dtype > 2) {
      snprintf(buf, sizeof buf, "tensor %d: bad dims/dtype", t);
      return fail(CSNET_E_INVALID, buf);
    }
    if (d.external < 0 && (d.arena_offset < 0 || d.arena_offset % 256 != 0)) {
      snprintf(buf, sizeof buf, "tensor %d: arena offset must be a non-negative multiple of 256", t);
      return fail(CSNET_E_INVALID, buf);
    }
  }
  for (size_t i = 0; i < P.ops.size(); ++i) {
    const csnet_op_desc& op = P.ops[i];
    auto bad = [&](const char* why) {
      snprintf(buf, sizeof buf, "op %zu: %s", i, why);
      return fail(CSNET_E_INVALID, buf);
    };
    if (op.kind != CSNET_OP_MIX && op.kind != CSNET_OP_DW && op.kind != CSNET_OP_ILBLOCK && op.kind != CSNET_OP_GN &&
        op.kind != CSNET_OP_MIXPROJ)
      return bad("unknown kind");
    if (op.dst < 0 || op.dst >= nt) return bad("dst out of range");
    if (op.kind == CSNET_OP_GN) {
      if (op.n_paths != 1) return bad("GN takes one input");
      const int a = op.paths[0].src, groups = op.paths[0].up;
      if (a < 0 || a >= nt || a == op.dst) return bad("GN input");
      const csnet_tensor_desc &X = P.tensors[a], &Y = P.tensors[op.dst];
      if (X.C != Y.C || X.H != Y.H || X.W != Y.W) return bad("GN shape");
      if (groups < 1 || X.C % groups) return bad("GN groups must divide the channels");
      if (op.ext_off[0] < 0 || op.ext_off[0] + X.C > P.blob_floats || op.ext_off[1] < 0 || op.ext_off[1] + X.C > P.blob_floats)
        return bad("GN gamma/beta outside blob");
      if (op.slope_off >= 0 && op.slope_off + X.C > P.blob_floats) return bad("slope outside blob");
      continue;
    }
    if (op.kind == CSNET_OP_ILBLOCK) {
      if (op.n_paths != 2) return bad("ILBLOCK takes two inputs");
      if (op.dst2 >= nt) return bad("dst2 out of range");
      const csnet_tensor_desc& Yh = P.tensors[op.dst];
      const int a = op.paths[0].src, b = op.paths[1].src;
      if (a < 0 || a >= nt || b < 0 || b >= nt) return bad("ILBLOCK input out of range");
      const csnet_tensor_desc &Xh = P.tensors[a], &Xl = P.tensors[b];
      if (a == op.dst || b == op.dst || a == op.dst2 || b == op.dst2) return bad("in-place op");
      const bool stem = op.paths[0].ksize == 3;          // stem form: both branches are 3x3 convs of one fp32 image
      if (Yh.dtype == CSNET_F32) return bad("ILBLOCK needs a 16-bit destination");
      if (Yh.W % 8 || Yh.H % 2) return bad("ILBLOCK needs W % 8 == 0 and H % 2 == 0");
      if (stem) {
        if (a != b || Xh.dtype != CSNET_F32 || Xh.C * 9 > 32) return bad("ILBLOCK stem form takes one fp32 image of at most 3 channels");
        if (Xh.H != Yh.H || Xh.W != Yh.W) return bad("ILBLOCK input/output resolutions");
        if (op.paths[1].ksize != 3 || op.paths[1].pool != 2) return bad("ILBLOCK stem form: lo path is a 3x3 conv of the 2x2 max-pool");
      } else {
        if (Xh.dtype != Yh.dtype || Xl.dtype != Yh.dtype) return bad("ILBLOCK needs one 16-bit dtype");
        if (Xh.H != Yh.H || Xh.W != Yh.W || Xl.H * 2 != Xh.H || Xl.W * 2 != Xh.W) return bad("ILBLOCK input/output resolutions");
      }
      if (op.paths[0].cin != Xh.C || op.paths[1].cin != Xl.C) return bad("ILBLOCK consumes whole input tensors");
      int Clo = 0;
      if (op.dst2 >= 0) {
        const csnet_tensor_desc& Yl = P.tensors[op.dst2];
        if (Yl.dtype != Yh.dtype || Yl.H * 2 != Yh.H || Yl.W * 2 != Yh.W) return bad("ILBLOCK lo output shape");
        Clo = Yl.C;
      }
      const int nreq = Clo > 0 ? 18 : 15;
      for (int e = 0; e < nreq; ++e) {
        if (Clo == 0 && (e == 4 || e == 5 || (e >= 9 && e <= 11))) continue;
        if (op.ext_off[e] < 0 || op.ext_off[e] >= P.blob_floats) return bad("ILBLOCK parameter offset outside blob");
      }
      continue;
    }
    if (op.n_paths < 1 || op.n_paths > CSNET_MAX_PATHS) return bad("n_paths out of range");
    const csnet_tensor_desc& D = P.tensors[op.dst];
    const int Cm = mix_channels(P, op);               // channels of the MIX result (== D.C unless projected away)
    if (op.kind == CSNET_OP_MIXPROJ) {
      if (D.C != 1 || Cm < 1 || Cm > 80) return bad("MIXPROJ projects 1..80 channels onto one");
      if (op.ext_off[0] < 0 || op.ext_off[0] + Cm > P.blob_floats) return bad("projection weights outside blob");
      if (op.ext_off[1] >= P.blob_floats) return bad("projection bias outside blob");
    }
    if (op.bias_off >= 0 && op.bias_off + Cm > P.blob_floats) return bad("bias outside blob");
    if (op.slope_off >= 0 && op.slope_off + Cm > P.blob_floats) return bad("slope outside blob");
    if (op.kind == CSNET_OP_DW && op.n_paths != 1) return bad("DW takes one path");
    for (int p = 0; p < op.n_paths; ++p) {
      const csnet_path_desc& q = op.paths[p];
      if (q.src < 0 || q.src >= nt) return bad("path src out of range");
      if (q.src == op.dst) return bad("in-place op");
      const csnet_tensor_desc& S = P.tensors[q.src];
      if (q.c0 < 0 || q.cin <= 0 || q.c0 + q.cin > S.C) return bad("path input channel slice");
      if (q.cout0 < 0 || q.cout <= 0 || q.cout0 + q.cout > Cm) return bad("path output channel slice");
      if (op.kind == CSNET_OP_DW) {
        if (q.ksize != 3 || q.dil != 1 || q.pad != 1 || q.stride != 1 || q.pre_avg || q.pool != 1 || q.up != 1)
          return bad("DW must be 3x3 pad 1");
        if (q.cin != D.C || q.cout != D.C || q.c0 != 0 || q.cout0 != 0 || S.C != D.C || S.H != D.H || S.W != D.W)
          return bad("DW shape");
        if (q.w_off < 0 || q.w_off + (int64_t)D.C * 9 > P.blob_floats) return bad("DW weights outside blob");
        continue;
      }
      if (q.ksize == 0) {
        if (q.up < 1 || q.cin != q.cout || q.pool < 1) return bad("resample path");
        if (q.pre_avg != 0 && q.pre_avg != 1 && q.pre_avg != 2 && q.pre_avg != 4 && q.pre_avg != 8) return bad("pre_avg must be 0, 1, 2, 4 or 8");
        const int div = csnet::pre_factor(q.pre_avg) * q.pool;
        if (div > 1 && q.up != 1) return bad("a resample path either up-samples or down-samples");
        if (S.H % div || S.W % div) return bad("pooling does not divide the source");
        if (S.H / div * q.up != D.H || S.W / div * q.up != D.W) return bad("resample path size");
      } else {
        if (q.ksize != 1 && q.ksize != 3) return bad("ksize must be 1 or 3");
        if (q.up < 1) return bad("conv path up < 1");
        if (q.up > 1 && (q.ksize != 1 || q.pool != 1 || q.pre_avg || q.stride != 1 || q.pad != 0))
          return bad("input-side up-sampling is only defined for plain 1x1 conv paths");
        if (q.pool < 1 || q.stride < 1 || q.dil < 1 || q.pad < 0) return bad("conv path params");
        if (q.pre_avg != 0 && q.pre_avg != 1 && q.pre_avg != 2 && q.pre_avg != 4 && q.pre_avg != 8) return bad("pre_avg must be 0, 1, 2, 4 or 8");
        const int div = csnet::pre_factor(q.pre_avg) * q.pool;
        if (S.H % div || S.W % div) return bad("pooling does not divide the source");
        const int Hc = q.up > 1 ? S.H * q.up : S.H / div, Wc = q.up > 1 ? S.W * q.up : S.W / div;
        const int Ho = (Hc + 2 * q.pad - q.dil * (q.ksize - 1) - 1) / q.stride + 1;
        const int Wo = (Wc + 2 * q.pad - q.dil * (q.ksize - 1) - 1) / q.stride + 1;
        if (Ho != D.H || Wo != D.W) return bad("conv path output size != dst");
        const int64_t nw = (int64_t)q.cout * q.cin * q.ksize * q.ksize;
        if (q.w_off < 0 || q.w_off + nw > P.blob_floats) return bad("weights outside blob");
      }
    }
  }
  return CSNET_OK;
}

csnet::MixArgs make_mix(const csnet_plan& P, const csnet_op_desc& op, int N, const void* const* ext) {
  csnet::MixArgs A{};
  const csnet_tensor_desc& D = P.tensors[op.dst];
  A.dst = P.tensor_ptr(op.dst, N, ext);
  A.bias = op.bias_off >= 0 ? P.blob + op.bias_off : nullptr;
  A.slope = op.slope_off >= 0 ? P.blob + op.slope_off : nullptr;
  A.dtype = D.dtype; A.C = mix_channels(P, op); A.H = D.H; A.W = D.W;
  A.n_paths = op.n_paths;
  if (op.kind == CSNET_OP_MIXPROJ) {
    A.proj_w = P.blob + op.ext_off[0];
    A.proj_b = op.ext_off[1] >= 0 ? P.blob + op.ext_off[1] : nullptr;
  }
  for (int p = 0; p < op.n_paths; ++p) {
    const csnet_path_desc& q = op.paths[p];
    const csnet_tensor_desc& S = P.tensors[q.src];
    csnet::MixPath& m = A.p[p];
    m.src = P.tensor_ptr(q.src, N, ext);
    m.w = q.ksize > 0 ? P.blob + q.w_off : nullptr;
    m.dtype = S.dtype; m.C = S.C; m.H = S.H; m.W = S.W;
    m.c0 = q.c0; m.cin = q.cin; m.pre_avg = q.pre_avg; m.pool = q.pool;
    m.ksize = q.ksize; m.dil = q.dil; m.stride = q.stride; m.pad = q.pad; m.up = q.up;
    m.cout0 = q.cout0; m.cout = q.cout;
  }
  return A;
}

int round_up(int v, int m) { return (v + m - 1) / m * m; }

// cuTensorMapEncodeTiled comes from the driver; resolve it through the runtime so the library links against
// cudart only.
typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                                  const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                                  CUtensorMapL2promotion, CUtensorMapFloatOOBfill);
EncodeTiledFn encode_tiled_fn() {
  static EncodeTiledFn fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    return reinterpret_cast<EncodeTiledFn>(p);
  }();
  return fn;
}

// Kernel arguments of a fused ILBlock op (the tensors are bound per launch) and its tile; false if no tile fits shared memory.
bool make_il(const csnet_plan& P, const csnet_op_desc& op, csnet::IlArgs* out) {
  csnet::IlArgs A{};
  const csnet_tensor_desc &Xh = P.tensors[op.paths[0].src], &Xl = P.tensors[op.paths[1].src], &Yh = P.tensors[op.dst];
  A.H = Yh.H; A.W = Yh.W;
  A.Chi = Xh.C; A.Cli = Xl.C; A.Cho = Yh.C; A.Clo = op.dst2 >= 0 ? P.tensors[op.dst2].C : 0;
  A.first = op.paths[0].ksize == 3;
  if (A.first) { A.Chi = Xh.C * 9; A.Cli = 0; }                  // im2col rows of the image; no lo input tensor
  auto f = [&](int e) { return op.ext_off[e] >= 0 ? P.blob + op.ext_off[e] : nullptr; };
  A.wh = reinterpret_cast<const uint32_t*>(f(0));
  A.wl = reinterpret_cast<const uint32_t*>(f(1));
  A.bias_h = f(2); A.slope_h = f(3); A.bias_l = f(4); A.slope_l = f(5);
  A.dw1h = {f(6), f(7), f(8)};   A.dw1l = {f(9), f(10), f(11)};
  A.dw2h = {f(12), f(13), f(14)}; A.dw2l = {f(15), f(16), f(17)};
  A.K8 = round_up(A.Chi + A.Cli, 8);
  if (A.K8 > 8 * csnet::kIlMaxK8) return false;
  A.MH16 = round_up(A.Cho, 16);
  A.ML16 = A.Clo > 0 ? round_up(A.Clo, 16) : 0;
  A.rowsAh = A.K8 > A.Cho ? A.K8 : A.Cho;
  A.rowsAl = A.Clo > 0 ? (A.K8 > A.Clo ? A.K8 : A.Clo) : A.Cli;
  static const int cand[][2] = {{32, 32}, {28, 32}, {16, 64}, {16, 32}, {8, 16}};   // the instantiated tile geometries
  double best = -1;
  for (int chunked = 0; chunked < 2; ++chunked) {
    for (auto& c : cand) {
      csnet::IlArgs T = A;
      T.TH = c[0]; T.TW = c[1];
      T.t2h = chunked ? 8 : A.Cho;                       // chunked: the depthwise tail runs 8 hi channels at a time
      if (chunked && A.Cho <= 8) continue;
      const int NPH = ((T.TH + 8) | 1) * (T.TW + 8), NPL = ((T.TH / 2 + 4) | 1) * (T.TW / 2 + 8);
      if (csnet::il_smem_bytes(T, NPH, NPL) > 227 * 1024) continue;
      // stem form: the fp32 image tile is staged in the T2 buffers before they are needed
      if (A.first && (size_t)Xh.C * (T.TH + 12) * (T.TW + 24) * 4 > ((size_t)T.t2h * NPH + (size_t)A.Clo * NPL) * 2) continue;
      const int ty = (A.H + T.TH - 1) / T.TH, tx = (A.W + T.TW - 1) / T.TW;
      const double cost = (double)ty * tx * NPH * (chunked ? 1.15 : 1.0);   // halo work, small penalty for the extra barriers
      if (best < 0 || cost < best) { best = cost; T.tiles_x = tx; *out = T; }
    }
  }
  return best >= 0;
}

size_t il_smem_of(const csnet::IlArgs& A) {
  return csnet::il_smem_bytes(A, ((A.TH + 8) | 1) * (A.TW + 8), ((A.TH / 2 + 4) | 1) * (A.TW / 2 + 8));
}

// 5-D map over a planar [N][C][H][W] 16-bit tensor with W split into (W/8, 8): dims (8 px, C, W/8, H, N).  A box
// (8, slots, groups, rows, 1) lands in shared memory as [row][group][slot][8 px] — the tensor-core operand layout of
// il_stream.cuh; slots past C are zero-filled.
bool encode_group_map(CUtensorMap* tm, const void* base, int N, int C, int H, int W, int slots, int groups, int rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return false;
  const cuuint64_t dims[5] = {8, (cuuint64_t)C, (cuuint64_t)(W / 8), (cuuint64_t)H, (cuuint64_t)N};
  const cuuint64_t strides[4] = {(cuuint64_t)H * W * 2, 16, (cuuint64_t)W * 2, (cuuint64_t)C * H * W * 2};
  const cuuint32_t box[5] = {8, (cuuint32_t)slots, (cuuint32_t)groups, (cuuint32_t)rows, 1};
  const cuuint32_t estr[5] = {1, 1, 1, 1, 1};
  return fn(tm, CU_TENSOR_MAP_DATA_TYPE_UINT16, 5, const_cast<void*>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// 4-D map over the planar fp32 image [N][C][H][W]: box (bw floats, rows, C, 1) -> [c][row][bw] in shared memory, zeros outside.
bool encode_image_map(CUtensorMap* tm, const void* base, int N, int C, int H, int W, int bw, int rows) {
  EncodeTiledFn fn = encode_tiled_fn();
  if (!fn) return false;
  const cuuint64_t dims[4] = {(cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)C, (cuuint64_t)N};
  const cuuint64_t strides[3] = {(cuuint64_t)W * 4, (cuuint64_t)H * W * 4, (cuuint64_t)C * H * W * 4};
  const cuuint32_t box[4] = {(cuuint32_t)bw, (cuuint32_t)rows, (cuuint32_t)C, 1};
  const cuuint32_t estr[4] = {1, 1, 1, 1};
  return fn(tm, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, const_cast<void*>(base), dims, strides, box, estr,
            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_NONE, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
            CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) == CUDA_SUCCESS;
}

// Geometry and parameter pointers of the streaming ILBlock kernel for an op; false if the op does not qualify (the tiled kernel
// runs it).  Picks the column-strip split: the fewest strips that fit the thread / shared-memory / TMEM limits (force_ns > 0:
// exactly that many).
bool make_ils(const csnet_plan& P, const csnet_op_desc& op, int force_ns, csnet::IlsArgs* out) {
  if (encode_tiled_fn() == nullptr) return false;
  const csnet_tensor_desc &Xh = P.tensors[op.paths[0].src], &Xl = P.tensors[op.paths[1].src], &Yh = P.tensors[op.dst];
  if (Yh.dtype != CSNET_F16) return false;
  const bool stem = op.paths[0].ksize == 3;                              // stem form: 3x3 convs of the fp32 image (im2col K = 9 Ci)
  csnet::IlsArgs A{};
  A.H = Yh.H; A.W = Yh.W;
  A.Chi = stem ? Xh.C * 9 : Xh.C; A.Cli = stem ? 0 : Xl.C; A.Cho = Yh.C; A.Clo = op.dst2 >= 0 ? P.tensors[op.dst2].C : 0;
  A.Ci = stem ? Xh.C : 0;
  if (stem && (Xh.dtype != CSNET_F32 || A.Chi > 32 || A.W % 4)) return false;
  if (A.W % 16 || A.H % 4 || A.Cho > csnet::kIlsMaxC || A.Clo > csnet::kIlsMaxC || A.Chi + A.Cli > 64) return false;
  A.K8 = stem ? 32 : round_up(A.Chi + A.Cli, 8);                      // the compiler packs the stem's weights as [M16][32]
  A.K16 = round_up(A.Chi + A.Cli, 16);
  A.NH = round_up(A.Cho, 16);
  A.NL = A.Clo > 0 ? round_up(A.Clo, 16) : 0;
  A.GH = A.W / 8; A.GL = A.W / 16;
  A.SH = (A.K16 > A.NH ? A.K16 : A.NH) + 1;            // odd: consecutive pixel groups start in different bank groups
  A.SL = A.Clo > 0 ? A.K16 + 1 : (A.Cli | 1);
  A.ST = A.NL + 1;
  A.cpi = A.H / 4;
  auto r128 = [](int v) { return (v + 127) / 128 * 128; };
  bool found = false;
  double best_cost = 0;
  csnet::IlsArgs best{};
  for (int ns = 1; ns <= 16; ++ns) {
    if (force_ns > 0 && ns != force_ns) continue;
    if (A.GH % ns || (A.GH / ns) % 2) continue;
    csnet::IlsArgs T = A;
    T.ns = ns; T.gsn = A.GH / ns; T.hl = ns > 1 ? 1 : 0;
    T.GR = T.gsn + 2 * T.hl; T.GLR = T.gsn / 2 + 2 * T.hl;
    T.dw_warps = (T.Cho * T.gsn + T.Clo * (T.gsn / 2) + 31) / 32;        // tail tasks are packed: hi (channel, column)s, then lo ones
    if (T.dw_warps < 4) T.dw_warps = 4;                                   // the epilogue needs one warp per TMEM lane quarter
    const int warps = T.dw_warps;
    if (warps * 32 > csnet::kIlsMaxThreads || T.SH > 256 || T.SL > 256 || T.GR > 256) continue;
    const int nbh = (4 * T.GR + 15) / 16, nbl = T.Clo > 0 ? (2 * T.GLR + 15) / 16 : 0;
    const int cols = nbh * T.NH + nbl * T.NL;                              // fp32 accumulators of a chunk: TMEM columns
    if (cols > 512 || nbh + nbl > 16) continue;
    T.tmem_cols = 32;
    while (T.tmem_cols < cols) T.tmem_cols *= 2;
    T.BW = 8 * T.GR + 8;                                                  // stem: image block row = the tile's pixels + 4 on each side
    if (stem && T.BW > 256) continue;
    T.lo_stage_bytes = stem ? r128(T.BW * 4 * T.Ci * 4) : r128(2 * T.GLR * T.SL * 16);
    T.hi_stage_bytes = r128(4 * T.GR * T.SH * 16);
    T.off_xl = 0;
    T.off_xh = csnet::kIlsLoStages * T.lo_stage_bytes;
    T.off_t1l = T.off_xh + csnet::kIlsHiStages * T.hi_stage_bytes;
    T.off_wbh = T.off_t1l + r128(2 * T.GLR * T.ST * 16);
    T.off_wbl = T.off_wbh + r128(T.NH * T.K16 * 2);
    T.off_bar = T.off_wbl + r128(T.NL * T.K16 * 2);
    T.off_zero = T.off_bar + 256;
    T.off_epi = T.off_zero + 128;                          // 4 tables of 64 floats + 512 bytes of scratch rows
    T.off_xlo = T.off_epi + 1536;                          // stem: GEMM operand of the lo chunk (the ring holds image blocks)
    int end = T.off_xlo + (stem ? r128(2 * T.GLR * T.SL * 16) : 0);
    // the last accumulator block of a chunk reads (never uses) up to 15 pixel groups past the chunk: keep them inside
    const int over_h = T.off_xh + T.hi_stage_bytes + nbh * 16 * T.SH * 16,
              over_l = (stem ? T.off_xlo : T.off_xl + 2 * T.lo_stage_bytes) + nbl * 16 * T.SL * 16;
    end = over_h > end ? over_h : end;
    end = over_l > end ? over_l : end;
    T.smem_bytes = end + 128;
    if (T.smem_bytes > 227 * 1024) continue;
    // cost model: the depthwise tail (~55 % of a chunk) does not see the halo groups, everything else scales with them.
    // (Narrow strips do NOT buy a second CTA per SM: a kernel that touches tcgen05 is resident once per SM — measured with
    // scripts/occ_probe.cu: occupancy 1 for any kernel with tcgen05.alloc / commit, whatever its shared memory.)
    const double cost = 0.55 + 0.45 * T.GR / T.gsn;
    if (!found || cost < best_cost) { best = T; best_cost = cost; found = true; }
  }
  if (!found) return false;
  auto f = [&](int e) { return op.ext_off[e] >= 0 ? P.blob + op.ext_off[e] : nullptr; };
  best.wh = reinterpret_cast<const uint32_t*>(f(0));
  best.wl = reinterpret_cast<const uint32_t*>(f(1));
  best.dw1h = {f(6), f(7), f(8)};   best.dw1l = {f(9), f(10), f(11)};
  best.dw2h = {f(12), f(13), f(14)}; best.dw2l = {f(15), f(16), f(17)};
  *out = best;
  return true;
}

// MSBlock form of a MIX op: every path a dilated 3x3 (pad == dil in {1, 2, 4, 8, 16}, stride 1) of the SAME whole fp16 tensor,
// at most 8 output channels per path, fp16 destination of the same size.  Each path's launch writes only its own cout slice and
// applies no accumulation across paths, so the slices must be disjoint and cover the destination (the MSBlock concat).
bool is_msd(const csnet_plan& P, const csnet_op_desc& op) {
  if (op.kind != CSNET_OP_MIX || op.ext_off[CSNET_EXT_NO_FAST] == 1 || op.n_paths < 1) return false;
  const csnet_tensor_desc& D = P.tensors[op.dst];
  if (D.dtype != CSNET_F16 || D.W % 8 || D.C > 64) return false;
  uint64_t covered = 0;                                  // (validate(): cout0 + cout <= D.C <= 64)
  for (int p = 0; p < op.n_paths; ++p) {
    const csnet_path_desc& q = op.paths[p];
    const csnet_tensor_desc& S = P.tensors[q.src];
    if (q.ksize != 3 || q.src != op.paths[0].src || q.c0 != 0 || q.cin != S.C || q.stride != 1 || q.pad != q.dil || q.pool != 1 || q.pre_avg ||
        q.up != 1 || S.dtype != CSNET_F16 || S.H != D.H || S.W != D.W || q.cout > 8 || q.cin > 128)
      return false;
    if (q.dil != 1 && q.dil != 2 && q.dil != 4 && q.dil != 8 && q.dil != 16) return false;
    const uint64_t slice = ((1ull << q.cout) - 1) << q.cout0;
    if (covered & slice) return false;
    covered |= slice;
  }
  return covered == (D.C == 64 ? ~0ull : (1ull << D.C) - 1);
}

// Kernel arguments of the streaming MIX kernel for an op (the tensors and N are bound per launch); false if the op does not qualify.
bool make_ms(const csnet_plan& P, const csnet_op_desc& op, csnet::MsArgs* out) {
  if ((op.kind != CSNET_OP_MIX && op.kind != CSNET_OP_MIXPROJ) || encode_tiled_fn() == nullptr) return false;
  if (op.kind == CSNET_OP_MIX && op.ext_off[CSNET_EXT_NO_FAST] == 1) return false;
  const csnet_tensor_desc& D = P.tensors[op.dst];
  csnet::MsArgs A{};
  A.C = mix_channels(P, op);
  A.has_proj = op.kind == CSNET_OP_MIXPROJ;
  if (A.C > csnet::kMsMaxC || D.W % 8 || D.H % csnet::kMsRows) return false;
  if (A.has_proj ? D.dtype != CSNET_F32 : D.dtype == CSNET_BF16) return false;
  A.dst_f32 = D.dtype == CSNET_F32;
  A.H = D.H; A.W = D.W; A.G = D.W / 8; A.NN = round_up(A.C, 16);
  int off = 0;
  auto r128 = [](int v) { return (v + 127) / 128 * 128; };
  for (int p = 0; p < op.n_paths; ++p) {
    const csnet_path_desc& q = op.paths[p];
    const csnet_tensor_desc& S = P.tensors[q.src];
    if (q.ksize == 0) {
      if (A.n_rs >= csnet::kMsMaxRs || q.up < 2 || q.pool != 1 || q.pre_avg || S.H * q.up != D.H || S.W * q.up != D.W || S.dtype != CSNET_F32 || q.cout0 != 0) return false;
      const int j = A.n_rs++;
      A.r_dtype[j] = S.dtype; A.r_up[j] = q.up; A.r_H[j] = S.H; A.r_W[j] = S.W; A.r_C[j] = S.C; A.r_c0[j] = q.c0; A.r_cout0[j] = q.cout0; A.r_n[j] = q.cout;
      continue;
    }
    const bool k3 = q.ksize == 3 && q.pad == 1 && q.dil == 1, k1 = q.ksize == 1 && q.pad == 0;
    if (A.n_in >= csnet::kMsMaxIn || !(k1 || k3) || (A.n_in > 0 && (int)k3 != A.k3) || q.stride != 1 || q.up != 1 || q.pool != 1 || q.pre_avg ||
        S.dtype != CSNET_F16 || S.H != D.H || S.W != D.W || q.cin > 64)
      return false;
    A.k3 = k3;
    const int trows = csnet::kMsRows + (k3 ? 2 : 0);
    const int i = A.n_in++;
    A.w[i] = P.blob + q.w_off;
    A.cin[i] = q.cin; A.cout0[i] = q.cout0; A.cout[i] = q.cout;
    A.K16[i] = round_up(q.cin, 16); A.S[i] = A.K16[i] + 1;
    A.in_off[i] = off;
    A.copy_bytes[i] = r128(trows * A.G * A.S[i] * 16);
    off += (k3 ? 3 : 1) * A.copy_bytes[i];
    if (q.c0 != 0) return false;                                            // (a channel-sliced source would need a c0 coordinate)
  }
  if (A.n_in == 0) return false;
  A.stage_bytes = off;
  A.tx_bytes = 0;
  for (int i = 0; i < A.n_in; ++i) A.tx_bytes += (csnet::kMsRows + (A.k3 ? 2 : 0)) * A.G * A.S[i] * 16;
  A.nb = (csnet::kMsRows * A.G + 15) / 16;
  A.n_acc = 512 / (A.nb * A.NN);
  A.n_acc = A.n_acc > 8 ? 8 : A.n_acc;
  if (A.n_acc < 2) return false;
  A.cpi = D.H / csnet::kMsRows;
  int wb = 0;
  const int taps = A.k3 ? 9 : 1;
  for (int i = 0; i < A.n_in; ++i) wb += r128(taps * A.NN * A.K16[i] * 2);
  const int fixed = wb + 512 + 1280 + 16 * 65 * 16 + 128;                  // weights, barriers, tables, tail slack, alignment
  A.n_stages = (227 * 1024 - fixed) / A.stage_bytes;
  A.n_stages = A.n_stages > 6 ? 6 : A.n_stages;
  if (A.n_stages < 2) return false;
  A.off_stage = 0;
  int o = A.n_stages * A.stage_bytes + 16 * 65 * 16;
  for (int i = 0; i < A.n_in; ++i) { A.off_wb[i] = o; o += r128(taps * A.NN * A.K16[i] * 2); }
  A.off_bar = o; o += 512;
  A.off_tab = o; o += 1280;
  A.smem_bytes = o + 128;
  A.has_slope = op.slope_off >= 0;
  *out = A;
  return true;
}

// The epilogue tables the streaming kernels carry in their arguments, from the host copy of the blob.
void fill_tables(const csnet_op_desc& op, const float* blob, OpRoute& R) {
  if (R.route == Route::MIX_STREAM) {
    csnet::MsArgs& A = R.ms;
    for (int c = 0; c < A.C; ++c) {
      A.bias[c] = op.bias_off >= 0 ? blob[op.bias_off + c] : 0.f;
      A.sm1[c] = op.slope_off >= 0 ? blob[op.slope_off + c] - 1.f : 0.f;
      A.proj[c] = A.has_proj ? blob[op.ext_off[0] + c] : 0.f;
    }
    A.proj_b = A.has_proj && op.ext_off[1] >= 0 ? blob[op.ext_off[1]] : 0.f;
  } else if (R.route == Route::IL_STREAM) {
    csnet::IlsArgs& A = R.ils;
    for (int c = 0; c < A.Cho; ++c) { A.bias_h[c] = blob[op.ext_off[2] + c]; A.sm1_h[c] = blob[op.ext_off[3] + c] - 1.f; }
    for (int c = 0; c < A.Clo; ++c) { A.bias_l[c] = blob[op.ext_off[4] + c]; A.sm1_l[c] = blob[op.ext_off[5] + c] - 1.f; }
  }
}

template <typename T>
void launch_il_t(const csnet::IlArgs& A, dim3 grid, size_t smem, cudaStream_t st) {
  if (A.TH == 32) csnet::il_block_kernel<T, 32, 32><<<grid, csnet::kIlThreads, smem, st>>>(A);
  else if (A.TH == 28) csnet::il_block_kernel<T, 28, 32><<<grid, csnet::kIlThreads, smem, st>>>(A);
  else if (A.TH == 16 && A.TW == 64) csnet::il_block_kernel<T, 16, 64><<<grid, csnet::kIlThreads, smem, st>>>(A);
  else if (A.TH == 16) csnet::il_block_kernel<T, 16, 32><<<grid, csnet::kIlThreads, smem, st>>>(A);
  else csnet::il_block_kernel<T, 8, 16><<<grid, csnet::kIlThreads, smem, st>>>(A);
}

template <typename T>
cudaError_t set_il_smem_t(int bytes) {
  cudaError_t e = cudaFuncSetAttribute(csnet::il_block_kernel<T, 32, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(csnet::il_block_kernel<T, 28, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(csnet::il_block_kernel<T, 16, 64>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(csnet::il_block_kernel<T, 16, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(csnet::il_block_kernel<T, 8, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  return e;
}

// Can this MIX op run on the tensor-core kernel (mix_tc.cuh)?  Needs 16-bit operands somewhere, stride-1 conv
// paths and at most 80 output channels.  enabled == false (CSNET_TC=0) keeps MIX ops off it.
TcChoice choose_tc(const csnet_plan& P, const csnet_op_desc& op, bool enabled) {
  TcChoice c;
  if (op.kind == CSNET_OP_MIXPROJ) { /* no other kernel implements it */ }
  else if (!enabled || op.kind != CSNET_OP_MIX || op.ext_off[CSNET_EXT_NO_FAST] == 1) return c;
  const csnet_tensor_desc& D = P.tensors[op.dst];
  const int Cm = mix_channels(P, op);
  int dt = D.dtype != CSNET_F32 ? D.dtype : -1, pad = 0, nconv = 0, kk = 1, cin_max = 0;
  for (int p = 0; p < op.n_paths; ++p) {
    const csnet_path_desc& q = op.paths[p];
    if (q.ksize == 0 && (q.pre_avg || q.pool > 1)) return c;     // down-sampling resample paths: generic kernels only
    if (q.ksize == 0) continue;
    ++nconv;
    if (q.stride != 1) return c;
    if (dt < 0 && P.tensors[q.src].dtype != CSNET_F32) dt = P.tensors[q.src].dtype;
    pad = q.pad > pad ? q.pad : pad;
    kk = q.ksize * q.ksize > kk ? q.ksize * q.ksize : kk;
    cin_max = q.cin > cin_max ? q.cin : cin_max;
  }
  if (dt < 0 || nconv == 0 || pad > csnet::kTcMaxPad) return c;
  c.mt = Cm > 80 ? 5 : (Cm + 15) / 16;               // more than 80 output channels: 80-channel slices over grid.y
  c.dtype = dt;
  // wide halos (dilated MS convs): taller tiles while the accumulators fit (MT * rows <= 4)
  c.rows = pad >= 4 ? (c.mt == 1 ? 4 : (c.mt == 2 ? 2 : 1)) : 1;
  c.xs_halves = csnet::tc_plane_halves(pad, c.rows);
  c.kk = kk;
  c.kc = 8;
  for (int kc : {32, 16}) {                       // the largest chunk that keeps two CTAs per SM resident
    TcChoice t = c;
    t.kc = kc;
    if (kc <= ((cin_max + 7) & ~7) && tc_smem_bytes(t) <= 100 * 1024) { c.kc = kc; break; }
  }
  return c;
}

template <typename T>
void launch_mix_tc_t(int mt, dim3 grid, size_t smem, cudaStream_t st, const csnet::MixArgs& A, const csnet::TcGeom& G) {
  if (G.rows == 4) { csnet::mix_tc_kernel<T, 1, 4><<<grid, csnet::kTcThreads, smem, st>>>(A, G); return; }
  if (G.rows == 2) { csnet::mix_tc_kernel<T, 2, 2><<<grid, csnet::kTcThreads, smem, st>>>(A, G); return; }
  switch (mt) {
    case 1: csnet::mix_tc_kernel<T, 1><<<grid, csnet::kTcThreads, smem, st>>>(A, G); break;
    case 2: csnet::mix_tc_kernel<T, 2><<<grid, csnet::kTcThreads, smem, st>>>(A, G); break;
    case 3: csnet::mix_tc_kernel<T, 3><<<grid, csnet::kTcThreads, smem, st>>>(A, G); break;
    case 4: csnet::mix_tc_kernel<T, 4><<<grid, csnet::kTcThreads, smem, st>>>(A, G); break;
    default: csnet::mix_tc_kernel<T, 5><<<grid, csnet::kTcThreads, smem, st>>>(A, G); break;
  }
}

void launch_mix_tc(const TcChoice& c, dim3 grid, size_t smem, cudaStream_t st, const csnet::MixArgs& A, const csnet::TcGeom& G) {
  if (c.dtype == CSNET_F16) launch_mix_tc_t<__half>(c.mt, grid, smem, st, A, G);
  else launch_mix_tc_t<__nv_bfloat16>(c.mt, grid, smem, st, A, G);
}

template <typename T>
cudaError_t set_tc_smem_t(int bytes) {
  cudaError_t e = cudaFuncSetAttribute(csnet::mix_tc_kernel<T, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(csnet::mix_tc_kernel<T, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(csnet::mix_tc_kernel<T, 3>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(csnet::mix_tc_kernel<T, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(csnet::mix_tc_kernel<T, 5>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(csnet::mix_tc_kernel<T, 1, 4>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  if (e == cudaSuccess) e = cudaFuncSetAttribute(csnet::mix_tc_kernel<T, 2, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, bytes);
  return e;
}

// The executor's switches, read from the environment when a plan is created.  They select the slower kernels, which the tests
// use as references for the fast ones.
struct Switches {
  bool tc, msd, ms, ils;     // CSNET_TC / CSNET_MSD / CSNET_MS / CSNET_ILS = 0: keep ops off that kernel
  int ils_ns;                // CSNET_ILS_NS = k: il_stream runs k column strips (0: automatic)
  int ils_min_chunks;        // CSNET_ILS_MIN_CHUNKS: fewer 4-row chunks per ILBlock at max_batch -> the tiled kernel
  int graph_max_n;           // CSNET_GRAPH_MAX_N: largest batch replayed from a CUDA graph (0: none)
};

Switches read_switches(int num_sms) {
  auto on = [](const char* name) { const char* e = getenv(name); return !(e && e[0] == '0'); };
  auto num = [](const char* name, int dflt) { const char* e = getenv(name); return e ? atoi(e) : dflt; };
  return {on("CSNET_TC"), on("CSNET_MSD"), on("CSNET_MS"), on("CSNET_ILS"), num("CSNET_ILS_NS", 0),
          num("CSNET_ILS_MIN_CHUNKS", 4 * num_sms), num("CSNET_GRAPH_MAX_N", 8)};
}

// Decide an op's route, first match in the order below, and fill what it needs (the caller allocates the packed weights);
// an error message if the op cannot run.
const char* route_op(const csnet_plan& P, const csnet_op_desc& op, const Switches& sw, OpRoute& R) {
  const csnet_tensor_desc& D = P.tensors[op.dst];
  if (op.kind == CSNET_OP_MIX || op.kind == CSNET_OP_MIXPROJ) {
    const TcChoice tc = choose_tc(P, op, sw.tc);
    const bool tc_ok = tc.mt > 0 && tc_smem_bytes(tc) <= 200 * 1024;
    if (op.kind == CSNET_OP_MIXPROJ && !tc_ok)
      return "MIXPROJ op does not qualify for the tensor-core kernel (16-bit sources, stride 1, pad <= limit)";
    const csnet_path_desc& q = op.paths[0];
    if (sw.msd && is_msd(P, op)) {
      R.route = Route::MSD;
    } else if (sw.ms && make_ms(P, op, &R.ms) && (int64_t)P.max_batch * (D.H / csnet::kMsRows) >= (int64_t)2 * P.num_sms) {
      R.route = Route::MIX_STREAM;
      R.smem = R.ms.smem_bytes;
    } else if (tc_ok) {
      R.route = Route::MIX_TC;
      R.tc = tc;
      R.smem = tc_smem_bytes(tc);
    } else if (op.n_paths == 1 && q.ksize == 0 && q.cout0 == 0 && q.cout == D.C) {
      const csnet_tensor_desc& S = P.tensors[q.src];
      const bool avg2 = q.pre_avg == 1 && q.pool == 1, max2 = q.pre_avg == 0 && q.pool == 2;
      const bool fast = S.dtype == D.dtype && D.dtype != CSNET_F32 && D.W % 4 == 0 && op.bias_off < 0 && op.slope_off < 0;
      if (fast && (avg2 || max2) && q.up == 1 && q.c0 == 0) R.route = Route::POOL2;
      else if (fast && q.up > 1 && !q.pre_avg && q.pool == 1) R.route = Route::UPSAMPLE;
      else R.route = Route::RESAMPLE;
    } else {
      R.route = Route::MIX_GENERIC;
    }
  } else if (op.kind == CSNET_OP_GN) {
    R.route = Route::GN;
  } else if (op.kind == CSNET_OP_ILBLOCK) {
    if (!make_il(P, op, &R.il)) return "ILBLOCK op does not fit shared memory";
    if (sw.ils && make_ils(P, op, sw.ils_ns, &R.ils) && (int64_t)P.max_batch * (D.H / 4) >= (int64_t)sw.ils_min_chunks) {
      R.route = Route::IL_STREAM;
      R.smem = R.ils.smem_bytes;
    } else {
      R.route = Route::IL_BLOCK;
      R.smem = il_smem_of(R.il);
    }
  } else {
    const csnet_tensor_desc& S = P.tensors[op.paths[0].src];
    const bool fast = op.ext_off[CSNET_EXT_NO_FAST] != 1 && S.dtype == D.dtype && D.dtype != CSNET_F32 && D.W % 4 == 0;
    R.route = fast ? Route::DW_FAST : Route::DW_GENERIC;
  }
  return nullptr;
}

}  // namespace

extern "C" {

int csnet_abi_version(void) { return CSNET_ABI_VERSION; }

const char* csnet_last_error(void) { return g_err.c_str(); }

int csnet_device_count(void) {
  int n = 0;
  cudaError_t e = cudaGetDeviceCount(&n);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return fail(CSNET_E_CUDA, std::string("cudaGetDeviceCount: ") + cudaGetErrorString(e));
  }
  return n;
}

int csnet_plan_create(csnet_plan** out, const csnet_tensor_desc* tensors, int32_t n_tensors,
                      const csnet_op_desc* ops, int32_t n_ops, int64_t blob_floats, int32_t max_batch,
                      int32_t device) {
  if (!out || !tensors || !ops || n_tensors <= 0 || n_ops <= 0 || blob_floats <= 0 || max_batch <= 0)
    return fail(CSNET_E_INVALID, "csnet_plan_create: null/empty argument");
  csnet_plan* P = new (std::nothrow) csnet_plan();
  if (!P) return fail(CSNET_E_NOMEM, "host allocation failed");
  P->device = device;
  P->max_batch = max_batch;
  P->tensors.assign(tensors, tensors + n_tensors);
  P->ops.assign(ops, ops + n_ops);
  P->blob_floats = blob_floats;
  int rc = validate(*P);
  if (rc != CSNET_OK) { delete P; return rc; }
  for (const auto& d : P->tensors) {
    if (d.external >= 0) { P->n_ext = d.external + 1 > P->n_ext ? d.external + 1 : P->n_ext; continue; }
    const int64_t end = d.arena_offset + (int64_t)d.C * d.H * d.W * (int64_t)dtype_size(d.dtype);
    P->arena_per_image = end > P->arena_per_image ? end : P->arena_per_image;
  }
  P->arena_per_image = (P->arena_per_image + 255) / 256 * 256;
  auto cleanup = [&](int code, const std::string& m) { csnet_plan_destroy(P); return fail(code, m); };
  DeviceGuard guard_(device);
  cudaError_t e = cudaSuccess;
  {
    int cur = -1;
    if (cudaGetDevice(&cur) != cudaSuccess || cur != device) return cleanup(CSNET_E_CUDA, "cudaSetDevice failed");
  }
  e = cudaMalloc(&P->blob, (size_t)blob_floats * sizeof(float));
  if (e != cudaSuccess) return cleanup(CSNET_E_NOMEM, std::string("cudaMalloc(blob): ") + cudaGetErrorString(e));
  const size_t arena_bytes = (size_t)P->arena_per_image * (size_t)max_batch + 256;
  e = cudaMalloc(&P->arena, arena_bytes);
  if (e != cudaSuccess) return cleanup(CSNET_E_NOMEM, std::string("cudaMalloc(arena): ") + cudaGetErrorString(e));
  for (const auto& op : P->ops)
    if (op.kind == CSNET_OP_GN && op.paths[0].up > P->gn_groups_max) P->gn_groups_max = op.paths[0].up;
  if (P->gn_groups_max > 0) {
    e = cudaMalloc(&P->gn_stats, (size_t)max_batch * P->gn_groups_max * 2 * sizeof(float));
    if (e != cudaSuccess) return cleanup(CSNET_E_NOMEM, std::string("cudaMalloc(gn stats): ") + cudaGetErrorString(e));
  }
  {
    cudaDeviceProp prop;
    if (cudaGetDeviceProperties(&prop, device) == cudaSuccess && prop.multiProcessorCount > 0) P->num_sms = prop.multiProcessorCount;
  }
  const Switches sw = read_switches(P->num_sms);
  P->graph_max_n = sw.graph_max_n;
  P->routes.resize(P->ops.size());
  bool uses[kRoutes] = {};
  for (size_t i = 0; i < P->ops.size(); ++i) {
    OpRoute& R = P->routes[i];
    if (const char* why = route_op(*P, P->ops[i], sw, R)) return cleanup(CSNET_E_UNSUPPORTED, why);
    uses[(int)R.route] = true;
    if (R.route != Route::MIX_TC) continue;
    const csnet_op_desc& op = P->ops[i];
    const int C = mix_channels(*P, op), slice = R.tc.mt * 16, m16t = (C + slice - 1) / slice * slice, WR = R.tc.kc + 8;
    R.w16.assign(op.n_paths, nullptr);
    for (int p = 0; p < op.n_paths; ++p) {
      const csnet_path_desc& q = op.paths[p];
      if (q.ksize == 0) continue;
      const size_t halves = (size_t)((q.cin + R.tc.kc - 1) / R.tc.kc) * q.ksize * q.ksize * m16t * WR;
      e = cudaMalloc(&R.w16[p], halves * 2);
      if (e != cudaSuccess) return cleanup(CSNET_E_NOMEM, std::string("cudaMalloc(packed weights): ") + cudaGetErrorString(e));
    }
  }
  // The shared-memory limit of every kernel the plan launches is the architectural maximum: plans created later must not lower
  // the limit an earlier plan relies on.
  constexpr int kMaxSmem = 227 * 1024;
  if (uses[(int)Route::MIX_TC]) {
    e = set_tc_smem_t<__half>(kMaxSmem);
    if (e == cudaSuccess) e = set_tc_smem_t<__nv_bfloat16>(kMaxSmem);
    if (e != cudaSuccess) return cleanup(CSNET_E_CUDA, std::string("cudaFuncSetAttribute(mix_tc): ") + cudaGetErrorString(e));
  }
  if (uses[(int)Route::MIX_STREAM]) {
    e = cudaFuncSetAttribute(csnet::mix_stream_kernel<__half>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e != cudaSuccess) return cleanup(CSNET_E_CUDA, std::string("cudaFuncSetAttribute(mix_stream): ") + cudaGetErrorString(e));
  }
  if (uses[(int)Route::IL_STREAM]) {
    e = cudaFuncSetAttribute(csnet::il_stream_kernel<__half, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(csnet::il_stream_kernel<__half, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(csnet::il_stream_kernel<__half, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem);
    // two CTAs of <= 113 KB share an SM only with the full shared-memory carve-out
    if (e == cudaSuccess) e = cudaFuncSetAttribute(csnet::il_stream_kernel<__half, false>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (e == cudaSuccess) e = cudaFuncSetAttribute(csnet::il_stream_kernel<__half, true>, cudaFuncAttributePreferredSharedMemoryCarveout, 100);
    if (e != cudaSuccess) return cleanup(CSNET_E_CUDA, std::string("cudaFuncSetAttribute(il_stream): ") + cudaGetErrorString(e));
  }
  if (uses[(int)Route::IL_BLOCK]) {
    e = set_il_smem_t<__half>(kMaxSmem);
    if (e == cudaSuccess) e = set_il_smem_t<__nv_bfloat16>(kMaxSmem);
    if (e != cudaSuccess) return cleanup(CSNET_E_CUDA, std::string("cudaFuncSetAttribute(il_block): ") + cudaGetErrorString(e));
  }
  *out = P;
  return CSNET_OK;
}

static void drop_graphs(csnet_plan* P);

int csnet_plan_set_blob(csnet_plan* P, const float* host_blob, int64_t n, void* stream) {
  if (!P || !host_blob || n != P->blob_floats) return fail(CSNET_E_INVALID, "csnet_plan_set_blob: size mismatch");
  DeviceGuard guard_(P->device);
  CU_CHECK(cudaMemcpyAsync(P->blob, host_blob, (size_t)n * sizeof(float), cudaMemcpyHostToDevice, (cudaStream_t)stream));
  drop_graphs(P);                                   // captured launches carry parameter tables of the old blob
  // tensor-core MIX ops read their weights as 16-bit [chunk][tap][m16_total][kc + 8] blocks: pack them here, once per
  // weight update, so the kernels stage them with plain 16-byte copies
  std::vector<std::vector<uint16_t>> keep;
  for (size_t i = 0; i < P->ops.size(); ++i) {
    OpRoute& R = P->routes[i];
    const csnet_op_desc& op = P->ops[i];
    fill_tables(op, host_blob, R);
    if (R.route != Route::MIX_TC) continue;
    const TcChoice& tc = R.tc;
    const int C = mix_channels(*P, op), slice = tc.mt * 16, m16t = (C + slice - 1) / slice * slice, WR = tc.kc + 8;
    for (int p = 0; p < op.n_paths; ++p) {
      const csnet_path_desc& q = op.paths[p];
      if (q.ksize == 0) continue;
      const int kk = q.ksize * q.ksize, nchunks = (q.cin + tc.kc - 1) / tc.kc;
      std::vector<uint16_t> h((size_t)nchunks * kk * m16t * WR, 0);
      const float* w = host_blob + q.w_off;                         // [cin][kk][cout]
      for (int ci = 0; ci < q.cin; ++ci)
        for (int tap = 0; tap < kk; ++tap)
          for (int co = 0; co < q.cout; ++co) {
            const float v = w[((size_t)ci * kk + tap) * q.cout + co];
            uint16_t bits;
            if (tc.dtype == CSNET_F16) { __half hv = __float2half_rn(v); memcpy(&bits, &hv, 2); }
            else { __nv_bfloat16 hv = __float2bfloat16_rn(v); memcpy(&bits, &hv, 2); }
            h[(((size_t)(ci / tc.kc) * kk + tap) * m16t + q.cout0 + co) * WR + ci % tc.kc] = bits;
          }
      CU_CHECK(cudaMemcpyAsync(R.w16[p], h.data(), h.size() * 2, cudaMemcpyHostToDevice, (cudaStream_t)stream));
      keep.push_back(std::move(h));
    }
  }
  CU_CHECK(cudaStreamSynchronize((cudaStream_t)stream));
  return CSNET_OK;
}

static int check_run_args(csnet_plan* P, int32_t N, const void* const* ext_ptrs, int32_t n_ext) {
  if (!P) return fail(CSNET_E_INVALID, "null plan");
  if (N <= 0 || N > P->max_batch) return fail(CSNET_E_INVALID, "batch size outside [1, max_batch]");
  if (n_ext < P->n_ext || (P->n_ext > 0 && !ext_ptrs)) return fail(CSNET_E_INVALID, "missing external tensor pointers");
  for (int i = 0; i < P->n_ext; ++i)
    if (!ext_ptrs[i]) return fail(CSNET_E_INVALID, "null external tensor pointer");
  return CSNET_OK;
}

static int launch_op(csnet_plan* P, size_t i, int32_t N, const void* const* ext_ptrs, cudaStream_t stream) {
  const csnet_op_desc& op = P->ops[i];
  const OpRoute& R = P->routes[i];
  const csnet_tensor_desc& D = P->tensors[op.dst];
  switch (R.route) {
    case Route::MSD:
      for (int p = 0; p < op.n_paths; ++p) {
        const csnet_path_desc& q = op.paths[p];
        csnet::MsdArgs A{};
        A.src = reinterpret_cast<const uint16_t*>(P->tensor_ptr(q.src, N, ext_ptrs));
        A.dst = reinterpret_cast<uint16_t*>(P->tensor_ptr(op.dst, N, ext_ptrs));
        A.w = P->blob + q.w_off;
        A.bias = op.bias_off >= 0 ? P->blob + op.bias_off : nullptr;
        A.slope = op.slope_off >= 0 ? P->blob + op.slope_off : nullptr;
        A.N = N; A.Cin = q.cin; A.H = D.H; A.W = D.W; A.Ctot = D.C; A.cout0 = q.cout0; A.cout = q.cout;
        csnet::msd_launch<__half>(q.dil, A, stream);
      }
      break;
    case Route::MIX_STREAM: {
      csnet::MsArgs A = R.ms;
      CUtensorMap maps[csnet::kMsMaxIn];
      memset(maps, 0, sizeof maps);
      for (int p = 0, in = 0, rs = 0; p < op.n_paths; ++p) {
        const csnet_path_desc& q = op.paths[p];
        const csnet_tensor_desc& S = P->tensors[q.src];
        void* src = P->tensor_ptr(q.src, N, ext_ptrs);
        if (q.ksize == 0) { A.rsrc[rs++] = src; continue; }
        if (!encode_group_map(&maps[in], src, N, S.C, S.H, S.W, A.S[in], A.G, csnet::kMsRows + (A.k3 ? 2 : 0)))
          return fail(CSNET_E_CUDA, "cuTensorMapEncodeTiled failed (streaming MIX)");
        ++in;
      }
      for (int k = A.n_in; k < csnet::kMsMaxIn; ++k) maps[k] = maps[0];
      A.dst = P->tensor_ptr(op.dst, N, ext_ptrs);
      A.N = N;
      A.total_chunks = N * A.cpi;
      int grid = A.total_chunks / 2;
      grid = grid < 1 ? 1 : (grid > P->num_sms ? P->num_sms : grid);
      csnet::mix_stream_kernel<__half><<<grid, csnet::kMsThreads, R.smem, stream>>>(A, maps[0], maps[1], maps[2]);
      break;
    }
    case Route::MIX_TC: {
      csnet::MixArgs A = make_mix(*P, op, N, ext_ptrs);
      const TcChoice& tc = R.tc;
      const int Cm = A.C;
      csnet::TcGeom G{};
      G.tiles_x = (D.W + csnet::kTcTW - 1) / csnet::kTcTW; G.xs_halves = tc.xs_halves; G.kc = tc.kc; G.rows = tc.rows;
      const int th = csnet::kTcTH * tc.rows;
      G.m16_total = (Cm + tc.mt * 16 - 1) / (tc.mt * 16) * (tc.mt * 16);
      for (int p = 0; p < op.n_paths; ++p) G.w16[p] = R.w16[p];
      dim3 grid(G.tiles_x * ((D.H + th - 1) / th), (Cm + tc.mt * 16 - 1) / (tc.mt * 16), N);
      launch_mix_tc(tc, grid, R.smem, stream, A, G);
      break;
    }
    case Route::POOL2:                          // avg_pool2d(2, 2) / max_pool2d(2, 2) of a 16-bit tensor
    case Route::UPSAMPLE: {                     // bilinear up-sampling, 16-bit to 16-bit
      csnet::MixArgs A = make_mix(*P, op, N, ext_ptrs);
      const dim3 grid((D.H * (D.W / 4) + 255) / 256, D.C, N);
      const bool max2 = op.paths[0].pool == 2, f16 = D.dtype == CSNET_F16;
      if (R.route == Route::POOL2 && f16) csnet::pool2_fast_kernel<__half><<<grid, 256, 0, stream>>>(A, max2);
      else if (R.route == Route::POOL2) csnet::pool2_fast_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(A, max2);
      else if (f16) csnet::upsample_fast_kernel<__half><<<grid, 256, 0, stream>>>(A);
      else csnet::upsample_fast_kernel<__nv_bfloat16><<<grid, 256, 0, stream>>>(A);
      break;
    }
    case Route::RESAMPLE:
      csnet::resample_fast_kernel<<<dim3((D.H * D.W + 255) / 256, D.C, N), 256, 0, stream>>>(make_mix(*P, op, N, ext_ptrs));
      break;
    case Route::MIX_GENERIC: {
      dim3 grid((D.H * D.W + kThreads - 1) / kThreads, (D.C + csnet::kMixCT - 1) / csnet::kMixCT, N);
      mix_generic_kernel<<<grid, kThreads, 0, stream>>>(make_mix(*P, op, N, ext_ptrs));
      break;
    }
    case Route::GN: {
      const csnet_tensor_desc& S = P->tensors[op.paths[0].src];
      csnet::GnArgs A{};
      A.src = P->tensor_ptr(op.paths[0].src, N, ext_ptrs);
      A.dst = P->tensor_ptr(op.dst, N, ext_ptrs);
      A.gamma = P->blob + op.ext_off[0];
      A.beta = P->blob + op.ext_off[1];
      A.slope = op.slope_off >= 0 ? P->blob + op.slope_off : nullptr;
      A.stats = P->gn_stats;
      A.src_dtype = S.dtype; A.dst_dtype = D.dtype; A.C = D.C; A.HW = D.H * D.W; A.groups = op.paths[0].up;
      gn_stats_kernel<<<dim3(A.groups, N), kThreads, 0, stream>>>(A);
      const int bx = (A.HW + kThreads * 4 - 1) / (kThreads * 4);
      gn_apply_kernel<<<dim3(bx < 1 ? 1 : bx, D.C, N), kThreads, 0, stream>>>(A);
      break;
    }
    case Route::IL_STREAM: {
      csnet::IlsArgs A = R.ils;
      A.yh = P->tensor_ptr(op.dst, N, ext_ptrs);
      A.yl = op.dst2 >= 0 ? P->tensor_ptr(op.dst2, N, ext_ptrs) : nullptr;
      A.N = N;
      A.total_chunks = N * A.ns * A.cpi;
      CUtensorMap tmH, tmL;
      const bool stem = A.Ci > 0;
      if (stem) {
        if (!encode_image_map(&tmL, P->tensor_ptr(op.paths[0].src, N, ext_ptrs), N, A.Ci, A.H, A.W, A.BW, 4))
          return fail(CSNET_E_CUDA, "cuTensorMapEncodeTiled failed (streaming ILBlock, image)");
        tmH = tmL;
      } else if (!encode_group_map(&tmH, P->tensor_ptr(op.paths[0].src, N, ext_ptrs), N, A.Chi, A.H, A.W, A.SH, A.GR, 4) ||
                 !encode_group_map(&tmL, P->tensor_ptr(op.paths[1].src, N, ext_ptrs), N, A.Cli, A.H / 2, A.W / 2, A.SL, A.GLR, 2))
        return fail(CSNET_E_CUDA, "cuTensorMapEncodeTiled failed (streaming ILBlock)");
      int grid = A.total_chunks / 4;
      grid = grid < 1 ? 1 : (grid > P->num_sms ? P->num_sms : grid);     // persistent: one CTA per SM
      static const bool dbg = [] { const char* e = getenv("CSNET_ILS_DBG"); return e && e[0] == '1'; }();
      static unsigned long long* dbg_buf = nullptr;
      if (dbg && !dbg_buf) cudaMalloc(&dbg_buf, 1024 * 8 * sizeof(unsigned long long));
      A.dbg = dbg ? dbg_buf : nullptr;
      if (stem) csnet::il_stream_kernel<__half, false, true><<<grid, A.dw_warps * 32, R.smem, stream>>>(A, tmH, tmL);
      else if (dbg) csnet::il_stream_kernel<__half, true><<<grid, A.dw_warps * 32, R.smem, stream>>>(A, tmH, tmL);
      else csnet::il_stream_kernel<__half, false><<<grid, A.dw_warps * 32, R.smem, stream>>>(A, tmH, tmL);
      if (dbg && !stem) {        // debugging aid: mean cycles per phase over the CTAs (synchronises)
        std::vector<unsigned long long> h((size_t)grid * 8);
        cudaStreamSynchronize(stream);
        cudaMemcpy(h.data(), dbg_buf, h.size() * sizeof(unsigned long long), cudaMemcpyDeviceToHost);
        double m[8] = {0, 0, 0, 0, 0, 0, 0, 0};
        for (int b = 0; b < grid; ++b) for (int k = 0; k < 8; ++k) m[k] += (double)h[(size_t)b * 8 + k] / grid;
        int occ = -1;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, csnet::il_stream_kernel<__half, true>, A.dw_warps * 32, A.smem_bytes);
        fprintf(stderr, "[ils ns %d grid %d threads %d smem %d tmem %d occupancy %d] ", A.ns, grid, A.dw_warps * 32, A.smem_bytes, A.tmem_cols, occ);
        fprintf(stderr, "[ils %dx%d C %d+%d->%d+%d] cycles/CTA: load-wait %.0f resample %.0f syncA %.0f issue %.0f epilogue %.0f syncB %.0f dw %.0f tail %.0f\n",
                A.H, A.W, A.Chi, A.Cli, A.Cho, A.Clo, m[0], m[1], m[2], m[3], m[4], m[5], m[6], m[7]);
      }
      break;
    }
    case Route::IL_BLOCK: {
      csnet::IlArgs A = R.il;
      A.xh = P->tensor_ptr(op.paths[0].src, N, ext_ptrs);
      A.xl = A.first ? nullptr : P->tensor_ptr(op.paths[1].src, N, ext_ptrs);
      A.yh = P->tensor_ptr(op.dst, N, ext_ptrs);
      A.yl = op.dst2 >= 0 ? P->tensor_ptr(op.dst2, N, ext_ptrs) : nullptr;
      const dim3 grid(A.tiles_x * ((A.H + A.TH - 1) / A.TH), 1, N);
      if (D.dtype == CSNET_F16) launch_il_t<__half>(A, grid, R.smem, stream);
      else launch_il_t<__nv_bfloat16>(A, grid, R.smem, stream);
      break;
    }
    case Route::DW_FAST:
    case Route::DW_GENERIC: {
      const csnet_path_desc& q = op.paths[0];
      const csnet_tensor_desc& S = P->tensors[q.src];
      csnet::DwArgs A{};
      A.src = P->tensor_ptr(q.src, N, ext_ptrs);
      A.dst = P->tensor_ptr(op.dst, N, ext_ptrs);
      A.w = P->blob + q.w_off;
      A.bias = op.bias_off >= 0 ? P->blob + op.bias_off : nullptr;
      A.slope = op.slope_off >= 0 ? P->blob + op.slope_off : nullptr;
      A.src_dtype = S.dtype; A.dst_dtype = D.dtype; A.C = D.C; A.H = D.H; A.W = D.W;
      if (R.route == Route::DW_FAST) {
        const int tasks = (D.W / 4) * ((D.H + csnet::kDwfRun - 1) / csnet::kDwfRun);
        dim3 grid((tasks + csnet::kDwfThreads - 1) / csnet::kDwfThreads, D.C, N);
        if (D.dtype == CSNET_F16) csnet::dw_fast_kernel<__half><<<grid, csnet::kDwfThreads, 0, stream>>>(A);
        else csnet::dw_fast_kernel<__nv_bfloat16><<<grid, csnet::kDwfThreads, 0, stream>>>(A);
      } else {
        const int strips = (D.H + csnet::kDwRows - 1) / csnet::kDwRows;
        dim3 grid((strips * D.W + kThreads - 1) / kThreads, D.C, N);
        dw_generic_kernel<<<grid, kThreads, 0, stream>>>(A);
      }
      break;
    }
  }
  CU_CHECK(cudaGetLastError());
  return CSNET_OK;
}

static int run_ops(csnet_plan* P, int32_t N, const void* const* ext_ptrs, cudaStream_t stream) {
  for (size_t i = 0; i < P->ops.size(); ++i) {
    const int rc = launch_op(P, i, N, ext_ptrs, stream);
    if (rc != CSNET_OK) return rc;
  }
  return CSNET_OK;
}

static void drop_graphs(csnet_plan* P) {
  for (auto& g : P->graphs) {
    if (g.exec) cudaGraphExecDestroy(g.exec);
    if (g.in) cudaFree(g.in);
    if (g.out) cudaFree(g.out);
    g = csnet_plan::GraphSlot();
  }
}

// Capture the op list for batch N into G.exec, over staging buffers allocated into G.
static int capture_graph(csnet_plan* P, int32_t N, csnet_plan::GraphSlot& G) {
  const csnet_tensor_desc *in = nullptr, *out = nullptr;
  for (const auto& d : P->tensors) {
    if (d.external == 0) in = &d;
    if (d.external == 1) out = &d;
  }
  G.in_bytes = (size_t)N * in->C * in->H * in->W * dtype_size(in->dtype);
  G.out_bytes = (size_t)N * out->C * out->H * out->W * dtype_size(out->dtype);
  CU_CHECK(cudaMalloc(&G.in, G.in_bytes));
  CU_CHECK(cudaMalloc(&G.out, G.out_bytes));
  const void* ext[2] = {G.in, G.out};
  cudaGraph_t graph = nullptr;
  // capture on a stream of our own: the caller's may be the legacy default stream, which cannot be captured
  if (!P->cap_stream) CU_CHECK(cudaStreamCreateWithFlags(&P->cap_stream, cudaStreamNonBlocking));
  CU_CHECK(cudaStreamBeginCapture(P->cap_stream, cudaStreamCaptureModeThreadLocal));
  const int rc = run_ops(P, N, ext, P->cap_stream);
  const cudaError_t e = cudaStreamEndCapture(P->cap_stream, &graph);
  if (rc != CSNET_OK || e != cudaSuccess || !graph) {
    if (graph) cudaGraphDestroy(graph);
    cudaGetLastError();
    return rc != CSNET_OK ? rc : fail(CSNET_E_CUDA, std::string("graph capture: ") + cudaGetErrorString(e));
  }
  const cudaError_t e2 = cudaGraphInstantiate(&G.exec, graph, 0);
  cudaGraphDestroy(graph);
  if (e2 != cudaSuccess) { G.exec = nullptr; return fail(CSNET_E_CUDA, std::string("cudaGraphInstantiate: ") + cudaGetErrorString(e2)); }
  return CSNET_OK;
}

// Small batches of a two-external plan (input, logits): copy the input into the plan's staging buffer, replay the captured
// graph, copy the logits out — three stream operations instead of one launch per op.
static int run_graph(csnet_plan* P, int32_t N, const void* const* ext_ptrs, cudaStream_t stream) {
  if ((int)P->graphs.size() <= N) P->graphs.resize((size_t)N + 1);
  csnet_plan::GraphSlot& G = P->graphs[N];
  if (!G.exec) {
    const int rc = capture_graph(P, N, G);
    if (rc != CSNET_OK) {                            // the slot stays empty; its staging buffers are not leaked
      if (G.in) cudaFree(G.in);
      if (G.out) cudaFree(G.out);
      G = csnet_plan::GraphSlot();
      return rc;
    }
  }
  CU_CHECK(cudaMemcpyAsync(G.in, ext_ptrs[0], G.in_bytes, cudaMemcpyDeviceToDevice, stream));
  CU_CHECK(cudaGraphLaunch(G.exec, stream));
  CU_CHECK(cudaMemcpyAsync(const_cast<void*>(ext_ptrs[1]), G.out, G.out_bytes, cudaMemcpyDeviceToDevice, stream));
  return CSNET_OK;
}

int csnet_plan_run(csnet_plan* P, int32_t N, const void* const* ext_ptrs, int32_t n_ext, void* stream_) {
  int rc = check_run_args(P, N, ext_ptrs, n_ext);
  if (rc != CSNET_OK) return rc;
  cudaStream_t stream = (cudaStream_t)stream_;
  DeviceGuard guard_(P->device);
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  if (N <= P->graph_max_n && P->n_ext == 2 && cudaStreamIsCapturing(stream, &cap) == cudaSuccess && cap == cudaStreamCaptureStatusNone)
    return run_graph(P, N, ext_ptrs, stream);
  return run_ops(P, N, ext_ptrs, stream);
}

int csnet_plan_profile(csnet_plan* P, int32_t N, const void* const* ext_ptrs, int32_t n_ext, void* stream_,
                       float* ms_per_op, int32_t n_ops) {
  int rc = check_run_args(P, N, ext_ptrs, n_ext);
  if (rc != CSNET_OK) return rc;
  if (!ms_per_op || n_ops != (int32_t)P->ops.size()) return fail(CSNET_E_INVALID, "csnet_plan_profile: n_ops mismatch");
  cudaStream_t stream = (cudaStream_t)stream_;
  DeviceGuard guard_(P->device);
  std::vector<cudaEvent_t> ev(P->ops.size() + 1);
  for (auto& e : ev) CU_CHECK(cudaEventCreate(&e));
  CU_CHECK(cudaEventRecord(ev[0], stream));
  for (size_t i = 0; i < P->ops.size() && rc == CSNET_OK; ++i) {
    rc = launch_op(P, i, N, ext_ptrs, stream);
    if (rc == CSNET_OK && cudaEventRecord(ev[i + 1], stream) != cudaSuccess) rc = fail(CSNET_E_CUDA, "cudaEventRecord");
  }
  cudaError_t e = cudaStreamSynchronize(stream);
  if (rc == CSNET_OK && e != cudaSuccess) rc = fail(CSNET_E_CUDA, std::string("sync: ") + cudaGetErrorString(e));
  if (rc == CSNET_OK)
    for (size_t i = 0; i < P->ops.size(); ++i) cudaEventElapsedTime(&ms_per_op[i], ev[i], ev[i + 1]);
  for (auto& e2 : ev) cudaEventDestroy(e2);
  return rc;
}

void* csnet_plan_tensor_ptr(csnet_plan* P, int32_t tensor, int32_t N) {
  if (!P || tensor < 0 || tensor >= (int)P->tensors.size() || N <= 0 || N > P->max_batch) return nullptr;
  if (P->tensors[tensor].external >= 0) return nullptr;
  return P->tensor_ptr(tensor, N, nullptr);
}

int csnet_plan_read_tensor(csnet_plan* P, int32_t tensor, int32_t N, void* dst, void* stream) {
  void* src = csnet_plan_tensor_ptr(P, tensor, N);
  if (!src || !dst) return fail(CSNET_E_INVALID, "csnet_plan_read_tensor: bad tensor / batch / destination");
  const csnet_tensor_desc& d = P->tensors[tensor];
  DeviceGuard guard_(P->device);
  CU_CHECK(cudaMemcpyAsync(dst, src, (size_t)N * d.C * d.H * d.W * dtype_size(d.dtype), cudaMemcpyDeviceToDevice,
                           (cudaStream_t)stream));
  return CSNET_OK;
}

const char* csnet_plan_op_kernel(const csnet_plan* P, int32_t i) {
  if (!P || i < 0 || i >= (int32_t)P->ops.size()) return "";
  return kRouteKernel[(int)P->routes[i].route];
}

int32_t csnet_plan_launches(const csnet_plan* P) {
  if (!P) return 0;
  int32_t n = 0;
  for (size_t i = 0; i < P->ops.size(); ++i) {
    const Route r = P->routes[i].route;
    n += r == Route::GN ? 2 : (r == Route::MSD ? P->ops[i].n_paths : 1);
  }
  return n;
}

int64_t csnet_plan_arena_bytes(const csnet_plan* P) { return P ? P->arena_per_image * (int64_t)P->max_batch : 0; }

void csnet_plan_destroy(csnet_plan* P) {
  if (!P) return;
  DeviceGuard guard_(P->device);
  drop_graphs(P);
  if (P->cap_stream) cudaStreamDestroy(P->cap_stream);
  if (P->blob) cudaFree(P->blob);
  if (P->arena) cudaFree(P->arena);
  if (P->gn_stats) cudaFree(P->gn_stats);
  for (const OpRoute& R : P->routes)
    for (uint16_t* q : R.w16)
      if (q) cudaFree(q);
  for (int b = 0; b < 2; ++b) {
    if (P->h_in[b]) cudaFree(P->h_in[b]);
    if (P->h_out[b]) cudaFree(P->h_out[b]);
    if (P->h_in8[b]) cudaFree(P->h_in8[b]);
    if (P->h_out8[b]) cudaFree(P->h_out8[b]);
    if (P->ev_h2d[b]) cudaEventDestroy(P->ev_h2d[b]);
    if (P->ev_comp[b]) cudaEventDestroy(P->ev_comp[b]);
    if (P->ev_d2h[b]) cudaEventDestroy(P->ev_d2h[b]);
  }
  if (P->s_h2d) cudaStreamDestroy(P->s_h2d);
  if (P->s_d2h) cudaStreamDestroy(P->s_d2h);
  delete P;
}

static int run_host_impl(csnet_plan* P, int32_t N, const void* x_host, void* y_host, void* stream_, bool u8, const float* mean, const float* stdv);

int csnet_plan_run_host(csnet_plan* P, int32_t N, const float* x_host, float* y_host, void* stream_) {
  return run_host_impl(P, N, x_host, y_host, stream_, false, nullptr, nullptr);
}

int csnet_plan_run_host_u8(csnet_plan* P, int32_t N, const uint8_t* x_hwc, uint8_t* y_u8, const float* mean, const float* stdv, void* stream_) {
  if (!mean || !stdv) return fail(CSNET_E_INVALID, "null mean / std");
  return run_host_impl(P, N, x_hwc, y_u8, stream_, true, mean, stdv);
}

// Chunks of a run_host batch.  fp32: a small first and last chunk (N/8 images) keep the exposed copies short — the first H2D
// and the last D2H are the only ones nothing overlaps — and one large middle chunk keeps the kernels at large-batch
// efficiency.  uint8: the copies are 4x smaller, so one chunk at full-batch kernel efficiency wins.  Batches under 64: one chunk.
static int host_chunks(int N, bool u8, int sizes[3]) {
  if (N < 64 || u8) {
    sizes[0] = N;
    return 1;
  }
  const int edge = N * 32 / 256;
  sizes[0] = edge; sizes[1] = N - 2 * edge; sizes[2] = edge;
  return 3;
}

static int run_host_impl(csnet_plan* P, int32_t N, const void* x_host, void* y_host, void* stream_, bool u8, const float* mean, const float* stdv) {
  if (!P || !x_host || !y_host) return fail(CSNET_E_INVALID, "null argument");
  if (N <= 0 || N > P->max_batch) return fail(CSNET_E_INVALID, "batch size outside [1, max_batch]");
  if (P->n_ext != 2) return fail(CSNET_E_INVALID, "run_host needs a plan with externals {0: input, 1: logits}");
  const csnet_tensor_desc *in = nullptr, *lo = nullptr;
  for (const auto& d : P->tensors) {
    if (d.external == 0) in = &d;
    if (d.external == 1) lo = &d;
  }
  if (!in || !lo || in->dtype != CSNET_F32 || lo->dtype != CSNET_F32)
    return fail(CSNET_E_INVALID, "run_host: externals must be fp32");
  cudaStream_t stream = (cudaStream_t)stream_;
  DeviceGuard guard_(P->device);
  // The batch is cut into chunks that flow through a three-stage pipeline: H2D copy (own stream) -> program
  // (caller's stream) -> D2H copy (own stream), with ping-pong device staging, so the PCIe copies of chunk i+1 / i-1
  // overlap the kernels of chunk i.  Pinned host memory is needed for the copies to be truly asynchronous.
  int sizes[3], n_sizes = host_chunks(N, u8, sizes);
  int chunk = 0;
  for (int i = 0; i < n_sizes; ++i) chunk = sizes[i] > chunk ? sizes[i] : chunk;
  const size_t xin = (size_t)in->C * in->H * in->W * sizeof(float), yout = (size_t)lo->C * lo->H * lo->W * sizeof(float);
  if (!P->s_h2d) {
    CU_CHECK(cudaStreamCreateWithFlags(&P->s_h2d, cudaStreamNonBlocking));
    CU_CHECK(cudaStreamCreateWithFlags(&P->s_d2h, cudaStreamNonBlocking));
    for (int b = 0; b < 2; ++b) {
      CU_CHECK(cudaEventCreateWithFlags(&P->ev_h2d[b], cudaEventDisableTiming));
      CU_CHECK(cudaEventCreateWithFlags(&P->ev_comp[b], cudaEventDisableTiming));
      CU_CHECK(cudaEventCreateWithFlags(&P->ev_d2h[b], cudaEventDisableTiming));
    }
  }
  if (P->h_in_bytes < (size_t)chunk * xin) {
    for (int b = 0; b < 2; ++b) {
      if (P->h_in[b]) cudaFree(P->h_in[b]);
      if (P->h_out[b]) cudaFree(P->h_out[b]);
      CU_CHECK(cudaMalloc(&P->h_in[b], (size_t)chunk * xin));
      CU_CHECK(cudaMalloc(&P->h_out[b], (size_t)chunk * yout));
    }
    P->h_in_bytes = (size_t)chunk * xin;
    P->h_out_bytes = (size_t)chunk * yout;
  }
  const size_t xin8 = xin / sizeof(float), yout8 = yout / sizeof(float);      // bytes per image of the uint8 forms
  if (u8 && P->h_in8_bytes < (size_t)chunk * xin8) {
    for (int b = 0; b < 2; ++b) {
      if (P->h_in8[b]) cudaFree(P->h_in8[b]);
      if (P->h_out8[b]) cudaFree(P->h_out8[b]);
      CU_CHECK(cudaMalloc(&P->h_in8[b], (size_t)chunk * xin8));
      CU_CHECK(cudaMalloc(&P->h_out8[b], (size_t)chunk * yout8));
    }
    P->h_in8_bytes = (size_t)chunk * xin8;
  }
  if (u8 && in->C != 3) return fail(CSNET_E_INVALID, "run_host_u8: the network input must have 3 channels");
  PreArgs PA{};
  if (u8) for (int c = 0; c < 3; ++c) { PA.mean[c] = (double)mean[c]; PA.std[c] = (double)stdv[c]; }
  int rc = CSNET_OK;
  for (int it = 0, n0 = 0; it < n_sizes && rc == CSNET_OK; n0 += sizes[it], ++it) {
    const int b = it & 1, nb = sizes[it];
    if (it >= 2) CU_CHECK(cudaStreamWaitEvent(P->s_h2d, P->ev_comp[b], 0));     // staging input b was consumed
    if (u8) CU_CHECK(cudaMemcpyAsync(P->h_in8[b], (const uint8_t*)x_host + (size_t)n0 * xin8, (size_t)nb * xin8, cudaMemcpyHostToDevice, P->s_h2d));
    else CU_CHECK(cudaMemcpyAsync(P->h_in[b], (const float*)x_host + (size_t)n0 * (xin / sizeof(float)), (size_t)nb * xin, cudaMemcpyHostToDevice, P->s_h2d));
    CU_CHECK(cudaEventRecord(P->ev_h2d[b], P->s_h2d));
    CU_CHECK(cudaStreamWaitEvent(stream, P->ev_h2d[b], 0));
    if (it >= 2) CU_CHECK(cudaStreamWaitEvent(stream, P->ev_d2h[b], 0));         // staging output b was drained
    if (u8) {
      const int64_t npix = (int64_t)nb * in->H * in->W;
      pre_u8_kernel<<<(unsigned)((npix + kThreads - 1) / kThreads), kThreads, 0, stream>>>((const uint8_t*)P->h_in8[b], (float*)P->h_in[b], npix, (int64_t)in->H * in->W, PA);
    }
    const void* ext[2] = {P->h_in[b], P->h_out[b]};
    rc = run_ops(P, nb, ext, stream);               // (its own staging: no graph path)
    if (rc != CSNET_OK) break;
    if (u8) {
      const int64_t nel = (int64_t)nb * lo->C * lo->H * lo->W;
      post_u8_kernel<<<(unsigned)((nel / 4 + kThreads - 1) / kThreads), kThreads, 0, stream>>>((const float*)P->h_out[b], (uint8_t*)P->h_out8[b], nel);
    }
    CU_CHECK(cudaEventRecord(P->ev_comp[b], stream));
    CU_CHECK(cudaStreamWaitEvent(P->s_d2h, P->ev_comp[b], 0));
    if (u8) CU_CHECK(cudaMemcpyAsync((uint8_t*)y_host + (size_t)n0 * yout8, P->h_out8[b], (size_t)nb * yout8, cudaMemcpyDeviceToHost, P->s_d2h));
    else CU_CHECK(cudaMemcpyAsync((float*)y_host + (size_t)n0 * (yout / sizeof(float)), P->h_out[b], (size_t)nb * yout, cudaMemcpyDeviceToHost, P->s_d2h));
    CU_CHECK(cudaEventRecord(P->ev_d2h[b], P->s_d2h));
  }
  cudaError_t e1 = cudaStreamSynchronize(P->s_d2h), e2 = cudaStreamSynchronize(stream), e3 = cudaStreamSynchronize(P->s_h2d);
  if (rc == CSNET_OK && (e1 != cudaSuccess || e2 != cudaSuccess || e3 != cudaSuccess))
    rc = fail(CSNET_E_CUDA, std::string("run_host sync: ") + cudaGetErrorString(e1 != cudaSuccess ? e1 : (e2 != cudaSuccess ? e2 : e3)));
  return rc;
}

}  // extern "C"
