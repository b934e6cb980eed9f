/*
 * csnet_b200.h — C ABI of libcsnet_b200.so, the B200 (sm_100a) CSNet forward/backward engine.
 *
 * The reference (ShangHua-Gao/SOD100K) has no FFI of its own: its hot path is Python calling
 * torch.nn.functional (ATen/cuDNN).  This header is the boundary a maintainer would bind instead of
 * those library calls; every entry point names the reference call site it replaces.  All arguments
 * are plain pointers and sizes; device pointers are raw CUdeviceptr-compatible addresses; `stream`
 * is a cudaStream_t passed as void*.  No torch types cross this boundary.
 *
 * Execution model: the host side (sod100k_b200/compiler.py, mirroring the reference's module tree
 * CSNet/model/csnet.py) lowers a CSNet `layer_config` + `state_dict` into a flat PROGRAM: a tensor
 * table, a list of fused ops and one fp32 parameter blob.  A plan owns the blob copy and the
 * activation arena on one device and replays the program for a batch.
 *
 * Data layout in HBM: activations are planar NCHW (batch stride C*H*W, plane stride H*W, row
 * stride W, all dense), element type per tensor (fp32 / fp16 / bf16).  Channel counts are never
 * padded (CSNet widths are 8..79 and differ per layer), so algorithmic bytes == allocated bytes.
 *
 * Errors: every function returns 0 on success or a negative CSNET_E_* code; csnet_last_error()
 * returns a thread-local message.  The reference's own convention is Python exceptions
 * (CSNet/test.py:24 `assert`); the Python wrapper turns non-zero codes into RuntimeError.
 * Threading: a plan is used by one host thread / one stream at a time; no global mutable state.
 * Ownership: the caller owns inputs, outputs and parameters; the plan owns its blob copy + arena.
 */
#ifndef CSNET_B200_H
#define CSNET_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define CSNET_ABI_VERSION 5

enum { CSNET_F32 = 0, CSNET_F16 = 1, CSNET_BF16 = 2 };

enum {
  CSNET_OK = 0,
  CSNET_E_INVALID = -1,   /* malformed program / argument */
  CSNET_E_CUDA = -2,      /* CUDA runtime error (message holds cudaGetErrorString) */
  CSNET_E_NOMEM = -3,
  CSNET_E_UNSUPPORTED = -4
};

#define CSNET_MAX_PATHS 8
#define CSNET_MAX_EXT 24
/* ext_off slot of CSNET_OP_MIX / CSNET_OP_DW: 1 keeps the op on the generic kernels (no fast kernel) */
#define CSNET_EXT_NO_FAST 23

/* One activation tensor of the program (per image: [C,H,W]; a run adds the batch dimension). */
typedef struct {
  int32_t C, H, W;
  int32_t dtype;          /* CSNET_F32 / F16 / BF16 */
  int32_t external;       /* >= 0: bound at run time to ext_ptrs[external]; -1: lives in the arena */
  int32_t _pad;
  int64_t arena_offset;   /* bytes PER IMAGE from the arena base (multiple of 256); the run address is
                             base + N * arena_offset, so tensors of a smaller batch stay disjoint */
} csnet_tensor_desc;

/*
 * One accumulation path of a MIX op.  out[cout0 : cout0+cout] += path(src[c0 : c0+cin]).
 *
 * ksize > 0 — convolution path, replaces the F.conv2d calls of gOctaveConv.forward
 *   (CSNet/model/csnet.py:702-717), Conv2dX100.forward (CSNet/model/conv2d.py:104) and
 *   MSBlock.forward (csnet.py:141-146), with the resampling the reference does around them folded
 *   into the read: pre_avg=f (1 means 2) down-samples by f first — avg_pool2d(2,2) for f=2 (csnet.py:679-680) and
 *   F.interpolate(bilinear) to 1/f size for f=2,4,8 (CSF+Res2Net/networks/gOctConv.py:101-102) —, pool=k applies
 *   max_pool2d(k,k) next (csnet.py:709-712); the convolution (cross-correlation, zero padding `pad`,
 *   dilation `dil`, stride `stride`) then runs on that pooled grid.
 *   A plain 1x1 conv path may carry up > 1: the source is bilinearly up-sampled FIRST (same linear map as the
 *   reference's conv-then-interpolate; used by 16-bit programs when cin <= cout).
 * ksize == 0 — resample-add path: channel c of src is bilinearly up-sampled by the integer factor
 *   `up` (align_corners=False, source index (dst+0.5)/up-0.5 clamped at 0 — F.interpolate at
 *   csnet.py:705-707 and :382-385) and added to out[cout0+c]; cin == cout.
 */
typedef struct {
  int32_t src;            /* tensor id */
  int32_t c0, cin;
  int32_t pre_avg, pool;
  int32_t ksize, dil, stride, pad;
  int32_t up;
  int32_t cout0, cout;
  int64_t w_off;          /* blob offset (floats) of weights laid out [cin][ksize*ksize][cout] (cout innermost,
                             the compiler transposes the reference's [cout][cin][k][k]); -1 if ksize==0 */
} csnet_path_desc;

enum {
  CSNET_OP_MIX = 1,       /* dst = prelu(sum_paths + bias)   — gOctaveCBR / MSBlock / cls_layer */
  CSNET_OP_DW = 2,        /* dst = prelu(dw3x3(src) + bias)  — SimplifiedGOctConvBR branch */
  CSNET_OP_GN = 4,        /* dst = prelu(GroupNorm(src)): per-image statistics over (C/groups, H, W), eps 1e-5 — the CSF+Res2Net
                             head (CSF+Res2Net/networks/gOctConv.py:133, csf_res2net.py:220).  paths[0].src = input,
                             paths[0].up = groups, ext_off[0] / ext_off[1] = gamma / beta, slope_off = PReLU slope. */
  CSNET_OP_ILBLOCK = 3,   /* whole ILBlock of the 1x1 kind in one kernel (ILBlock.forward, csnet.py:72-76):
                             paths[0].src / paths[1].src = high / low resolution inputs (cin = channels),
                             dst / dst2 = high / low resolution outputs (dst2 = -1 for a 2->1 block);
                             16-bit activations only.  ext_off[] (blob offsets, floats):
                               0 WH  packed 16-bit [ru16(Cho)][K8], K8 = ru8(Chi+Cli): columns [W_hh | W_lh]
                                     (the kernel up-samples x_l before the conv: same linear map), BN scale folded
                               1 WL  packed 16-bit [ru16(Clo)][K8]: columns [W_ll | W_hl] (x_l, then max-pooled x_h)
                               2,3   conv bias / PReLU slope of the hi branch      4,5  of the lo branch
                               6-8   conv3x3_1 hi: weights [C][9], bias, slope     9-11 conv3x3_1 lo
                               12-14 conv3x3_2 hi                                  15-17 conv3x3_2 lo
                             Stem form (the first block, `first=True`, csnet.py:60-71): paths[0] and paths[1] both name
                             the fp32 input image (cin <= 3) with ksize = 3, pad = 1, paths[1].pool = 2; both branches are
                             3x3 convs of it (lo: of its 2x2 max-pool).  WH / WL are then [ru16(C)][32] with column
                             k = ci*9 + ky*3 + kx; the kernel builds the im2col planes in shared memory. */
  CSNET_OP_MIXPROJ = 5     /* a MIX op whose Cmid-channel result is never stored: a 1x1 projection to the single dst channel
                             runs in the epilogue, dst = proj_b + sum_c proj_w[c] * prelu(mix[c] + bias[c])  (CSNet.forward,
                             csnet.py:383-384: fuse1x1 -> cls_layer).  paths / bias_off / slope_off describe the Cmid-channel
                             MIX; ext_off[0] = proj_w offset (Cmid floats), ext_off[1] = proj_b offset or -1,
                             ext_off[2] = Cmid (<= 80).  Tensor-core kernel only: 16-bit sources, stride-1 conv paths. */
};

/*
 * One fused op.  Epilogue (both kinds): y = acc + bias[c] (bias_off >= 0), then PReLU with
 * per-channel slope (slope_off >= 0): y > 0 ? y : slope[c]*y  (F.batch_norm + F.prelu,
 * csnet.py:786,791,846-847,148; eval-mode BN scale is folded into the weights by the compiler).
 * CSNET_OP_DW uses paths[0] with ksize=3, dil=1, pad=1, cin==cout, weights [C][9]
 * (Conv2dX100 groups=C, csnet.py:817-824).
 */
typedef struct {
  int32_t kind;
  int32_t dst;            /* tensor id */
  int32_t n_paths;
  int32_t dst2;           /* second destination (CSNET_OP_ILBLOCK) or -1 */
  int64_t bias_off;       /* blob offset of bias[dst.C] or -1 */
  int64_t slope_off;      /* blob offset of PReLU slope[dst.C] or -1 */
  csnet_path_desc paths[CSNET_MAX_PATHS];
  int64_t ext_off[CSNET_MAX_EXT];   /* kind-specific blob offsets, -1 when unused.  CSNET_OP_MIX / CSNET_OP_DW:
                                       ext_off[CSNET_EXT_NO_FAST] == 1 forbids the fast kernels (not requested, or the
                                       weights do not fit the 16-bit operand type) */
} csnet_op_desc;

typedef struct csnet_plan csnet_plan;

/* ABI version of the loaded library (== CSNET_ABI_VERSION of the header it was built from). */
int csnet_abi_version(void);

/* Thread-local description of the last error returned on this thread ("" if none). */
const char* csnet_last_error(void);

/* Number of CUDA devices visible; < 0 on error.  Used by the wrapper to fail loudly without a GPU. */
int csnet_device_count(void);

/*
 * Build a plan on `device` for batches up to `max_batch`.  Validates the program (shapes of every
 * path against its destination, blob bounds) and allocates blob + arena.
 * Replaces: model construction + `.cuda()` (CSNet/test.py:39-40, CSNet_training/train.py:77-92).
 */
int csnet_plan_create(csnet_plan** out, const csnet_tensor_desc* tensors, int32_t n_tensors,
                      const csnet_op_desc* ops, int32_t n_ops, int64_t blob_floats,
                      int32_t max_batch, int32_t device);

/* Upload the fp32 parameter blob (host pointer, `n` floats == blob_floats) on `stream`.
 * Replaces: load_state_dict + per-call `100.0 * weight` / BN arithmetic (conv2d.py:104, csnet.py:786). */
int csnet_plan_set_blob(csnet_plan* plan, const float* host_blob, int64_t n, void* stream);

/*
 * Run the program for a batch of N images.  ext_ptrs[i] is the DEVICE address bound to tensors with
 * external == i (network input fp32 NCHW, logits fp32 NCHW, ...).  Asynchronous on `stream`.
 * Replaces: CSNet.forward (CSNet/model/csnet.py:365-387) == `model(input_var)` at CSNet/test.py:90.
 */
int csnet_plan_run(csnet_plan* plan, int32_t N, const void* const* ext_ptrs, int32_t n_ext, void* stream);

/*
 * Same as csnet_plan_run, but records a CUDA event on `stream` around every op and writes each op's device
 * time in milliseconds to ms_per_op[n_ops] (synchronises the stream).  Measurement aid for bench.py's roofline.
 */
int csnet_plan_profile(csnet_plan* plan, int32_t N, const void* const* ext_ptrs, int32_t n_ext, void* stream,
                       float* ms_per_op, int32_t n_ops);

/* Device address of an arena tensor for a batch of N (for tests / taps); NULL if external/invalid. */
void* csnet_plan_tensor_ptr(csnet_plan* plan, int32_t tensor, int32_t N);

/* Copy an arena tensor of the last run of batch N into caller-owned DEVICE memory (same dtype, dense). */
int csnet_plan_read_tensor(csnet_plan* plan, int32_t tensor, int32_t N, void* dst_device, void* stream);

/* Name of the kernel (family) csnet_plan_run launches for op `op_index` of this plan — measurement aid: bench.py groups the per-op
 * times of csnet_plan_profile by kernel to find the dominant one.  "" for an invalid index. */
const char* csnet_plan_op_kernel(const csnet_plan* plan, int32_t op_index);

/* Number of kernel launches one csnet_plan_run issues (bench.py reports it as gpu_launches). */
int32_t csnet_plan_launches(const csnet_plan* plan);

/* Bytes of arena the plan holds. */
int64_t csnet_plan_arena_bytes(const csnet_plan* plan);

void csnet_plan_destroy(csnet_plan* plan);

/*
 * Convenience for hosts that keep their data in pageable/pinned HOST memory (the e2e path of
 * bench.py and of CSNet/test.py:86-93): copies x (fp32 NCHW, N*3*H*W floats) to the device, runs,
 * copies the logits (N*H*W floats) back and returns when y_host is complete.  Batches of 64 or more are cut into
 * three chunks (N/8, the rest, N/8) that pipeline H2D copy / kernels / D2H copy on separate streams (use pinned host memory).
 * The plan must bind external 0 = input, external 1 = logits.
 */
int csnet_plan_run_host(csnet_plan* plan, int32_t N, const float* x_host, float* y_host, void* stream);

/*
 * Same pipeline with the reference's pre- and post-processing moved onto the device (CSNet/test.py:68-69,86-96; SURVEY §8 f3):
 * x_hwc = uint8 [N][H][W][3] images as io.imread returns them (already at the network size), y_u8 = uint8 [N][H][W] saliency maps
 * = (sigmoid(logits) * 255) truncated, exactly what test.py writes to png.  The input becomes (x / 255 - mean[c]) / std[c]
 * (evaluated in float64, rounded to fp32, like the host code).  4x fewer bytes over PCIe in both directions.
 */
int csnet_plan_run_host_u8(csnet_plan* plan, int32_t N, const uint8_t* x_hwc, uint8_t* y_u8, const float* mean, const float* std,
                           void* stream);

/* ------------------------------------------------------------------------------------------------------------
 * Training primitives (fp32 planar NCHW device tensors).  The reference trains through torch autograd
 * (CSNet_training/train.py:203-216); train-mode BatchNorm makes the reference MODULE the closed unit, so the
 * boundary is one call per module piece.  sod100k_b200/train_ops.py wraps them in torch.autograd.Function s.
 * All return 0 / CSNET_E_*; csnet_train_last_error() holds the message.
 * ------------------------------------------------------------------------------------------------------------ */

/* One path of a raw (pre-BN) conv mix, device pointers resolved.  Same semantics as csnet_path_desc; `w` is the
 * path's weight in kernel layout [cin][ksize*ksize][cout] (fp32), NULL for resample-add paths (ksize == 0). */
typedef struct {
  const void* src;        /* fp32 [N, C, H, W] */
  const float* w;
  int32_t C, H, W;
  int32_t c0, cin;
  int32_t pre_avg, pool;
  int32_t ksize, dil, stride, pad;
  int32_t up;
  int32_t cout0, cout;
} csnet_train_path;

const char* csnet_train_last_error(void);

/* F.batch_norm(training=True) statistics: per-channel mean and BIASED variance over (N, H*W)  (csnet.py:786,846). */
int csnet_train_bn_stats(const float* z, int32_t N, int32_t C, int32_t HW, float* mean, float* var, void* stream);
/* y = PReLU(gamma*(z-mean)/sqrt(var+eps)+beta); gap (optional, [N*C]) = per-image channel means of y, the quantity
 * Oct_bn_hook pools (csnet.py:403-404). */
int csnet_train_bn_prelu_fwd(const float* z, float* y, int32_t N, int32_t C, int32_t HW, const float* mean, const float* var,
                             const float* gamma, const float* beta, const float* slope, float eps, float* gap, void* stream);
/* autograd of the above: dz plus dgamma / dbeta / dslope ([C] each).  frozen=1: mean / var were constants (eval-mode
 * BatchNorm inside a training graph, as CSF+Res2Net/solver.py keeps its net), so the batch-statistic terms vanish. */
int csnet_train_bn_prelu_bwd(const float* z, const float* dy, float* dz, int32_t N, int32_t C, int32_t HW, const float* mean,
                             const float* var, const float* gamma, const float* beta, const float* slope, float eps,
                             float* dgamma, float* dbeta, float* dslope, int32_t frozen, void* stream);
/* Depthwise 3x3 pad 1 with effective weight scale*w (Conv2dX100, conv2d.py:104); transposed=1 gives the data gradient. */
int csnet_train_dw_conv(const float* x, const float* w, float* y, int32_t N, int32_t C, int32_t H, int32_t W, float scale,
                        int32_t transposed, void* stream);
int csnet_train_dw_wgrad(const float* x, const float* dy, float* dw, int32_t N, int32_t C, int32_t H, int32_t W, float scale,
                         void* stream);
/* Both gradients of the depthwise conv in one pass over dy (autograd of F.conv2d(x, 100 * w, groups=C), conv2d.py:104): dx [N,C,H,W], dw [C][9]. */
int csnet_train_dw_bwd(const float* x, const float* dy, const float* w, float* dx, float* dw, int32_t N, int32_t C, int32_t H, int32_t W,
                       float scale, void* stream);
/* Raw conv mix (gOctaveConv.forward csnet.py:664-726 for one output branch; MSBlock :141-146): dst = sum of paths. */
int csnet_train_mix_fwd(float* dst, int32_t N, int32_t C, int32_t H, int32_t W, const csnet_train_path* paths, int32_t n_paths,
                        void* stream);
/* Gradient of one path w.r.t. its source slice: dsrc is [N, cin, path.H, path.W] (through max/avg pooling, the conv,
 * or the bilinear up-sample for resample paths). */
int csnet_train_mix_dgrad(const float* ddst, int32_t N, int32_t C, int32_t H, int32_t W, const csnet_train_path* path, float* dsrc,
                          void* stream);
/* Gradient of one conv path w.r.t. its weight, kernel layout [cin][k*k][cout]. */
int csnet_train_mix_wgrad(const float* ddst, int32_t N, int32_t C, int32_t H, int32_t W, const csnet_train_path* path, float* dw,
                          void* stream);
/* The down-sampling a path carries, materialised once (F.avg_pool2d(2) of a stride-2 gOctaveConv, csnet.py:683-686, then F.max_pool2d(pool)
 * of a high -> low path, :692-698): dst [N, cin, Hs/f, Ws/f] from channels [c0, c0+cin) of src [N, Cs, Hs, Ws], f = (pre_avg ? 2 : 1) * pool;
 * idx (uint8, same shape, required when pool > 1) = position of the first maximum in the window.  _bwd routes the gradient of dst back to
 * dsrc [N, cin, Hs, Ws] the way autograd does (max: to the recorded position; average: a quarter to each). */
int csnet_train_pool_fwd(const float* src, int32_t N, int32_t Cs, int32_t c0, int32_t cin, int32_t Hs, int32_t Ws, int32_t pre_avg, int32_t pool,
                         float* dst, uint8_t* idx, void* stream);
int csnet_train_pool_bwd(const float* dpool, const uint8_t* idx, int32_t N, int32_t cin, int32_t Hs, int32_t Ws, int32_t pre_avg, int32_t pool,
                         float* dsrc, void* stream);
/* Channel slimming on the device (SURVEY 8 f4; build_model_with_weight and its loaders, CSNet_training/model/csnet.py:571-818):
 * dst[i][j][:] = src[out_idx[i]][in_idx[j]][:] for i < n_out, j < n_in; src is [Co][Ci][kk] fp32, dst [dCo][dCi][kk] (the caller zeroes it:
 * the reference fills torch.zeros), the index lists are device int64 (torch.nonzero of the BatchNorm-gamma masks). */
int csnet_slim_gather(const float* src, int32_t Co, int32_t Ci, int32_t kk, const int64_t* out_idx, int32_t n_out, const int64_t* in_idx, int32_t n_in,
                      float* dst, int32_t dCo, int32_t dCi, void* stream);
/* F.binary_cross_entropy_with_logits (mean) and its gradient * grad_scale (train.py:209). */
int csnet_train_bce(const float* logits, const float* target, float* dlogits, float* loss, int64_t n, float grad_scale, void* stream);
/* torch.optim.Adam step (train.py:108-123) over many tensors: `chunk_table_device` = n_chunks records
 * {float* p; const float* g; float* m; float* v; int32 n; float weight_decay} (40 bytes each). */
int csnet_train_adam(const void* chunk_table_device, int32_t n_chunks, float lr, float beta1, float beta2, float eps, int32_t step,
                     float grad_scale, void* stream);

/* ---- evaluation: the counting part of SalMetric on the device (CSNet_training/SalMetric/src/sal_metric.cpp:86-120) ----
 * prob: device float32 [N][HW] saliency in [0,1] (after sigmoid); gt: device uint8 [N][HW] ground truth.  Per image:
 * q = (uint8)(prob * 255) (CSNet/test.py:94-96), hist_all[q]++, hist_pos[q]++ where gt > 128, abs_sum += |q - gt|.
 * hist_all / hist_pos: device uint32 [N][256], abs_sum: device uint64 [N]; all three are zeroed by the call.  The caller
 * turns them into precision / recall per threshold (suffix sums), F-measure and MAE (sod100k_b200/salmetric.py). */
int csnet_salmetric_hist(const float* prob, const uint8_t* gt, int32_t N, int64_t HW, uint32_t* hist_all, uint32_t* hist_pos,
                         unsigned long long* abs_sum, void* stream);

#ifdef __cplusplus
}
#endif
#endif /* CSNET_B200_H */
