"""Lower a CSNet (layer_config + parameters) to the engine's program IR.

Host-side mirror of the reference's module tree: the walk below visits exactly the modules that
`CSNet.__init__` builds (CSNet/model/csnet.py:209-311) and emits, for each reference module call, the
fused op(s) that replace it:

    gOctaveCBR   (csnet.py:729-792)  -> one MIX op per output branch (+ one raw low-res MIX per up path)
    SimplifiedGOctConvBR (:795-851)  -> one DW op per branch
    MSBlock      (:116-149)          -> one MIX op with a conv path per live dilation (concat = cout0 offsets)
    cls_layer + F.interpolate (:381-385) -> MIX (1x1 + bias, at H/2) then MIX (resample x2, fp32 logits)

Eval-mode folding done here, once per weight update, instead of per call in the reference:
  * BatchNorm (running stats, eps 1e-5): y = s*x + t with s = gamma/sqrt(var+eps), t = beta - mean*s;
    s is multiplied into the conv weights (bilinear resampling is linear with weights summing to 1 and
    max/avg pooling happen before the conv, so s commutes with every path); t becomes the op bias.
  * the `100.0 * weight` of Conv2dX100 (CSNet/model/conv2d.py:104) is multiplied into dw / dilated /
    single-branch conv weights.
"""
from __future__ import annotations

from typing import Dict, List, Mapping, Optional

import numpy as np

from . import ir, splits

BN_EPS = 1e-5


def to_bits16(a: np.ndarray, dtype: int) -> np.ndarray:
    """float array -> raw fp16 / bf16 bit patterns (round to nearest even)."""
    a = np.ascontiguousarray(a, np.float32)
    if dtype == ir.F16:
        return a.astype(np.float16).view(np.uint16)
    u = a.view(np.uint32).astype(np.uint64)
    u = (u + 0x7FFF + ((u >> 16) & 1)) >> 16
    return u.astype(np.uint16)


def _ru(v: int, m: int) -> int:
    return (v + m - 1) // m * m


def _padded_region(n: int) -> int:
    n = _ru(n, 8)
    return n + 8 if (n // 8) % 2 == 0 else n


def il_block_fits(Chi, Cli, Cho, Clo) -> bool:
    """Mirror of make_il() in csrc/plan.cu: K = Chi + Cli must fit the register-resident B fragments (<= 64) and the
    smallest candidate tile (8 x 16) must fit 227 KB of shared memory."""
    K8, MH16, ML16 = _ru(Chi + Cli, 8), _ru(Cho, 16), (_ru(Clo, 16) if Clo else 0)
    if K8 > 64:
        return False
    TH, TW = 8, 16
    NPH, NPL = ((TH + 8) | 1) * (TW + 8), ((TH // 2 + 4) | 1) * (TW // 2 + 8)
    rows_l = max(K8, Clo) if Clo else Cli
    halves = max(K8, Cho) * NPH + Cho * NPH + rows_l * NPL + Clo * NPL + MH16 * K8 + ML16 * K8
    return halves * 2 + 512 <= 227 * 1024


def upsample_input_side(cin: int, cout: int, up: int) -> bool:
    """A 1x1 up path can up-sample its INPUT (conv at the high resolution over cin channels, cin bilinear evaluations per
    output pixel at staging) or its OUTPUT (the reference's order: conv at the low resolution, cout bilinear evaluations per
    output pixel in the epilogue).  Cost model in issued-instruction equivalents per output pixel: a MAC on the tensor-core
    path ~0.16, a staged bilinear evaluation ~30, an epilogue one ~20.  Narrow layers (CSNet: 24 -> 79) win on the input
    side; wide ones (CSF+Res2Net: 256 -> 1408) must keep the conv at the low resolution."""
    cost_in = 0.16 * cin * cout + 30.0 * cin
    cost_out = 0.16 * cin * cout / (up * up) + 20.0 * cout
    return cost_in < cost_out


def _np(v) -> np.ndarray:
    if hasattr(v, "detach"):
        v = v.detach().cpu().numpy()
    return np.asarray(v)


class _Lowering:
    def __init__(self, layer_config, params: Mapping[str, object], H: int, W: int, act_dtype: int, fuse=True,
                 tensor_core=True, upsample_inputs=None):
        if H % 16 or W % 16:
            # the reference's own callers enforce this (CSNet/test.py:80-85); its branch sums fail otherwise
            raise ValueError(f"input size {H}x{W} must be a multiple of 16")
        self.cfg = layer_config
        self.P = params
        self.H, self.W = H, W
        self.dt = act_dtype
        # fuse: True / False, or a collection of block prefixes to fuse (tests isolate one block that way)
        self.fuse = fuse if act_dtype in (ir.F16, ir.BF16) else False
        self.tensor_core = tensor_core       # True / False / collection of op-name prefixes allowed on the fast kernels
        # 1x1 up-paths with cin <= cout: up-sample the conv input instead of its output (default: 16-bit programs)
        self.upsample_inputs = (act_dtype != ir.F32) if upsample_inputs is None else upsample_inputs
        self._pooled: Dict[tuple, int] = {}            # (source tensor, factor) -> materialised max-pooled tensor
        self.b = ir.Builder()
        self._wmax: Dict[int, float] = {}

    def finalize_flags(self, prog: ir.Program):
        """Keep MIX and DW ops off the fast kernels when they are not requested, and MIX ops whose folded weights do not fit
        the 16-bit operand type."""
        lim = 6.0e4 if self.dt == ir.F16 else 3.0e38
        ir.veto_fast_kernels(prog.ops, self.tensor_core, (ir.OP_MIX, ir.OP_DW),
                             lambda o: o.kind == ir.OP_MIX and any(self._wmax.get(q.w_off, 0.0) >= lim for q in o.paths if q.ksize > 0))

    # ---- parameters -----------------------------------------------------------------------------
    def p(self, key: str) -> np.ndarray:
        if key not in self.P:
            raise KeyError(f"missing parameter '{key}' (state_dict does not match layer_config)")
        return _np(self.P[key]).astype(np.float64)

    def bn_fold(self, prefix: str):
        s = self.p(prefix + ".weight") / np.sqrt(self.p(prefix + ".running_var") + BN_EPS)
        t = self.p(prefix + ".bias") - self.p(prefix + ".running_mean") * s
        return s, t

    def conv_w(self, w: np.ndarray) -> int:
        """[cout][cin][k][k] -> blob layout [cin][k*k][cout]."""
        co, ci, kh, kw = w.shape
        off = self.b.param(np.transpose(w.reshape(co, ci, kh * kw), (1, 2, 0)))
        self._wmax[off] = float(np.abs(w).max()) if w.size else 0.0
        return off

    def dims(self, t: int):
        d = self.b.prog.tensors[t]
        return d.C, d.H, d.W

    # ---- modules --------------------------------------------------------------------------------
    def goct_cbr(self, prefix: str, xs: List[Optional[int]], a_in, a_out, ksize: int, stride: int):
        """gOctaveCBR.forward (csnet.py:778-792) incl. gOctaveConv.forward (:664-726)."""
        W4 = self.p(prefix + ".conv.weight")
        cout_t, cin_t = W4.shape[0], W4.shape[1]
        pad = 1 if ksize == 3 else 0
        if len(a_in) == 1 and len(a_out) == 1:                      # plain Conv2dX100 (csnet.py:751-754)
            s, t = self.bn_fold(prefix + ".bns.0")
            C_, H_, W_ = self.dims(xs[0])
            Ho, Wo = (H_ + 2 * pad - ksize) // stride + 1, (W_ + 2 * pad - ksize) // stride + 1
            dst = self.b.tensor(cout_t, Ho, Wo, self.dt, name=prefix + "/0")
            path = ir.Path(xs[0], cin_t, cout_t, ksize=ksize, pad=pad, stride=stride,
                           w_off=self.conv_w(100.0 * W4 * s[:, None, None, None]))
            self.b.op(ir.OP_MIX, dst, [path], bias=t, slope=self.p(prefix + ".prelus.0.weight"), name=prefix)
            return [dst]
        ci, co = splits.cuts(cin_t, a_in), splits.cuts(cout_t, a_out)
        pool_once = self.dt != ir.F32 and (self.fuse is True or bool(self.fuse and prefix in self.fuse))
        if stride == 2 and pool_once:
            # gOctaveConv's stride 2 is avg_pool2d(2, 2) of every input branch followed by a stride-1 conv (:679-680).
            # 16-bit programs materialise the pooled branches once (one bandwidth-bound pass) instead of averaging in the
            # staging loop of each of the 2-3 conv ops that read them; the stored value is the one they would stage.
            pooled: List[Optional[int]] = []
            for i, x in enumerate(xs):
                if x is None or ci[i] == ci[i + 1]:
                    pooled.append(x)
                    continue
                C_, H_, W_ = self.dims(x)
                t = self.b.tensor(C_, H_ // 2, W_ // 2, self.dt, name=f"{prefix}/pool{i}")
                self.b.op(ir.OP_MIX, t, [ir.Path(x, C_, C_, ksize=0, pre_avg=1)], name=f"{prefix}.pool{i}")
                pooled.append(t)
            xs, stride = pooled, 1
        base = None                                                   # resolution of branch 0 after the stride-2 pool
        for i, x in enumerate(xs):
            if x is not None:
                _, H_, W_ = self.dims(x)
                base = (H_ * 2 ** i // stride, W_ * 2 ** i // stride)
                break
        outs: List[Optional[int]] = []
        for j in range(len(a_out)):
            cj = co[j + 1] - co[j]
            if cj == 0:
                outs.append(None)
                continue
            Hj, Wj = base[0] // 2 ** j, base[1] // 2 ** j
            s, t = self.bn_fold(f"{prefix}.bns.{j}")
            paths = []
            for i, x in enumerate(xs):
                if x is None or ci[i] == ci[i + 1]:
                    continue
                cin = ci[i + 1] - ci[i]
                w = W4[co[j]:co[j + 1], ci[i]:ci[i + 1]] * s[:, None, None, None]
                common = dict(pre_avg=int(stride == 2), ksize=ksize, pad=pad, w_off=self.conv_w(w))
                if i > j and ksize == 1 and stride == 1 and self.upsample_inputs and upsample_input_side(cin, cj, 2 ** (i - j)):
                    # 16-bit programs, 1x1, fewer input than output channels: up-sample the conv INPUT instead of its
                    # output (identical linear map, cin instead of cout bilinear evaluations, no scratch tensor)
                    if pool_once:                                    # ... and do it once, in a bandwidth-bound op of its own
                        paths.append(ir.Path(self.upsampled(x, 2 ** (i - j), prefix), cin, cj, ksize=1, w_off=self.conv_w(w)))
                    else:
                        paths.append(ir.Path(x, cin, cj, ksize=1, up=2 ** (i - j), w_off=self.conv_w(w)))
                elif i > j:                                          # conv at low res, then bilinear (:702-707)
                    _, Hi, Wi = self.dims(x)
                    low = self.b.tensor(cj, Hi // stride, Wi // stride, ir.F32, name=f"{prefix}/low{i}to{j}")
                    self.b.op(ir.OP_MIX, low, [ir.Path(x, cin, cj, **common)], name=f"{prefix}.low{i}to{j}")
                    paths.append(ir.Path(low, cj, cj, ksize=0, up=2 ** (i - j)))
                elif j > i and pool_once and not common["pre_avg"]:   # max-pool first (:708-717), materialised once per source
                    paths.append(ir.Path(self.maxpooled(x, 2 ** (j - i), prefix), cin, cj, **common))
                else:                                                # same res, or max-pool in the consumer's staging loop
                    paths.append(ir.Path(x, cin, cj, pool=2 ** (j - i), **common))
            if not paths:
                outs.append(None)
                continue
            dst = self.b.tensor(cj, Hj, Wj, self.dt, name=f"{prefix}/{j}")
            self.b.op(ir.OP_MIX, dst, paths, bias=t, slope=self.p(f"{prefix}.prelus.{j}.weight"), name=f"{prefix}.{j}")
            outs.append(dst)
        return outs

    def maxpooled(self, x: int, f: int, prefix: str) -> int:
        """max_pool2d(f, f) of a whole 16-bit tensor as its own bandwidth-bound op(s) (a chain of 2x2 steps, exact for a
        maximum), cached per source: several conv paths (oct_fuse.fuse.1 / .2) read the same pooled branch."""
        if f == 1:
            return x
        key = (x, f)
        if key not in self._pooled:
            src = self.maxpooled(x, f // 2, prefix)
            C_, H_, W_ = self.dims(src)
            t = self.b.tensor(C_, H_ // 2, W_ // 2, self.dt, name=f"{prefix}/maxpool{f}of{x}")
            self.b.op(ir.OP_MIX, t, [ir.Path(src, C_, C_, ksize=0, pool=2)], name=f"{prefix}.maxpool{f}of{x}")
            self._pooled[key] = t
        return self._pooled[key]

    def upsampled(self, x: int, f: int, prefix: str) -> int:
        """F.interpolate(scale_factor=f, bilinear) of a whole 16-bit tensor as its own op: the stored 16-bit value is the one
        the tensor-core kernel would stage for an input-side up-sampled 1x1 path, computed once instead of once per tile."""
        C_, H_, W_ = self.dims(x)
        t = self.b.tensor(C_, H_ * f, W_ * f, self.dt, name=f"{prefix}/up{f}of{x}")
        self.b.op(ir.OP_MIX, t, [ir.Path(x, C_, C_, ksize=0, up=f)], name=f"{prefix}.up{f}of{x}")
        return t

    def dw_cbr(self, prefix: str, xs: List[Optional[int]]):
        """SimplifiedGOctConvBR.forward (csnet.py:838-851)."""
        outs = []
        for b_, x in enumerate(xs):
            if x is None:
                outs.append(None)
                continue
            C_, H_, W_ = self.dims(x)
            s, t = self.bn_fold(f"{prefix}.bns.{b_}")
            w = 100.0 * self.p(f"{prefix}.convs.{b_}.weight").reshape(C_, 9) * s[:, None]
            dst = self.b.tensor(C_, H_, W_, self.dt, name=f"{prefix}/{b_}")
            path = ir.Path(x, C_, C_, ksize=3, pad=1, w_off=self.b.param(w))
            self.b.op(ir.OP_DW, dst, [path], bias=t, slope=self.p(f"{prefix}.prelus.{b_}.weight"), name=f"{prefix}.{b_}")
            outs.append(dst)
        return outs

    def dw_params(self, prefix: str, b_: int):
        s, t = self.bn_fold(f"{prefix}.bns.{b_}")
        w = 100.0 * self.p(f"{prefix}.convs.{b_}.weight").reshape(-1, 9) * s[:, None]
        return [self.b.param(w), self.b.param(t), self.b.param(self.p(f"{prefix}.prelus.{b_}.weight"))]

    def il_block_fused(self, prefix, xs, a_in, a_out):
        """Whole 1x1-kind ILBlock as one CSNET_OP_ILBLOCK (csrc/il_block.cuh); None if it does not qualify."""
        if len(a_in) != 2 or len(a_out) not in (1, 2) or xs[0] is None or xs[1] is None:
            return None
        W4 = self.p(prefix + ".conv1x1.conv.weight")
        ci, co = splits.cuts(W4.shape[1], a_in), splits.cuts(W4.shape[0], a_out)
        Chi, Cli = ci[1] - ci[0], ci[2] - ci[1]
        Cho, Clo = co[1] - co[0], (co[2] - co[1]) if len(a_out) == 2 else 0
        (c_h, H_, W_), (c_l, Hl, Wl) = self.dims(xs[0]), self.dims(xs[1])
        if min(Chi, Cli, Cho) <= 0 or (len(a_out) == 2 and Clo <= 0) or (c_h, c_l) != (Chi, Cli):
            return None
        if W_ % 8 or H_ % 2 or (Hl * 2, Wl * 2) != (H_, W_) or not il_block_fits(Chi, Cli, Cho, Clo):
            return None
        s_h, t_h = self.bn_fold(prefix + ".conv1x1.bns.0")
        W2 = W4[:, :, 0, 0]
        K8 = _ru(Chi + Cli, 8)
        WH = np.zeros((_ru(Cho, 16), K8))                    # columns: [x_h | bilinear_x2(x_l)]
        WH[:Cho, :Chi] = W2[co[0]:co[1], ci[0]:ci[1]] * s_h[:, None]
        WH[:Cho, Chi:Chi + Cli] = W2[co[0]:co[1], ci[1]:ci[2]] * s_h[:, None]
        WL = np.zeros((max(_ru(Clo, 16), 16), K8))           # columns: [x_l | maxpool2(x_h)]
        ext = [0, 0, self.b.param(t_h), self.b.param(self.p(prefix + ".conv1x1.prelus.0.weight")), -1, -1]
        if Clo > 0:
            s_l, t_l = self.bn_fold(prefix + ".conv1x1.bns.1")
            WL[:Clo, :Cli] = W2[co[1]:co[2], ci[1]:ci[2]] * s_l[:, None]
            WL[:Clo, Cli:Cli + Chi] = W2[co[1]:co[2], ci[0]:ci[1]] * s_l[:, None]
            ext[4], ext[5] = self.b.param(t_l), self.b.param(self.p(prefix + ".conv1x1.prelus.1.weight"))
        lim = 6.0e4 if self.dt == ir.F16 else 3.0e38
        if not (np.isfinite(WH).all() and np.isfinite(WL).all() and max(np.abs(WH).max(), np.abs(WL).max()) < lim):
            return None
        ext[0] = self.b.param_bits16(to_bits16(WH, self.dt))
        ext[1] = self.b.param_bits16(to_bits16(WL, self.dt))
        none3 = [-1, -1, -1]
        ext += self.dw_params(prefix + ".conv3x3_1", 0) + (self.dw_params(prefix + ".conv3x3_1", 1) if Clo else none3)
        ext += self.dw_params(prefix + ".conv3x3_2", 0) + (self.dw_params(prefix + ".conv3x3_2", 1) if Clo else none3)
        yh = self.b.tensor(Cho, H_, W_, self.dt, name=f"{prefix}/0")
        yl = self.b.tensor(Clo, Hl, Wl, self.dt, name=f"{prefix}/1") if Clo else -1
        op = self.b.op(ir.OP_ILBLOCK, yh, [ir.Path(xs[0], Chi, Cho, ksize=1), ir.Path(xs[1], Cli, Cho, ksize=1)], name=prefix)
        op.dst2, op.ext_off = yl, ext
        return [yh] + ([yl] if Clo else [])

    def il_block_stem_fused(self, prefix, xs, a_in, a_out):
        """The first ILBlock (one fp32 image in, 3x3 gOctaveCBR, csnet.py:60-76) as one CSNET_OP_ILBLOCK in its stem
        form: the kernel builds im2col planes of the image / its 2x2 max-pool and reuses the 1x1 machinery."""
        if len(a_in) != 1 or len(a_out) not in (1, 2) or xs[0] is None:
            return None
        W4 = self.p(prefix + ".conv1x1.conv.weight")
        co = splits.cuts(W4.shape[0], a_out)
        Cho, Clo = co[1] - co[0], (co[2] - co[1]) if len(a_out) == 2 else 0
        Ci, H_, W_ = self.dims(xs[0])
        if self.b.prog.tensors[xs[0]].dtype != ir.F32 or Ci * 9 > 32 or W4.shape[1] != Ci or Cho <= 0 or (len(a_out) == 2 and Clo <= 0):
            return None
        if W_ % 8 or H_ % 2 or not il_block_fits(Ci * 9, 0, Cho, Clo):
            return None
        K8 = 32
        s_h, t_h = self.bn_fold(prefix + ".conv1x1.bns.0")
        WH = np.zeros((_ru(Cho, 16), K8))
        WH[:Cho, :Ci * 9] = (W4[co[0]:co[1]] * s_h[:, None, None, None]).reshape(Cho, -1)
        WL = np.zeros((max(_ru(Clo, 16), 16), K8))
        ext = [0, 0, self.b.param(t_h), self.b.param(self.p(prefix + ".conv1x1.prelus.0.weight")), -1, -1]
        if Clo > 0:
            s_l, t_l = self.bn_fold(prefix + ".conv1x1.bns.1")
            WL[:Clo, :Ci * 9] = (W4[co[1]:co[2]] * s_l[:, None, None, None]).reshape(Clo, -1)
            ext[4], ext[5] = self.b.param(t_l), self.b.param(self.p(prefix + ".conv1x1.prelus.1.weight"))
        lim = 6.0e4 if self.dt == ir.F16 else 3.0e38
        if not (np.isfinite(WH).all() and np.isfinite(WL).all() and max(np.abs(WH).max(), np.abs(WL).max()) < lim):
            return None
        ext[0] = self.b.param_bits16(to_bits16(WH, self.dt))
        ext[1] = self.b.param_bits16(to_bits16(WL, self.dt))
        none3 = [-1, -1, -1]
        ext += self.dw_params(prefix + ".conv3x3_1", 0) + (self.dw_params(prefix + ".conv3x3_1", 1) if Clo else none3)
        ext += self.dw_params(prefix + ".conv3x3_2", 0) + (self.dw_params(prefix + ".conv3x3_2", 1) if Clo else none3)
        yh = self.b.tensor(Cho, H_, W_, self.dt, name=f"{prefix}/0")
        yl = self.b.tensor(Clo, H_ // 2, W_ // 2, self.dt, name=f"{prefix}/1") if Clo else -1
        op = self.b.op(ir.OP_ILBLOCK, yh, [ir.Path(xs[0], Ci, Cho, ksize=3, pad=1),
                                           ir.Path(xs[0], Ci, max(Clo, 1), ksize=3, pad=1, pool=2)], name=prefix)
        op.dst2, op.ext_off = yl, ext
        return [yh] + ([yl] if Clo else [])

    def il_block(self, prefix, xs, in_split, out_split, stride, first):
        """ILBlock.forward (csnet.py:72-76)."""
        a_in, a_out = splits.alphas(in_split), splits.alphas(out_split)
        k = 3 if (first or stride == 2) else 1
        if (k == 1 or (first and stride == 1)) and (self.fuse is True or (self.fuse and prefix in self.fuse)):
            y = self.il_block_fused(prefix, xs, a_in, a_out) if k == 1 else self.il_block_stem_fused(prefix, xs, a_in, a_out)
            if y is not None:
                for b_, t in enumerate(y):
                    self.b.prog.taps[f"{prefix}/{b_}"] = t
                return y
        y = self.goct_cbr(prefix + ".conv1x1", xs, a_in, a_out, k, stride)
        y = self.dw_cbr(prefix + ".conv3x3_1", y)
        y = self.dw_cbr(prefix + ".conv3x3_2", y)
        for b_, t in enumerate(y):
            if t is not None:
                self.b.prog.taps[f"{prefix}/{b_}"] = t
        return y

    def ms_block(self, prefix: str, x: int, dil_channels):
        """MSBlock.forward (csnet.py:141-149)."""
        C_, H_, W_ = self.dims(x)
        s, t = self.bn_fold(prefix + ".bn")
        cout_t = int(s.shape[0])
        dst = self.b.tensor(cout_t, H_, W_, self.dt, name=prefix)
        paths, c = [], 0
        for d, dil in enumerate(splits.DILATIONS):
            n = int(dil_channels[d])
            if n == 0:
                continue
            w = 100.0 * self.p(f"{prefix}.msconv.{d}.weight") * s[c:c + n, None, None, None]
            paths.append(ir.Path(x, C_, n, cout0=c, ksize=3, dil=dil, pad=dil, w_off=self.conv_w(w)))
            c += n
        if c != cout_t:
            raise ValueError(f"{prefix}: dilation split sums to {c}, BN has {cout_t} channels")
        self.b.op(ir.OP_MIX, dst, paths, bias=t, slope=self.p(prefix + ".prelu.weight"), name=prefix)
        return dst

    def csf_head(self, prefix: str, xs, cfg3):
        """CSFHead.forward (csnet.py:202-206), PallMSBlock.forward (:102-113)."""
        a_in, a_mid_in, a_mid_out = splits.alphas(cfg3[0][0]), splits.alphas(cfg3[1][0]), splits.alphas(cfg3[1][1])
        dils = np.asarray(cfg3[1][2])
        y = self.goct_cbr(prefix + ".fuse", xs, a_in, a_mid_in, 1, 1)
        z = []
        for b_ in range(len(a_mid_in)):
            z.append(self.ms_block(f"{prefix}.ms.convs.{b_}", y[b_], dils[b_]) if max(dils[b_]) != 0 else None)
        out = self.goct_cbr(prefix + ".fuse1x1", z, a_mid_out, [1], 1, 1)
        for name, ts in ((".fuse", y), (".ms", z), (".fuse1x1", out)):
            for b_, t in enumerate(ts):
                if t is not None:
                    self.b.prog.taps[f"{prefix}{name}/{b_}"] = t
        return out

    def project_cls(self, feat: int, low: int, cls_w: np.ndarray) -> bool:
        """cls_layer (a 1x1 conv to one channel, csnet.py:383) folded into the epilogue of the op that produces its
        input: that op becomes a CSNET_OP_MIXPROJ and the feature tensor is never written.  16-bit tensor-core
        programs only; `fuse` / `tensor_core` name sets gate it like the other fused kernels ("cls_layer")."""
        ops = self.b.prog.ops
        prod = next((o for o in reversed(ops) if o.dst == feat), None)
        C_ = self.dims(feat)[0]
        want = self.fuse is True or (self.fuse and "cls_layer" in self.fuse)
        if not want or self.dt == ir.F32 or prod is None or prod.kind != ir.OP_MIX or cls_w.shape[0] != 1 or C_ > 80:
            return False
        if not (self.tensor_core is True or (self.tensor_core and any(prod.name.startswith(x) for x in self.tensor_core))):
            return False
        if any(feat in (q.src for q in o.paths) for o in ops):
            return False                                   # somebody else reads the feature tensor
        lim = 6.0e4 if self.dt == ir.F16 else 3.0e38
        conv = [q for q in prod.paths if q.ksize > 0]
        if not conv or any(q.stride != 1 or self._wmax.get(q.w_off, 0.0) >= lim for q in conv):
            return False
        prod.kind, prod.dst, prod.name = ir.OP_MIXPROJ, low, prod.name + "+cls_layer"
        prod.ext_off = [self.b.param(cls_w.reshape(-1)), self.b.param(self.p("cls_layer.bias")), C_]
        for key in [k for k, t in self.b.prog.taps.items() if t == feat]:
            del self.b.prog.taps[key]                      # the tapped tensor no longer exists
        return True

    def run(self, reuse: bool) -> ir.Program:
        """CSNet.forward (csnet.py:365-387)."""
        b = self.b
        x = b.tensor(3, self.H, self.W, ir.F32, external=0, name="input")
        walk, idx = splits.block_walk(self.cfg)
        feats: Dict[str, List[Optional[int]]] = {}
        cur: List[Optional[int]] = [x]
        for prefix, ci, stride, first in walk:
            in_split = np.array([3]) if first else self.cfg[ci][0]
            cur = self.il_block(prefix, cur, in_split, self.cfg[ci][1], stride, first)
            feats[prefix] = cur
        stages = [int(s) for s in self.cfg[-1]]
        ends = [f"stage{s + 1}.{stages[s] - 1}" for s in (1, 2, 3)]
        fuse = self.csf_head("oct_fuse", [feats[e][0] for e in ends], self.cfg[idx:idx + 3])
        C_, Hf, Wf = self.dims(fuse[0])
        cls_w = self.p("cls_layer.weight")
        low = b.tensor(cls_w.shape[0], Hf, Wf, ir.F32, name="cls/low")
        if not self.project_cls(fuse[0], low, cls_w):
            b.op(ir.OP_MIX, low, [ir.Path(fuse[0], C_, cls_w.shape[0], ksize=1, w_off=self.conv_w(cls_w))],
                 bias=self.p("cls_layer.bias"), name="cls_layer")
        if self.H % Hf or self.W % Wf or self.H // Hf != self.W // Wf:
            raise ValueError("final resample factor is not an integer")
        out = b.tensor(cls_w.shape[0], self.H, self.W, ir.F32, external=1, name="logits")
        b.op(ir.OP_MIX, out, [ir.Path(low, cls_w.shape[0], cls_w.shape[0], ksize=0, up=self.H // Hf)], name="upsample")
        prog = b.finish(reuse=reuse)
        self.finalize_flags(prog)
        prog.input, prog.output = x, out
        return prog


def compile_csnet(layer_config, params: Mapping[str, object], H: int, W: int, dtype="fp32",
                  reuse_arena: bool = True, fuse=True, tensor_core=True, upsample_inputs=None) -> ir.Program:
    """layer_config: the reference's pickle structure (list of [in_split, out_split(, dil_split)] + stages);
    params: state_dict-like mapping (torch tensors or numpy arrays); returns the eval-mode program."""
    dt = ir.DTYPE_NAMES[dtype] if isinstance(dtype, str) else int(dtype)
    return _Lowering(layer_config, params, H, W, dt, fuse, tensor_core, upsample_inputs).run(reuse_arena)
