"""Lower the CSF head of CSF+Res2Net (config 5) to the engine's program IR.

Mirrors `CSFNet.forward` after the backbone (/root/reference/CSF+Res2Net/networks/csf_res2net.py:253-258):
    fuse     gOctaveCBR 4 -> 4, 1x1, GroupNorm(32)   (networks/gOctConv.py:60-152)
    ms       PallMSBlock: per branch five dilated 3x3 convs, concat, GroupNorm(32), PReLU   (csf_res2net.py:190-225)
    fuse1x1  gOctaveCBR 4 -> 1 (1408 channels at 1/4 resolution)
    cls_layer + bilinear x4
GroupNorm statistics are per image, so nothing folds: every conv mix writes its raw sum and a CSNET_OP_GN op
normalises it.  Differences to the CSNet lowering: the down paths resize the conv INPUT bilinearly (pre_avg = 2/4/8:
for exact integer ratios `F.interpolate` to a smaller size is the mean of the centre 2x2 of every cell), the weight
parameter is called `weights`, and widths are 128...2048, so the tensor-core MIX kernel runs 80-channel output slices.
The Res2Net-50 backbone is NOT lowered: it runs on torch (cuDNN) — a library call, see DESIGN.md.
"""
from __future__ import annotations

from typing import Mapping, Sequence, Tuple

import numpy as np

from . import ir, splits
from .compiler import _np, upsample_input_side

FUSE_IN_SPLIT = [1 / 15, 2 / 15, 4 / 15, 8 / 15]       # csf_res2net.py:240
FUSE_OUT_SPLIT = [1 / 11, 2 / 11, 4 / 11, 4 / 11]      # :242
GN_GROUPS = 32


def compile_csf_head(params: Mapping[str, object], feat_dims: Sequence[Tuple[int, int, int]], H: int, W: int, dtype="fp32",
                     reuse_arena: bool = True, tensor_core=True) -> ir.Program:
    """feat_dims: (C, h, w) of the four backbone stages (externals 0..3, in the plan dtype); external 4 = fp32 logits."""
    dt = ir.DTYPE_NAMES[dtype] if isinstance(dtype, str) else int(dtype)
    b = ir.Builder()
    p = lambda k: _np(params[k]).astype(np.float64)

    def conv_w(w):
        co, ci, kh, kw = w.shape
        return b.param(np.transpose(w.reshape(co, ci, kh * kw), (1, 2, 0)))

    def gn(src, prefix_gn, prefix_prelu, name):
        C_, h, w = (b.prog.tensors[src].C, b.prog.tensors[src].H, b.prog.tensors[src].W)
        dst = b.tensor(C_, h, w, dt, name=name)
        op = b.op(ir.OP_GN, dst, [ir.Path(src, C_, C_, ksize=0, up=GN_GROUPS)], slope=p(prefix_prelu + ".weight"), name=name)
        op.ext_off = [b.param(p(prefix_gn + ".weight")), b.param(p(prefix_gn + ".bias"))]
        return dst

    feats = [b.tensor(c, h, w, dt, external=i, name=f"feat{i}") for i, (c, h, w) in enumerate(feat_dims)]
    for i in range(1, 4):
        if feat_dims[i][1] * 2 ** i != feat_dims[0][1] or feat_dims[i][2] * 2 ** i != feat_dims[0][2]:
            raise ValueError("backbone stages must halve exactly (input size multiple of 32)")
    # ---- fuse -----------------------------------------------------------------------------------------------------
    Wf = p("fuse.conv.weights")
    ci, co = splits.cuts(Wf.shape[1], FUSE_IN_SPLIT), splits.cuts(Wf.shape[0], FUSE_OUT_SPLIT)
    y = []
    for j in range(4):
        cj, (_, hj, wj) = co[j + 1] - co[j], feat_dims[j]
        paths = []
        for i in range(4):
            cin = ci[i + 1] - ci[i]
            w = Wf[co[j]:co[j + 1], ci[i]:ci[i + 1]]
            if i == j:
                paths.append(ir.Path(feats[i], cin, cj, ksize=1, w_off=conv_w(w)))
            elif i < j:                                   # resize the input down, then conv (gOctConv.py:101-103)
                paths.append(ir.Path(feats[i], cin, cj, ksize=1, pre_avg=2 ** (j - i), w_off=conv_w(w)))
            else:                                         # conv at low resolution, resize the output up (:98-100)
                low = b.tensor(cj, feat_dims[i][1], feat_dims[i][2], ir.F32, name=f"fuse/low{i}to{j}")
                b.op(ir.OP_MIX, low, [ir.Path(feats[i], cin, cj, ksize=1, w_off=conv_w(w))], name=f"fuse.low{i}to{j}")
                paths.append(ir.Path(low, cj, cj, ksize=0, up=2 ** (i - j)))
        z = b.tensor(cj, hj, wj, dt, name=f"fuse/raw{j}")
        b.op(ir.OP_MIX, z, paths, name=f"fuse.{j}")
        y.append(gn(z, f"fuse.bns.{j}", f"fuse.prelus.{j}", f"fuse/{j}"))
        b.prog.taps[f"fuse/{j}"] = y[-1]
    # ---- ms -------------------------------------------------------------------------------------------------------
    zs = []
    for br in range(4):
        C_, h, w = b.prog.tensors[y[br]].C, b.prog.tensors[y[br]].H, b.prog.tensors[y[br]].W
        paths, c = [], 0
        for d, dil in enumerate(splits.DILATIONS):
            wd = p(f"ms.convs.{br}.msconv.{d}.weight")
            paths.append(ir.Path(y[br], C_, wd.shape[0], cout0=c, ksize=3, dil=dil, pad=dil, w_off=conv_w(wd)))
            c += wd.shape[0]
        raw = b.tensor(c, h, w, dt, name=f"ms/raw{br}")
        b.op(ir.OP_MIX, raw, paths, name=f"ms.convs.{br}")
        zs.append(gn(raw, f"ms.convs.{br}.bn", f"ms.convs.{br}.prelu", f"ms/{br}"))
        b.prog.taps[f"ms/{br}"] = zs[-1]
    # ---- fuse1x1: 4 -> 1 (up paths: input- or output-side resampling by the cost model in compiler.upsample_input_side) ----
    W1 = p("fuse1x1.conv.weights")
    c1 = splits.cuts(W1.shape[1], FUSE_OUT_SPLIT)
    cout = W1.shape[0]
    paths = []
    for i in range(4):
        cin_i, w_i = c1[i + 1] - c1[i], W1[:, c1[i]:c1[i + 1]]
        if i == 0 or (dt != ir.F32 and upsample_input_side(cin_i, cout, 2 ** i)):
            paths.append(ir.Path(zs[i], cin_i, cout, ksize=1, up=2 ** i, w_off=conv_w(w_i)))
        else:                                             # wide layers: conv at the low resolution, resample the output
            low = b.tensor(cout, feat_dims[i][1], feat_dims[i][2], ir.F32, name=f"fuse1x1/low{i}")
            b.op(ir.OP_MIX, low, [ir.Path(zs[i], cin_i, cout, ksize=1, w_off=conv_w(w_i))], name=f"fuse1x1.low{i}")
            paths.append(ir.Path(low, cout, cout, ksize=0, up=2 ** i))
    raw = b.tensor(cout, feat_dims[0][1], feat_dims[0][2], dt, name="fuse1x1/raw")
    b.op(ir.OP_MIX, raw, paths, name="fuse1x1.0")
    f0 = gn(raw, "fuse1x1.bns.0", "fuse1x1.prelus.0", "fuse1x1/0")
    b.prog.taps["fuse1x1/0"] = f0
    # ---- cls + final bilinear -------------------------------------------------------------------------------------
    wc = p("cls_layer.weight")
    low = b.tensor(wc.shape[0], feat_dims[0][1], feat_dims[0][2], ir.F32, name="cls/low")
    b.op(ir.OP_MIX, low, [ir.Path(f0, cout, wc.shape[0], ksize=1, w_off=conv_w(wc))], bias=p("cls_layer.bias"), name="cls_layer")
    if H % feat_dims[0][1] or H // feat_dims[0][1] != W // feat_dims[0][2]:
        raise ValueError("final resample factor is not an integer")
    out = b.tensor(wc.shape[0], H, W, ir.F32, external=4, name="logits")
    b.op(ir.OP_MIX, out, [ir.Path(low, wc.shape[0], wc.shape[0], ksize=0, up=H // feat_dims[0][1])], name="upsample")
    prog = b.finish(reuse=reuse_arena)
    ir.veto_fast_kernels(prog.ops, tensor_core, (ir.OP_MIX,))
    prog.input, prog.output = feats[0], out
    return prog
