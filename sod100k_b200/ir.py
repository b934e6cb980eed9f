"""Program IR — ctypes mirrors of include/csnet_b200.h plus a small builder with arena planning."""
from __future__ import annotations

import ctypes as C
from dataclasses import dataclass, field
from typing import Dict, List, Optional

import numpy as np

F32, F16, BF16 = 0, 1, 2
DTYPE_BYTES = {F32: 4, F16: 2, BF16: 2}
DTYPE_NAMES = {"fp32": F32, "float32": F32, "fp16": F16, "float16": F16, "half": F16, "bf16": BF16, "bfloat16": BF16}
MAX_PATHS = 8
MAX_EXT = 24
EXT_NO_FAST = 23          # CSNET_EXT_NO_FAST: the ext_off slot that keeps a MIX / DW op on the generic kernels
OP_MIX, OP_DW, OP_ILBLOCK, OP_GN, OP_MIXPROJ = 1, 2, 3, 4, 5


class TensorDesc(C.Structure):
    _fields_ = [("C", C.c_int32), ("H", C.c_int32), ("W", C.c_int32), ("dtype", C.c_int32),
                ("external", C.c_int32), ("_pad", C.c_int32), ("arena_offset", C.c_int64)]


class PathDesc(C.Structure):
    _fields_ = [("src", C.c_int32), ("c0", C.c_int32), ("cin", C.c_int32), ("pre_avg", C.c_int32),
                ("pool", C.c_int32), ("ksize", C.c_int32), ("dil", C.c_int32), ("stride", C.c_int32),
                ("pad", C.c_int32), ("up", C.c_int32), ("cout0", C.c_int32), ("cout", C.c_int32),
                ("w_off", C.c_int64)]


class OpDesc(C.Structure):
    _fields_ = [("kind", C.c_int32), ("dst", C.c_int32), ("n_paths", C.c_int32), ("dst2", C.c_int32),
                ("bias_off", C.c_int64), ("slope_off", C.c_int64), ("paths", PathDesc * MAX_PATHS),
                ("ext_off", C.c_int64 * MAX_EXT)]


@dataclass
class Path:
    src: int
    cin: int
    cout: int
    c0: int = 0
    cout0: int = 0
    pre_avg: int = 0
    pool: int = 1
    ksize: int = 1
    dil: int = 1
    stride: int = 1
    pad: int = 0
    up: int = 1
    w_off: int = -1


@dataclass
class Op:
    kind: int
    dst: int
    paths: List[Path]
    bias_off: int = -1
    slope_off: int = -1
    name: str = ""
    dst2: int = -1
    ext_off: List[int] = field(default_factory=list)

    @property
    def dsts(self):
        return [self.dst] + ([self.dst2] if self.dst2 >= 0 else [])


def veto_fast_kernels(ops, tensor_core, kinds, forced=lambda o: False):
    """Keep the ops of `kinds` on the generic kernels (ext_off[EXT_NO_FAST] = 1) unless `tensor_core` allows them (True: all,
    a collection of op-name prefixes: those ops, falsy: none) and `forced(op)` is false."""
    for o in ops:
        if o.kind not in kinds:
            continue
        allowed = tensor_core is True or (tensor_core and any(o.name.startswith(x) for x in tensor_core))
        if not allowed or forced(o):
            o.ext_off = [-1] * EXT_NO_FAST + [1]


@dataclass
class Tensor:
    C: int
    H: int
    W: int
    dtype: int
    external: int = -1
    arena_offset: int = 0
    name: str = ""

    @property
    def bytes_per_image(self) -> int:
        return self.C * self.H * self.W * DTYPE_BYTES[self.dtype]


@dataclass
class Program:
    tensors: List[Tensor] = field(default_factory=list)
    ops: List[Op] = field(default_factory=list)
    blob: Optional[np.ndarray] = None
    taps: Dict[str, int] = field(default_factory=dict)
    input: int = -1
    output: int = -1

    # ---- ctypes views -----------------------------------------------------------------------
    def tensor_array(self):
        arr = (TensorDesc * len(self.tensors))()
        for i, t in enumerate(self.tensors):
            arr[i] = TensorDesc(t.C, t.H, t.W, t.dtype, t.external, 0, t.arena_offset)
        return arr

    def op_array(self):
        arr = (OpDesc * len(self.ops))()
        for i, o in enumerate(self.ops):
            d = OpDesc()
            d.kind, d.dst, d.n_paths, d.bias_off, d.slope_off = o.kind, o.dst, len(o.paths), o.bias_off, o.slope_off
            d.dst2 = o.dst2
            for k in range(MAX_EXT):
                d.ext_off[k] = o.ext_off[k] if k < len(o.ext_off) else -1
            for k, p in enumerate(o.paths):
                d.paths[k] = PathDesc(p.src, p.c0, p.cin, p.pre_avg, p.pool, p.ksize, p.dil, p.stride, p.pad,
                                      p.up, p.cout0, p.cout, p.w_off)
            arr[i] = d
        return arr

    def signature(self) -> bytes:
        """Everything a plan freezes at creation: the tensor table, the op list (kinds, paths, parameter offsets, flags) and the
        blob size.  Two programs with equal signatures differ only in parameter VALUES (csnet_plan_set_blob suffices)."""
        import hashlib

        h = hashlib.sha256()
        h.update(bytes(self.tensor_array()))
        h.update(bytes(self.op_array()))
        h.update(str(0 if self.blob is None else int(self.blob.size)).encode())
        return h.digest()

    @property
    def arena_bytes_per_image(self) -> int:
        return max([t.arena_offset + t.bytes_per_image for t in self.tensors if t.external < 0] + [0])


class Builder:
    """Accumulates tensors / ops / blob segments; `finish()` plans the arena."""

    def __init__(self):
        self.prog = Program()
        self._blob: List[np.ndarray] = []
        self._blob_len = 0

    def tensor(self, C_, H, W, dtype, external=-1, name="") -> int:
        self.prog.tensors.append(Tensor(int(C_), int(H), int(W), int(dtype), int(external), 0, name))
        return len(self.prog.tensors) - 1

    def param(self, arr) -> int:
        """Append a float32 array to the blob (16-byte aligned start); returns its offset in floats."""
        a = np.ascontiguousarray(np.asarray(arr, dtype=np.float32)).reshape(-1)
        off = self._blob_len
        pad = (-a.size) % 4
        self._blob.append(a)
        if pad:
            self._blob.append(np.zeros(pad, np.float32))
        self._blob_len += a.size + pad
        return off

    def param_bits16(self, arr_u16) -> int:
        """Append a uint16 array (raw fp16/bf16 bits) packed two per blob word; returns its offset in floats."""
        a = np.ascontiguousarray(np.asarray(arr_u16, dtype=np.uint16)).reshape(-1)
        if a.size % 2:
            a = np.concatenate([a, np.zeros(1, np.uint16)])
        return self.param(a.view(np.float32))

    def op(self, kind, dst, paths, bias=None, slope=None, name="") -> Op:
        if len(paths) > MAX_PATHS:
            raise ValueError(f"{name}: {len(paths)} paths exceed CSNET_MAX_PATHS")
        o = Op(kind, dst, list(paths), -1 if bias is None else self.param(bias),
               -1 if slope is None else self.param(slope), name)
        self.prog.ops.append(o)
        return o

    def finish(self, reuse: bool = True) -> Program:
        p = self.prog
        p.blob = np.concatenate(self._blob) if self._blob else np.zeros(4, np.float32)
        plan_arena(p, reuse)
        return p


def plan_arena(p: Program, reuse: bool = True) -> None:
    """Assign per-image arena offsets (multiples of 256 B).  With `reuse`, a tensor's bytes are recycled
    after its last reader (first-fit over the live set); taps are then only valid right after their op."""
    last_use: Dict[int, int] = {}
    first_def: Dict[int, int] = {}
    for k, o in enumerate(p.ops):
        for d in o.dsts:
            first_def.setdefault(d, k)
            last_use[d] = max(last_use.get(d, k), k)
        for q in o.paths:
            last_use[q.src] = k
    align = lambda v: (v + 255) // 256 * 256
    live: List[tuple] = []          # (offset, size, tensor)
    top = 0
    for k, o in enumerate(p.ops):
        for dst in o.dsts:
            t = p.tensors[dst]
            if t.external >= 0 or first_def[dst] != k:
                continue
            size = align(t.bytes_per_image)
            if reuse:
                live.sort()
                off = 0
                for lo, sz, _ in live:
                    if lo - off >= size:
                        break
                    off = max(off, lo + sz)
                t.arena_offset = off
            else:
                t.arena_offset = top
            top = max(top, t.arena_offset + size)
            live.append((t.arena_offset, size, dst))
        if reuse:
            live = [e for e in live if last_use.get(e[2], k) > k]
