"""Which kernel runs each op of the shipped programs, and how many launches a run issues.  The executor decides both once,
at plan creation; these lists pin that decision so a change to the executor cannot move an op to another kernel unnoticed
(bench.py groups its per-op times by these names).  `python tests/test_gpu_routes.py` prints the current lists."""
import json
import os
import sys

import numpy as np
import pytest

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))

from sod100k_b200 import compiler, compiler_r, runtime, synth  # noqa: E402
from tests import fixtures  # noqa: E402

pytestmark = pytest.mark.gpu

KERNELS = {
    "msd": "msd_kernel (ms_direct.cuh, FP32 pipe)",
    "ms": "mix_stream_kernel (TMA + tcgen05)",
    "tc": "mix_tc_kernel (mma.sync)",
    "rs": "pool2 / upsample / resample kernels",
    "mix": "mix_generic_kernel",
    "gn": "gn kernels",
    "ils": "il_stream_kernel (TMA + tcgen05 + TMEM)",
    "il": "il_block_kernel (mma.sync, tiled)",
    "dw": "dw kernels",
}

# name: (checkpoint, dtype, max_batch, tensor_core); "csf-head" is the CSF+Res2Net head on case "b" backbone features
CONFIGS = {
    "x2-fp16-bs256": ("csnet-L-x2", "fp16", 256, True),
    "x2-fp16-bs1": ("csnet-L-x2", "fp16", 1, True),
    "x2-fp32": ("csnet-L-x2", "fp32", 256, True),
    "x1-bf16": ("csnet-L-x1", "bf16", 256, True),
    "x2-fp16-no-tc": ("csnet-L-x2", "fp16", 256, False),
    "csf-head": (None, "fp16", 2, True),
}

# name: (kernel of every op in launch order, as KERNELS keys; launches of one run)
EXPECTED = {
    "x2-fp16-bs256": (
        "ils ils ils ils rs rs ms ms rs ms dw dw dw dw ils ils ils rs ms rs tc dw dw dw dw il il il il il rs tc rs tc "
        "dw dw dw dw tc tc rs tc dw dw dw dw tc tc rs tc dw dw dw dw tc tc dw dw ms tc ms rs tc ms rs rs tc msd msd tc "
        "rs rs ms rs", 81),
    "x2-fp16-bs1": (
        "il il il il rs rs tc tc rs tc dw dw dw dw il il il rs tc rs tc dw dw dw dw il il il il il rs tc rs tc dw dw dw "
        "dw tc tc rs tc dw dw dw dw tc tc rs tc dw dw dw dw tc tc dw dw tc tc tc rs tc tc rs rs tc msd msd tc rs rs tc "
        "rs", 81),
    "x2-fp32": (
        "mix mix dw dw dw dw mix mix mix dw dw dw dw mix mix mix dw dw dw dw mix mix mix dw dw dw dw mix mix mix dw dw "
        "dw dw mix mix mix dw dw dw dw mix mix mix dw dw dw dw mix mix dw dw mix mix dw dw dw dw mix mix mix dw dw dw "
        "dw mix mix mix dw dw dw dw mix mix mix dw dw dw dw mix mix mix dw dw dw dw mix mix dw dw mix mix dw dw dw dw "
        "mix mix mix dw dw dw dw mix mix mix dw dw dw dw mix mix dw dw mix mix mix mix mix mix mix mix mix mix mix mix "
        "mix rs", 128),
    "x1-bf16": (
        "il il il il rs rs tc tc rs tc dw dw dw dw il il il rs tc rs tc dw dw dw dw il il il il il rs tc rs tc dw dw dw "
        "dw tc tc rs tc dw dw dw dw tc tc rs tc dw dw dw dw rs tc dw dw tc tc tc rs tc tc rs rs tc tc tc tc rs rs tc rs", 74),
    "x2-fp16-no-tc": (
        "ils ils ils ils rs rs mix mix rs mix dw dw dw dw ils ils ils rs mix rs mix dw dw dw dw il il il il il rs mix "
        "rs mix dw dw dw dw mix mix rs mix dw dw dw dw mix mix rs mix dw dw dw dw mix mix dw dw mix mix mix rs mix mix "
        "rs rs mix mix mix mix rs rs mix mix rs", 75),
    "csf-head": (
        "tc tc tc tc gn tc tc tc gn tc tc gn tc gn tc gn tc gn tc gn tc gn tc tc tc tc gn tc rs", 38),
}


def _plan(name):
    tag, dtype, max_batch, tc = CONFIGS[name]
    if tag is None:
        z = np.load(os.path.join(fixtures.GOLDEN, "csf_res2net.npz"))
        meta = json.loads(str(z["__meta__"]))
        sd = synth.synth_state_r({k: tuple(v) for k, v in meta["shapes"].items()}, meta["seed"])
        h, w, _ = meta["cases"]["b"]
        feats = [(256, h // 4, w // 4), (512, h // 8, w // 8), (1024, h // 16, w // 16), (2048, h // 32, w // 32)]
        prog = compiler_r.compile_csf_head(sd, feats, h, w, dtype, tensor_core=tc)
    else:
        cfg, sd = fixtures.checkpoint(tag)
        prog = compiler.compile_csnet(cfg, sd, 224, 224, dtype, tensor_core=tc)
    return runtime.Plan(prog, max_batch=max_batch)


def _routes(name):
    plan = _plan(name)
    try:
        codes = {v: k for k, v in KERNELS.items()}
        return " ".join(codes[plan.op_kernel(i)] for i in range(len(plan.prog.ops))), plan.launches
    finally:
        plan.close()


@pytest.mark.parametrize("name", sorted(CONFIGS))
def test_op_kernels_and_launches(name):
    assert _routes(name) == EXPECTED[name]


if __name__ == "__main__":
    print(json.dumps({name: _routes(name) for name in CONFIGS}, indent=1))
