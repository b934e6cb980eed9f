"""Print the op list of the bench program (kind, name, dst dims) in launch order."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from sod100k_b200 import checkpoints, compiler, ir
cfg, sd = checkpoints.load_npz("csnet-L-x2")
prog = compiler.compile_csnet(cfg, sd, 224, 224, "fp16")
for i, o in enumerate(prog.ops):
    d = prog.tensors[o.dst]
    veto = len(o.ext_off) > ir.EXT_NO_FAST and o.ext_off[ir.EXT_NO_FAST] == 1
    print(i, {1: "MIX", 2: "DW", 3: "IL", 4: "GN", 5: "MIXPROJ"}[o.kind], o.name, f"{d.C}@{d.H}x{d.W}", "veto" if veto else "")
