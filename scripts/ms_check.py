"""GPU check of the streaming 1x1 MIX kernel (csrc/mix_stream.cuh): the fp16 program with CSNET_MS=1 vs CSNET_MS=0 (taps of the
CSF head + logits), then per-op times."""
import os, sys
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import numpy as np, torch
from sod100k_b200 import compiler, runtime, synth, checkpoints

def plan(prog, nb, ms):
    os.environ["CSNET_MS"] = "1" if ms else "0"
    return runtime.Plan(prog, max_batch=nb)

for tag, h, w, nb in (("csnet-L-x2", 224, 224, 24), ("csnet-L-x1", 224, 224, 24), ("csnet-L-x2", 96, 160, 40)):
    cfg, sd = checkpoints.load_npz(tag)
    sd = {k: torch.from_numpy(v) for k, v in sd.items()}
    x = torch.from_numpy(synth.randn_images(nb, h, w, 3)).cuda()
    prog = compiler.compile_csnet(cfg, sd, h, w, "fp16", reuse_arena=False)
    p1, p0 = plan(prog, nb, True), plan(prog, nb, False)
    y1, y0 = p1.forward(x), p0.forward(x)
    torch.cuda.synchronize()
    print(f"{tag} {h}x{w} bs{nb}: logits max diff {(y1 - y0).abs().max().item():.3e} (|y| max {y0.abs().max().item():.2f}) finite {bool(torch.isfinite(y1).all())}", flush=True)
    for name, tid in prog.taps.items():
        if not (name.startswith("oct_fuse") or name.startswith("stage2.0") or name.startswith("stage3.0") or name.startswith("stage2.1")):
            continue
        a, b = p1.read_tensor(tid, nb), p0.read_tensor(tid, nb)
        print(f"   {name:22s} rel diff {(a - b).abs().max().item() / max(1.0, b.abs().max().item()):.2e}", flush=True)
    p1.close(); p0.close()

# MSBlock direct kernel (csrc/ms_direct.cuh): compare against the tap values of the all-generic program
print("MSBlock taps vs the all-generic program:")
for tag, h, w, nb in (("csnet-L-x2", 224, 224, 4), ("csnet-L-x1", 224, 224, 3), ("csnet-L-x2", 96, 160, 2)):
    cfg, sd = checkpoints.load_npz(tag)
    sd = {k: torch.from_numpy(v) for k, v in sd.items()}
    x = torch.from_numpy(synth.randn_images(nb, h, w, 5)).cuda()
    base = compiler.compile_csnet(cfg, sd, h, w, "fp16", reuse_arena=False, fuse=False, tensor_core=False)
    prog = compiler.compile_csnet(cfg, sd, h, w, "fp16", reuse_arena=False, fuse=False, tensor_core={"oct_fuse.ms"})
    p0, p1 = runtime.Plan(base, max_batch=nb), runtime.Plan(prog, max_batch=nb)
    p0.forward(x); p1.forward(x)
    for name in ("oct_fuse.ms/0", "oct_fuse.ms/1", "oct_fuse.ms/2"):
        if name in prog.taps:
            a, b = p1.read_tensor(prog.taps[name], nb), p0.read_tensor(base.taps[name], nb)
            print(f"   {tag} {h}x{w} {name}: rel diff {(a - b).abs().max().item() / max(1.0, b.abs().max().item()):.2e} finite {bool(torch.isfinite(a).all())}", flush=True)
