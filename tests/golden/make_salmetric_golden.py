"""Runs the reference's own SalMetric (oracle/_ref/salmetric = /root/reference/CSNet_training/SalMetric/src/sal_metric.cpp compiled
unmodified with oracle/cvshim, see oracle/build_ref.py) on seeded 8-bit maps and stores its report in tests/golden/salmetric_ref.json.
    python tests/golden/make_salmetric_golden.py"""
import json
import os
import subprocess
import sys
import tempfile

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)


def seeded_maps(seed, n, h, w):
    """Blob-like saliency maps and binary ground truth (uint8), one image without any foreground."""
    rng = np.random.default_rng(seed)
    yy, xx = np.mgrid[0:h, 0:w]
    sal, gt = [], []
    for i in range(n):
        cy, cx, r = rng.uniform(0.3, 0.7) * h, rng.uniform(0.3, 0.7) * w, rng.uniform(0.15, 0.3) * min(h, w)
        d = np.sqrt((yy - cy) ** 2 + (xx - cx) ** 2)
        g = (d < r).astype(np.uint8) * 255
        s = np.clip(255 * np.exp(-(d / (1.2 * r)) ** 2) + rng.normal(0, 25, (h, w)), 0, 255).astype(np.uint8)
        if i == n - 1:
            g[:] = 0
        sal.append(s)
        gt.append(g)
    return sal, gt


def write_pgm(path, a):
    with open(path, "wb") as f:
        f.write(b"P5\n%d %d\n255\n" % (a.shape[1], a.shape[0]))
        f.write(np.ascontiguousarray(a, np.uint8).tobytes())


def run_reference(binary, sal, gt, threads=3):
    with tempfile.TemporaryDirectory() as d:
        lines = []
        for i, (s, g) in enumerate(zip(sal, gt)):
            write_pgm(os.path.join(d, f"{i}_sal.pgm"), s)
            write_pgm(os.path.join(d, f"{i}_gt.pgm"), g)
            lines.append(f"{d}/{i}_sal.pgm {d}/{i}_gt.pgm")
        lst = os.path.join(d, "list.txt")
        open(lst, "w").write("\n".join(lines) + "\n")
        out = subprocess.run([binary, lst, str(threads)], capture_output=True, text=True, check=True).stdout
    rep = {}
    for line in out.strip().splitlines()[-7:]:
        k, v = line.split(":")
        rep[k.strip()] = float(v)
    return rep


if __name__ == "__main__":
    from oracle import build_ref

    binary = build_ref.build()
    cases = {}
    for name, (seed, n, h, w) in {"a": (11, 5, 24, 32), "b": (12, 3, 40, 40), "c": (13, 7, 16, 48)}.items():
        sal, gt = seeded_maps(seed, n, h, w)
        cases[name] = {"args": [seed, n, h, w], "report": run_reference(binary, sal, gt)}
    # the maps of test_restatement_matches_the_reference_binary_live, on two threads as that test runs the binary
    sal, gt = seeded_maps(21, 6, 20, 28)
    cases["d"] = {"args": [21, 6, 20, 28], "threads": 2, "report": run_reference(binary, sal, gt, threads=2)}
    json.dump(cases, open(os.path.join(HERE, "salmetric_ref.json"), "w"), indent=1)
    print(json.dumps(cases, indent=1))
