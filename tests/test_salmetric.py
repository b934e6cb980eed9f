"""Pins oracle/salmetric.py (the histogram restatement of the reference's SalMetric) two ways: against a literal
loop-for-loop restatement of CSNet_training/SalMetric/src/sal_metric.cpp:86-120,164-185 on small random maps, and
against cases worked out by hand.  The reference binary itself needs OpenCV 3.4 and cannot be built here."""
import numpy as np
import pytest

from oracle import salmetric as sm


def _literal(sal_maps, gt_maps):
    """sal_metric.cpp restated loop for loop (float32 accumulators as in the C++)."""
    n = len(sal_maps)
    prec, rec, mae = [np.float32(0)] * 256, [np.float32(0)] * 256, np.float32(0)
    for sal, gt in zip(sal_maps, gt_maps):
        m = np.float32(0)
        for s, g in zip(sal.reshape(-1), gt.reshape(-1)):
            m += np.float32(abs(float(s) - float(g)) / 255.0)
        mae += m / np.float32(sal.size)
        for th in range(256):
            a_sum = b_sum = ab = 0
            for s, g in zip(sal.reshape(-1), gt.reshape(-1)):
                a, b = int(float(s) > th), int(float(g) > 256 / 2)
                ab += a & b
                a_sum += a
                b_sum += b
            prec[th] += (np.float32(ab) + np.float32(1e-4)) / (np.float32(a_sum) + np.float32(1e-4))
            rec[th] += (np.float32(ab) + np.float32(1e-4)) / (np.float32(b_sum) + np.float32(1e-4))
    p = np.asarray(prec, np.float64) / n
    r = np.asarray(rec, np.float64) / n
    f = (1.3 * p * r) / (0.3 * p + r)
    k = int(np.argmax(f))
    return dict(max_f=f[k], mean_f=f.mean(), precision=p[k], recall=r[k], mae=float(mae) / n, argmax=k)


def test_histogram_form_equals_literal_loops():
    rng = np.random.default_rng(7)
    sal = [rng.integers(0, 256, (6, 5), dtype=np.uint8) for _ in range(3)]
    gt = [(rng.random((6, 5)) > 0.6).astype(np.uint8) * 255 for _ in range(3)]
    gt[2][:] = 0                                                   # an image without foreground (b_sum = 0)
    a, b = sm.evaluate(sal, gt), _literal(sal, gt)
    for key in ("max_f", "mean_f", "precision", "recall", "mae"):
        assert a[key] == pytest.approx(b[key], rel=2e-6, abs=2e-7), key
    assert a["argmax"] == b["argmax"]


def test_perfect_prediction():
    gt = np.zeros((4, 4), np.uint8)
    gt[1:3, 1:3] = 255
    out = sm.evaluate([gt.copy()], [gt])
    assert out["max_f"] == pytest.approx(1.0, abs=1e-6) and out["mae"] == 0.0
    # th = 255: nothing is > 255, precision = eps/eps = 1, recall = eps / (4 + eps)
    p, r = sm.precision_recall(gt, gt)
    assert p[255] == pytest.approx(1.0) and r[255] == pytest.approx(1e-4 / 4.0001, rel=1e-4)
    assert np.all(p[:255] == 1.0) and np.all(r[:255] == 1.0)


def test_half_overlap_by_hand():
    sal = np.array([[255, 255, 0, 0]], np.uint8)
    gt = np.array([[255, 0, 255, 0]], np.uint8)
    out = sm.evaluate([sal], [gt])
    pr = (1 + 1e-4) / (2 + 1e-4)                                   # ab = 1, |a| = |b| = 2 for every th < 255
    assert out["precision"] == pytest.approx(pr, rel=1e-6) and out["recall"] == pytest.approx(pr, rel=1e-6)
    assert out["max_f"] == pytest.approx(pr, rel=1e-6)            # F = 1.3 p r / (0.3 p + r) = p when p == r
    assert out["mae"] == pytest.approx(0.5)


def test_gt_threshold_is_strictly_above_128_and_quantisation_truncates():
    sal = np.full((1, 2), 200, np.uint8)
    gt = np.array([[128, 129]], np.uint8)                          # only 129 counts as foreground
    p, r = sm.precision_recall(sal, gt)
    assert p[0] == pytest.approx((1 + 1e-4) / (2 + 1e-4)) and r[0] == pytest.approx(1.0)
    assert p[200] == pytest.approx(1.0) and r[200] == pytest.approx(1e-4 / (1 + 1e-4), rel=1e-3)   # sal > 200 is empty
    assert sm.quantise(np.array([0.0, 0.999, 1.0, 0.5])).tolist() == [0, 254, 255, 127]


def _golden_cases():
    import json
    import os

    from tests import fixtures
    return json.load(open(os.path.join(fixtures.GOLDEN, "salmetric_ref.json")))


def _maps(args):
    import importlib.util
    import os

    from tests import fixtures
    spec = importlib.util.spec_from_file_location("make_salmetric_golden", os.path.join(fixtures.GOLDEN, "make_salmetric_golden.py"))
    mod = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mod)
    return mod, mod.seeded_maps(*args)


@pytest.mark.parametrize("case", ["a", "b", "c"])
def test_restatement_matches_the_reference_binary_golden(case):
    """tests/golden/salmetric_ref.json = the report of the reference's OWN sal_metric.cpp (compiled unmodified against the
    header shim in oracle/cvshim, oracle/build_ref.py) on seeded maps.  The binary prints 6 significant digits."""
    g = _golden_cases()[case]
    _, (sal, gt) = _maps(g["args"])
    e, r = sm.evaluate(sal, gt), g["report"]
    for mine, theirs in (("max_f", "Max_F-measre"), ("mean_f", "Mean_F-measre"), ("precision", "Precision"), ("recall", "Recall"),
                         ("mean_precision", "Mean_Precision"), ("mean_recall", "Mean_Recall"), ("mae", "MAE")):
        assert abs(e[mine] - r[theirs]) <= 2e-6 + 2e-6 * abs(r[theirs]), (mine, e[mine], r[theirs])


def test_restatement_matches_the_reference_binary_live():
    """Same comparison on other maps with the binary on two threads: against its report stored as golden case "d", and
    against the binary itself as well when __graft_entry__.build() could compile it into oracle/_ref/salmetric."""
    import os

    g = _golden_cases()["d"]
    mod, (sal, gt) = _maps(g["args"])
    reports = [g["report"]]
    binary = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "oracle", "_ref", "salmetric")
    if os.path.exists(binary):
        reports.append(mod.run_reference(binary, sal, gt, threads=g["threads"]))
    e = sm.evaluate(sal, gt)
    for r in reports:
        for mine, theirs in (("max_f", "Max_F-measre"), ("mean_f", "Mean_F-measre"), ("mae", "MAE"), ("precision", "Precision"), ("recall", "Recall")):
            assert abs(e[mine] - r[theirs]) <= 2e-6 + 2e-6 * abs(r[theirs]), (mine, e[mine], r[theirs])
