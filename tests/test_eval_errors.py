"""calc_error (a-tvsnet_b200/eval_errors.py) against the ONLY reference-produced known answers the repository
ships: example/{0,1,2}/result/pred.npy evaluated against 0_gt.npy by the reference itself and written to
result/error.xlsx (example.py:196-216).  The xlsx values are committed in tests/golden/reference_error_xlsx.json;
the 2.4 MB arrays per scene are not: they are read from the reference checkout named by ATVS_REFERENCE_DIR (a clone of
daiszh/A-TVSNet), and the test is skipped without one.  test_calc_error_known_answers pins every metric without it."""
import importlib.util
import json
import os

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = os.environ.get('ATVS_REFERENCE_DIR', '')


def _mod():
    spec = importlib.util.spec_from_file_location('atvs_eval_errors', os.path.join(ROOT, 'a-tvsnet_b200', 'eval_errors.py'))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


@pytest.mark.parametrize('ex', [0, 1, 2])
def test_calc_error_matches_reference_xlsx(ex):
    pred_p = os.path.join(REF, 'example/%d/result/pred.npy' % ex)
    if not REF or not os.path.exists(pred_p):
        pytest.skip('set ATVS_REFERENCE_DIR to a reference checkout with its example/ outputs')
    m = _mod()
    gold = json.load(open(os.path.join(ROOT, 'tests/golden/reference_error_xlsx.json')))['example/%d' % ex]
    pred = np.squeeze(np.load(pred_p))
    gt = np.squeeze(np.load(os.path.join(REF, 'example/%d/0_gt.npy' % ex)))
    err, info = m.calc_error(pred, gt)
    names = m.err_metrics_namelist + m.acc_metrics_namelist
    assert len(err) == len(names) == 14
    for k, v in zip(names, err):
        assert abs(float(v) - gold[k]) <= 2e-6 * max(1.0, abs(gold[k])), (k, float(v), gold[k])


def _restated(pred, gt, num_depths=100, thresholds=(1, 3, 5, 10)):
    """the 14 metrics of the reference's calc_error restated directly from their definitions, in float64, over the
    pixels where both depths lie in (0, 1e10); the interval is the range of the valid ground truth / num_depths."""
    pred = np.nan_to_num(pred.astype(np.float64), nan=0.0)
    gt = np.nan_to_num(gt.astype(np.float64), nan=0.0)
    gt_ok = (gt > 0) & (gt < 1e10)
    interval = (gt[gt_ok].max() - gt[gt_ok].min()) / num_depths
    ok = gt_ok & (pred > 0) & (pred < 1e10)
    g, p = gt[ok], pred[ok]
    d, inv, lg = np.abs(g - p), np.abs(1 / g - 1 / p), np.log(g) - np.log(p)
    e = [d.mean(), np.sqrt((d ** 2).mean()), inv.mean(), np.sqrt((inv ** 2).mean()), np.abs(lg).mean(),
         np.sqrt((lg ** 2).mean()), np.sqrt((lg ** 2).mean() - lg.mean() ** 2), (d / g).mean(), (d ** 2 / g ** 2).mean(),
         d.mean() / interval]
    return np.array(e + [(d / interval < t).mean() for t in thresholds]), interval


def test_calc_error_known_answers():
    m = _mod()
    names = m.err_metrics_namelist + m.acc_metrics_namelist
    # by hand: gt (1, 2, 4), pred 2 everywhere, interval (4 - 1) / 100
    l2 = np.log(2.0)
    hand = [1.0, np.sqrt(5 / 3), 0.25, np.sqrt(0.3125 / 3), 2 * l2 / 3, l2 * np.sqrt(2 / 3), l2 * np.sqrt(2 / 3), 0.5,
            1.25 / 3, 1 / 0.03, 1 / 3, 1 / 3, 1 / 3, 1 / 3]
    e, info = m.calc_error(np.float32([[2, 2, 2]]), np.float32([[1, 2, 4]]))
    for k, got, want in zip(names, e, hand):
        assert abs(got - want) <= 1e-6 * max(1.0, want), (k, got, want)
    assert abs(info[1] - 0.03) < 1e-7
    # seeded map: multiplicative error with a bias (the scale-invariant term differs from log rmse), spread so that
    # every inlier ratio lies strictly between 0 and 1, and invalid pixels of every kind
    rng = np.random.default_rng(3)
    gt = rng.uniform(2.0, 12.0, (60, 80)).astype(np.float32)
    pred = (gt * np.exp(0.05 + 0.1 * rng.standard_normal(gt.shape))).astype(np.float32)
    pred[0, :5] = np.nan
    pred[1, :5] = -1.0
    gt[0, 0], gt[1, 0] = 1.0, 15.0      # the interval spans the valid ground truth, also where the prediction is not
    gt[2, :5] = 0.0
    gt[3, :5] = 1e11
    gt[4, :5] = np.nan
    want, interval = _restated(pred, gt)
    assert all(0.05 < r < 0.95 for r in want[10:]) and want[6] < 0.99 * want[5]
    e, info = m.calc_error(pred, gt)
    for k, got, w in zip(names, e, want):
        assert abs(got - w) <= 2e-5 * max(1.0, abs(w)), (k, got, w)
    assert abs(info[1] - interval) < 1e-6


def test_calc_error_properties():
    m = _mod()
    rng = np.random.default_rng(0)
    gt = rng.uniform(2.0, 12.0, (40, 50)).astype(np.float32)
    e, info = m.calc_error(gt.copy(), gt)
    assert np.all(e[:10] == 0) and np.all(e[10:] == 1.0)
    pred = gt + 0.5
    pred[0, 0] = np.nan          # NaN prediction and non-positive / huge ground truth are excluded
    g2 = gt.copy()
    g2[1, 1] = 0.0
    g2[2, 2] = 1e11
    e, info = m.calc_error(pred, g2)
    assert abs(e[0] - 0.5) < 1e-6 and abs(e[1] - 0.5) < 1e-6
    interval = (g2[(g2 > 0) & (g2 < 1e10)].max() - g2[(g2 > 0) & (g2 < 1e10)].min()) / 100.0
    assert abs(info[1] - interval) < 1e-9 and abs(e[9] - 0.5 / interval) < 1e-3
    with pytest.raises(AssertionError):
        m.calc_error(pred[:5], g2)
