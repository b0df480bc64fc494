"""GPU: the probability (confidence) maps the schedules return with ``confidence=True`` (get_propability_map,
model.py:13-65, through prob2depth(_upsample)(out_prob_map=True), model.py:80-129), against the CPU oracle, and the
promise that the flag changes nothing else.

Two comparisons per map:
  * soft-argmin parity: the map against the oracle's prob2depth(out_prob_map=True) applied to the volume the CUDA
    schedule itself produced (returned beside it), i.e. the right map from the right launch;
  * end to end: the map against the oracle's prob2depth applied to the oracle's own volume.
Where the estimate sits close to an integer plane index, a last-bit difference in the depth moves the 4-tap window of
get_propability_map by one plane, and that pixel's confidence by a whole tap: such pixels are counted, not bounded.
A confidence lies in [0, 3] (to fp32 rounding of the 4-tap sum): the window is clamped to the swept planes, so at an end
plane three of its taps coincide."""
import os

import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
MV_KEYS = {'depth', 'depth_up', 'prob_volume_agg', 'cost_volume_agg', 'depth_views'}
CONF_KEYS = {'prob_map', 'prob_map_up', 'depth_view_probs'}
CONF_MAX = 3 + 1e-5


def cu(x):
    return torch.from_numpy(np.ascontiguousarray(x)).cuda()


def npy(t):
    return t.detach().float().cpu().numpy()


@pytest.fixture(scope='module')
def A():
    import atvsnet_b200 as A_
    assert torch.cuda.is_available()
    return A_


def _ranges(cams):
    return cams[:, 0, 1, 3, 0], cams[:, 0, 1, 3, 1]


def _precision(A, prec, fn):
    A.FLAGS.precision = prec
    try:
        out = fn()
        torch.cuda.synchronize()
    finally:
        A.FLAGS.precision = A.flags.DEFAULT_PRECISION
    return out


def _stats(got, want):
    """(max |diff|, mean |diff|, fraction of pixels off by more than 1e-5)"""
    d = np.abs(npy(got) - want)
    return float(d.max()), float(d.mean()), float((d > 1e-5).mean())


def _oracle_reverse_probs(om, feats, cams, D, weights):
    """the confidence of every depth_view: the reverse pass of oracle TVSNet_base_siamese (view_i as reference)
    with prob2depth(out_prob_map=True)"""
    ds, di = _ranges(cams)
    probs = []
    for v in range(1, cams.shape[1]):
        cvv = om.build_cost_volume(feats[:, v], feats[:, 0], cams, D, ds, di, ref_id=v, view_id=0)
        probs.append(om.prob2depth(om.cost_volume_reasoning(cvv, weights), D, ds, di, out_prob_map=True)[1])
    return probs


def _multiview_case(A, D, h, w, gain):
    """_e2e_inputs of test_gpu_parity.py (3 views) with the oracle's stage-II and reverse-pass confidence maps"""
    from oracle import model as om
    cams = A.synthetic.orbit_cams(3, h, w, D)[None]
    feats = A.synthetic.smooth_features(3, h, w, 32, seed=3)[None]
    weights = A.variables.synthetic_weights(seed=11, logit_gain=gain)
    ds, di = _ranges(cams)
    ref = om.run_multiview_stage12(feats, cams, D, weights, siamese=True)
    _, _, pm, pm_up = om.prob2depth_upsample(ref['prob_volume_agg'], D, ds, di, out_prob_map=True)
    return dict(D=D, cams=cams, feats=feats, weights=weights, ref=ref, prob_map=pm, prob_map_up=pm_up,
                depth_view_probs=_oracle_reverse_probs(om, feats, cams, D, weights))


@pytest.fixture(scope='module')
def small_case(A):
    """D = 16, 16x24, logit gain 2: the case of test_gpu_parity.py::test_multiview_pipeline_fp32_and_16bit"""
    return _multiview_case(A, 16, 16, 24, 2.0)


@pytest.fixture(scope='module')
def large_case(A):
    """D = 64, 64x80 with the weights bench.py times (logit gain 4): the case of
    test_gpu_parity.py::test_multiview_pipeline_16bit_depth_mae.  The 16-bit path is checked here, where the deepest
    U-Net level keeps 8x8x10 voxels for its batch statistics (8 at 16x24x16)."""
    return _multiview_case(A, 64, 64, 80, 4.0)


def _check_run_multiview(A, c, prec):
    from oracle import model as om
    D, cams = c['D'], c['cams']
    ds, di = _ranges(cams)
    A.variables.load_weights(c['weights'])
    out = _precision(A, prec, lambda: A.pipeline.run_multiview(cu(c['feats']), cu(cams), D, siamese=True, confidence=True))
    assert set(out) == MV_KEYS | CONF_KEYS
    assert tuple(out['prob_map'].shape) == tuple(out['depth'].shape)
    assert tuple(out['prob_map_up'].shape) == tuple(out['depth_up'].shape)
    assert len(out['depth_view_probs']) == len(out['depth_views']) == 2
    for m in (out['prob_map'], out['prob_map_up']) + tuple(out['depth_view_probs']):
        assert float(m.min()) >= 0 and float(m.max()) <= CONF_MAX
    # soft-argmin parity on the schedule's own volume
    _, _, opm, opm_up = om.prob2depth_upsample(npy(out['prob_volume_agg']), D, ds, di, out_prob_map=True)
    k4 = [_stats(out['prob_map'], opm), _stats(out['prob_map_up'], opm_up)]
    # end to end against the oracle's volumes
    e2e = [_stats(out['prob_map'], c['prob_map']), _stats(out['prob_map_up'], c['prob_map_up'])]
    e2e += [_stats(a, b) for a, b in zip(out['depth_view_probs'], c['depth_view_probs'])]
    print("%s D=%d confidence (max, mean, fraction > 1e-5): on its own volume %s; against the oracle's volumes "
          "prob_map, prob_map_up, depth_view_probs %s" % (prec, D, k4, e2e))
    for mx, mean, frac in k4:
        assert frac < 1e-3, k4
    return e2e


def test_run_multiview_confidence_fp32(A, small_case):
    for mx, mean, frac in _check_run_multiview(A, small_case, 'fp32'):
        assert mx < 1e-5


@pytest.mark.parametrize('prec,tol,tol_views', [('fp16', 1e-3, 2e-3), ('bf16', 8e-3, 1.6e-2)])
def test_run_multiview_confidence_16bit(A, large_case, prec, tol, tol_views):
    """mean error bounded, not the max: a 16-bit estimate that crosses an integer plane index moves that pixel's
    confidence by a whole tap.  fp16 (the default): stage-II maps within 1e-3 (measured 6.0e-4, 4.4e-4 x4), the maps
    of the single-pair reverse passes within 2e-3 (measured 1.0e-3, 1.5e-3).  bf16 storage is held to 8x those bounds,
    the ratio of its rounding unit to fp16's (2^-8 / 2^-11; measured 5.2e-3, 3.0e-3 and 1.1e-2, 1.0e-2)."""
    e2e = _check_run_multiview(A, large_case, prec)
    for mx, mean, frac in e2e[:2]:
        assert mean < tol, e2e
    for mx, mean, frac in e2e[2:]:
        assert mean < tol_views, e2e


def test_run_multiview_flag_changes_nothing_else(A, small_case):
    c = small_case
    A.variables.load_weights(c['weights'])
    f, cm = cu(c['feats']), cu(c['cams'])
    for siamese in (True, False):
        off = A.pipeline.run_multiview(f, cm, c['D'], siamese=siamese)
        on = A.pipeline.run_multiview(f, cm, c['D'], siamese=siamese, confidence=True)
        assert set(off) == MV_KEYS and set(on) == MV_KEYS | CONF_KEYS
        for k in ('depth', 'depth_up', 'prob_volume_agg', 'cost_volume_agg'):
            assert torch.equal(off[k], on[k]), k
        if siamese:
            assert all(torch.equal(a, b) for a, b in zip(off['depth_views'], on['depth_views']))
        else:
            assert off['depth_views'] == on['depth_views'] == on['depth_view_probs'] == [None, None]
    low = A.pipeline.run_multiview(f, cm, c['D'], upsample=False, confidence=True)
    assert set(low) == MV_KEYS - {'depth_up'} | CONF_KEYS - {'prob_map_up'}


@pytest.mark.parametrize('prec,case', [('fp32', 'small_case'), ('fp16', 'large_case')])
def test_confidence_feeds_probability_filter(A, request, prec, case):
    """fusion.probability_filter (depth_fusion.py:183-202, threshold 0.8 as in reproduce_pc.sh) keeps the same pixels
    on the schedule's maps as on the oracle's; on the 16-bit path pixels near the threshold may flip."""
    c = request.getfixturevalue(case)
    A.variables.load_weights(c['weights'])
    out = _precision(A, prec, lambda: A.pipeline.run_multiview(cu(c['feats']), cu(c['cams']), c['D'], confidence=True))
    got = A.fusion.probability_filter(out['depth_up'], out['prob_map_up'], 0.8) > 0
    want = A.fusion.probability_filter(cu(c['ref']['depth_agg_init_up']), cu(c['prob_map_up']), 0.8) > 0
    kept = float(want.float().mean())
    differ = float((got != want).float().mean())
    print("%s D=%d probability filter at 0.8: oracle keeps %.3f of the pixels, masks differ on %.2e"
          % (prec, c['D'], kept, differ))
    assert 0.02 < kept < 0.98          # the threshold splits the map: the comparison is not vacuous
    if prec == 'fp32':
        assert torch.equal(got, want)
    else:
        assert differ < 2e-3, differ           # measured 1.6e-4


def _same_depth_without_map(A, volume, cams, depth, depth_up):
    """the depth maps a confidence run returned equal the soft-argmin WITHOUT the map on the same volume.  (Two runs of
    the refinement schedules are not compared bit for bit: the fp32 CUDA-core layers and the 2-D feature extractor sum
    their batch statistics with atomics, in no fixed order.)"""
    from atvsnet_b200.model import _prob2depth
    ds, di = (cu(r) for r in _ranges(cams))
    assert torch.equal(depth, _prob2depth(volume, ds, di, 1, False)[0])
    assert torch.equal(depth_up, _prob2depth(volume, ds, di, 4, False)[0])


@pytest.fixture(scope='module')
def refine_case(A):
    """the 3-view images-in case of test_gpu_refine.py::test_four_stage_schedule_fp32_against_oracle"""
    from gen_common import fem_weights, named_weights
    rng = np.random.default_rng(17)
    nv, H, W, D = 3, 32, 64, 8
    imgs = (127.5 + 50 * rng.standard_normal((1, nv, H, W, 3))).clip(0, 255).astype(np.float32)
    cams = A.synthetic.orbit_cams(nv, H // 4, W // 4, D)[None]
    allw = A.variables.synthetic_weights(seed=11, logit_gain=2.0)
    allw.update(fem_weights(7))
    allw.update(named_weights('refine_variables.json', 5))
    return dict(D=D, imgs=imgs, cams=cams, weights=allw)


def test_four_stage_schedule_confidence_fp32(A, refine_case):
    from oracle import model as om
    from oracle import schedule as osch
    c = refine_case
    D, imgs, cams = c['D'], c['imgs'], c['cams']
    ds, di = _ranges(cams)
    ref = osch.run_multiview(imgs, cams, D, c['weights'])
    _, _, rpm, rpm_up = om.prob2depth_upsample(ref['refined_prob_volume_agg'], D, ds, di, out_prob_map=True)
    A.variables.load_weights(c['weights'])
    out = _precision(A, 'fp32', lambda: A.pipeline.run_example_schedule(cu(imgs), cu(cams), D, confidence=True))
    off = _precision(A, 'fp32', lambda: A.pipeline.run_example_schedule(cu(imgs), cu(cams), D))
    assert set(out) - set(off) == {'prob_map', 'depth_view_probs', 'refined_prob_map', 'refined_prob_map_up'}
    assert tuple(out['refined_prob_map_up'].shape) == tuple(out['depth_refined_up'].shape)
    _same_depth_without_map(A, out['refined_prob_volume_agg'], cams, out['depth_refined'], out['depth_refined_up'])
    _, _, opm, opm_up = om.prob2depth_upsample(npy(out['refined_prob_volume_agg']), D, ds, di, out_prob_map=True)
    k4 = [_stats(out['refined_prob_map'], opm), _stats(out['refined_prob_map_up'], opm_up)]
    e2e = [_stats(out['refined_prob_map'], rpm), _stats(out['refined_prob_map_up'], rpm_up)]
    print("four-stage refined confidence (max, mean, fraction > 1e-5): on its own volume %s; against the oracle's %s"
          % (k4, e2e))
    for mx, mean, frac in k4:
        assert frac < 1e-3, k4
    for mx, mean, frac in e2e:
        assert mean < 1e-3, e2e


def test_twoview_confidence_fp32(A, refine_case):
    from oracle import model as om
    from oracle import schedule as osch
    c = refine_case
    D, imgs, cams = c['D'], c['imgs'][:, :2], c['cams'][:, :2]
    ds, di = _ranges(cams)
    ref = osch.run_twoview(imgs, cams, D, c['weights'])
    _, _, rpm, rpm_up = om.prob2depth_upsample(ref['refined_prob_volume'], D, ds, di, out_prob_map=True)
    A.variables.load_weights(c['weights'])
    out = _precision(A, 'fp32', lambda: A.pipeline.run_twoview(cu(imgs), cu(cams), D, confidence=True))
    assert set(out) == {'refined_prob_volume', 'depth_refined', 'depth_refined_up', 'refined_prob_map',
                        'refined_prob_map_up'}
    _same_depth_without_map(A, out['refined_prob_volume'], cams, out['depth_refined'], out['depth_refined_up'])
    _, _, opm, opm_up = om.prob2depth_upsample(npy(out['refined_prob_volume']), D, ds, di, out_prob_map=True)
    k4 = [_stats(out['refined_prob_map'], opm), _stats(out['refined_prob_map_up'], opm_up)]
    e2e = [_stats(out['refined_prob_map'], rpm), _stats(out['refined_prob_map_up'], rpm_up)]
    print("two-view refined confidence (max, mean, fraction > 1e-5): on its own volume %s; against the oracle's %s"
          % (k4, e2e))
    for mx, mean, frac in k4:
        assert frac < 1e-3, k4
    for mx, mean, frac in e2e:
        assert mean < 1e-3, e2e


def test_run_example_twoview_returns_prob(A):
    """tests/golden/example/2 (two views, 640x480): ``prob`` beside ``pred``, the depth map unchanged by the flag.  With
    these synthetic weights some pixels sit at an end of the swept range, where the confidence reaches 3."""
    D = 128
    images, cams, _ = A.pipeline.load_example(os.path.join(ROOT, 'tests', 'golden', 'example', '2'), view_num=3)
    w = A.variables.synthetic_weights()
    w.update(A.variables.synthetic_fem_weights())
    w.update(A.variables.synthetic_refine_weights())
    A.variables.load_weights(w)
    out = A.pipeline.run_example(cu(images), cu(cams), D, confidence=True)
    off = A.pipeline.run_example(cu(images), cu(cams), D)
    torch.cuda.synchronize()
    assert set(out) - set(off) == {'refined_prob_map', 'refined_prob_map_up', 'prob'}
    assert tuple(out['prob'].shape) == tuple(out['pred'].shape) == (1, 480, 640, 1)
    assert torch.equal(out['prob'], out['refined_prob_map_up'])
    _same_depth_without_map(A, out['refined_prob_volume'], cams, out['depth_refined'], out['depth_refined_up'])
    assert torch.equal(out['pred'], A.pipeline.inverse_to_depth(out['depth_refined_up'], twoview=True))
    p = npy(out['prob'])
    print("example/2 confidence: min %.3f mean %.3f max %.3f" % (p.min(), p.mean(), p.max()))
    assert np.isfinite(p).all() and p.min() >= 0 and p.max() <= CONF_MAX


def test_frame_stream_confidence_matches_run_multiview(A):
    """FrameStream(confidence=True): every (depth, confidence) pair, in order, equals the eager call on that frame"""
    D, h, w, nv = 16, 16, 24, 3
    A.variables.load_weights(A.variables.synthetic_weights(seed=11, logit_gain=2.0))
    assert A.FLAGS.precision == A.flags.DEFAULT_PRECISION
    cams = torch.from_numpy(A.synthetic.orbit_cams(nv, h, w, D)[None])
    frames = [(torch.from_numpy(A.synthetic.smooth_features(nv, h, w, 32, seed=s)[None]).pin_memory(), cams.pin_memory())
              for s in range(5)]
    fs = A.pipeline.FrameStream(tuple(frames[0][0].shape), tuple(cams.shape), D, 'cuda:0', siamese=True, confidence=True)
    got = []
    for pair in fs.run(frames):
        assert isinstance(pair, tuple) and len(pair) == 2 and all(t.is_pinned() for t in pair)
        got.append(tuple(t.clone() for t in pair))
    assert len(got) == 5
    for (fh, ch), (dm, pm) in zip(frames, got):
        ref = A.pipeline.run_multiview(fh.cuda(), ch.cuda(), D, siamese=True, confidence=True)
        assert torch.equal(dm, ref['depth_up'].cpu()) and torch.equal(pm, ref['prob_map_up'].cpu())
    # a second pass through the same object reuses the captured graph
    graph = fs.graph
    again = [tuple(t.clone() for t in pair) for pair in fs.run(frames[:2])]
    assert fs.graph is graph
    for a, b in zip(again, got[:2]):
        assert torch.equal(a[0], b[0]) and torch.equal(a[1], b[1])
    # without the flag the stream still yields bare depth maps, the same ones
    plain = A.pipeline.FrameStream(tuple(frames[0][0].shape), tuple(cams.shape), D, 'cuda:0', siamese=True)
    bare = [dm.clone() for dm in plain.run(frames[:3])]
    assert all(isinstance(dm, torch.Tensor) for dm in bare)
    assert all(torch.equal(a, b[0]) for a, b in zip(bare, got[:3]))
