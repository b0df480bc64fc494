"""GPU: the device rule (every entry point runs on the device of its CUDA inputs, whatever device is current, and leaves
the caller's current device as it was), per-device weight copies and library state, and FrameStream over several
devices.  Tests that need two devices skip on a machine with one."""
import os
import subprocess
import sys
import textwrap

import pytest
import torch

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
two_devices = pytest.mark.skipif(torch.cuda.device_count() < 2, reason="needs two CUDA devices")
EXAMPLE = os.path.join(ROOT, 'tests', 'golden', 'example')
STAGE2_KEYS = ('depth', 'prob_volume_agg', 'cost_volume_agg', 'depth_views', 'prob_map', 'depth_view_probs')


@pytest.fixture(scope='module')
def A():
    import atvsnet_b200 as A_
    assert torch.cuda.is_available()
    return A_


def _frame(A, seed=0, D=16, h=16, w=24, nv=3):
    cams = torch.from_numpy(A.synthetic.orbit_cams(nv, h, w, D)[None])
    feats = torch.from_numpy(A.synthetic.smooth_features(nv, h, w, 32, seed=seed)[None])
    return feats, cams


def _equal(a, b):
    """torch.equal over the (nested) results of a schedule, on the host"""
    if isinstance(a, dict):
        return set(a) == set(b) and all(_equal(a[k], b[k]) for k in a)
    if isinstance(a, (list, tuple)):
        return len(a) == len(b) and all(_equal(x, y) for x, y in zip(a, b))
    if a is None or b is None:
        return a is None and b is None
    return torch.equal(a.cpu(), b.cpu())


def _all_weights(A):
    w = A.variables.synthetic_weights()
    w.update(A.variables.synthetic_fem_weights())
    w.update(A.variables.synthetic_refine_weights())
    return w


@two_devices
def test_every_kernel_family_runs_on_each_device():
    """in a fresh process, weights loaded once on cuda:0: the fp16 run_multiview with the fused attention kernel, the
    tensor FEM and the four-stage schedule (deconvolution rings, conv3d_tc, conv2d_tc, k_attention_ring) on cuda:0
    and then on cuda:1.  The shared-memory attribute of a kernel is set per device: set once per process, the first
    ring launch on the second device fails."""
    script = textwrap.dedent("""
        import os, sys
        import torch
        sys.path.insert(0, %r)
        import atvsnet_b200 as A
        w = A.variables.synthetic_weights()
        w.update(A.variables.synthetic_fem_weights())
        w.update(A.variables.synthetic_refine_weights())
        A.variables.load_weights(w, device='cuda:0')
        images, cams, _ = A.pipeline.load_example(os.path.join(%r, '0'), view_num=3)
        D = 32
        cf = torch.from_numpy(A.synthetic.orbit_cams(3, 32, 48, D)[None])
        ff = torch.from_numpy(A.synthetic.smooth_features(3, 32, 48, 32, seed=1)[None])
        assert A.network.attention_fused_ok([torch.empty((1, D, 32, 48, 8), dtype=torch.float16)] * 2)
        for dev in ('cuda:0', 'cuda:1'):
            A.pipeline.run_multiview(ff.to(dev), cf.to(dev), D, confidence=True)
            A.FLAGS.fem_tensor = True
            A.fem.extract_features(torch.from_numpy(images).to(dev))
            A.FLAGS.fem_tensor = False
            A.pipeline.run_example_schedule(torch.from_numpy(images).to(dev), torch.from_numpy(cams).to(dev), D)
            torch.cuda.synchronize(dev)
            assert torch.cuda.current_device() == 0
            print('ran on', dev)
        print('ok')
    """ % (ROOT, EXAMPLE))
    r = subprocess.run([sys.executable, '-c', script], capture_output=True, text=True, cwd=ROOT, timeout=900)
    assert r.returncode == 0 and r.stdout.strip().endswith('ok'), r.stdout[-2000:] + r.stderr[-4000:]


@two_devices
def test_run_multiview_on_another_device_than_the_current_one(A):
    A.variables.load_weights(A.variables.synthetic_weights(seed=11, logit_gain=2.0), device='cuda:0')
    f, c = _frame(A)
    torch.cuda.set_device(0)
    for conf in (False, True):
        ref = A.pipeline.run_multiview(f.cuda(0), c.cuda(0), 16, confidence=conf)
        got = A.pipeline.run_multiview(f.cuda(1), c.cuda(1), 16, confidence=conf)
        assert torch.cuda.current_device() == 0
        assert got['depth_up'].device == torch.device('cuda', 1)
        assert _equal(got, ref)


def _max_diff(a, b):
    return float((a.cpu().double() - b.cpu().double()).abs().max())


def _refined_within_spread(runs0, run1, keys):
    """the refined maps are not bit-reproducible even on one device (the FEM and the fp32 statistics sum with atomics):
    cuda:1 against cuda:0 is held to twice the spread of two cuda:0 runs, with a floor of 1e-6 of the value range so
    that two runs that happen to agree exactly do not demand bit equality from the third"""
    for k in keys:
        spread = _max_diff(runs0[0][k], runs0[1][k])
        floor = 1e-6 * float(runs0[0][k].abs().max())
        diff = _max_diff(run1[k], runs0[0][k])
        print("%s: cuda:1 vs cuda:0 %.3e, two cuda:0 runs %.3e" % (k, diff, spread))
        assert diff <= 2 * max(spread, floor), (k, diff, spread)


@two_devices
def test_example_schedules_on_the_second_device(A):
    """example/0 through the four-stage schedule and example/2 through the two-view one, on cuda:1 with cuda:0 current.
    The FEM sums its batch statistics with atomics, so stage II is held to torch.equal on one feature tensor (computed
    once and copied to both devices), and the maps behind the FEM to the spread of two cuda:0 runs."""
    A.variables.load_weights(_all_weights(A), device='cuda:0')
    torch.cuda.set_device(0)
    D = 64
    images, cams, _ = A.pipeline.load_example(os.path.join(EXAMPLE, '0'), view_num=3)
    images, cams = torch.from_numpy(images), torch.from_numpy(cams)
    feats = A.fem.extract_features(images.cuda(0))
    runs0 = [A.pipeline.run_example_schedule(images.cuda(0), cams.cuda(0), D, features=feats, confidence=True)
             for _ in range(2)]
    run1 = A.pipeline.run_example_schedule(images.cuda(1), cams.cuda(1), D, features=feats.to(1), confidence=True)
    assert torch.cuda.current_device() == 0
    for k in STAGE2_KEYS:
        assert _equal(run1[k], runs0[0][k]), k
    _refined_within_spread(runs0, run1, ('depth_refined', 'depth_refined_up', 'refined_prob_map_up'))

    images, cams, _ = A.pipeline.load_example(os.path.join(EXAMPLE, '2'), view_num=3)
    images, cams = torch.from_numpy(images), torch.from_numpy(cams)
    runs0 = [A.pipeline.run_twoview(images.cuda(0), cams.cuda(0), D, confidence=True) for _ in range(2)]
    run1 = A.pipeline.run_twoview(images.cuda(1), cams.cuda(1), D, confidence=True)
    _refined_within_spread(runs0, run1, ('depth_refined', 'depth_refined_up', 'refined_prob_map_up'))


@two_devices
def test_load_weights_replaces_the_copies_on_every_device(A):
    f, c = _frame(A)
    A.variables.load_weights(A.variables.synthetic_weights(seed=11, logit_gain=2.0), device='cuda:0')
    old = A.pipeline.run_multiview(f.cuda(1), c.cuda(1), 16)        # copies and packs the weights on cuda:1
    A.variables.load_weights(A.variables.synthetic_weights(seed=12, logit_gain=2.0), device='cuda:0')
    got = A.pipeline.run_multiview(f.cuda(1), c.cuda(1), 16)
    ref = A.pipeline.run_multiview(f.cuda(0), c.cuda(0), 16)
    assert _equal(got, ref)
    assert not torch.equal(old['depth_up'].cpu(), got['depth_up'].cpu())


@two_devices
def test_inputs_on_different_devices_raise_before_any_launch(A):
    A.variables.load_weights(A.variables.synthetic_weights(seed=11, logit_gain=2.0), device='cuda:0')
    f, c = _frame(A)
    f0, c1 = f.cuda(0), c.cuda(1)
    lib = A._lib.load()
    torch.cuda.synchronize(0)
    torch.cuda.synchronize(1)
    n = lib.atvs_launch_count()
    with pytest.raises(ValueError, match='different devices'):
        A.pipeline.run_multiview(f0, c1, 16)
    with pytest.raises(ValueError, match='different devices'):
        A.model.build_cost_volume(f0[:, 0], f0[:, 1], c1, 16, c1[:, 0, 1, 3, 0], c1[:, 0, 1, 3, 1], 0, 1)
    with pytest.raises(ValueError, match='different devices'):
        A.homography_warping.get_homographies(c.cuda(0)[:, 0], c1[:, 1], 16, 0.1, 0.01)
    assert lib.atvs_launch_count() == n
    assert torch.cuda.current_device() == 0


@two_devices
def test_frame_stream_on_another_device_than_the_current_one(A):
    A.variables.load_weights(A.variables.synthetic_weights(seed=11, logit_gain=2.0), device='cuda:0')
    torch.cuda.set_device(0)
    frames = [tuple(t.pin_memory() for t in _frame(A, seed=s)) for s in range(4)]
    fs = A.pipeline.FrameStream(tuple(frames[0][0].shape), tuple(frames[0][1].shape), 16, 'cuda:1', confidence=True)
    got = [tuple(t.clone() for t in pair) for pair in fs.run(frames)]
    assert torch.cuda.current_device() == 0
    for (fh, ch), (dm, pm) in zip(frames, got):
        ref = A.pipeline.run_multiview(fh.cuda(1), ch.cuda(1), 16, confidence=True)
        assert torch.equal(dm, ref['depth_up'].cpu()) and torch.equal(pm, ref['prob_map_up'].cpu())


def _stream_matches_one_device(A, devices):
    """3K+1 frames over ``devices`` with and without confidence, run twice on the same object: every frame equals what
    a single-device FrameStream returns for it, in order"""
    A.variables.load_weights(A.variables.synthetic_weights(seed=11, logit_gain=2.0), device='cuda:0')
    K = len(devices)
    frames = [tuple(t.pin_memory() for t in _frame(A, seed=s)) for s in range(3 * K + 1)]
    shapes = tuple(frames[0][0].shape), tuple(frames[0][1].shape)
    for conf in (False, True):
        one = A.pipeline.FrameStream(*shapes, 16, 'cuda:0', confidence=conf)
        want = [tuple(t.clone() for t in r) if conf else r.clone() for r in one.run(frames)]
        fs = A.pipeline.FrameStream(*shapes, 16, devices, confidence=conf)
        for _ in range(2):
            got = [tuple(t.clone() for t in r) if conf else r.clone() for r in fs.run(frames)]
            assert len(got) == len(frames)
            assert all(_equal(g, w) for g, w in zip(got, want))
        assert all(lane.graph is not None for lane in fs.lanes)


def test_frame_stream_over_all_visible_devices(A):
    _stream_matches_one_device(A, ['cuda:%d' % i for i in range(torch.cuda.device_count())])


def test_frame_stream_with_a_device_listed_twice(A):
    """a device named twice gets two graphs and two sets of buffers; frames alternate between them"""
    _stream_matches_one_device(A, ['cuda:0', 'cuda:0'])


def test_frame_stream_keeps_the_last_k_results(A):
    """the pinned buffers of frame i are reused by frame i + 2K: the K results a consumer received last stay intact
    while it asks for the next ones"""
    A.variables.load_weights(A.variables.synthetic_weights(seed=11, logit_gain=2.0), device='cuda:0')
    devices = ['cuda:0', 'cuda:0', 'cuda:0']
    K = len(devices)
    frames = [tuple(t.pin_memory() for t in _frame(A, seed=s)) for s in range(3 * K)]
    shapes = tuple(frames[0][0].shape), tuple(frames[0][1].shape)
    want = [r.clone() for r in A.pipeline.FrameStream(*shapes, 16, 'cuda:0').run(frames)]
    held = []
    for i, r in enumerate(A.pipeline.FrameStream(*shapes, 16, devices).run(frames)):
        held = (held + [(i, r)])[-K:]
        for j, buf in held:
            assert torch.equal(buf, want[j]), (i, j)
