"""python tools/confidence_cost.py [--rounds R] [--steps K] [--workload cfg2]

What the confidence maps cost (pipeline.run_multiview(confidence=True), pipeline.FrameStream(confidence=True)) on
bench.py's inputs and weights, one JSON line:
  * the step as a CUDA graph with and without the flag (stage I siamese + stage II + x4 soft-argmin), the two graphs
    replayed alternately (A B B A ...) in R rounds of K steps, so that clock and neighbour drift hit both alike;
  * the soft-argmin launches alone (atvs_prob2depth at x1 and x4 on the step's own aggregated volume) with and without
    the probability-map store, 50 launches per CUDA graph so that host overhead stays out of the time per launch;
  * the same for FrameStream (pinned host frames in, pinned host maps out) and the extra device-to-host bytes per frame.
The card name and power limit are read in the same run."""
import argparse
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import numpy as np  # noqa: E402
import torch  # noqa: E402

import atvsnet_b200 as A  # noqa: E402
from atvsnet_b200.model import _prob2depth  # noqa: E402
from bench import WORKLOADS, capture, make_inputs  # noqa: E402


def card():
    q = subprocess.run(["nvidia-smi", "-i", str(torch.cuda.current_device()), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True)
    return dict(torch_name=torch.cuda.get_device_name(), nvidia_smi=q.stdout.strip() if q.returncode == 0 else None)


def alternate(arms, rounds, steps):
    """arms: dict name -> fn running ONE step; returns name -> list of ms per step, one entry per round"""
    ms = {k: [] for k in arms}
    names = list(arms)
    for r in range(rounds):
        for name in (names if r % 2 == 0 else names[::-1]):
            torch.cuda.synchronize()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record()
            for _ in range(steps):
                arms[name]()
            e1.record()
            torch.cuda.synchronize()
            ms[name].append(e0.elapsed_time(e1) / steps)
    return ms


def summary(t, base='off', other='on'):
    """per arm: mean / min / max over the rounds; other - base paired by round: mean, standard deviation, percent"""
    a, b = np.array(t[base]), np.array(t[other])
    d = b - a
    out = {k: dict(mean=float(np.mean(v)), min=float(np.min(v)), max=float(np.max(v))) for k, v in t.items()}
    out['delta'] = dict(mean=float(d.mean()), std=float(d.std(ddof=1)) if len(d) > 1 else None,
                        pct=float(100 * d.mean() / a.mean()))
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--workload', default='cfg2', choices=list(WORKLOADS))
    ap.add_argument('--rounds', type=int, default=10)
    ap.add_argument('--steps', type=int, default=20)
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit("confidence_cost.py needs a CUDA device")
    dev = torch.device('cuda', 0)
    torch.cuda.set_device(dev)
    A.variables.load_weights(A.variables.synthetic_weights(), device=dev)
    feats, cams, D = make_inputs(args.workload, 0)
    feats_d, cams_d = torch.from_numpy(feats).to(dev), torch.from_numpy(cams).to(dev)

    def step(confidence):
        return A.pipeline.run_multiview(feats_d, cams_d, D, siamese=True, upsample=True, confidence=confidence)

    for _ in range(3):
        step(False)
        step(True)
    g_off, out_off = capture(lambda: step(False), torch)
    g_on, out_on = capture(lambda: step(True), torch)
    same = all(torch.equal(out_off[k], out_on[k]) for k in ('depth', 'depth_up'))
    graph_ms = alternate({'off': g_off.replay, 'on': g_on.replay}, args.rounds, args.steps)

    # the soft-argmin launches alone, on the aggregated volume of the step (10 MB at cfg2: L2-resident, as in the step
    # where the output convolution has just written it)
    vol = out_on['prob_volume_agg']
    ds, di = cams_d[:, 0, 1, 3, 0].contiguous(), cams_d[:, 0, 1, 3, 1].contiguous()
    n = 50
    k4 = {}
    for up in (1, 4):
        for k in ('off', 'on'):
            g, _ = capture(lambda: [_prob2depth(vol, ds, di, up, k == 'on') for _ in range(n)], torch)
            k4['x%d_%s' % (up, k)] = g
    k4_ms = alternate({k: g.replay for k, g in k4.items()}, args.rounds, args.steps)
    k4_us = {k: [1e3 * v / n for v in vs] for k, vs in k4_ms.items()}
    g_off = g_on = out_off = out_on = vol = k4 = None
    torch.cuda.synchronize()
    torch.cuda.empty_cache()

    # FrameStream: pinned host frames in, pinned host depth (and confidence) maps out
    feats_h, cams_h = torch.from_numpy(feats).pin_memory(), torch.from_numpy(cams).pin_memory()
    streams = {k: A.pipeline.FrameStream(tuple(feats_h.shape), tuple(cams_h.shape), D, dev, siamese=True,
                                         confidence=(k == 'on')) for k in ('off', 'on')}
    for fs in streams.values():
        for _ in fs.run([(feats_h, cams_h)] * 3):
            pass
    d2h = {k: sum(t.numel() * t.element_size() for t in fs.lanes[0].host_o[0]) for k, fs in streams.items()}

    def stream_arm(fs):
        def run():
            for _ in fs.run([(feats_h, cams_h)] * args.steps):
                pass
        return run
    fs_ms = alternate({k: stream_arm(fs) for k, fs in streams.items()}, args.rounds, 1)
    fs_ms = {k: [v / args.steps for v in vs] for k, vs in fs_ms.items()}

    nv, H, W, _ = WORKLOADS[args.workload]
    print(json.dumps(dict(
        workload="%s: 1 ref + %d src, %dx%d features, D=%d, stage I siamese + II + x4 soft-argmin, bench.py weights"
                 % (args.workload, nv - 1, H // 4, W // 4, D),
        precision=A.FLAGS.precision, card=card(), rounds=args.rounds, steps_per_round=args.steps,
        depth_equal_with_and_without=same,
        graph_step_ms=summary(graph_ms),
        soft_argmin_alone_us_per_launch=dict(x1=summary({k: k4_us['x1_' + k] for k in ('off', 'on')}),
                                             x4=summary({k: k4_us['x4_' + k] for k in ('off', 'on')})),
        frame_stream_ms_per_frame=summary(fs_ms),
        frame_stream_d2h_bytes_per_frame=d2h, frame_stream_extra_d2h_bytes_per_frame=d2h['on'] - d2h['off'])))


if __name__ == '__main__':
    main()
