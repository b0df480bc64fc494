"""python tools/multi_device_stream.py [--ks 1,2,4,8] [--frames F] [--rounds R] [--workload cfg2]

Frames per second of ONE process streaming bench.py's cfg2 frames over K devices (pipeline.FrameStream with a device
list: frame i on device i mod K, one host thread), end to end from pinned host frames to pinned host depth maps, one
JSON line:
  * per K: maps/s of R runs of F frames per device (K * F frames a run), the order of K alternating between rounds
    (1 2 4 8, 8 4 2 1, ...) so that clock and neighbour drift hit every K alike; host wall clock around FrameStream.run,
    which ends once the last depth map is in host memory;
  * per K, the host side: the time FrameStream spends enqueueing a frame (H2D staging, graph replay, D2H; the pushes of
    the timed runs, timed with the host clock) and the share of the run's wall time the host spends there;
  * per K, the copies alone: one frame's H2D and one depth map's D2H on every device at once, host clock around the
    copies and a synchronise of every device, so that a shared host-memory or PCIe limit shows;
  * the single-process numbers beside the torchrun data-parallel e2e line of profiles/r02d_bench_8gpu.json.
K larger than the visible device count is reported as not measured.  The card names and power limits are read in the
same run."""
import argparse
import json
import os
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

import atvsnet_b200 as A  # noqa: E402
from bench import WORKLOADS, make_inputs  # noqa: E402


def cards(n):
    q = subprocess.run(["nvidia-smi", "--query-gpu=index,name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True)
    return dict(torch_names=[torch.cuda.get_device_name(i) for i in range(n)],
                nvidia_smi=q.stdout.strip().splitlines() if q.returncode == 0 else None)


def summary(xs):
    xs = sorted(xs)
    return dict(median=xs[len(xs) // 2], min=xs[0], max=xs[-1], spread_pct=100.0 * (xs[-1] - xs[0]) / xs[len(xs) // 2],
                runs=len(xs))


def timed_pushes(fs, sink):
    """wrap every device's push so that the host time it takes lands in ``sink``"""
    for lane in fs.lanes:
        def push(fh, ch, _push=lane.push):
            t0 = time.perf_counter()
            r = _push(fh, ch)
            sink.append(time.perf_counter() - t0)
            return r
        lane.push = push


def copy_ms(devices, feats_h, out_h, reps):
    """ms per frame of one H2D frame copy + one D2H depth-map copy issued on every device at once"""
    dev_in = [torch.empty(feats_h.shape, dtype=feats_h.dtype, device=d) for d in devices]
    dev_out = [torch.empty(out_h.shape, dtype=out_h.dtype, device=d) for d in devices]
    hosts = [torch.empty_like(out_h).pin_memory() for _ in devices]
    streams = [torch.cuda.Stream(device=d) for d in devices]

    def once():
        for di, do, ho, s in zip(dev_in, dev_out, hosts, streams):
            with torch.cuda.stream(s):
                di.copy_(feats_h, non_blocking=True)
                ho.copy_(do, non_blocking=True)
        for d in devices:
            torch.cuda.synchronize(d)
    once()
    t0 = time.perf_counter()
    for _ in range(reps):
        once()
    return 1e3 * (time.perf_counter() - t0) / reps


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--ks', default='1,2,4,8')
    ap.add_argument('--frames', type=int, default=100, help='frames per device per run')
    ap.add_argument('--rounds', type=int, default=4)
    ap.add_argument('--workload', default='cfg2', choices=list(WORKLOADS))
    args = ap.parse_args()
    if not torch.cuda.is_available():
        raise RuntimeError("multi_device_stream.py needs CUDA devices")
    n_dev = torch.cuda.device_count()
    ks = [int(k) for k in args.ks.split(',')]
    run_ks = [k for k in ks if k <= n_dev]

    A.variables.load_weights(A.variables.synthetic_weights(), device='cuda:0')     # copied to the others on first use
    feats, cams, D = make_inputs(args.workload, 0)
    feats_h, cams_h = torch.from_numpy(feats).pin_memory(), torch.from_numpy(cams).pin_memory()
    streams, pushes = {}, {}
    for k in run_ks:
        fs = A.pipeline.FrameStream(tuple(feats_h.shape), tuple(cams_h.shape), D, ['cuda:%d' % i for i in range(k)])
        for _ in fs.run([(feats_h, cams_h)] * (3 * k)):      # captures every device's graph
            pass
        pushes[k] = []
        timed_pushes(fs, pushes[k])
        streams[k] = fs

    rate, host_us, host_share = {k: [] for k in run_ks}, {k: [] for k in run_ks}, {k: [] for k in run_ks}
    for r in range(args.rounds):
        for k in (run_ks if r % 2 == 0 else run_ks[::-1]):
            n = k * args.frames
            del pushes[k][:]
            for d in range(k):
                torch.cuda.synchronize(d)
            t0 = time.perf_counter()
            for _ in streams[k].run((feats_h, cams_h) for _ in range(n)):
                pass
            wall = time.perf_counter() - t0
            rate[k].append(n / wall)
            host_us[k].append(1e6 * sum(pushes[k]) / n)
            host_share[k].append(100.0 * sum(pushes[k]) / wall)
    out_h = streams[run_ks[0]].lanes[0].host_o[0][0] if run_ks else None
    copies = {k: copy_ms(['cuda:%d' % i for i in range(k)], feats_h, out_h, 50) for k in run_ks}

    one = summary(rate[1])['median'] if 1 in rate else None
    per_k = {}
    for k in ks:
        if k not in rate:
            per_k[k] = "not measured: %d visible device(s)" % n_dev
            continue
        s = summary(rate[k])
        per_k[k] = dict(maps_per_s=s, vs_one_device=None if one is None else s['median'] / one,
                        host_us_per_frame=summary(host_us[k]), host_share_of_wall_pct=summary(host_share[k]),
                        copies_ms_per_frame_all_devices_at_once=copies[k])
    torchrun = None
    p = os.path.join(ROOT, 'profiles', 'r02d_bench_8gpu.json')
    if os.path.exists(p):
        for line in open(p):
            if line.strip().startswith('{'):
                e2e = json.loads(line).get('e2e', {})
                torchrun = dict(source='profiles/r02d_bench_8gpu.json (bench.py --gpus 8 under torchrun, one process '
                                       'per GPU)', e2e_maps_per_s=e2e.get('value'), ms_per_step=e2e.get('ms_per_step'))
    nv, H, W, _ = WORKLOADS[args.workload]
    print(json.dumps(dict(
        workload="%s: 1 ref + %d src, %dx%d features, D=%d, stage I siamese + II + x4 soft-argmin, bench.py weights, "
                 "FrameStream from pinned host frames to pinned host depth maps" % (args.workload, nv - 1, H // 4, W // 4, D),
        precision=A.FLAGS.precision, cards=cards(n_dev), visible_devices=n_dev, frames_per_device_per_run=args.frames,
        rounds=args.rounds, h2d_bytes_per_frame=feats_h.numel() * 4 + cams_h.numel() * 4,
        d2h_bytes_per_frame=None if out_h is None else out_h.numel() * 4, per_k=per_k, torchrun_dp_8gpu=torchrun)))


if __name__ == '__main__':
    main()
