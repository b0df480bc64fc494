#!/usr/bin/env python
"""bench.py - depth maps / s of the A-TVSNet inference hot path on B200.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference]
                    [--workload cfg2|cfg3|cfg4] [--precision fp16|bf16|fp32] [--no-graph] [--dump-outputs DIR]
                    [--ref-budget-s S]

One "step" = one depth map of the workload: stage I (TVSNet_base_siamese: fused warp + cost volume -> 3-D CNN
regularisation -> soft-argmin, forward and reverse direction) for every source view, stage II (attention aggregation
-> output conv) and the final x4 upsampled soft-argmin, i.e. example.py:144-158 + :109 with features in.

N = 1   : cfg2 (1 ref + 4 src, 640x512 images -> 128x160 features, D = 128).  The line also carries, as declared extra
          fields, the same depth map FROM IMAGES (2-D feature extractor included) and the whole four-stage example.py
          schedule (refinement included), the roofline of the dominant kernel, K1 / K4 against the HBM peak and the CPU
          oracle timed on the host cores.
N > 1   : independent reference frames data-parallel, one frame stream per rank, no data-path collective ("scaling":
          "weak");  the SAME invocation then also runs cfg3 - ONE 1920x1056, D=256 frame whose 8 source views are
          sharded over the ranks, completed with an NCCL max + reduce-scatter + all-gather - and reports it under
          "sharded" (with the same frame on rank 0 alone beside it).  --workload cfg3 makes that the headline instead.
--impl reference : the CPU oracle (NumPy/torch-CPU restatement of the TF-1.5 reference, which cannot be installed
          offline) on all host cores; each step is the FULL workload (every depth plane, every view, ~30 s at cfg2); all
          --steps are timed unless --ref-budget-s S stops the run once the next step would end after S seconds (the
          JSON line says how many were timed).
--dump-outputs DIR : after the timed steps, rank 0 writes what the last timed step returned (the run_multiview dict)
          as DIR/<name>.npy, so that two builds can be compared output for output on the same seeded inputs.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

WORKLOADS = {
    # name: (n_views, H, W, D)   image resolution; features are H/4 x W/4 x 32
    'cfg2': (5, 512, 640, 128),
    'cfg3': (9, 1056, 1920, 256),
    'cfg4': (5, 512, 640, 192),
}
METRIC = "depth maps/sec"
CRM_MAC_PER_VOXEL = 29592          # SURVEY.md 8(a) a6
# --dump-outputs: an array above DUMP_MAX_ELEMS elements is stored as a seeded sample of that many (8 MB as float32);
# the five arrays of a step then stay under DUMP_MAX_BYTES even at cfg3
DUMP_MAX_ELEMS = 1 << 21
DUMP_MAX_BYTES = 64 << 20


def peaks():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return dict(hbm=d['hbm_gbs'], bf16=d['bf16_tflops'], bf16_sustained=d['bf16_tflops_sustained'], src='measured')
    return dict(hbm=6650.0, bf16=1590.0, bf16_sustained=1400.0, src='fallback')


class ClockSampler(object):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.rows, self.proc, self.idx, self.skip = [], None, gpu_index, 0

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.idx), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(',')])

    def wait_first(self, timeout=8.0):
        """block until nvidia-smi delivers its first sample (its start-up takes 0.1-1 s, longer with 8 ranks starting one
        each), then forget what was sampled so far: everything kept from here on falls inside the timed region."""
        if self.proc is None:
            return
        t0 = time.time()
        while not self.rows and time.time() - t0 < timeout:
            time.sleep(0.01)
        self.skip = len(self.rows)

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        for r in self.rows[self.skip:]:
            try:
                sm.append(float(r[1]))
                mx = float(r[2])
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                pass
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def make_inputs(workload, frame_seed):
    import atvsnet_b200 as A
    nv, H, W, D = WORKLOADS[workload]
    h, w = H // 4, W // 4
    cams = A.synthetic.orbit_cams(nv, h, w, D)[None]
    feats = A.synthetic.smooth_features(nv, h, w, 32, seed=frame_seed)[None]
    return feats, cams, D


def common_config(workload, world, sharded):
    """the `config` object BOTH arms print: names the workload and how it is spread over the GPUs, nothing arm-specific"""
    nv, H, W, D = WORKLOADS[workload]
    return {"workload": "%s: 1 ref + %d src, %dx%d images -> %dx%dx32 features in, D=%d, stages I (siamese) + II + x4 "
                        "soft-argmin" % (workload, nv - 1, W, H, H // 4, W // 4, D),
            "frames_per_step": 1 if sharded else world,
            "parallelism": ("source views of one frame sharded over %d ranks, NCCL all-reduce(max) + reduce-scatter(sum) + "
                            "all-gather" % world) if sharded else ("dp%d: independent frames per rank, no collective" % world),
            "l2": "no explicit flush: every step streams > 3 GB of intermediate volumes through HBM (L2 = 126 MB)"}


# ============================================================================ reference arm
def run_reference(args, rank, world):
    """The reference's CPU implementation of the path = the oracle port (TF 1.5 / py2.7 cannot be installed offline), all
    host cores, FULL workload per step (all depth planes, all source views, siamese stage I + stage II + x4 soft-argmin)."""
    if rank != 0:
        return
    import numpy as np
    import torch
    import atvsnet_b200 as A
    from oracle import model as om
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)            # torchrun exports OMP_NUM_THREADS=1: undo it, rank 0 owns the host here
    workload = args.workload or 'cfg2'
    sharded = workload == 'cfg3' and world > 1
    feats, cams, D = make_inputs(workload, 0)
    weights = A.variables.synthetic_weights()
    nv, H, W, _ = WORKLOADS[workload]
    ds, di = cams[:, 0, 1, 3, 0], cams[:, 0, 1, 3, 1]
    om.TVSNet_base(feats[:, :2, :16, :16], cams, 8, ds, di, 1, weights)          # touch the code paths (not a step)
    times, warm = [], []
    t_run = time.perf_counter()
    nwarm = min(args.warmup, 1)             # a full-size CPU step is ~30 s: one warm-up step at most
    steps = args.steps
    i = 0
    while i < nwarm + steps:
        t0 = time.perf_counter()
        om.run_multiview_stage12(feats, cams, D, weights, siamese=True)
        dt = time.perf_counter() - t0
        (warm if i < nwarm else times).append(dt)
        i += 1
        if (args.ref_budget_s is not None and i >= nwarm + 1
                and time.perf_counter() - t_run + dt > args.ref_budget_s):
            break                           # opt-in bounded run: stop once the next step would cross the budget
    t = float(np.mean(times))
    value = 1.0 / t
    budget = "" if args.ref_budget_s is None else " inside a %.0f s budget" % args.ref_budget_s
    sample = ("full %s workload per step (all %d depth planes, %d source views, %dx%d features), %d of %d requested steps "
              "timed%s, %d warm-up step(s)" % (workload, D, nv - 1, H // 4, W // 4, len(times), args.steps, budget,
                                               len(warm)))
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": value, "unit": "depth maps/s", "n_gpus": args.gpus,
        "steps": len(times), "steps_requested": args.steps, "warmup": len(warm), "ms_per_step": 1e3 * t,
        "higher_is_better": True, "scaling": "strong" if sharded else "weak", "vs_baseline": None, "dtype": "f32",
        "data": "synthetic", "config": common_config(workload, world, sharded),
        "cpu_baseline": {"value": value, "unit": "depth maps/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "depth maps/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }))


# ============================================================================ our arm
def capture(step_fn, torch):
    """CUDA-graph capture of one step (after eager warm-up by the caller) -> (graph, output tensor)."""
    torch.cuda.synchronize()
    torch.cuda.empty_cache()        # the eager warm-up's cached blocks would sit beside the graph's private pool (cfg3: 2 x 80 GB)
    s = torch.cuda.Stream()
    s.wait_stream(torch.cuda.current_stream())
    with torch.cuda.stream(s):
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph, stream=s):
            out = step_fn()
    torch.cuda.current_stream().wait_stream(s)
    for _ in range(2):
        graph.replay()
    torch.cuda.synchronize()
    return graph, out


def dump_outputs(out, directory):
    """write one step's result (the run_multiview dict) as directory/<name>.npy, float32 (float64 stays float64);
    depth_views is stacked along a new leading axis.  An array of more than DUMP_MAX_ELEMS elements is replaced by
    that many of its flattened elements at sorted indices drawn with a fixed seed: the same indices in every run."""
    import numpy as np
    import torch
    arrays = {}
    for name, t in out.items():
        if isinstance(t, list):
            if any(x is None for x in t):
                continue                    # depth_views of a step without the reverse passes
            t = torch.stack(t)
        t = t.detach()
        if t.numel() > DUMP_MAX_ELEMS:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), DUMP_MAX_ELEMS, replace=False))
            t = t.reshape(-1)[torch.from_numpy(idx).to(t.device)]
        t = t.double() if t.dtype == torch.float64 else t.float()
        arrays[name] = t.cpu().numpy()
    total = sum(a.nbytes for a in arrays.values())
    if total > DUMP_MAX_BYTES:
        raise RuntimeError("bench: %d bytes of outputs exceed the %d-byte dump limit" % (total, DUMP_MAX_BYTES))
    os.makedirs(directory, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(directory, name + '.npy'), a)


def timed_steps(fn, steps, torch, barrier):
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        res = fn()
    e1.record()
    barrier()
    return e0.elapsed_time(e1), res


def run_ours(args, rank, world, local_rank):
    import numpy as np
    import torch
    import torch.distributed as dist
    import atvsnet_b200 as A
    from atvsnet_b200 import network as N

    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    lib = A._lib.load()
    A.FLAGS.precision = args.precision
    A.FLAGS.raw_dtype = args.raw_dtype
    workload = args.workload or 'cfg2'
    sharded = workload == 'cfg3' and world > 1
    group = dist.group.WORLD if sharded else None
    allw = A.variables.synthetic_weights()
    allw.update(A.variables.synthetic_fem_weights())
    allw.update(A.variables.synthetic_refine_weights())
    A.variables.load_weights(allw, device=dev)
    feats, cams, D = make_inputs(workload, frame_seed=rank if not sharded else 0)
    nv, H, W, _ = WORKLOADS[workload]
    h, w = H // 4, W // 4
    V = D * h * w

    # pinned host buffers (end-to-end path) and resident device inputs (kernel path)
    feats_h = torch.from_numpy(feats).pin_memory()
    cams_h = torch.from_numpy(cams).pin_memory()
    feats_d = torch.empty_like(feats_h, device=dev)
    cams_d = torch.empty_like(cams_h, device=dev)
    feats_d.copy_(feats_h)
    cams_d.copy_(cams_h)
    depth_h = torch.empty((1, H, W, 1), dtype=torch.float32).pin_memory()

    def step():
        return A.pipeline.run_multiview(feats_d, cams_d, D, siamese=True, upsample=True, group=group, rank=rank,
                                        world=world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # warm-up (eager): compiles nothing, but sets kernel attributes, packs weights, fills the allocator
    for _ in range(max(args.warmup, 3)):
        out = step()
    torch.cuda.synchronize()
    n0 = lib.atvs_launch_count()
    out = step()
    torch.cuda.synchronize()
    launches_per_step = lib.atvs_launch_count() - n0

    use_graph = not args.no_graph and not sharded
    graph = None
    if use_graph:
        graph, out = capture(step, torch)

    value_graphed = graph is not None

    def run_step():
        if graph is not None:
            graph.replay()
            return out
        return step()

    # ---------------- timed region 1: inputs resident in HBM ----------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.wait_first()
    barrier()
    ms_total, res = timed_steps(run_step, args.steps, torch, barrier)
    dumped = None
    if args.dump_outputs and rank == 0:
        # a device copy now (the graph and its buffers are released below); the files are written once the clock
        # sampler has stopped, so that the host work of the dump does not enter the clocks of the timed regions
        dumped = {k: [x if x is None else x.clone() for x in v] if isinstance(v, list) else v.clone()
                  for k, v in res.items()}

    # ---------------- timed region 2: end to end from / to pinned host memory ----------------
    # the public streaming call (pipeline.FrameStream): frames arrive in pinned host memory, every step copies its
    # inputs H2D and its depth map D2H; the copies of neighbouring frames overlap the step on their own streams
    fstream = None
    if graph is not None:
        # the device-resident graph is done: release its private pool before FrameStream captures its own (cfg3 holds
        # ~100 GB of intermediate volumes per captured step)
        graph, res, out = None, None, None
        torch.cuda.synchronize()
        torch.cuda.empty_cache()
        fstream = A.pipeline.FrameStream(tuple(feats_h.shape), tuple(cams_h.shape), D, dev, siamese=True)
        for dm in fstream.run([(feats_h, cams_h)] * 3):
            pass
    barrier()
    f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    f0.record()
    if fstream is not None:
        for dm in fstream.run((feats_h, cams_h) for _ in range(args.steps)):
            depth_h = dm
    else:
        for _ in range(args.steps):
            feats_d.copy_(feats_h, non_blocking=True)
            cams_d.copy_(cams_h, non_blocking=True)
            res = run_step()
            depth_h.copy_(res['depth_up'], non_blocking=True)
    f1.record()
    barrier()
    clocks = sampler.stop()
    if dumped is not None:
        dump_outputs(dumped, args.dump_outputs)
        dumped = None
    ms_e2e = f0.elapsed_time(f1)
    # sanity of what was timed: the depth map must be finite and inside the swept inverse-depth range
    dmin, dmax = float(cams[0, 0, 1, 3, 0]), float(cams[0, 0, 1, 3, 0] + (D - 1) * cams[0, 0, 1, 3, 1])
    dm = depth_h.clone()
    if not bool(torch.isfinite(dm).all()) or float(dm.min()) < dmin - 1e-4 or float(dm.max()) > dmax + 1e-4:
        raise RuntimeError("bench: depth map not finite / outside the depth sweep [%g, %g]: min %g max %g"
                           % (dmin, dmax, float(dm.min()), float(dm.max())))
    saturated = A.pipeline.check_saturation(action='count') if args.precision != 'fp32' else 0
    h2d = feats_h.numel() * 4 + cams_h.numel() * 4
    d2h = depth_h.numel() * 4

    # ---------------- dominant kernel, timed with CUDA events on its launch stream ----------------
    roof = None
    if args.precision != 'fp32':
        # Three clocks on the same launch (conv_b0_0_1 of the step, the step's own tensors):
        #  (a) ms_per_launch: the launch re-issued back to back, alone on the GPU, as a CUDA graph on its stream, CUDA
        #      events around the replay (the microbenchmark form also used for K1 / K4 below) - the roofline number;
        #  (b) ms_per_launch_in_step: CUDA events around each of the step's own launches while the step's streams
        #      share the SMs (eager pass of the same work: events cannot be recorded inside a graph replay);
        #  (c) ms_per_launch_events_alone: as (b) with the passes run one after the other on one stream; it carries the
        #      idle-GPU launch latency of an eager launch on top of (a).
        is_dom = lambda key: key in ('conv_b0_0_1/conv3d/kernel', 'conv_b0_0_1/conv3d/kernel/warp')
        timings = {}
        for label, nstreams in (('alone', 1), ('in_step', A.pipeline.CONCURRENT_PASSES)):
            sink = []
            saved = A.pipeline.CONCURRENT_PASSES
            A.pipeline.CONCURRENT_PASSES = nstreams
            N.PROFILE = (is_dom, sink)
            try:
                for _ in range(2):
                    step()
                torch.cuda.synchronize()
            finally:
                N.PROFILE = None
                A.pipeline.CONCURRENT_PASSES = saved
            timings[label] = [r[1].elapsed_time(r[2]) for r in sink]
        nvox, cin, cout, again = sink[-1][3], sink[-1][4], sink[-1][5], sink[-1][6]
        reps = 10
        gk, _ = capture(lambda: [again() for _ in range(reps)][-1][0], torch)
        gk.replay()
        torch.cuda.synchronize()
        ts = []
        for _ in range(3):
            k0, k1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            k0.record()
            gk.replay()
            k1.record()
            torch.cuda.synchronize()
            ts.append(k0.elapsed_time(k1) / reps)
        del gk
        t_ms = float(np.mean(ts))
        # (d) steady state: the same layer on a volume 8 x deeper (launch ramp / drain and the per-CTA prologue are
        #     <3 % of such a launch; what a batch of 8 passes in one launch would cost per pass)
        t_steady = None
        try:
            t_steady = steady_state_ms(A, torch, cin, cout, nvox, D, h, w)
        except Exception:
            torch.cuda.synchronize()
        flops = 2.0 * 27 * cin * cout * nvox
        pk = peaks()
        ach = flops / (t_ms * 1e-3) / 1e12
        roof = {"bound": "tensor",
                "kernel": "k_conv3d_ring<%d,8,2> (conv_b0_0_1, %d->8 stride 1 on %d voxels%s)"
                          % (cin, cin, nvox, "; the 32 tiled-reference channels enter as an epilogue bias" if cin == 32 else ""),
                "achieved": ach, "peak": pk['bf16_sustained'], "unit": "TFLOP/s", "frac": ach / pk['bf16_sustained'],
                "traffic": None, "peak_source": pk['src'] + " (sustained bf16 = fp16 rate of tcgen05.mma.kind::f16)",
                "ms_per_launch": t_ms, "launches_timed": 3 * reps, "algorithmic_flops_per_launch": flops,
                "timing": "the step's conv_b0_0_1 launch (its own tensors) re-issued %d times back to back as a CUDA graph, "
                          "alone on the GPU (grid as the library sizes it for a lone launch, atvs_set_concurrency(1)), CUDA events "
                          "around the replay on the launch stream, mean of 3 replays; "
                          "ms_per_launch_in_step = CUDA events around each of the step's %d launches of this layer with the "
                          "step's %d streams sharing the SMs (eager pass); ms_per_launch_events_alone = the same with the "
                          "passes one after the other" % (reps, len(timings['in_step']) // 2, A.pipeline.CONCURRENT_PASSES),
                "ms_per_launch_in_step": float(np.mean(timings['in_step'])),
                "ms_per_launch_events_alone": float(np.mean(timings['alone'])),
                "frac_in_step": flops / (float(np.mean(timings['in_step'])) * 1e-3) / 1e12 / pk['bf16_sustained']}
        if t_steady is not None:
            roof["ms_per_launch_steady_state"] = t_steady
            roof["frac_steady_state"] = flops / (t_steady * 1e-3) / 1e12 / pk['bf16_sustained']
            roof["timing"] += ("; ms_per_launch_steady_state = the same layer (random 16-bit input, same weights) on a volume "
                               "8 x deeper, time / 8: the kernel without its launch ramp / drain")

    # ---------------- the HBM-bound kernels of the path (K1, K4) on this workload's shapes ----------------
    kernels = None
    if rank == 0 and args.precision != 'fp32':
        kernels = hbm_kernel_lines(A, feats_d, cams_d, D, h, w, N.act_dtype())
        if roof is not None:
            roof["traffic"], roof["traffic_source"] = ncu_traffic("k_conv3d_ring<32, 8, 2, 2,")

    # ---------------- N = 1: the same depth map from IMAGES, and the whole four-stage schedule ----------------
    extras = {}
    if world == 1 and not args.no_extras and args.precision != 'fp32':
        rng = np.random.default_rng(1000)
        imgs_h = torch.from_numpy((127.5 + 50.0 * rng.standard_normal((1, nv, H, W, 3))).clip(0, 255).astype(np.float32)).pin_memory()
        imgs_d = imgs_h.to(dev)

        def step_images():
            return A.pipeline.run_multiview(A.fem.extract_features(imgs_d), cams_d, D, siamese=True)['depth_up']

        def step_four():
            return A.pipeline.run_example_schedule(imgs_d, cams_d, D)['depth_refined_up']

        for name, fn, what in (("from_images", step_images, "IMAGES in: 2-D feature extractor (ResNetDS2SPP, fp32 CUDA-core path: the parity default) on the 5 views + stages I + II + x4 soft-argmin"),
                               ("four_stage", step_four, "IMAGES in: the whole example.py:144-181 schedule (FEM, stages I-IV with refinement)"),
                               ("from_images_tensor_fem", step_images, "as from_images with FLAGS.fem_tensor = True: the FEM's stride-1 convolutions on tcgen05 (fp16 operands); opt-in, costs 0.09-0.24 % of the depth range in accuracy (tools/fem_accuracy.py)"),
                               ("four_stage_tensor_fem", step_four, "as four_stage with FLAGS.fem_tensor = True")):
            A.FLAGS.fem_tensor = name.endswith("tensor_fem")
            try:
                for _ in range(2):
                    o = fn()
                torch.cuda.synchronize()
                k = max(3, min(args.steps, 10))
                graphed = not args.no_graph
                if graphed:
                    try:
                        g, o = capture(fn, torch)
                    except Exception:          # a step that cannot be captured is timed as eager launches
                        torch.cuda.synchronize()
                        graphed = False
                if graphed:
                    ms, _ = timed_steps(lambda: g.replay(), k, torch, barrier)
                    del g
                else:
                    ms, o = timed_steps(fn, k, torch, barrier)
                extras[name] = {"what": what, "ms_per_step": ms / k, "value": k / (ms * 1e-3), "unit": "depth maps/s",
                                "steps": k, "cuda_graph": graphed, "finite": bool(torch.isfinite(o).all())}
                del o
                A.FLAGS.fem_tensor = False
            except Exception as e:       # an extra must never take the headline line down with it
                A.FLAGS.fem_tensor = False
                extras[name] = {"what": what, "error": "%s: %s" % (type(e).__name__, str(e)[:200])}
                torch.cuda.synchronize()
        del imgs_d

    # ---------------- N > 1: ONE cfg3 frame with its source views sharded over the ranks ----------------
    sharded_line = None
    if world > 1 and not sharded and not args.no_extras:
        sharded_line = run_sharded_cfg3(A, dist, torch, dev, rank, world, local_rank, barrier)

    # max over ranks
    t = torch.tensor([ms_total, ms_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, ms_e2e = float(t[0]), float(t[1])
    maps_per_step = 1 if sharded else world
    value = maps_per_step * args.steps / (ms_total * 1e-3)
    e2e_value = maps_per_step * args.steps / (ms_e2e * 1e-3)
    all_clocks = [clocks]
    if world > 1:
        all_clocks = [None] * world
        dist.all_gather_object(all_clocks, clocks)

    if rank != 0:
        return
    crm_passes = 2 * (nv - 1)
    flops_step = 2.0 * CRM_MAC_PER_VOXEL * V * crm_passes + 2.0 * 2 * 27 * 64 * V * (nv - 1) + 2.0 * 216 * V
    # the line's clocks: the slowest rank's median, the union of the reasons, per-rank detail beside it
    sm = [c.get("sm_mhz") for c in all_clocks if c.get("sm_mhz") is not None]
    clk = {"sm_mhz": min(sm) if sm else None, "sm_max_mhz": all_clocks[0].get("sm_max_mhz"),
           "reasons": sorted(set(r for c in all_clocks for r in c.get("reasons", []))),
           "samples": min(c.get("samples", 0) for c in all_clocks), "per_rank": all_clocks}
    line = {
        "metric": METRIC, "value": value, "unit": "depth maps/s", "n_gpus": world, "steps": args.steps,
        "warmup": max(args.warmup, 3), "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "strong" if sharded else "weak", "vs_baseline": None,
        "dtype": {"fp16": "fp16 operands / fp32 accumulate (tcgen05 kind::f16)", "bf16": "bf16", "fp32": "f32"}[args.precision],
        "data": "synthetic",
        "config": common_config(workload, world, sharded),
        "details": {"cuda_graph": value_graphed, "tensor_flops_per_step": flops_step,
                    "tensor_tflops_whole_step": flops_step * maps_per_step * args.steps / (ms_total * 1e-3) / 1e12 / world,
                    "weights": "variables.synthetic_weights() (seeded He-normal under the checkpoint names, logit gain 4); "
                               "tests/test_gpu_parity.py::test_cfg2_full_size_against_oracle checks this exact workload "
                               "against the CPU oracle (0.1 % of the depth range)"},
        "e2e": {"value": e2e_value, "unit": "depth maps/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                "ms_per_step": ms_e2e / args.steps,
                "api": "pipeline.FrameStream.run (pinned host frames in, pinned host depth maps out; copies of "
                       "neighbouring frames overlap the step)" if fstream is not None else
                       "pipeline.run_multiview bracketed by the H2D / D2H copies on one stream"},
        "gpu_launches": int(launches_per_step * args.steps),
        "gpu_launches_per_step": int(launches_per_step),
        "clocks": clk,
        "output_check": "depth map finite and inside the inverse-depth sweep; fp16 raw rows clamped: %d" % saturated,
    }
    if roof is not None:
        line["roofline"] = roof
    if kernels is not None:
        line["hbm_kernels"] = kernels
    line.update(extras)
    if sharded_line is not None:
        line["sharded"] = sharded_line
    if world == 1 and not args.no_cpu_baseline:
        line["cpu_baseline"] = cpu_baseline(workload)
    print(json.dumps(line))


def run_sharded_cfg3(A, dist, torch, dev, rank, world, local_rank, barrier, steps=5):
    """cfg3 = ONE 1920x1056, D = 256 frame with 8 source views: stage I of view v on rank (v-1) % world, aggregation
    completed across ranks (all-reduce(max) of the local logit max, reduce-scatter(sum) of [num || den], all-gather of
    the 8-channel result), output conv + soft-argmin replicated.  Timed on every rank, max over ranks; then the same
    frame on rank 0 alone (all 8 views) for the 1-GPU time of the same build in the same run."""
    feats, cams, D = make_inputs('cfg3', 0)
    nv, H, W, _ = WORKLOADS['cfg3']
    V = D * (H // 4) * (W // 4)
    f = torch.from_numpy(feats).to(dev)
    c = torch.from_numpy(cams).to(dev)
    torch.cuda.empty_cache()

    def step_sh():
        return A.pipeline.run_multiview(f, c, D, siamese=True, upsample=True, group=dist.group.WORLD, rank=rank,
                                        world=world)['depth_up']

    def step_one():
        return A.pipeline.run_multiview(f, c, D, siamese=True, upsample=True)['depth_up']

    for _ in range(2):
        o = step_sh()
    # enough steps for >= ~0.7 s of timed region (the 50 ms clock sampler must see it: 5 steps at 8 GPUs are 0.12 s)
    barrier()
    w0, w1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    w0.record()
    o = step_sh()
    w1.record()
    torch.cuda.synchronize()
    est = torch.tensor([w0.elapsed_time(w1)], dtype=torch.float64, device=dev)
    dist.all_reduce(est, op=dist.ReduceOp.MAX)
    steps = int(min(40, max(steps, 700.0 / max(float(est[0]), 1.0) + 1)))
    sampler = ClockSampler(local_rank)
    sampler.start()
    sampler.wait_first()
    barrier()
    ms, o = timed_steps(step_sh, steps, torch, barrier)
    clocks = sampler.stop()
    t = torch.tensor([ms], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms = float(t[0])
    finite = bool(torch.isfinite(o).all())
    ms1 = None
    if rank == 0:
        torch.cuda.empty_cache()
        for _ in range(1):
            o1 = step_one()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(2):
            o1 = step_one()
        e1.record()
        torch.cuda.synchronize()
        ms1 = e0.elapsed_time(e1) / 2
        same = float((o1 - o).abs().max())
    barrier()
    allc = [None] * world
    dist.all_gather_object(allc, clocks)
    if rank != 0:
        return None
    per_rank_views = [len(A.pipeline.shard_views(nv, r, world)) for r in range(world)]
    return {"workload": "cfg3: 1 ref + 8 src, 1920x1056 images -> 264x480x32 features in, D=256, stages I (siamese) + II + x4 "
                        "soft-argmin, ONE frame, source views sharded over the ranks",
            "n_gpus": world, "steps": steps, "ms_per_step": ms / steps, "value": steps / (ms * 1e-3), "unit": "depth maps/s",
            "scaling": "strong", "ms_per_step_1gpu_same_run": ms1, "views_per_rank": per_rank_views,
            "collective_bytes_per_rank": {"all_reduce_max_bf16": 2 * 8 * V, "reduce_scatter_sum_f32": 4 * 16 * V,
                                          "all_gather_result_f16": 2 * 8 * V},
            "max_abs_diff_vs_1gpu_depth": same, "finite": finite,
            "clocks": {"per_rank": allc, "samples": min(x.get("samples", 0) for x in allc),
                       "reasons": sorted(set(r for x in allc for r in x.get("reasons", [])))},
            "what_limits_it": "one rank's share of stage I (ceil(8/N) views x ~17 ms), the replicated stage II at full "
                              "resolution and the reduce-scatter payload; see DESIGN.md section 7"}


def ncu_traffic(kernel_substr):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of the named kernel, from the committed
    `ncu --set full` capture (profiles/*_traffic.json, written by tools/ncu_traffic.py), newest round first."""
    import glob
    for f in sorted(glob.glob(os.path.join(ROOT, 'profiles', '*_traffic.json')), reverse=True):
        try:
            for row in json.load(open(f)):
                if kernel_substr in row['kernel']:
                    return row['dram_bytes'], os.path.relpath(f, ROOT)
        except Exception:
            pass
    return None, None


def steady_state_ms(A, torch, cin, cout, nvox, D, h, w):
    """conv_b0_0_1's kernel on a (8D, h, w, cin) volume, per cfg-sized eighth (ms)."""
    from atvsnet_b200 import network as N
    if nvox != D * h * w or 8 * nvox * max(cin, cout) >= 2 ** 31:
        return None
    dt = N.act_dtype()
    x = torch.randn(1, 8 * D, h, w, cin, device='cuda').to(dt)
    wk = A.variables.get_variable('conv_b0_0_1/conv3d/kernel')[..., -cin:, :].contiguous()
    stats = torch.zeros(2 * cout, dtype=torch.float64, device='cuda')
    fn = lambda: N.conv3d_raw(x, 'bench/steady_state', wk, cout, 1, False, True, stats_buf=stats, raw_dtype=torch.float16)[0]
    fn()
    torch.cuda.synchronize()
    g, _ = capture(lambda: [fn() for _ in range(3)][-1], torch)
    g.replay()
    torch.cuda.synchronize()
    a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    a.record()
    g.replay()
    b.record()
    torch.cuda.synchronize()
    del g, x
    return a.elapsed_time(b) / 3 / 8


def hbm_kernel_lines(A, feats_d, cams_d, D, h, w, act_dtype):
    """K1 (fused homography + bilinear + cost slice, 16-bit warped-only as the step uses it) and K4 (soft-argmin
    with the fused x4 logit upsample) timed alone with CUDA events on the current stream; algorithmic bytes
    per SURVEY.md 8(d) over the measured HBM copy peak."""
    import torch
    pk = peaks()
    ds, di = cams_d[:, 0, 1, 3, 0].contiguous(), cams_d[:, 0, 1, 3, 1].contiguous()
    F = feats_d.shape[-1]
    V = D * h * w
    logits = torch.randn(1, D, h, w, device=feats_d.device)

    feats16 = A.pipeline.features_act(feats_d)      # once per frame in the step (pipeline.run_multiview)
    hv = A.get_homographies(cams_d[:, 0].contiguous(), cams_d[:, 1].contiguous(), depth_num=D, depth_start=ds,
                            depth_interval=di)
    cv_out = torch.empty((1, D, h, w, F), dtype=act_dtype, device=feats_d.device)
    ref0, v16 = feats_d[:, 0].contiguous(), feats16[:, 1].contiguous()

    def k1():       # the K1 kernel itself, through its C-ABI entry (homographies: a 4.7 us helper launch per pass)
        A._lib.call("atvs_build_cost_volume_src16", A._lib.ptr(ref0), A._lib.ptr(v16), A._lib.ptr(hv), 1, D, h, w, F, 1,
                    A._lib.dtype_code(cv_out), A._lib.ptr(cv_out), A._lib.stream())
        return cv_out

    def k4up():
        return A.model._prob2depth(logits, ds, di, 4, False)

    def k4():
        return A.model._prob2depth(logits, ds, di, 1, False)

    def timed(fn, iters=10):
        # CUDA-graph replay of `iters` back-to-back launches, CUDA events around the replay on the replay stream
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        g = torch.cuda.CUDAGraph()
        st = torch.cuda.Stream()
        st.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(st):
            with torch.cuda.graph(g, stream=st):
                for _ in range(iters):
                    fn()
        torch.cuda.current_stream().wait_stream(st)
        g.replay()
        torch.cuda.synchronize()
        ts = []
        for _ in range(5):
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            g.replay()
            b.record()
            b.synchronize()
            ts.append(a.elapsed_time(b))
        ts.sort()
        return ts[len(ts) // 2] * 1e-3 / iters

    # K2: the attention aggregation module of stage II on this workload's view count (one kernel, conv_attn_ring.cu)
    nsrc = feats_d.shape[1] - 1
    views = [torch.randn(1, D, h, w, 8, device=feats_d.device).clamp_(min=-0.5).to(act_dtype) for _ in range(nsrc)]

    def k2():
        return A.cost_volume_aggregation(views, keepchannel=True)

    out = {}
    if A.network.attention_fused_ok(views):
        t = timed(k2)
        nb = nsrc * V * 8 * 2 + V * 8 * 4
        fl = 2.0 * 27 * 8 * 16 * V * nsrc
        out["K2 k_attention_ring (attention convolutions of all views + softmax over views + weighted sum)"] = {
            "bound": "hbm", "achieved": nb / t / 1e9, "peak": pk['hbm'], "unit": "GB/s", "frac": nb / t / 1e9 / pk['hbm'],
            "algorithmic_bytes": nb, "us_per_launch": t * 1e6,
            "tensor_tflops": fl / t / 1e12, "tensor_frac": fl / t / 1e12 / pk['bf16_sustained'],
            "note": "reads the %d filtered 8-channel volumes once, writes the fp32 aggregate; the 2 x 3x3x3 8->8 attention "
                    "convolutions per view (%.1f GFLOP) run on tcgen05 with their logits kept in TMEM, so the kernel is bound "
                    "by the tensor pipe's operand fetch (tensor_frac of the sustained peak), not by HBM; the two-kernel path it "
                    "replaces (8->16 convolution per view + atvs_attention_raw) moved 922 MB for these %.0f MB; graph replay "
                    "of 10 launches, CUDA events" % (nsrc, fl / 1e9, nb / 1e6)}
    del views
    for name, fn, nbytes, note in (
            ("K1 k_build_cost_volume_h (16-bit, warped-only)", k1, 2 * h * w * F + 2 * V * F,
             "reads the 16-bit source feature map (converted once per frame for all passes), writes the (D,h,w,32) 16-bit "
             "slice; one launch of atvs_build_cost_volume_src16"),
            ("K4 k_prob2depth_up_sliced<4> (x4 upsample fused)", k4up, 4 * V + 4 * 16 * h * w,
             "reads the low-res logits once, writes the 4h x 4w depth map; instruction bound by construction (16*V "
             "interpolations + exponentials per 4*V bytes), see equivalent_unfused_gbs"),
            ("K4 k_prob2depth_sliced (volume resolution)", k4, 4 * V + 4 * h * w,
             "reads the logits once; a 10 MB volume: launch-latency sized at this workload (see the cfg5 sweep under "
             "profiles/ for the large planes)")):
        t = timed(fn)
        out[name] = {"bound": "hbm", "achieved": nbytes / t / 1e9, "peak": pk['hbm'], "unit": "GB/s",
                     "frac": nbytes / t / 1e9 / pk['hbm'], "algorithmic_bytes": nbytes, "us_per_launch": t * 1e6,
                     "note": note + "; graph replay of 10 launches, CUDA events"}
        if 'up_sliced' in name:
            # what the reference formulation moves for the same result: write + read of the x16 upsampled logit volume
            out[name]["equivalent_unfused_gbs"] = (2 * 4 * 16 * V + 4 * V) / t / 1e9
    return out


def cpu_baseline(workload):
    """the oracle port timed on the host cores: ONE full step of the workload (all depth planes, all source views,
    siamese stage I + stage II + x4 soft-argmin), ~30 s of CPU work at cfg2."""
    import torch
    import atvsnet_b200 as A
    from oracle import model as om
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    feats, cams, D = make_inputs(workload, 0)
    nv = cams.shape[1]
    weights = A.variables.synthetic_weights()
    ds, di = cams[:, 0, 1, 3, 0], cams[:, 0, 1, 3, 1]
    om.TVSNet_base(feats[:, :2, :16, :16], cams, 8, ds, di, 1, weights)          # touch the code paths
    t0 = time.perf_counter()
    om.run_multiview_stage12(feats, cams, D, weights, siamese=True)
    dt = time.perf_counter() - t0
    return {"value": 1.0 / dt, "unit": "depth maps/s", "cores": cores, "kind": "port",
            "sample": "one full %s step (stages I siamese + II + x4 soft-argmin, all %d source views, all %d depth planes): "
                      "%.1f s of CPU work" % (workload, nv - 1, D, dt)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=30)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--workload', default=None, choices=[None] + list(WORKLOADS))
    ap.add_argument('--precision', default='fp16', choices=['fp16', 'bf16', 'fp32'])
    ap.add_argument('--raw-dtype', default='f16', choices=['f16', 'f32'],
                    help='storage of the raw (pre-BN) convolution outputs on the tensor-core path')
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--no-extras', action='store_true',
                    help='skip the extra fields (from-images / four-stage at N=1, sharded cfg3 at N>1)')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--ref-budget-s', type=float, default=None, metavar='S',
                    help='--impl reference: time fewer than --steps steps if the run would otherwise pass S seconds')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step returned as DIR/<name>.npy (rank 0)')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs writes the outputs of --impl ours only')

    rank = int(os.environ.get('RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    if args.impl == 'reference':
        run_reference(args, rank, world)
        return
    if world > 1:
        import torch
        import torch.distributed as dist
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        os.environ.setdefault('MASTER_PORT', '29511')
        torch.cuda.set_device(local_rank)
        # NCCL prints its version banner to stdout when the communicator is created: keep fd 1 pointed at stderr until
        # that has happened (rank 0's stdout carries ONE JSON line)
        sys.stdout.flush()
        saved_stdout = os.dup(1)
        os.dup2(2, 1)
        try:
            dist.init_process_group('nccl', rank=rank, world_size=world, device_id=torch.device('cuda', local_rank))
            dist.barrier()
            torch.cuda.synchronize()
        finally:
            sys.stdout.flush()
            os.dup2(saved_stdout, 1)
            os.close(saved_stdout)
    try:
        run_ours(args, rank, world, local_rank)
    finally:
        if world > 1:
            import torch.distributed as dist
            dist.destroy_process_group()


if __name__ == '__main__':
    main()
