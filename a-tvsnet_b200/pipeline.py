"""The multi-view schedule of /root/reference/atvsnet/example.py:144-158 (stage I per source
view, stage II = AAM1 -> output_conv -> prob2depth) run entirely on the device: the
filtered cost volumes stay in HBM (no np.stack / feed_dict round trips), and source views
can be sharded over ranks with one max + one sum all-reduce of the attention partials
(SURVEY.md section 8(e)).  run_example_schedule adds stages III/IV (refinement, example.py:163-181),
run_twoview is the single-shot two-view schedule (example.py:219-303).  Entry points take IMAGES
(B,N,H,W,3) or, to skip the 2-D feature extractor, FEATURES (B,N,h,w,32)."""
import torch

from . import _lib as L
from . import network as N
from .atvsnet import OutputConv, StackedUNet_prob
from .model import _prob2depth, build_cost_volume

# tensor-core path: run the first CRM layers on the warped half only (network.SplitCostVolume)
SPLIT_COST_VOLUME = True
# number of CUDA streams the independent stage-I passes are spread over
CONCURRENT_PASSES = 8


def _cost_volume(r, v, cams, depth_num, depth_start, depth_interval, rid, vid, v16=None):
    """``v16``: the view's feature map already in the activation dtype (features_act): K1 gathers from it directly."""
    dt = N.act_dtype()
    if dt in N.HALF_DTYPES and v16 is not None and v16.dtype == dt and v.shape[-1] in (8, 16, 32, 64, 128):
        v = v16
    if dt in N.HALF_DTYPES and SPLIT_COST_VOLUME:
        # [tile(ref) | warped] kept as its halves: K1 writes only the warped 32 channels
        warped = build_cost_volume(r, v, cams, depth_num, depth_start, depth_interval, ref_id=rid, view_id=vid,
                                   mode='warped_only', out_dtype=dt)
        return N.SplitCostVolume(r, warped)
    return build_cost_volume(r, v, cams, depth_num, depth_start, depth_interval, ref_id=rid, view_id=vid, out_dtype=dt)


@L.on_input_device
def features_act(features):
    """(B,N,h,w,F) fp32 feature maps -> the same in the 16-bit activation dtype, ONE conversion per frame for all the
    passes that warp a view (forward passes warp the sources, reverse passes the reference); None on the fp32 path."""
    return N.to_act(features) if N.act_dtype() in N.HALF_DTYPES else None


@L.on_input_device
def stage1_forward(features, cams, depth_num, depth_start, depth_interval, view_i, features16=None):
    """forward half of TVSNet_base_siamese (model.py:409-411): ref <- view_i.  Returns the 8-ch
    filtered volume (activation dtype) and the prob logits (fp32)."""
    cv = _cost_volume(features[:, 0], features[:, view_i], cams, depth_num, depth_start, depth_interval, 0, view_i,
                      None if features16 is None else features16[:, view_i])
    tower = StackedUNet_prob({'data': cv}, outputs=('conv_b2_6_1', 'conv_b2_6_2'))
    return tower.get_output_by_name('conv_b2_6_1'), tower.get_output().squeeze(-1)


@L.on_input_device
def stage1_reverse(features, cams, depth_num, depth_start, depth_interval, view_i, features16=None, confidence=False):
    """reverse half (model.py:413-415): view_i as reference -> depth_view (B,h,w,1); with ``confidence`` the pair
    (depth_view, its probability map (B,h,w,1)), both from the same soft-argmin launch."""
    cvv = _cost_volume(features[:, view_i], features[:, 0], cams, depth_num, depth_start, depth_interval, view_i, 0,
                       None if features16 is None else features16[:, 0])
    pv = StackedUNet_prob({'data': cvv}, outputs=('conv_b2_6_2',)).get_output().squeeze(-1)
    depth_view, prob_map = _prob2depth(pv, depth_start, depth_interval, 1, confidence)
    return (depth_view, prob_map) if confidence else depth_view


@L.on_input_device
def stage1_view(features, cams, depth_num, depth_start, depth_interval, view_i, siamese=True):
    """TVSNet_base_siamese (model.py:398-417) keeping the 8-ch filtered volume in the activation
    dtype.  Returns (filtered (B,D,h,w,8), prob logits (B,D,h,w) fp32, depth_view | None)."""
    filtered, prob = stage1_forward(features, cams, depth_num, depth_start, depth_interval, view_i)
    depth_view = stage1_reverse(features, cams, depth_num, depth_start, depth_interval, view_i) if siamese else None
    return filtered, prob, depth_view


_STREAMS = {}
_WARM = set()      # (weights generation, precision, raw dtypes, split mode, device) whose weight images are packed


def _side_streams(device, n):
    key = (device.index, n)
    if key not in _STREAMS:
        _STREAMS[key] = [torch.cuda.Stream(device=device) for _ in range(n)]
    return _STREAMS[key]


def reduce_partials(nd, world, rank, group, finish, gather_dtype):
    """Complete the view softmax across ranks from the local partials ``nd`` (V,2C) fp32 = [sum_n e^{l_n-m} x_n | sum_n
    e^{l_n-m}]: reduce-scatter(SUM) so that every rank owns V/world voxels of the summed partials, ``finish`` (slab
    (v,2C) -> (v,C) = num / den) on the owned slab, all-gather of the RESULT in ``gather_dtype``.  Against one
    all-reduce of the partials this moves (2C*4 + C*s) instead of 2*2C*4 bytes per voxel over the links (40 vs 128 for
    C = 8, bf16) and divides the finish work by ``world``.  Backends without reduce-scatter (gloo, CPU tests) take the
    equivalent all-reduce + slice."""
    import torch.distributed as dist
    V, c2 = nd.shape
    per = -(-V // world)
    if per * world != V:                                   # pad to a multiple of world (tail rows are dropped again)
        pad = torch.zeros((per * world, c2), dtype=nd.dtype, device=nd.device)
        pad[:V] = nd
        nd = pad
    if dist.get_backend(group) == 'nccl':
        slab = torch.empty((per, c2), dtype=nd.dtype, device=nd.device)
        dist.reduce_scatter_tensor(slab, nd, op=dist.ReduceOp.SUM, group=group)
    else:
        dist.all_reduce(nd, op=dist.ReduceOp.SUM, group=group)
        slab = nd[rank * per:(rank + 1) * per].contiguous()
    mine = finish(slab).to(gather_dtype).contiguous()
    full = torch.empty((per * world, mine.shape[1]), dtype=gather_dtype, device=nd.device)
    dist.all_gather_into_tensor(full, mine, group=group)
    return full[:V]


@L.on_input_device
def aggregate(filtered_views, scope='attention_aggregate', group=None, rank=0, world=1, raw=None):
    """AAM (network.py:379-408) over this rank's views; with ``group`` the softmax over views is completed across
    ranks: all-reduce(MAX) of the local logit max (as bf16: any shift that is the same on every rank is exact for the
    softmax), then reduce_partials() of [numerator || denominator] (V,16) fp32.  Sharded result: activation dtype."""
    if group is None:
        return N.attention_aggregation(filtered_views, scope, raw=raw)
    import torch.distributed as dist
    views = N.split_views(filtered_views)
    shape = views[0].shape
    c = shape[-1]
    nvox = views[0].numel() // c
    if raw is None:
        raw = N.attention_activations_raw(views, scope)
    x = views[0]
    xp = N.view_pointers(views)
    lmax = torch.empty((nvox, c), dtype=torch.float32, device=x.device)
    L.call("atvs_attention_raw", L.ptr(raw), N._raw_code(raw), None, len(views), nvox, c, L.dtype_code(x), 1, None, L.ptr(lmax), L.stream())
    lmax16 = lmax.to(torch.bfloat16)
    dist.all_reduce(lmax16, op=dist.ReduceOp.MAX, group=group)
    lmax.copy_(lmax16)
    del lmax16
    nd = torch.empty((nvox, 2 * c), dtype=torch.float32, device=x.device)
    L.call("atvs_attention_raw", L.ptr(raw), N._raw_code(raw), xp, len(views), nvox, c, L.dtype_code(x), 2, L.ptr(lmax), L.ptr(nd),
           L.stream())
    del raw, lmax

    def finish(slab):
        out = torch.empty((slab.shape[0], c), dtype=torch.float32, device=slab.device)
        L.call("atvs_attention_finish", L.ptr(slab), slab.shape[0], c, L.ptr(out), L.stream())
        return out

    out = reduce_partials(nd, world, rank, group, finish, x.dtype)
    return out.reshape(shape)


def check_saturation(reset=True, action='raise'):
    """fp16 raw-output rows that had to be clamped to +-65504 by the tensor-path epilogues since the last reset
    (atvs_saturation_count; synchronises the device, so call it once per batch of frames, not per kernel).  A non-zero
    count means the feature scale of the loaded checkpoint does not fit fp16 raw storage: ``action='raise'`` raises,
    ``'fallback'`` switches FLAGS.raw_dtype / first_raw_dtype to 'f32' for the following frames and returns the count."""
    n = int(L.load().atvs_saturation_count(1 if reset else 0))
    if n < 0:
        raise RuntimeError("atvs_saturation_count failed")
    if n > 0:
        if action == 'fallback':
            N.FLAGS.raw_dtype = N.FLAGS.first_raw_dtype = 'f32'
        elif action == 'raise':
            raise RuntimeError("%d fp16 raw-output rows were clamped to +-65504: the feature scale of these weights does "
                               "not fit fp16 raw storage; set FLAGS.raw_dtype = FLAGS.first_raw_dtype = 'f32'" % n)
    return n


def shard_views(n_views, rank, world):
    """source views 1..N-1 dealt round-robin to ranks (SURVEY.md 8(e))."""
    return [v for v in range(1, n_views) if (v - 1) % world == rank]


@L.on_input_device
def run_multiview(features, cams, depth_num, siamese=True, upsample=True, group=None, rank=0, world=1, confidence=False):
    """features (B,N,h,w,F) fp32, cams (B,N,2,4,4) -> dict(depth (B,h,w,1), depth_up (B,4h,4w,1),
    prob_volume_agg, cost_volume_agg, depth_views).  example.py:144-158 + :109 (x4 upsample).
    ``confidence`` adds the probability maps of prob2depth_upsample(out_prob_map=True) (model.py:113-129, :13-65),
    each from the soft-argmin launch of its depth map: prob_map (B,h,w,1), prob_map_up (B,4h,4w,1) with ``upsample``,
    and depth_view_probs beside depth_views (None entries without ``siamese``)."""
    L.require_cuda(features, cams)
    cams = L.f32c(cams)
    n_views = cams.shape[1]
    ds = cams[:, 0, 1, 3, 0].contiguous()
    di = cams[:, 0, 1, 3, 1].contiguous()
    mine = shard_views(n_views, rank, world) if group is not None else list(range(1, n_views))
    # the 2*(N-1) regularisation passes of stage I are independent: spread them over a few streams so that
    # the many small kernels of the coarse U-Net levels (40-tile launches) overlap with other passes.
    tasks = [(v, 'f') for v in mine] + ([(v, 'r') for v in mine] if siamese else [])
    nstreams = max(1, min(CONCURRENT_PASSES, len(tasks)))
    main = torch.cuda.current_stream()
    results = {}
    # attention logits (N,V,16), allocated on the calling stream before the passes fan out: every view's 8->16
    # attention convolution runs on that view's stream right behind its forward pass instead of in the serial tail
    B_, _, h_, w_, _ = features.shape
    like = torch.empty((B_, int(depth_num), h_, w_, 8), dtype=N.act_dtype(), device='meta')
    # one-kernel AAM (atvs_attention_fused): no per-view logits at all; the sharded aggregation needs them
    fused_att = group is None and N.attention_fused_ok([like] * len(mine))
    att_raw = None if fused_att else N.attention_raw_alloc(len(mine), like, device=features.device)

    feats16 = features_act(features)     # on the calling stream, before the passes fan out
    # scheduling hint for the persistent tensor kernels: `nstreams` passes share the SMs (fewer, longer CTAs per launch)
    L.call("atvs_set_concurrency", nstreams)

    def run_task(v, kind):
        if kind == 'r':
            return stage1_reverse(features, cams, depth_num, ds, di, v, feats16, confidence)
        out = stage1_forward(features, cams, depth_num, ds, di, v, feats16)
        if att_raw is not None:
            N.attention_raw_view(att_raw, mine.index(v), N.to_act(out[0]), 'attention_aggregate')
        return out

    if nstreams == 1:
        for v, kind in tasks:
            results[(v, kind)] = run_task(v, kind)
    else:
        warm = (N.V.generation(), N.FLAGS.precision, N.FLAGS.raw_dtype, N.FLAGS.first_raw_dtype, SPLIT_COST_VOLUME,
                features.device.index)
        if tasks and warm not in _WARM:
            # first call with these weights in this precision / split mode: run one forward pass on the calling stream,
            # so that every packed 16-bit weight image it needs (CRM, split halves, attention pair) is produced by
            # kernels the side streams are ordered behind (st.wait_stream(main) below) before they read the cache
            v, kind = tasks.pop(0)
            results[(v, kind)] = run_task(v, kind)
            _WARM.add(warm)
        streams = _side_streams(features.device, nstreams)
        for st in streams:
            st.wait_stream(main)
        for i, (v, kind) in enumerate(tasks):
            with torch.cuda.stream(streams[i % nstreams]):
                out = run_task(v, kind)
                for t in (out if isinstance(out, tuple) else (out,)):
                    t.record_stream(main)
                results[(v, kind)] = out
        for st in streams:
            main.wait_stream(st)
    L.call("atvs_set_concurrency", 1)      # stage II runs alone on the calling stream
    filtered = [results[(v, 'f')][0] for v in mine]
    reverse = [results[(v, 'r')] if siamese else None for v in mine]
    depth_views = [r[0] if confidence and r is not None else r for r in reverse]
    cost_agg = aggregate(filtered, 'attention_aggregate', group, rank, world, raw=att_raw)
    prob_agg = OutputConv({'data': cost_agg}).get_output().squeeze(-1)
    depth, prob_map = _prob2depth(prob_agg, ds, di, 1, confidence)
    out = dict(depth=depth, prob_volume_agg=prob_agg, cost_volume_agg=cost_agg, depth_views=depth_views)
    if confidence:
        out.update(prob_map=prob_map, depth_view_probs=[None if r is None else r[1] for r in reverse])
    if upsample:
        out['depth_up'], prob_map_up = _prob2depth(prob_agg, ds, di, 4, confidence)
        if confidence:
            out['prob_map_up'] = prob_map_up
    return out


@L.on_input_device
def run_example_schedule(images, cams, depth_num, features=None, confidence=False):
    """The whole four-stage schedule of example.py:144-181 on the device, images in:
      I   per source view: FEM features -> TVSNet_base_siamese -> (filtered cost, prob volume, depth_view)
      II  AAM1 (keepchannel) -> output_conv -> prob2depth                              (run_multiview)
      III per source view: TVSNet_refine(depth_agg_init, depth_view_n, prob_agg, cost_agg, images, cams)   (refine.py, fp32)
      IV  AAM2 (keepchannel) -> output_conv_refine -> prob2depth_upsample -> final x4 inverse-depth map
    images (B,N,H,W,3) fp32 0..255, cams (B,N,2,4,4) at feature resolution.  ``features`` (B,N,h,w,32) skips the FEM.
    ``confidence`` adds the stage-II keys of run_multiview(confidence=True) and the stage-IV probability maps
    refined_prob_map (B,h,w,1) and refined_prob_map_up (B,4h,4w,1)."""
    from . import fem, refine
    from .atvsnet import OutputConv_refine
    L.require_cuda(images, cams)
    cams = L.f32c(cams)
    feats = features if features is not None else fem.extract_features(images)
    out = run_multiview(feats, cams, depth_num, siamese=True, upsample=False, confidence=confidence)
    ds = cams[:, 0, 1, 3, 0].contiguous()
    di = cams[:, 0, 1, 3, 1].contiguous()
    n_views = cams.shape[1]
    refined_costs, refined_probs = [], []
    images = L.f32c(images)
    with refine.shallow_cache():       # the reference view's shallow features once, not once per source
        for n, v in enumerate(range(1, n_views)):
            rp, rc = refine.TVSNet_refine(out['depth'], out['depth_views'][n], out['prob_volume_agg'], out['cost_volume_agg'],
                                          images, cams, depth_num, ds, di, v)
            refined_probs.append(rp)
            refined_costs.append(rc)
    cost_ref = N.attention_aggregation(refined_costs, 'attention_aggregate_refine')
    prob_ref = OutputConv_refine({'data': cost_ref}).get_output().squeeze(-1)
    out['depth_refined'], pm = _prob2depth(prob_ref, ds, di, 1, confidence)
    out['depth_refined_up'], pm_up = _prob2depth(prob_ref, ds, di, 4, confidence)
    out.update(refined_cost_volume_agg=cost_ref, refined_prob_volume_agg=prob_ref, refined_prob_volumes=refined_probs)
    if confidence:
        out.update(refined_prob_map=pm, refined_prob_map_up=pm_up)
    return out


@L.on_input_device
def run_twoview(images, cams, depth_num, confidence=False):
    """The two-view driver of example.py:219-272 (run_test_twoview; taken when only two views exist, example.py:344-347):
    TVSNet (FEM on both images, both directions, refinement) -> prob2depth_upsample.  images (B,2,H,W,3) raw 0..255 BGR,
    cams (B,2,2,4,4) at feature resolution -> dict(refined_prob_volume, depth_refined, depth_refined_up), with
    ``confidence`` also refined_prob_map (B,h,w,1) and refined_prob_map_up (B,4h,4w,1)."""
    from .model import TVSNet
    L.require_cuda(images, cams)
    cams = L.f32c(cams)
    ds = cams[:, 0, 1, 3, 0].contiguous()
    di = cams[:, 0, 1, 3, 1].contiguous()
    refined = TVSNet(images, cams, depth_num, ds, di, view_i=1, ref_i=0)
    est, pm = _prob2depth(refined, ds, di, 1, confidence)
    est_up, pm_up = _prob2depth(refined, ds, di, 4, confidence)
    out = dict(refined_prob_volume=refined, depth_refined=est, depth_refined_up=est_up)
    if confidence:
        out.update(refined_prob_map=pm, refined_prob_map_up=pm_up)
    return out


def inverse_to_depth(out, twoview=False):
    """host epilogue of example.py:183-186 (multi-view: values below 1e-10 become inf) / :269-272 (two-view: values <= 0
    become inf), then depth = 1 / inverse depth.  Tensor in, tensor out (same device)."""
    out = out.clone()
    out[(out <= 0) if twoview else (out < 1e-10)] = float('inf')
    return 1.0 / out


@L.on_input_device
def run_example(images, cams, depth_num=None, confidence=False):
    """example.py:main dispatch (:344-347): the multi-view schedule for more than two views, the two-view network
    otherwise.  Returns the final x4 inverse-depth map (B,H,W,1) and ``pred`` = depth (what example.py saves); with
    ``confidence`` also ``prob`` = the x4 probability map of that final depth map (refined_prob_map_up)."""
    n_views = cams.shape[1]
    D = int(depth_num if depth_num is not None else N.FLAGS.max_d)
    if n_views > 2:
        out = run_example_schedule(images, cams, D, confidence=confidence)
    else:
        out = run_twoview(images, cams, D, confidence=confidence)
    inv = out['depth_refined_up']
    out['pred'] = inverse_to_depth(inv, twoview=n_views <= 2)
    if confidence:
        out['prob'] = out['refined_prob_map_up']
    if N.act_dtype() in N.HALF_DTYPES:
        check_saturation()
    return out


def load_example(data_root, view_num=5):
    """input loading of example.py:312-342: ``{i}.jpg`` (cv2.imread: BGR uint8, fed un-normalised) and ``{i}_cam.npy``
    (2,4,4: extrinsic; intrinsic at feature resolution with depth_start / depth_interval in row 3) for i < view_num,
    shrunk to the views that exist.  Returns (images (1,N,H,W,3) float32, cams (1,N,2,4,4) float32, depth_gt | None)
    as NumPy arrays (host side, as in the reference)."""
    import os
    import cv2
    import numpy as np
    images, cams = [], []
    for i in range(view_num):
        ip, cp = os.path.join(data_root, '%d.jpg' % i), os.path.join(data_root, '%d_cam.npy' % i)
        if not (os.path.exists(ip) and os.path.exists(cp)):
            break
        images.append(cv2.imread(ip))
        cams.append(np.load(cp))
    if not images:
        raise FileNotFoundError("no {i}.jpg / {i}_cam.npy pairs under %s" % data_root)
    gt = os.path.join(data_root, '0_gt.npy')
    return (np.stack(images)[None].astype(np.float32), np.stack(cams)[None].astype(np.float32),
            np.load(gt) if os.path.exists(gt) else None)


class _DeviceStream(object):
    """What FrameStream keeps on one device: the step captured as a CUDA graph over fixed device buffers, the
    double-buffered staging of inputs and outputs, the two copy streams and the pinned host outputs."""

    def __init__(self, feats_shape, cams_shape, depth_num, device, siamese, confidence):
        self.device = device
        self.depth_num = int(depth_num)
        with torch.cuda.device(device):
            self.feats = torch.zeros(feats_shape, dtype=torch.float32, device=device)
            self.cams = torch.zeros(cams_shape, dtype=torch.float32, device=device)
            self.stage_f = [torch.empty_like(self.feats) for _ in range(2)]
            self.stage_c = [torch.empty_like(self.cams) for _ in range(2)]
            self.s_in, self.s_out = torch.cuda.Stream(device=device), torch.cuda.Stream(device=device)
        self.siamese = siamese
        self.confidence = confidence
        self.graph = None
        self.out = None

    def _step(self):
        return run_multiview(self.feats, self.cams, self.depth_num, siamese=self.siamese, confidence=self.confidence)

    def _capture(self):
        for _ in range(3):      # eager warm-up: copies and packs the weights, sets kernel attributes, fills the allocator
            self._step()
        torch.cuda.synchronize(self.device)
        s = torch.cuda.Stream(device=self.device)
        s.wait_stream(torch.cuda.current_stream(self.device))
        with torch.cuda.stream(s):
            self.graph = torch.cuda.CUDAGraph()
            with torch.cuda.graph(self.graph, stream=s):
                res = self._step()
                self.out = [res[k] for k in (('depth_up', 'prob_map_up') if self.confidence else ('depth_up',))]
        torch.cuda.current_stream(self.device).wait_stream(s)
        # per output: staging slot k on the device and its pinned host copy, k = this device's frame index & 1
        self.stage_o = [[torch.empty_like(o) for o in self.out] for _ in range(2)]
        self.host_o = [[torch.empty(o.shape, dtype=torch.float32).pin_memory() for o in self.out] for _ in range(2)]

    def begin(self):
        """start of a FrameStream.run: frames dealt to this device are counted from 0 again"""
        self.n = 0
        self.free = [None, None]     # staging slot reusable once the step that read it has copied it out
        self.done = [None, None]     # D2H of slot complete
        self.main = torch.cuda.current_stream(self.device)

    def push(self, fh, ch):
        """enqueue one frame (nothing here waits for the device once the graph exists) -> (event, pinned result),
        the result complete once the event is"""
        k = self.n & 1
        self.n += 1
        main, free, done = self.main, self.free, self.done
        with torch.cuda.device(self.device):
            if self.graph is None:
                # captured on real data of the first frame dealt to this device (BN statistics of zeros are degenerate)
                self.feats.copy_(fh, non_blocking=True)
                self.cams.copy_(ch, non_blocking=True)
                self._capture()
            with torch.cuda.stream(self.s_in):
                if free[k] is not None:
                    self.s_in.wait_event(free[k])
                self.stage_f[k].copy_(fh, non_blocking=True)
                self.stage_c[k].copy_(ch, non_blocking=True)
                ready = torch.cuda.Event()
                ready.record(self.s_in)
            main.wait_event(ready)
            self.feats.copy_(self.stage_f[k], non_blocking=True)
            self.cams.copy_(self.stage_c[k], non_blocking=True)
            free[k] = torch.cuda.Event()
            free[k].record(main)
            self.graph.replay()
            if done[k] is not None:
                main.wait_event(done[k])          # stage_o[k] / host_o[k] of this device's frame before last are drained
            for so, o in zip(self.stage_o[k], self.out):
                so.copy_(o, non_blocking=True)
            computed = torch.cuda.Event()
            computed.record(main)
            with torch.cuda.stream(self.s_out):
                self.s_out.wait_event(computed)
                for ho, so in zip(self.host_o[k], self.stage_o[k]):
                    ho.copy_(so, non_blocking=True)
                done[k] = torch.cuda.Event()
                done[k].record(self.s_out)
        return done[k], tuple(self.host_o[k]) if self.confidence else self.host_o[k][0]


class FrameStream(object):
    """Depth maps for a stream of frames that live in PINNED HOST memory (what a reader thread hands over): the step is
    captured once per device as a CUDA graph over fixed device buffers, and the host->device copy of a device's next
    frame and the device->host copy of its previous depth map run on their own streams while the frame computes
    (double-buffered staging).

        fs = FrameStream(feats_shape, cams_shape, depth_num, device)
        for depth_h in fs.run(frames):      # frames: iterable of (feats_pinned, cams_pinned)
            ...                              # depth_h: pinned (B,4h,4w,1) fp32, valid until two frames later

    ``device`` is one device or a sequence of K devices: frame i then runs on device i mod K, every device with its
    own graph (captured on the first frame dealt to it), staging buffers, copy streams and weight copies, all driven
    from the calling thread, and ``run`` still yields the results in frame order.  The pinned buffers of frame i are
    reused by frame i + 2K, which is enqueued when the consumer asks for frame i + K: a result stays valid until two
    frames later on one device, and a consumer may hold the last K results it received.

    With ``confidence=True`` the graph also computes the x4 probability map (run_multiview's prob_map_up) and ``run``
    yields pinned (depth_h, confidence_h) pairs of that shape, copied and kept valid like the depth map alone.
    """

    def __init__(self, feats_shape, cams_shape, depth_num, device, siamese=True, confidence=False):
        devices = [device] if isinstance(device, (str, int, torch.device)) else list(device)
        if not devices:
            raise ValueError("FrameStream: no device given")
        self.devices = []
        for d in devices:
            d = torch.device('cuda', d) if isinstance(d, int) else torch.device(d)
            if d.type != 'cuda':
                raise ValueError("FrameStream runs on CUDA devices, got %s" % d)
            self.devices.append(torch.device('cuda', torch.cuda.current_device()) if d.index is None else d)
        self.confidence = confidence
        self.lanes = [_DeviceStream(feats_shape, cams_shape, depth_num, d, siamese, confidence) for d in self.devices]

    @property
    def graph(self):
        """the captured graph of the first device (None before its first frame)"""
        return self.lanes[0].graph

    def run(self, frames):
        """generator over pinned host depth maps, one per frame, in order (each is yielded once its copy is complete);
        (depth, confidence) pairs with ``confidence=True``."""
        K = len(self.lanes)
        for lane in self.lanes:
            lane.begin()
        pending = []
        for i, (fh, ch) in enumerate(frames):
            pending.append(self.lanes[i % K].push(fh, ch))
            if len(pending) > K:      # every device keeps a frame queued behind the one the host waits for
                ev, buf = pending.pop(0)
                ev.synchronize()
                yield buf
        for ev, buf in pending:
            ev.synchronize()
            yield buf
