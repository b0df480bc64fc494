"""Layer DSL of /root/reference/cnn_wrapper/network.py (Network :37-119 and the hot-path
layers conv :142, conv_bn :173, attention_aggregation :379, deconv_bn :511, add :696) on
torch CUDA tensors, executing hand-written sm_100a kernels through libatvs.so.

Differences that are deliberate and invisible at the call surface:
  * ``setup()`` records the layer graph; it is executed on the first ``get_output*()`` so
    that batch-norm (batch statistics, no affine: network.py:206-212 with
    ``training=True, center=False, scale=False``), ReLU and the ``add`` skip joins run as ONE
    fused elementwise kernel per conv layer instead of separate graph ops;
  * activations between layers are fp16 (default) or bf16 when ``FLAGS.precision`` is
    ``'fp16'`` / ``'bf16'`` (tcgen05 path) and fp32 when ``'fp32'`` (CUDA-core parity path); BN
    moments always come from the fp32 accumulators;
  * variables are looked up by their TF checkpoint names in ``variables``.
"""
from collections import OrderedDict

import torch

from . import _lib as L
from . import variables as V
from .flags import FLAGS

BN_EPS = 1e-3   # tf.layers.batch_normalization default (network.py:206)

# measurement hook (bench.py): when set to (predicate, sink), conv launches whose weight key
# satisfies predicate(key) are bracketed by CUDA events on the launching stream.
PROFILE = None


_ACT = {'fp32': torch.float32, 'bf16': torch.bfloat16, 'fp16': torch.float16}
HALF_DTYPES = (torch.bfloat16, torch.float16)


def act_dtype():
    try:
        return _ACT[FLAGS.precision]
    except KeyError:
        raise ValueError("FLAGS.precision must be 'fp16', 'bf16' or 'fp32' (got %r)" % (FLAGS.precision,))


def _same_shape(who, tensors):
    """every operand of a skip join must have the lead tensor's shape (TF raises on a mismatch; the fused kernels size
    their launch from the lead tensor)."""
    lead = tuple(tensors[0].shape)
    for t in tensors[1:]:
        if t is not None and tuple(t.shape) != lead:
            raise ValueError("%s: operand shapes differ: %s vs %s (volumes must be divisible by 8 in D, H and W for the "
                             "stride-2 down / up path to line up)" % (who, lead, tuple(t.shape)))


def to_act(t):
    """fp32/bf16 NDHWC tensor -> contiguous tensor in the activation dtype."""
    L.require_cuda(t)
    dt = act_dtype()
    t = t.contiguous()
    if t.dtype == dt:
        return t
    if t.dtype not in (torch.float32, torch.bfloat16, torch.float16):
        t = t.float()
    if t.dtype in HALF_DTYPES and dt in HALF_DTYPES:      # bf16 <-> fp16: through fp32
        t = to_dtype(t, torch.float32)
    return to_dtype(t, dt)


def to_dtype(t, dt):
    if t.dtype == dt:
        return t
    out = torch.empty(t.shape, dtype=dt, device=t.device)
    L.call("atvs_cast", L.ptr(t), L.dtype_code(t), L.ptr(out), L.dtype_code(out), t.numel(), L.stream())
    return out


def _dt_code(dt):
    return {torch.float32: L.F32, torch.bfloat16: L.BF16, torch.float16: L.F16}[dt]


def _packed_weight(key, w, cin, cout, transposed, dt):
    """16-bit weight images of one layer (all kernel formulations), cached per (variable, format)."""
    cache = V.packed_cache()
    key = key + ('|bf16' if dt == torch.bfloat16 else '|f16')
    if key not in cache:
        nbytes = L.load().atvs_packed_weight_bytes(cin, cout, transposed)
        buf = torch.empty(nbytes, dtype=torch.uint8, device=w.device)
        L.call("atvs_pack_conv_weights_tc", L.ptr(w), cin, cout, transposed, _dt_code(dt), L.ptr(buf), L.stream())
        cache[key] = buf
    return cache[key]


class SplitCostVolume(object):
    """The two-view cost volume of model.py:186-195, ``concat([tile(ref, D), warped], -1)``, kept as
    its two parts: ``ref`` (B,h,w,F) and ``warped`` (B,D,h,w,F).  A convolution over the concatenation
    is linear in the halves, and the ``tile(ref, D)`` half is the same 2-D result on every interior
    plane, so the first CRM layers run on the F warped channels only and add the reference part as a
    per-plane-class bias in their epilogue (atvs_conv3d_tc_bias).  Halves the dominant layer's work
    and the volume K1 has to write; results equal the concatenated form up to fp32 summation order."""

    def __init__(self, ref, warped):
        if warped.dtype not in HALF_DTYPES:
            raise ValueError("SplitCostVolume is a tensor-core path construct (fp16 / bf16 volumes)")
        self.ref, self.warped = ref, warped
        self.shape = tuple(warped.shape[:-1]) + (warped.shape[-1] + ref.shape[-1],)
        self.device = warped.device
        self.dtype = warped.dtype
        self._tiled = {}

    def ref_tiled(self, planes):
        if planes not in self._tiled:
            B, h, w, F = self.ref.shape
            r = to_dtype(self.ref.contiguous(), self.warped.dtype)
            self._tiled[planes] = r[:, None].expand(B, planes, h, w, F).contiguous()
        return self._tiled[planes]


def _split_weights(wkey, w, F):
    cache = V.packed_cache()
    k = wkey + '/split'
    if k not in cache:
        cache[k] = (w[..., :F, :].contiguous(), w[..., F:, :].contiguous())
    return cache[k]


def conv3d_split(cv, wkey, w, cout, stride, stats_buf):
    """first-layer convolution on a SplitCostVolume: bias from the reference half, main conv on the
    warped half.  Returns (raw fp32 (B,Do,ho,wo,Cout), moments)."""
    F = cv.ref.shape[-1]
    w_ref, w_warp = _split_weights(wkey, w, F)
    bias = _split_bias(cv, wkey, w_ref, cout, stride)
    return conv3d_raw(cv.warped, wkey + '/warp', w_warp, cout, stride, False, True, stats_buf, bias=bias,
                      raw_dtype=raw_dtype_for_bn(cv.warped, first=True))


def _split_bias(cv, wkey, w_ref, cout, stride):
    """depth-invariant part of a first-layer convolution (the tiled reference half): 3 plane classes."""
    planes = 3 if stride == 1 else 4
    bias, _ = conv3d_raw(cv.ref_tiled(planes), wkey + '/ref', w_ref, cout, stride, False, False)
    if stride == 2:                      # planes (interior, last) -> classes (first == interior, interior, last)
        bias = torch.cat([bias[:, :1], bias[:, :1], bias[:, 1:2]], dim=1).contiguous()
    return bias


def raw_dtype_for_bn(x, first=False):
    """dtype of a raw convolution output that only feeds the BN pass: fp16 on the tensor-core path
    (FLAGS.raw_dtype = 'f16': saturated, moments still from the fp32 accumulators), fp32 otherwise.
    ``first``: the layer reads the un-normalised cost volume (FLAGS.first_raw_dtype)."""
    flag = getattr(FLAGS, 'first_raw_dtype', 'f32') if first else getattr(FLAGS, 'raw_dtype', 'f16')
    if x.dtype in HALF_DTYPES and flag == 'f16':
        return torch.float16
    return torch.float32


def _raw_code(t):
    return L.F16 if t.dtype == torch.float16 else L.F32


def conv3d_raw(x, wkey, w, cout, stride, transposed, want_stats, stats_buf=None, bias=None, out=None,
               raw_dtype=torch.float32):
    """x (B,D,H,W,Cin) fp32|bf16 -> raw (B,Do,Ho,Wo,Cout) fp32 (or fp16 on request, bf16 inputs only)
    [+ fp64 moments (2*Cout)].
    ``stats_buf``: pre-zeroed fp64 buffer of >= 2*Cout elements to accumulate the moments into."""
    B, D, H, W, cin = x.shape
    if transposed:
        od, oh, ow = 2 * D, 2 * H, 2 * W
    else:
        od, oh, ow = -(-D // stride), -(-H // stride), -(-W // stride)
    if x.dtype == torch.float32:
        raw_dtype = torch.float32
    raw = out if out is not None else torch.empty((B, od, oh, ow, cout), dtype=raw_dtype, device=x.device)
    if not want_stats:
        stats = None
    elif stats_buf is not None:
        stats = stats_buf[:2 * cout]
    else:
        stats = torch.zeros(2 * cout, dtype=torch.float64, device=x.device)
    prof = PROFILE is not None and PROFILE[0](wkey)
    if prof:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
    if x.dtype == torch.float32:
        L.call("atvs_conv3d_fp32", L.ptr(x), L.ptr(w), B, D, H, W, cin, cout, stride, int(transposed),
               L.ptr(raw), L.ptr(stats), L.stream())
    else:
        pk = _packed_weight(wkey, w, cin, cout, int(transposed), x.dtype)
        if bias is not None:
            L.call("atvs_conv3d_tc_bias", L.ptr(x), L.dtype_code(x), L.ptr(pk), B, D, H, W, cin, cout, stride, L.ptr(bias),
                   L.ptr(raw), _raw_code(raw), L.ptr(stats), L.stream())
        else:
            L.call("atvs_conv3d_tc", L.ptr(x), L.dtype_code(x), L.ptr(pk), B, D, H, W, cin, cout, stride, int(transposed),
                   L.ptr(raw), _raw_code(raw), L.ptr(stats), L.stream())
    if prof:
        e1.record()
        # last field: re-issues exactly this launch (same tensors), for back-to-back replays of one layer
        again = lambda: conv3d_raw(x, wkey, w, cout, stride, transposed, want_stats, stats_buf=stats, bias=bias, out=raw,
                                   raw_dtype=raw_dtype)
        PROFILE[1].append((wkey, e0, e1, raw.numel() // cout, cin, cout, again))
    return raw, stats


def bn_relu_add(raw, stats, relu, skips, want_plain, want_sum, dtype):
    count = raw.numel() // raw.shape[-1]
    plain = torch.empty(raw.shape, dtype=dtype, device=raw.device) if want_plain else None
    summ = torch.empty(raw.shape, dtype=dtype, device=raw.device) if want_sum else None
    s1 = skips[0] if len(skips) > 0 else None
    s2 = skips[1] if len(skips) > 1 else None
    _same_shape("add", [raw, s1, s2])
    for sk in (s1, s2):
        if sk is not None and sk.dtype != dtype:
            raise RuntimeError("bn_relu_add: skip dtype %s != activation dtype %s" % (sk.dtype, dtype))
    L.call("atvs_bn_relu_add", L.ptr(raw), _raw_code(raw), L.ptr(stats), count, raw.shape[-1], BN_EPS, int(relu), L.ptr(s1),
           L.ptr(s2), L.ptr(plain), L.ptr(summ), _dt_code(dtype), L.stream())
    return plain, summ


class _PendingRaw(object):
    """raw convolution output + moments of a conv_bn layer whose only consumer is an `add` led by a
    later layer: normalised inside that layer's fused pass (atvs_bn_relu_add_pair)."""
    __slots__ = ('raw', 'stats', 'relu')

    def __init__(self, raw, stats, relu):
        self.raw, self.stats, self.relu = raw, stats, relu


def bn_relu_add_pair(raw_a, stats_a, pend, relu, skip, want_plain, dtype):
    count = raw_a.numel() // raw_a.shape[-1]
    plain = torch.empty(raw_a.shape, dtype=dtype, device=raw_a.device) if want_plain else None
    summ = torch.empty(raw_a.shape, dtype=dtype, device=raw_a.device)
    if pend.raw.dtype != raw_a.dtype:
        raise RuntimeError("bn_relu_add_pair: raw dtypes differ")
    _same_shape("add", [raw_a, pend.raw, skip])
    L.call("atvs_bn_relu_add_pair", L.ptr(raw_a), L.ptr(stats_a), L.ptr(pend.raw), L.ptr(pend.stats), _raw_code(raw_a), count,
           raw_a.shape[-1], BN_EPS, int(relu), L.ptr(skip), L.ptr(plain), L.ptr(summ), _dt_code(dtype), L.stream())
    return plain, summ


class _Node(object):
    __slots__ = ('name', 'kind', 'inputs', 'params', 'value')

    def __init__(self, name, kind, inputs, params, value=None):
        self.name, self.kind, self.inputs, self.params, self.value = name, kind, inputs, params, value


class Network(object):
    """cnn_wrapper/network.py:37-119.  ``Cls({'data': t}, is_training=True, reuse=...)``."""

    def __init__(self, inputs, is_training=True, dropout_rate=0.9, seed=None, reuse=False, scope_name=None,
                 outputs=()):
        self.inputs = inputs
        self.training = is_training     # accepted; BN always uses batch statistics (F4)
        self.reuse = reuse              # accepted and ignored
        self.nodes = OrderedDict()
        self.terminals = []
        self._wanted = set(outputs)
        self._ran = False
        for k, v in inputs.items():
            self.nodes[k] = _Node(k, 'input', [], {}, v)
        self.setup()
        self._last = self.terminals[-1] if self.terminals else None

    def setup(self):
        raise NotImplementedError('Must be implemented by the subclass.')

    # -- graph recording ---------------------------------------------------------
    def feed(self, *args):
        assert args
        self.terminals = []
        for a in args:
            if a not in self.nodes:
                raise KeyError('Unknown layer name fed: %s' % a)
            self.terminals.append(a)
        return self

    def _add_node(self, name, kind, **params):
        if not self.terminals:
            raise RuntimeError('No input variables found for layer %s.' % name)
        self.nodes[name] = _Node(name, kind, list(self.terminals), params)
        self.terminals = [name]
        return self

    def conv(self, kernel_size, filters, strides, name, relu=True, padding='SAME', biased=False, rate=1):
        self._check(kernel_size, padding, biased, rate)
        return self._add_node(name, 'conv', filters=filters, stride=strides, relu=relu)

    def conv_bn(self, kernel_size, filters, strides, name, relu=True, center=False, padding='SAME', biased=False,
                rate=1):
        self._check(kernel_size, padding, biased, rate)
        if center:
            raise NotImplementedError('conv_bn(center=True) is not on the 3-D hot path')
        return self._add_node(name, 'conv_bn', filters=filters, stride=strides, relu=relu)

    def deconv_bn(self, kernel_size, filters, strides, name, relu=True, center=False, padding='SAME', biased=False):
        self._check(kernel_size, padding, biased, 1)
        if strides != 2 or center:
            raise NotImplementedError('deconv_bn: only stride 2, center=False')
        return self._add_node(name, 'deconv_bn', filters=filters, stride=strides, relu=relu)

    def add(self, name):
        return self._add_node(name, 'add')

    def attention_aggregation(self, kernel_size, name, filters=None, second_weight=False, relu=True, padding='SAME',
                              biased=False, n_view=None):
        self._check(kernel_size, padding, biased, 1)
        if not (second_weight and relu) or filters is not None:
            raise NotImplementedError('attention_aggregation: only second_weight=True, relu=True, filters=None')
        return self._add_node(name, 'attention_aggregation')

    @staticmethod
    def _check(kernel_size, padding, biased, rate):
        if kernel_size != 3 or padding != 'SAME' or biased or rate != 1:
            raise NotImplementedError('hot-path 3-D layers are kernel 3, SAME, no bias, rate 1')

    def get_shape_by_name(self, layer_name):
        n = self.nodes[layer_name]
        if n.value is None:
            self._run()
        v = self.nodes[layer_name].value
        return tuple(v[0].shape) + (len(v),) if isinstance(v, (list, tuple)) else tuple(v.shape)

    # -- outputs -----------------------------------------------------------------
    def get_output(self):
        return self.get_output_by_name(self._last)

    def get_output_by_name(self, layer_name):
        if layer_name not in self.nodes:
            raise KeyError(layer_name)
        if not self._ran or self.nodes[layer_name].value is None:
            self._wanted.add(layer_name)
            self._wanted.add(self._last)
            self._run()
        return self.nodes[layer_name].value

    # -- execution ---------------------------------------------------------------
    def _run(self):
        with L.input_device(self.inputs, type(self).__name__):
            self._execute()

    def _execute(self):
        nodes = self.nodes
        order = list(nodes.keys())
        pos = {n: i for i, n in enumerate(order)}
        consumers = {n: [] for n in order}
        for n in order:
            for i in nodes[n].inputs:
                consumers[i].append(n)
        remaining = {n: len(consumers[n]) for n in order}
        done = set(n for n in order if nodes[n].kind == 'input')
        for n in order:
            if nodes[n].kind != 'input':
                nodes[n].value = None
        dt = act_dtype()
        # one zero-filled arena for the batch-norm moments of every conv_bn / deconv_bn layer
        bn_nodes = [n for n in order if nodes[n].kind in ('conv_bn', 'deconv_bn')]
        first = next(v.value for v in nodes.values() if v.kind == 'input')
        dev = (first[0] if isinstance(first, (list, tuple)) else first).device   # tensors and SplitCostVolume have .device
        arena = torch.zeros((max(len(bn_nodes), 1), 128), dtype=torch.float64, device=dev)
        arena_slot = {n: i for i, n in enumerate(bn_nodes)}

        def release(names):
            for i in names:
                remaining[i] -= 1
                if remaining[i] == 0 and i not in self._wanted and nodes[i].kind != 'input':
                    nodes[i].value = None

        def act_in(name):
            v = nodes[name].value
            if isinstance(v, SplitCostVolume):
                return v
            if isinstance(v, _PendingRaw):     # deferred normalisation that no fused add picked up
                v, _ = bn_relu_add(v.raw, v.stats, v.relu, [], True, False, dt)
                nodes[name].value = v
                return v
            if nodes[name].kind == 'input':
                v = to_act(v)
                nodes[name].value = v      # cast once
            return v

        for name in order:
            node = nodes[name]
            if name in done:
                continue
            if node.kind in ('conv_bn', 'deconv_bn'):
                x = act_in(node.inputs[0])
                transposed = node.kind == 'deconv_bn'
                wname = name + ('/conv3d_transpose/kernel' if transposed else '/conv3d/kernel')
                if isinstance(x, SplitCostVolume):
                    raw, stats = conv3d_split(x, wname, V.get_variable(wname), node.params['filters'],
                                              node.params['stride'], arena[arena_slot[name]])
                else:
                    raw, stats = conv3d_raw(x, wname, V.get_variable(wname), node.params['filters'],
                                            node.params['stride'], transposed, True, arena[arena_slot[name]],
                                            raw_dtype=raw_dtype_for_bn(x, first=nodes[node.inputs[0]].kind == 'input'))
                # a layer that only feeds an `add` led by a LATER conv layer is normalised inside that
                # layer's fused pass: keep its raw output and moments until then
                cons = consumers[name]
                if (len(cons) == 1 and name not in self._wanted and nodes[cons[0]].kind == 'add'
                        and nodes[cons[0]].inputs[0] != name and len(nodes[cons[0]].inputs) <= 3
                        and nodes[nodes[cons[0]].inputs[0]].kind in ('conv_bn', 'deconv_bn')
                        and pos[nodes[cons[0]].inputs[0]] > pos[name]
                        and not any(isinstance(nodes[i].value, _PendingRaw) for i in nodes[cons[0]].inputs)
                        and nodes[nodes[cons[0]].inputs[0]].params['relu'] == node.params['relu']
                        and raw.dtype == raw_dtype_for_bn(x)):
                    node.value = _PendingRaw(raw, stats, node.params['relu'])
                    done.add(name)
                    release(node.inputs)
                    continue
                # fuse a following add(name, older...) into the normalisation pass
                fused = None
                for c in consumers[name]:
                    cn = nodes[c]
                    if cn.kind == 'add' and cn.inputs[0] == name and len(cn.inputs) <= 3 and \
                            all(i in done for i in cn.inputs[1:]):
                        fused = cn
                        break
                others = [c for c in consumers[name] if fused is None or c != fused.name]
                want_plain = bool(others) or name in self._wanted or fused is None
                skips = [nodes[i].value for i in fused.inputs[1:]] if fused is not None else []
                pend = [v for v in skips if isinstance(v, _PendingRaw)]
                if pend:
                    rest = [v for v in skips if not isinstance(v, _PendingRaw)]
                    plain, summ = bn_relu_add_pair(raw, stats, pend[0], node.params['relu'], rest[0] if rest else None,
                                                   want_plain, dt)
                else:
                    plain, summ = bn_relu_add(raw, stats, node.params['relu'], skips, want_plain, fused is not None, dt)
                node.value = plain
                done.add(name)
                release(node.inputs)
                if fused is not None:
                    fused.value = summ
                    done.add(fused.name)
                    release(fused.inputs)
            elif node.kind == 'conv':
                x = act_in(node.inputs[0])
                wname = name + '/kernel'
                raw, _ = conv3d_raw(x, wname, V.get_variable(wname), node.params['filters'], node.params['stride'],
                                    False, False)
                if node.params['relu']:
                    raw = torch.relu_(raw)
                node.value = raw               # fp32 (network outputs are fp32 at the API)
                done.add(name)
                release(node.inputs)
            elif node.kind == 'add':
                vals = [act_in(i) for i in node.inputs]
                _same_shape("add(%s)" % name, vals)
                out = torch.empty_like(vals[0])
                L.call("atvs_add", L.ptr(vals[0]), L.ptr(vals[1]), L.ptr(out), L.dtype_code(out), out.numel(),
                       L.stream())
                for v in vals[2:]:
                    L.call("atvs_add", L.ptr(out), L.ptr(v), L.ptr(out), L.dtype_code(out), out.numel(), L.stream())
                node.value = out
                done.add(name)
                release(node.inputs)
            elif node.kind == 'attention_aggregation':
                node.value = attention_aggregation(nodes[node.inputs[0]].value, name)
                done.add(name)
                release(node.inputs)
            else:
                raise RuntimeError('unknown layer kind %s' % node.kind)
        self._ran = True


def split_views(cost_volumes):
    """(B,D,H,W,C,N) (reference layout: view innermost, example.py:150) or a list of N
    (B,D,H,W,C) tensors -> list of N contiguous activation-dtype tensors."""
    if isinstance(cost_volumes, (list, tuple)):
        return [to_act(v) for v in cost_volumes]
    L.require_cuda(cost_volumes)
    n = cost_volumes.shape[-1]
    return [to_act(cost_volumes[..., i]) for i in range(n)]


def _attention_weights(scope):
    key = scope + '/attention_activation/weight_unique||weight_shared'
    cache = V.packed_cache()
    if key not in cache:
        wu = V.get_variable(scope + '/attention_activation/weight_unique')
        ws = V.get_variable(scope + '/attention_activation/weight_shared')
        cache[key] = torch.cat([wu, ws], dim=-1).contiguous()
    return key, cache[key]


def attention_raw_alloc(n_views, like, device=None):
    """raw logits buffer (N,V,16) for n_views volumes shaped (and typed) like ``like`` (B,D,H,W,C)."""
    c = like.shape[-1]
    nvox = like.numel() // c
    return torch.empty((n_views, nvox, 2 * c), dtype=raw_dtype_for_bn(like), device=device or like.device)


def attention_raw_view(raw, n, x, scope):
    """network.py:313-344 for ONE view: the pair [conv(x,W_unique) | conv(x,W_shared)] as one 8->16 convolution into
    raw[n], NOT yet activated (the ReLU is applied by the combine kernel).  Independent per view, so the stage-I
    stream of a view can run it right behind that view's regularisation pass."""
    key, w = _attention_weights(scope)
    B, D, H, W_, _ = x.shape
    conv3d_raw(x, key + '/packed', w, w.shape[-1], 1, False, False, out=raw[n].view(B, D, H, W_, w.shape[-1]))


def attention_activations_raw(views, scope):
    """network.py:282-351: per view the pair [conv(x,W_unique) | conv(x,W_shared)] as one 8->16
    convolution, NOT yet activated: raw (N,V,16), fp16 on the tensor path (raw_dtype_for_bn) else fp32.
    The ReLU is applied by the combine kernel."""
    raw = attention_raw_alloc(len(views), views[0])
    for n, x in enumerate(views):
        attention_raw_view(raw, n, x, scope)
    return raw


def view_pointers(views):
    """HOST array of the N per-view device pointers (atvs_attention_raw reads the views where they are)."""
    import ctypes
    for v in views:
        if not v.is_contiguous() or v.dtype != views[0].dtype:
            raise RuntimeError("attention views must be contiguous and of one dtype")
    return (ctypes.c_void_p * len(views))(*[v.data_ptr() for v in views])


def attention_activations(views, scope):
    """activated pairs [relu(conv(x,W_unique)) | relu(conv(x,W_shared))] (N,V,16) in the activation dtype."""
    raw = attention_activations_raw(views, scope)
    dt = views[0].dtype
    act = torch.empty(raw.shape, dtype=dt, device=raw.device)
    L.call("atvs_bn_relu_add", L.ptr(raw), _raw_code(raw), None, raw.shape[0] * raw.shape[1], raw.shape[2], BN_EPS, 1, None, None,
           L.ptr(act), None, _dt_code(dt), L.stream())
    return act


def stack_views(views):
    c = views[0].shape[-1]
    nvox = views[0].numel() // c
    return torch.stack([v.reshape(nvox, c) for v in views], dim=0) if len(views) > 1 else views[0].reshape(1, nvox, c)


def attention_fused_ok(views):
    """the one-kernel AAM (atvs_attention_fused) covers 2..8 views of 8 channels in a 16-bit dtype, D >= 3, H, W >= 8"""
    if not getattr(FLAGS, 'attention_fused', True) or not isinstance(views, (list, tuple)) or not 2 <= len(views) <= 8:
        return False
    v = views[0]
    return (v.dtype in HALF_DTYPES and v.dim() == 5 and v.shape[-1] == 8 and v.shape[1] >= 3 and v.shape[2] >= 8
            and v.shape[3] >= 8)


def attention_aggregation(cost_volumes, scope, raw=None):
    """network.py:379-408 -> (B,D,H,W,C) fp32.  ``raw``: logits already produced by attention_raw_view()."""
    views = split_views(cost_volumes)
    shape = views[0].shape
    c = shape[-1]
    nvox = views[0].numel() // c
    out = torch.empty((nvox, c), dtype=torch.float32, device=views[0].device)
    if raw is None and attention_fused_ok(views):
        key, w = _attention_weights(scope)
        B, D, H, W_, _ = shape
        pk = _packed_weight(key + '/packed', w, c, 2 * c, 0, views[0].dtype)
        L.call("atvs_attention_fused", view_pointers(views), len(views), L.dtype_code(views[0]), L.ptr(pk), B, D, H, W_, c,
               L.ptr(out), L.stream())
    elif c % 8 == 0:
        if raw is None:
            raw = attention_activations_raw(views, scope)
        L.call("atvs_attention_raw", L.ptr(raw), _raw_code(raw), view_pointers(views), len(views), nvox, c,
               L.dtype_code(views[0]), 0, None, L.ptr(out), L.stream())
    else:
        x = stack_views(views)
        act = attention_activations(views, scope)
        L.call("atvs_attention_combine", L.ptr(act), L.ptr(x), len(views), nvox, c, L.dtype_code(x), L.ptr(out),
               L.stream())
    return out.reshape(shape)
