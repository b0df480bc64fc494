"""Variable store keyed by the TF checkpoint variable names (SURVEY.md Appendix B).

The reference restores ``tf.global_variables()`` from ``model.ckpt`` (example.py:121-125)
and its ops find weights through TF variable scopes; here the same names index a dict of
CUDA tensors.  The released checkpoint is not available offline, so
``synthetic_weights`` generates seeded He-normal kernels with the reference's names and
shapes."""
import numpy as np
import torch

_STORE = {}
_COPIES = {}            # device index -> {name: copy of _STORE[name] on that device}
_PACKED = {}            # device index -> {key: packed weight image derived from that device's variables}
_GENERATION = [0]


def load_weights(weights, device='cuda'):
    """weights: dict name -> array (TF layouts), or a path to an .npz with those keys.  The store lives on ``device``;
    a call on another device's inputs copies each variable it reads there once (get_variable).  Loading drops every
    copy and packed image on every device."""
    if isinstance(weights, str):
        weights = dict(np.load(weights))
    _STORE.clear()
    _COPIES.clear()
    _PACKED.clear()
    _GENERATION[0] += 1
    for k, v in weights.items():
        _STORE[k] = torch.as_tensor(np.asarray(v, dtype=np.float32)).to(device).contiguous()


def _current_device():
    return torch.cuda.current_device() if torch.cuda.is_initialized() else None


def get_variable(name):
    """the variable on the current device (the device of the call's inputs, _lib.input_device): the loaded tensor, or
    its copy made on first use there."""
    try:
        t = _STORE[name]
    except KeyError:
        raise KeyError("variable %r not loaded (call variables.load_weights first)" % name)
    dev = _current_device()
    if not t.is_cuda or t.device.index == dev:
        return t
    copies = _COPIES.setdefault(dev, {})
    if name not in copies:
        copies[name] = t.to(torch.device('cuda', dev))
    return copies[name]


def has_variable(name):
    return name in _STORE


def packed_cache():
    """the cache of images derived from the variables (packed weights, split and padded kernels) of the current
    device."""
    return _PACKED.setdefault(_current_device(), {})


def generation():
    """bumped by every load_weights(): consumers that derive state from the store (packed weight images, warm-up
    bookkeeping) key it on this."""
    return _GENERATION[0]


def crm_layer_table():
    """(name, kind, Cin, Cout, stride) for StackedUNet_prob, cnn_wrapper/atvsnet.py:100-192."""
    t = []
    for b in range(3):
        p = 'conv_b%d' % b
        cin0 = 64 if b == 0 else 8
        t += [(p + '_1_0', 'conv_bn', cin0, 16, 2), (p + '_2_0', 'conv_bn', 16, 32, 2),
              (p + '_3_0', 'conv_bn', 32, 64, 2), (p + '_0_1', 'conv_bn', cin0, 8, 1),
              (p + '_1_1', 'conv_bn', 16, 16, 1), (p + '_2_1', 'conv_bn', 32, 32, 1),
              (p + '_3_1', 'conv_bn', 64, 64, 1), (p + '_4_0', 'deconv_bn', 64, 32, 2),
              (p + '_5_0', 'deconv_bn', 32, 16, 2), (p + '_6_0', 'deconv_bn', 16, 8, 2)]
    t.append(('conv_b2_6_2', 'conv', 8, 1, 1))
    return t


def synthetic_weights(seed=1234, logit_gain=4.0):
    """Seeded He-normal weights with the checkpoint's names/shapes for the CRM
    (StackedUNet_prob), AAM1/AAM2 and the output convs.  ``logit_gain`` scales the two 8->1
    output kernels so that the soft-argmin is peaked (trained-like), SURVEY.md section 8(d)."""
    rng = np.random.default_rng(seed)
    w = {}

    def he(shape, fan_in):
        return (rng.standard_normal(shape) * np.sqrt(2.0 / fan_in)).astype(np.float32)

    for name, kind, cin, cout, _ in crm_layer_table():
        if kind == 'conv_bn':
            w[name + '/conv3d/kernel'] = he((3, 3, 3, cin, cout), 27 * cin)
        elif kind == 'deconv_bn':
            w[name + '/conv3d_transpose/kernel'] = he((3, 3, 3, cout, cin), 27 * cin / 8.0)
        else:
            w[name + '/kernel'] = he((3, 3, 3, cin, cout), 27 * cin) * np.float32(logit_gain)
        if kind != 'conv':
            w[name + '/batch_normalization/moving_mean'] = np.zeros((cout,), np.float32)
            w[name + '/batch_normalization/moving_variance'] = np.ones((cout,), np.float32)
    for scope, outc in (('attention_aggregate', 'attention_prob_vol'),
                        ('attention_aggregate_refine', 'attention_prob_vol_refine')):
        w[scope + '/attention_activation/weight_unique'] = he((3, 3, 3, 8, 8), 27 * 8)
        w[scope + '/attention_activation/weight_shared'] = he((3, 3, 3, 8, 8), 27 * 8)
        w[outc + '/kernel'] = he((3, 3, 3, 8, 1), 27 * 8) * np.float32(logit_gain)
    return w


def fem_variable_shapes():
    """name -> shape of the FEM (ResNetDS2SPP) variables, cnn_wrapper/atvsnet.py:254-292 + network.py:552-616 naming
    (SURVEY.md Appendix B); tests/test_host_logic.py holds it equal to the list recorded from the reference's own
    graph code (tests/golden/fem_variables.json)."""
    s = {'conv0_0/conv2d/kernel': (3, 3, 3, 32), 'conv0_1/conv2d/kernel': (3, 3, 32, 32),
         'conv0_2/conv2d/kernel': (3, 3, 32, 32)}
    cin = 32
    for name, depth, nblock in (('conv0_x', 32, 3), ('conv1_x', 64, 8), ('conv2_x', 128, 3), ('conv3_x', 128, 3)):
        for i in range(nblock):
            scope = name + '_%d' % i if i != nblock - 1 else name
            s[scope + '/preact/beta'] = (cin,)
            if cin != depth:
                s[scope + '/shortcut/weights'] = (1, 1, cin, depth)
                s[scope + '/shortcut/biases'] = (depth,)
            s[scope + '/conv1/weights'] = (1, 1, cin, depth)
            s[scope + '/conv2/weights'] = (3, 3, depth, depth)
            s[scope + '/conv3/weights'] = (1, 1, depth, depth)
            for c in ('conv1', 'conv2', 'conv3'):
                s[scope + '/' + c + '/biases'] = (depth,)
            cin = depth
    for i in range(4):
        s['branch_%d_conv/conv2d/kernel' % i] = (3, 3, 128, 32)
    s['fusion0/conv2d/kernel'] = (3, 3, 320, 128)
    s['fusion1/kernel'] = (1, 1, 128, 32)
    return s


def synthetic_fem_weights(seed=4321):
    """seeded FEM weights under the checkpoint names: He-normal kernels, small biases / betas."""
    w = {}
    for i, (name, shape) in enumerate(sorted(fem_variable_shapes().items())):
        rng = np.random.default_rng([seed, i])
        if len(shape) == 4:
            w[name] = (rng.standard_normal(shape) * np.sqrt(2.0 / np.prod(shape[:-1]))).astype(np.float32)
        else:
            w[name] = (rng.standard_normal(shape) * 0.1).astype(np.float32)
    return w


def refine_variable_shapes():
    """name -> shape of the refinement-stage variables (shallow feature net model.py:143-154 / atvsnet.py:245-251 and
    CostVolRefineNet atvsnet.py:295-336); tests/test_host_logic.py holds it equal to the list recorded from the
    reference's own code (tests/golden/refine_variables.json)."""
    s = {}
    cin = 3
    for i in range(3):
        scope = 'global_refine_conv0_x' + ('_%d' % i if i != 2 else '')
        s[scope + '/preact/beta'] = (cin,)
        if cin != 16:
            s[scope + '/shortcut/weights'] = (1, 1, cin, 16)
            s[scope + '/shortcut/biases'] = (16,)
        s[scope + '/conv1/weights'] = (1, 1, cin, 16)
        s[scope + '/conv2/weights'] = (3, 3, 16, 16)
        s[scope + '/conv3/weights'] = (1, 1, 16, 16)
        for c in ('conv1', 'conv2', 'conv3'):
            s[scope + '/' + c + '/biases'] = (16,)
        cin = 16
    s['global_refine_shallow_feature/kernel'] = (1, 1, 16, 16)
    p = 'global_refine_'
    for name, ci, co in (('photo_3dconv', 48, 8), ('geo_3dconv', 19, 8), ('prob_3dconv', 1, 8), ('vishull_3dconv', 1, 8),
                         ('3dconv1_0', 32, 16), ('3dconv2_0', 16, 32), ('3dconv3_0', 32, 64), ('3dconv0_1', 32, 8),
                         ('3dconv1_1', 16, 16), ('3dconv2_1', 32, 32), ('3dconv3_1', 64, 64)):
        s[p + name + '/conv3d/kernel'] = (3, 3, 3, ci, co)
    for name, ci, co in (('3dconv4_0', 64, 32), ('3dconv5_0', 32, 16), ('3dconv6_0', 16, 8)):
        s[p + name + '/conv3d_transpose/kernel'] = (3, 3, 3, co, ci)
    s['global_refined_cost_vol/kernel'] = (3, 3, 3, 8, 1)
    return s


def synthetic_refine_weights(seed=2468):
    """seeded refinement-stage weights under the checkpoint names."""
    w = {}
    for i, (name, shape) in enumerate(sorted(refine_variable_shapes().items())):
        rng = np.random.default_rng([seed, i])
        if len(shape) >= 4:
            fan_in = np.prod(shape[:-2]) * (shape[-1] if 'transpose' in name else shape[-2])
            w[name] = (rng.standard_normal(shape) * np.sqrt(2.0 / fan_in)).astype(np.float32)
        else:
            w[name] = (rng.standard_normal(shape) * 0.1).astype(np.float32)
    return w


def expected_variable_shapes(parts=('crm', 'fem', 'refine')):
    """name -> shape of every variable the inference graphs read (SURVEY.md Appendix B): 'crm' = StackedUNet_prob, both
    attention modules and both output convolutions (the hot path), 'fem' = ResNetDS2SPP, 'refine' = the refinement stage."""
    s = {}
    if 'crm' in parts:
        for name, kind, cin, cout, _ in crm_layer_table():
            if kind == 'conv_bn':
                s[name + '/conv3d/kernel'] = (3, 3, 3, cin, cout)
            elif kind == 'deconv_bn':
                s[name + '/conv3d_transpose/kernel'] = (3, 3, 3, cout, cin)
            else:
                s[name + '/kernel'] = (3, 3, 3, cin, cout)
        for scope, outc in (('attention_aggregate', 'attention_prob_vol'), ('attention_aggregate_refine', 'attention_prob_vol_refine')):
            s[scope + '/attention_activation/weight_unique'] = (3, 3, 3, 8, 8)
            s[scope + '/attention_activation/weight_shared'] = (3, 3, 3, 8, 8)
            s[outc + '/kernel'] = (3, 3, 3, 8, 1)
    if 'fem' in parts:
        s.update(fem_variable_shapes())
    if 'refine' in parts:
        s.update(refine_variable_shapes())
    return s


def check_variables(weights, parts=('crm', 'fem', 'refine')):
    """raise a ValueError that lists every missing or mis-shaped variable of ``parts`` (a wrong or partial checkpoint
    would otherwise surface as a KeyError mid-pipeline or a mis-shaped kernel handed to a CUDA launch)."""
    exp = expected_variable_shapes(parts)
    missing = sorted(n for n in exp if n not in weights)
    wrong = sorted("%s: %s, expected %s" % (n, tuple(np.shape(weights[n])), exp[n]) for n in exp
                   if n in weights and tuple(np.shape(weights[n])) != tuple(exp[n]))
    if missing or wrong:
        raise ValueError("checkpoint does not hold the variables of %s: %d missing %s%s; %d mis-shaped %s"
                         % ('+'.join(parts), len(missing), missing[:8], ' ...' if len(missing) > 8 else '', len(wrong), wrong[:8]))


def load_checkpoint(prefix, device='cuda', parts=('crm', 'fem', 'refine')):
    """restore every variable of a TensorFlow V2 checkpoint (``prefix.index`` / ``prefix.data-*``, example.py:121-125)
    by name, without TensorFlow (ckpt.read_checkpoint): optimizer slots and non-float entries are ignored; the variables
    of ``parts`` must all be present with the right shapes (check_variables), every tensor's CRC-32C is verified."""
    from . import ckpt
    exp = expected_variable_shapes(parts)
    w = {k: v for k, v in ckpt.read_checkpoint(prefix, required=exp).items()
         if v.dtype == np.float32 and not k.endswith(('/Adam', '/Adam_1', '/Momentum', '/RMSProp', '/RMSProp_1'))}
    if not w:
        raise RuntimeError("no float variables found in checkpoint %r" % prefix)
    check_variables(w, parts)
    load_weights(w, device=device)
    return sorted(w)
