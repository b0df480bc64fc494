"""2-D feature extraction module ``ResNetDS2SPP`` (/root/reference/cnn_wrapper/atvsnet.py:254-292 on the layers of
cnn_wrapper/network.py:142-215 conv / conv_bn, :552-616 bottleneck / res_block, :650-671 image_resize / avg_pool,
:690-697 concat / add) on torch CUDA tensors, NHWC fp32, through the C ABI (csrc/fem2d.cu).

SURVEY.md 8(f) row N1: checked against oracle/fem.py and the reference-graph golden vectors.  Variables are looked up
under the checkpoint names (tests/golden/fem_variables.json).  ``extract_features`` is the image-side entry that feeds
the hot path (model.py:420-425 TVSNet_feature_extraction over all views)."""
import torch

from . import _lib as L
from . import variables as V
from .flags import FLAGS

BN_EPS = 1e-3


def tensor_path():
    """the stride-1 convolutions run on the tcgen05 kernel (fp16 operands, fp32 accumulation) when asked to
    (FLAGS.fem_tensor, opt-in: see flags.py for the accuracy it costs) and the hot path is in fp16."""
    return FLAGS.precision == 'fp16' and getattr(FLAGS, 'fem_tensor', False)


def _packed2d(kernel):
    cache = V.packed_cache()
    key = ('fem2d', kernel.data_ptr(), tuple(kernel.shape))
    if key not in cache:
        k, _, cin, cout = kernel.shape
        buf = torch.empty(L.load().atvs_packed_weight2d_bytes(cin, cout, k), dtype=torch.uint8, device=kernel.device)
        L.call("atvs_pack_conv2d_weights_tc", L.ptr(kernel), cin, cout, k, L.F16, L.ptr(buf), L.stream())
        cache[key] = buf
    return cache[key]


def tc_supported(x, kernel, stride, explicit_pad):
    cin, cout = kernel.shape[2], kernel.shape[3]
    return (stride == 1 and explicit_pad is None and kernel.shape[0] in (1, 3) and (cin == 32 or cin % 64 == 0)
            and cin <= 320 and cout <= 256 and x.shape[1] * x.shape[2] >= 128)


@L.on_input_device
def conv2d_tc(x, kernel, rate=1, bias=None, relu=False, out_dtype=torch.float32, stats=None):
    """stride-1 'SAME' convolution on the tensor cores: x (B,H,W,Cin) fp16 -> (B,H,W,Cout) fp32 | fp16
    = [relu](conv + bias); ``stats`` (2*Cout fp64, zeroed) receives the per-channel moments (conv_bn layers)."""
    B, H, W, cin = x.shape
    k, cout = kernel.shape[0], kernel.shape[-1]
    out = torch.empty((B, H, W, cout), dtype=out_dtype, device=x.device)
    L.call("atvs_conv2d_tc", L.ptr(x), L.F16, L.ptr(_packed2d(kernel)), L.ptr(bias), B, H, W, cin, cout, k, rate, int(relu),
           L.ptr(out), L.F16 if out_dtype == torch.float16 else L.F32, L.ptr(stats), L.stream())
    return out


@L.on_input_device
def to_half(x):
    if x.dtype == torch.float16:
        return x
    out = torch.empty(x.shape, dtype=torch.float16, device=x.device)
    L.call("atvs_cast", L.ptr(x), L.F32, L.ptr(out), L.F16, x.numel(), L.stream())
    return out


def _same_pad(n, k_eff, s):
    out = -(-n // s)
    total = max((out - 1) * s + k_eff - n, 0)
    return total // 2, out


@L.on_input_device
def conv2d(x, kernel, stride=1, rate=1, bias=None, relu=False, padding='SAME', explicit_pad=None):
    """x (B,H,W,Cin) fp32 cuda, kernel [k,k,Cin,Cout].  padding 'SAME' (TF) or 'VALID' after ``explicit_pad`` =
    (begin, end) zero rows/cols on both axes (the bottleneck's tf.pad + VALID, network.py:589-595)."""
    L.require_cuda(x, kernel)
    if tensor_path() and tc_supported(x, kernel, stride, explicit_pad) and padding == 'SAME':
        return conv2d_tc(to_half(x.contiguous()), kernel, rate, bias, relu)
    x = L.f32c(x)
    B, H, W, cin = x.shape
    k, cout = kernel.shape[0], kernel.shape[-1]
    k_eff = (k - 1) * rate + 1
    if explicit_pad is not None:
        pb, pe = explicit_pad
        pt = pl = pb
        Ho = (H + pb + pe - k_eff) // stride + 1
        Wo = (W + pb + pe - k_eff) // stride + 1
    elif padding == 'SAME':
        pt, Ho = _same_pad(H, k_eff, stride)
        pl, Wo = _same_pad(W, k_eff, stride)
    else:
        pt = pl = 0
        Ho, Wo = (H - k_eff) // stride + 1, (W - k_eff) // stride + 1
    out = torch.empty((B, Ho, Wo, cout), dtype=torch.float32, device=x.device)
    L.call("atvs_conv2d_fp32", L.ptr(x), L.ptr(kernel), L.ptr(bias), B, H, W, cin, cout, k, stride, rate, pt, pl, Ho, Wo,
           int(relu), L.ptr(out), L.stream())
    return out


BATCH_VIEWS = True       # extract_features: one batch over the views (fp32 path)

# independent statistic groups along the batch dimension (extract_features runs the towers of all views as ONE batch:
# 5 x the pixels per convolution launch fills the SMs, the batch statistics stay per view as in the reference)
_GROUPS = 1


@L.on_input_device
def batch_norm(x, beta=None, relu=False, stats=None, out_dtype=torch.float32):
    """batch statistics over (B,H,W), biased variance, eps 1e-3, optional ``+ beta``, optional ReLU.  ``stats``: moments
    already accumulated by the producing convolution's epilogue; ``out_dtype`` fp16 feeds a tensor-core convolution.
    With ``_GROUPS`` = G > 1 the batch is G groups of B / G samples, each normalised with its own statistics."""
    x = L.f32c(x)
    C = x.shape[-1]
    count = x.numel() // C
    G = _GROUPS
    if G > 1:
        if stats is not None or x.shape[0] % G:
            raise RuntimeError("batch_norm: grouped statistics need a batch divisible by %d and no precomputed moments" % G)
        out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
        st = torch.zeros((G, 2 * C), dtype=torch.float64, device=x.device)
        bg = x.shape[0] // G
        for g in range(G):
            xs, os_ = x[g * bg:(g + 1) * bg], out[g * bg:(g + 1) * bg]
            L.call("atvs_channel_moments", L.ptr(xs), count // G, C, L.ptr(st[g]), L.stream())
            L.call("atvs_bn2d_apply", L.ptr(xs), L.ptr(st[g]), L.ptr(beta), count // G, C, BN_EPS, int(relu), L.ptr(os_),
                   L.F16 if out_dtype == torch.float16 else L.F32, L.stream())
        return out
    if stats is None:
        stats = torch.zeros(2 * C, dtype=torch.float64, device=x.device)
        L.call("atvs_channel_moments", L.ptr(x), count, C, L.ptr(stats), L.stream())
    out = torch.empty(x.shape, dtype=out_dtype, device=x.device)
    L.call("atvs_bn2d_apply", L.ptr(x), L.ptr(stats), L.ptr(beta), count, C, BN_EPS, int(relu), L.ptr(out),
           L.F16 if out_dtype == torch.float16 else L.F32, L.stream())
    return out


@L.on_input_device
def conv_bn(x, name, stride=1, rate=1, out_dtype=torch.float32):
    """network.py:173-215 on a 4-D tensor: name/conv2d/kernel, BN without affine, ReLU."""
    kernel = V.get_variable(name + '/conv2d/kernel')
    if tensor_path() and tc_supported(x, kernel, stride, None):
        stats = torch.zeros(2 * kernel.shape[-1], dtype=torch.float64, device=x.device)
        raw = conv2d_tc(to_half(x.contiguous()), kernel, rate, stats=stats)        # moments from the fp32 accumulators
        return batch_norm(raw, None, True, stats=stats, out_dtype=out_dtype)
    return batch_norm(conv2d(x, kernel, stride, rate), None, True, out_dtype=out_dtype)


@L.on_input_device
def add(a, b):
    if tuple(a.shape) != tuple(b.shape) or a.dtype != torch.float32 or b.dtype != torch.float32:
        raise ValueError("add: operands must be fp32 tensors of one shape, got %s %s and %s %s"
                         % (tuple(a.shape), a.dtype, tuple(b.shape), b.dtype))
    a, b = a.contiguous(), b.contiguous()
    out = torch.empty_like(a)
    L.call("atvs_add", L.ptr(a), L.ptr(b), L.ptr(out), L.F32, a.numel(), L.stream())
    return out


@L.on_input_device
def bottleneck(x, scope, depth, stride=1, rate=1):
    """network.py:552-603."""
    g = V.get_variable
    depth_in = x.shape[-1]
    if tensor_path() and stride == 1 and (depth_in == 32 or depth_in % 64 == 0) and x.shape[1] * x.shape[2] >= 128:
        # tensor-core bottleneck: the residual stream x stays fp32, everything a convolution reads is fp16
        preact = batch_norm(x, g(scope + '/preact/beta'), True, out_dtype=torch.float16)
        shortcut = x if depth == depth_in else conv2d_tc(preact, g(scope + '/shortcut/weights'), 1,
                                                         g(scope + '/shortcut/biases'))
        r = conv2d_tc(preact, g(scope + '/conv1/weights'), 1, g(scope + '/conv1/biases'), True, torch.float16)
        r = conv2d_tc(r, g(scope + '/conv2/weights'), rate, g(scope + '/conv2/biases'), True, torch.float16)
        r = conv2d_tc(r, g(scope + '/conv3/weights'), 1, g(scope + '/conv3/biases'))
        return add(shortcut, r)
    preact = batch_norm(x, g(scope + '/preact/beta'), True)
    if depth == depth_in:
        shortcut = x if stride == 1 else x[:, ::stride, ::stride, :].contiguous()
    else:
        shortcut = conv2d(preact, g(scope + '/shortcut/weights'), stride, 1, g(scope + '/shortcut/biases'))
    r = conv2d(preact, g(scope + '/conv1/weights'), 1, 1, g(scope + '/conv1/biases'), relu=True)
    if stride == 1:
        r = conv2d(r, g(scope + '/conv2/weights'), 1, rate, g(scope + '/conv2/biases'), relu=True)
    else:
        k_eff = 3 + 2 * (rate - 1)
        beg = (k_eff - 1) // 2
        r = conv2d(r, g(scope + '/conv2/weights'), stride, rate, g(scope + '/conv2/biases'), relu=True,
                   explicit_pad=(beg, k_eff - 1 - beg))
    r = conv2d(r, g(scope + '/conv3/weights'), 1, 1, g(scope + '/conv3/biases'))
    return add(shortcut, r)


@L.on_input_device
def res_block(x, name, depth, num_block, stride=1, rate=1):
    """network.py:605-616."""
    if num_block == 1:
        return bottleneck(x, name, depth, stride, rate)
    out = bottleneck(x, name + '_0', depth, stride, rate)
    for i in range(1, num_block):
        out = bottleneck(out, name + '_%d' % i if i != num_block - 1 else name, depth, 1, rate)
    return out


@L.on_input_device
def avg_pool(x, k, s):
    B, H, W, C = x.shape
    out = torch.empty((B, -(-H // s), -(-W // s), C), dtype=torch.float32, device=x.device)
    L.call("atvs_avg_pool_same", L.ptr(x), B, H, W, C, k, s, L.ptr(out), L.stream())
    return out


@L.on_input_device
def image_resize(x, Ho, Wo):
    B, H, W, C = x.shape
    out = torch.empty((B, Ho, Wo, C), dtype=torch.float32, device=x.device)
    L.call("atvs_resize_bilinear_align", L.ptr(x), B, H, W, C, Ho, Wo, L.ptr(out), L.stream())
    return out


@L.on_input_device
def ResNetDS2SPP(image, return_layers=False):
    """cnn_wrapper/atvsnet.py:254-292: image (B,H,W,3) fp32 cuda -> feature (B,H/4,W/4,32) fp32."""
    L.require_cuda(image)
    layers = {}
    x = conv_bn(L.f32c(image), 'conv0_0', stride=2)
    x = conv_bn(x, 'conv0_1')
    x = layers['conv0_2'] = conv_bn(x, 'conv0_2')
    x = layers['conv0_x'] = res_block(x, 'conv0_x', 32, 3, 1, 1)
    c1 = layers['conv1_x'] = res_block(x, 'conv1_x', 64, 8, 2, 1)
    x = layers['conv2_x'] = res_block(c1, 'conv2_x', 128, 3, 1, 2)
    c3 = layers['conv3_x'] = res_block(x, 'conv3_x', 128, 3, 1, 4)
    h, w = c3.shape[1], c3.shape[2]
    branches = []
    for i, k in enumerate((64, 32, 16, 8)):
        b = image_resize(conv_bn(avg_pool(c3, k, k), 'branch_%d_conv' % i), h, w)
        layers['branch_%d' % i] = b
        branches.append(b)
    cat = torch.cat([c1, c3] + branches, dim=-1).contiguous()
    f0 = layers['fusion0'] = conv_bn(cat, 'fusion0')
    out = layers['fusion1'] = conv2d(f0, V.get_variable('fusion1/kernel'))
    return (out, layers) if return_layers else out


@L.on_input_device
def extract_features(images):
    """model.py:420-425 TVSNet_feature_extraction over all views: images (B,N,H,W,3) -> features (B,N,H/4,W/4,32).
    One tower per VIEW on the (B,H,W,3) slice, as in the reference: batch statistics are taken over the whole batch B
    of that view (B = 1 in example.py), never across views."""
    global _GROUPS
    B, N = images.shape[0], images.shape[1]
    if tensor_path() or N == 1 or not BATCH_VIEWS:
        return torch.stack([ResNetDS2SPP(images[:, n]) for n in range(N)], dim=1)
    # all views as one batch (view-major), statistics per view: the same numbers as one tower per view, with 5 x the
    # pixels per convolution launch (the 1/4-resolution layers leave most SMs idle on one 640x512 image)
    stacked = L.f32c(images).transpose(0, 1).reshape((N * B,) + tuple(images.shape[2:])).contiguous()
    _GROUPS = N
    try:
        feat = ResNetDS2SPP(stacked)
    finally:
        _GROUPS = 1
    return feat.reshape((N, B) + tuple(feat.shape[1:])).transpose(0, 1).contiguous()
