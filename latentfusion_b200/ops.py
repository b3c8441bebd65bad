"""torch.autograd bindings of the lfb200 C ABI.

Every function here enqueues hand-written sm_100a kernels from ``liblfb200.so`` on the current CUDA
stream; none has a PyTorch/CPU fallback (CPU tensors raise).  Feature maps keep the reference's
logical shapes (``[N,C,D,H,W]`` / ``[N,C,H,W]``) but live in channels-last memory, which is what the
kernels index (``[N][D][H][W][C]``).
"""
import ctypes
import math
import weakref

import torch

from . import _lib as L

PRECISION_FP32 = 0      # exact fp32 FFMA path
PRECISION_BF16X3 = 1    # tcgen05, bf16 hi/lo split (3 MMAs), ~2^-16 relative
PRECISION_BF16 = 2      # tcgen05, plain bf16 operands, fp32 accumulate
PRECISION_MIXED = 3     # forward bf16x3 (fp32-grade outputs), backward-data single-pass bf16

import os as _os

_default_precision = int(_os.environ.get('LFB200_PRECISION', PRECISION_FP32))


def set_default_precision(p):
    global _default_precision
    _default_precision = int(p)


def get_default_precision():
    return _default_precision


_active_device = None      # device of the tensors of the op being issued (set by _need_cuda)


def _stream():
    return ctypes.c_void_p(torch.cuda.current_stream(_active_device).cuda_stream)


class KernelTrace:
    """Optional per-call CUDA-event trace of the library entry points (used by bench.py to measure each
    kernel's average launch duration live, on the launching stream).  Off by default: zero overhead."""
    enabled = False
    records = []          # (name, start_event, end_event, algorithmic_bytes, flops)
    launches = 0          # kernels launched through the C ABI since reset (always counted)

    @classmethod
    def reset(cls, enabled=False):
        cls.enabled, cls.records, cls.launches = enabled, [], 0

    @classmethod
    def summary(cls):
        """{name: dict(calls, ms_total, ms_avg, bytes, flops)}; call after a device synchronize."""
        out = {}
        for name, e0, e1, nbytes, flops in cls.records:
            d = out.setdefault(name, dict(calls=0, ms_total=0.0, bytes=0, flops=0))
            d['calls'] += 1
            d['ms_total'] += e0.elapsed_time(e1)
            d['bytes'] += nbytes
            d['flops'] += flops
        for d in out.values():
            d['ms_avg'] = d['ms_total'] / d['calls']
        return out


def _call(name, fn, args, kernels=1, nbytes=0, flops=0):
    """Invoke one C-ABI entry point, optionally bracketed by CUDA events on the current stream.  The library launches
    on the CUDA runtime's current device: when the tensors live elsewhere (model on cuda:1 without set_device), the
    call is issued under a device guard, like a PyTorch op would."""
    if _active_device is not None and _active_device.index != torch.cuda.current_device():
        with torch.cuda.device(_active_device):
            return _call(name, fn, args, kernels, nbytes, flops)
    KernelTrace.launches += kernels
    if KernelTrace.enabled:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        status = fn(*args)
        e1.record()
        KernelTrace.records.append((name, e0, e1, nbytes, flops))
    else:
        status = fn(*args)
    L.check(status, name)


def _p(t):
    return None if t is None else ctypes.c_void_p(t.data_ptr())


def _need_cuda(*tensors):
    """every tensor argument must be on ONE CUDA device; remembers it for the launches that follow"""
    global _active_device
    dev = None
    for t in tensors:
        if t is None:
            continue
        if not t.is_cuda:
            raise RuntimeError("latentfusion_b200: tensors must live on a CUDA device "
                               "(the hot path is sm_100a CUDA only; there is no CPU fallback)")
        if dev is None:
            dev = t.device
        elif t.device != dev:
            raise RuntimeError(f"latentfusion_b200: tensors of one op live on different devices ({dev} and {t.device})")
    if dev is not None:
        _active_device = dev


def _mf(ndim):
    return torch.channels_last_3d if ndim == 5 else torch.channels_last


def to_cl(x):
    """Dense fp32 channels-last view/copy of a [N,C,(D),H,W] tensor (no-op when already so)."""
    if x.dtype != torch.float32:
        x = x.float()
    return x.contiguous(memory_format=_mf(x.dim()))


def empty_cl(shape, device):
    return torch.empty(shape, device=device, dtype=torch.float32, memory_format=_mf(len(shape)))


# ------------------------------------------------------------------------------------------------
# K1 / K2: voxel resamplers
# ------------------------------------------------------------------------------------------------
class _ResampleO2C(torch.autograd.Function):
    """ObjectToCameraTransform (reference modules/geometry.py:669-690)."""

    last_split = None     # split_only: the SplitVol that holds the result (the returned dense tensor is NOT written)

    @staticmethod
    def forward(ctx, vol, cam, split_only=False):
        _need_cuda(vol, cam)
        vol = to_cl(vol)
        cam = cam.detach().float().contiguous()
        B, C, S = vol.shape[0], vol.shape[1], vol.shape[-1]
        N = cam.shape[0]
        if vol.shape[2:] != (S, S, S):
            raise ValueError(f"object volume must be a cube, got {tuple(vol.shape)}")
        if cam.shape[1] != L.CAM_STRIDE:
            raise ValueError("camera block must be [N, LF_CAM_STRIDE]")
        out = empty_cl((N, C, S, S, S), vol.device)
        _ResampleO2C.last_split = None
        if split_only:
            # the volumes go straight into the split-planar layout the consumer's TMA staging reads; `out` only carries
            # the shape and the autograd edge (the caller guarantees its single reader is that convolution)
            sv = SplitVol.empty(N, C, S, S, S, vol.device)
            _call('lf_resample_o2c_fwd', L.lib().lf_resample_o2c_fwd_split,
                  (_p(vol), _p(cam), _p(sv.buf), B, N, C, S, _stream()), kernels=2, nbytes=4 * C * S ** 3 * (B + N))
            _ResampleO2C.last_split = sv
        else:
            _call('lf_resample_o2c_fwd', L.lib().lf_resample_o2c_fwd, (_p(vol), _p(cam), _p(out), B, N, C, S, _stream()),
                  nbytes=4 * C * S ** 3 * (B + N))
        ctx.save_for_backward(vol, cam)
        return out

    @staticmethod
    def backward(ctx, gout):
        vol, cam = ctx.saved_tensors
        _need_cuda(gout, vol)
        gout = to_cl(gout)
        B, C, S = vol.shape[0], vol.shape[1], vol.shape[-1]
        N = cam.shape[0]
        gvol = gcam = None
        if ctx.needs_input_grad[0]:
            gvol = torch.zeros_like(vol)
            _call('lf_resample_o2c_bwd_vol', L.lib().lf_resample_o2c_bwd_vol,
                  (_p(gout), _p(cam), _p(gvol), B, N, C, S, _stream()), nbytes=4 * C * S ** 3 * (B + N))
        if ctx.needs_input_grad[1]:
            ws = torch.empty(L.lib().lf_resample_o2c_bwd_cam_ws(N, S), device=vol.device, dtype=torch.float32)
            # the finishing kernel writes the gradient in the camera block's own layout (zeros where no term lands)
            gcam = torch.empty(N, L.CAM_STRIDE, device=vol.device, dtype=torch.float32)
            _call('lf_resample_o2c_bwd_cam', L.lib().lf_resample_o2c_bwd_cam_block,
                  (_p(gout), _p(vol), _p(cam), _p(gcam), _p(ws), B, N, C, S, _stream()), kernels=2,
                  nbytes=4 * C * S ** 3 * (B + N))
        return gvol, gcam, None


class _ResampleC2O(torch.autograd.Function):
    """CameraToObjectTransform (reference modules/geometry.py:625-657).  As in the reference the
    camera is not differentiated on this direction (its grid is built with an in-place divide)."""

    @staticmethod
    def forward(ctx, vol, cam):
        _need_cuda(vol, cam)
        vol = to_cl(vol)
        cam = cam.detach().float().contiguous()
        V, C, S = vol.shape[0], vol.shape[1], vol.shape[-1]
        if vol.shape[2:] != (S, S, S):
            raise ValueError(f"camera volume must be a cube, got {tuple(vol.shape)}")
        if cam.shape != (V, L.CAM_STRIDE):
            raise ValueError(f"batch dimension of volume ({V}) and camera ({cam.shape[0]}) must match")
        out = empty_cl((V, C, S, S, S), vol.device)
        _call('lf_resample_c2o_fwd', L.lib().lf_resample_c2o_fwd, (_p(vol), _p(cam), _p(out), V, C, S, _stream()),
              nbytes=4 * C * S ** 3 * 2 * V)
        ctx.save_for_backward(cam)
        ctx.shape = (V, C, S)
        return out

    @staticmethod
    def backward(ctx, gout):
        (cam,) = ctx.saved_tensors
        _need_cuda(gout, cam)
        V, C, S = ctx.shape
        gvol = None
        if ctx.needs_input_grad[0]:
            gout = to_cl(gout)
            gvol = torch.zeros((V, C, S, S, S), device=gout.device, dtype=torch.float32).contiguous(
                memory_format=torch.channels_last_3d)
            _call('lf_resample_c2o_bwd_vol', L.lib().lf_resample_c2o_bwd_vol,
                  (_p(gout), _p(cam), _p(gvol), V, C, S, _stream()), nbytes=4 * C * S ** 3 * 2 * V)
        return gvol, None


def resample_o2c(vol, cam_block, split_only=False):
    """split_only: the result is written ONLY in split-planar form (attached as `_lf_split`, which eq_conv's depth-batched
    path stages from); the dense tensor returned is uninitialised.  For callers that know the single reader is such a
    convolution (o2c_split_ok) — the Photographer's first camera block in the pose loop."""
    out = _ResampleO2C.apply(vol, cam_block, bool(split_only))
    if _ResampleO2C.last_split is not None:
        out._lf_split = _ResampleO2C.last_split
        _ResampleO2C.last_split = None
    return out


def o2c_split_ok(channels, size, n_cams, conv):
    """may the object->camera volumes feeding `conv` (an EqualizedConv3d) exist in split-planar form only?  Yes when that
    convolution runs on the depth-batched tcgen05 kernel (which stages the split form and never reads the dense tensor)
    and its weights are frozen (a weight gradient would want the dense input)."""
    if _O2C_SPLIT_OFF or getattr(conv, 'ndim', 0) != 3:
        return False
    w = conv.module.weight
    if w.dim() != 5 or w.shape[-1] != 3 or w.shape[1] != channels:
        return False
    if torch.is_grad_enabled() and (w.requires_grad or (conv.bias is not None and conv.bias.requires_grad)):
        return False
    precision = conv.precision if conv.precision is not None else _default_precision
    if precision not in (1, 2, 3):
        return False
    desc = _desc(KIND_CONV, 3, n_cams, size, size, size, channels, w.shape[0], 3, 1.0, False, 0.0, False,
                 1 if precision == 3 else precision)
    return _dz_ok(desc) and bool(L.lib().lf_resample_o2c_fwd_split_supported(channels, size))


def resample_c2o(vol, cam_block):
    return _ResampleC2O.apply(vol, cam_block)


# ------------------------------------------------------------------------------------------------
# K3/K5/K6: equalised convolution with fused scale/bias/LeakyReLU/PixelNorm
# ------------------------------------------------------------------------------------------------
KIND_CONV, KIND_COLLAPSE, KIND_EXPAND = 0, 1, 2


_PACK_CACHE = {}


def _cache_put(cache, key, value, limit):
    """insert; when the cache is over its limit, drop the entries whose parameter object is dead (never a live
    entry: captured CUDA graphs and saved-for-backward tensors hold raw pointers into live packs)."""
    if len(cache) >= limit:
        for k in [k for k, v in cache.items() if v[0]() is None]:
            del cache[k]
    cache[key] = value


def _pack_weight_cached(weight, kind, depth):
    """_pack_weight memoised per live parameter object and version (weights are frozen in the pose loop, so the
    flip/permute kernels run once, not once per convolution call)."""
    key = (id(weight), weight._version, kind, depth)
    hit = _PACK_CACHE.get(key)
    if hit is not None and hit[0]() is weight:
        return hit[1], hit[2]
    wf, wb = _pack_weight(weight.detach(), kind, depth)
    _cache_put(_PACK_CACHE, key, (weakref.ref(weight), wf, wb), 512)
    return wf, wb


def _pack_weight(weight, kind, depth):
    """[Cout,Cin,k..] (reference layout) -> packed [taps][Cin][Cout] and its bwd-data twin."""
    if kind == KIND_CONV:
        nd = weight.dim() - 2
        sp = tuple(range(2, 2 + nd))
        taps = int(math.prod(weight.shape[2:]))
        fwd = weight.permute(*sp, 1, 0).reshape(taps, weight.shape[1], weight.shape[0])
        bwd = weight.flip(sp).permute(*sp, 0, 1).reshape(taps, weight.shape[0], weight.shape[1])
    elif kind == KIND_COLLAPSE:       # weight [Cout, C*S, 1, 1], channel index c*S + d
        cout = weight.shape[0]
        w3 = weight.reshape(cout, -1, depth)                 # [co][c][d]
        fwd = w3.permute(2, 1, 0)                            # [d][c][co]
        bwd = w3.permute(2, 0, 1)                            # [d][co][c]   (an expand)
    else:                             # weight [C*S, Cin, 1, 1], output index c*S + d
        cin = weight.shape[1]
        w3 = weight.reshape(-1, depth, cin)                  # [c][d][ci]
        fwd = w3.permute(1, 2, 0)                            # [d][ci][c]
        bwd = w3.permute(1, 0, 2)                            # [d][c][ci]   (a collapse)
    return fwd.contiguous().float(), bwd.contiguous().float()


def _unpack_weight_grad(gw, weight_shape, kind, depth):
    """inverse of the forward packing for a gradient [taps][Cin][Cout]."""
    if kind == KIND_CONV:
        cout, cin = weight_shape[:2]
        ks = tuple(weight_shape[2:])
        nd = len(ks)
        g = gw.reshape(*ks, cin, cout)
        return g.permute(nd + 1, nd, *range(nd)).contiguous()
    if kind == KIND_COLLAPSE:
        cout = weight_shape[0]
        return gw.permute(2, 1, 0).reshape(cout, -1, 1, 1).contiguous()       # [co][c][d]
    cin = weight_shape[1]
    return gw.permute(2, 0, 1).reshape(-1, cin, 1, 1).contiguous()            # [c][d][ci]


_bwd_precision_override = None     # dev/experiments: force the precision of every bwd-data convolution
_FUSE_BWD = _os.environ.get('LFB200_FUSE_BWD', '0') == '1'
# K1 writing the split-planar layout itself (lf_resample_o2c_fwd_split) instead of dense fp32 + lf_split_pack: measured
# at config B 182 us against 100 + 100 us (the 8-byte pieces of 8 planes double the kernel's store wavefronts, and its L1
# data pipe was already the co-limiter) -> 352.5 vs 352.8 iters/s, no gain, so it stays opt-in (LFB200_O2C_SPLIT=1)
_O2C_SPLIT_OFF = _os.environ.get('LFB200_O2C_SPLIT', '0') != '1'
_TC_PACK_CACHE = {}


def _cache_put(cache, key, value, limit):
    """insert; when the cache is over its limit, drop the entries whose parameter object is dead (never a live
    entry: captured CUDA graphs and saved-for-backward tensors hold raw pointers into live packs)."""
    if len(cache) >= limit:
        for k in [k for k, v in cache.items() if v[0]() is None]:
            del cache[k]
    cache[key] = value


def _tc_pack(wf, key):
    """fp32 packed weights [taps][Cin][Cout] -> bf16 hi|lo UMMA layout for the tcgen05 kernel (cached per
    parameter version; the pack itself is one small kernel)."""
    hit = _TC_PACK_CACHE.get(key[1:])
    if hit is not None and hit[0]() is key[0]:          # same live tensor object, same version
        return hit[1]
    taps, cin, cout = wf.shape
    nbytes = L.lib().lf_conv_tc_weight_bytes(taps, cin, cout)
    out = torch.empty(nbytes // 2, device=wf.device, dtype=torch.int16)
    _call('lf_conv_tc_pack_weights', L.lib().lf_conv_tc_pack_weights, (_p(wf), _p(out), taps, cin, cout, _stream()))
    _cache_put(_TC_PACK_CACHE, key[1:], (weakref.ref(key[0]), out), 256)
    return out


def _tc_passes(desc):
    """kernel launches the library makes for this convolution on the tcgen05 path (1 bf16, 2|3 bf16x3)."""
    return max(1, int(L.lib().lf_conv_tc_passes(ctypes.byref(desc))))


def _tc_ok(desc):
    return desc.precision != 0 and bool(L.lib().lf_conv_tc_supported(ctypes.byref(desc)))


def _desc(kind, nd, n, d, h, w, cin, cout, k, scale, act, slope, norm, precision):
    ndim = {KIND_CONV: nd, KIND_COLLAPSE: 1, KIND_EXPAND: -1}[kind]
    return L.ConvDesc(ndim, n, d, h, w, cin, cout, k, scale, int(act), slope, int(norm), int(precision))


def _conv_name(kind, nd, k, what):
    tag = {KIND_CONV: f'conv{nd}d_k{k}', KIND_COLLAPSE: 'collapse', KIND_EXPAND: 'expand'}[kind]
    return f'lf_conv_{what}[{tag}]'


# ------------------------------------------------------------------------------------------------
# depth-batched tcgen05 3x3x3 convolution on split-planar activations (csrc/conv3d_dz.cu)
# ------------------------------------------------------------------------------------------------
class SplitVol:
    """A feature volume in the library's internal split-planar layout ([hi|lo][N][D][C_pad/8][H+2][W+2][8] bf16,
    zero halo): what the depth-batched convolution stages with bulk TMA copies.  `buf` is an int16 device tensor."""
    __slots__ = ('buf', 'n', 'c', 'd', 'h', 'w')

    def __init__(self, buf, n, c, d, h, w):
        self.buf, self.n, self.c, self.d, self.h, self.w = buf, n, c, d, h, w

    @staticmethod
    def empty(n, c, d, h, w, device):
        nbytes = L.lib().lf_split_bytes(n, d, h, w, c)
        return SplitVol(torch.empty(nbytes // 2, device=device, dtype=torch.int16), n, c, d, h, w)

    def to_dense(self):
        """fp32 [N,C,D,H,W] (tests / debugging): hi + lo of the interior."""
        cp = (self.c + 15) // 16 * 16
        v = self.buf.view(torch.bfloat16).view(2, self.n, self.d, cp // 8, self.h + 2, self.w + 2, 8).float()
        v = (v[0] + v[1])[:, :, :, 1:-1, 1:-1, :]                       # [n, d, kc, h, w, 8]
        return v.permute(0, 2, 5, 1, 3, 4).reshape(self.n, cp, self.d, self.h, self.w)[:, :self.c]


def split_pack(x):
    """dense fp32 [N,C,D,H,W] (any memory format) -> SplitVol."""
    _need_cuda(x)
    x = to_cl(x)
    n, c, d, h, w = x.shape
    out = SplitVol.empty(n, c, d, h, w, x.device)
    _call('lf_split_pack', L.lib().lf_split_pack, (_p(x), _p(out.buf), n, d, h, w, c, _stream()),
          nbytes=4 * x.numel() + out.buf.numel() * 2)
    return out


def _dz_pack(wf, key):
    """[27][Cin][Cout] fp32 -> the depth-batched kernel's bf16 hi|lo weight layout (cached like _tc_pack)."""
    hit = _TC_PACK_CACHE.get(key[1:])
    if hit is not None and hit[0]() is key[0]:
        return hit[1]
    taps, cin, cout = wf.shape
    out = torch.empty(L.lib().lf_conv3d_dz_weight_bytes(cin, cout) // 2, device=wf.device, dtype=torch.int16)
    _call('lf_conv3d_dz_pack_weights', L.lib().lf_conv3d_dz_pack_weights, (_p(wf), _p(out), cin, cout, _stream()))
    _cache_put(_TC_PACK_CACHE, key[1:], (weakref.ref(key[0]), out), 256)
    return out


def _ws_pack(wf, key):
    """[27][Cin][Cout] fp32 -> the weight-streaming kernel's tile order (cached per parameter version)"""
    hit = _TC_PACK_CACHE.get(key[1:])
    if hit is not None and hit[0]() is key[0]:
        return hit[1]
    taps, cin, cout = wf.shape
    out = torch.empty(L.lib().lf_conv3d_ws_weight_bytes(taps, cin, cout) // 2, device=wf.device, dtype=torch.int16)
    _call('lf_conv3d_ws_pack_weights', L.lib().lf_conv3d_ws_pack_weights, (_p(wf), _p(out), taps, cin, cout, _stream()))
    _cache_put(_TC_PACK_CACHE, key[1:], (weakref.ref(key[0]), out), 256)
    return out


def _ct_pack(wf, key):
    """collapse weights [depth][Cin][Cout] fp32 -> the tensor-core collapse kernel's per-plane tiles (cached)"""
    hit = _TC_PACK_CACHE.get(key[1:])
    if hit is not None and hit[0]() is key[0]:
        return hit[1]
    depth, cin, cout = wf.shape
    out = torch.empty(L.lib().lf_collapse_tc_weight_bytes(depth, cin, cout) // 2, device=wf.device, dtype=torch.int16)
    _call('lf_collapse_tc_pack_weights', L.lib().lf_collapse_tc_pack_weights, (_p(wf), _p(out), depth, cin, cout, _stream()))
    _cache_put(_TC_PACK_CACHE, key[1:], (weakref.ref(key[0]), out), 256)
    return out


def _ex_ok(desc):
    return desc.precision in (1, 2) and bool(L.lib().lf_expand_tc_supported(ctypes.byref(desc)))


def _ex_pack(wf, key):
    """collapse weights [depth][Cin][Cout] fp32 -> the fused collapse-backward kernel's tile order (cached)"""
    hit = _TC_PACK_CACHE.get(key[1:])
    if hit is not None and hit[0]() is key[0]:
        return hit[1]
    depth, cin, cout = wf.shape
    out = torch.empty(L.lib().lf_expand_tc_weight_bytes(depth, cin, cout) // 2, device=wf.device, dtype=torch.int16)
    _call('lf_expand_tc_pack_weights', L.lib().lf_expand_tc_pack_weights, (_p(wf), _p(out), depth, cin, cout, _stream()))
    _cache_put(_TC_PACK_CACHE, key[1:], (weakref.ref(key[0]), out), 256)
    return out


def _ws_ok(desc):
    return desc.precision in (1, 2) and bool(L.lib().lf_conv3d_ws_supported(ctypes.byref(desc)))


def conv3d_ws(xs, wpk, bias, desc, name='lf_conv3d_ws'):
    """wide 3x3x3 (or, with a one-plane volume and desc.ndim == 2, 3x3) layer with streamed weights:
    SplitVol -> (dense fp32 channels-last [N,Cout,D,H,W], rnorm | None)"""
    lib = L.lib()
    dev = xs.buf.device
    y = empty_cl((xs.n, desc.cout, xs.d, xs.h, xs.w), dev)
    positions = xs.n * xs.d * xs.h * xs.w
    rnorm = torch.empty(positions, device=dev, dtype=torch.float32) if desc.norm else None
    scratch = torch.empty(lib.lf_conv3d_ws_scratch(ctypes.byref(desc)), device=dev, dtype=torch.float32) if desc.norm else None
    _call(name, lib.lf_conv3d_ws,
          (ctypes.byref(desc), _p(xs.buf), _p(wpk), _p(bias), _p(y), _p(rnorm), _p(scratch), _stream()),
          kernels=2 if desc.norm else 1, nbytes=xs.buf.numel() * 2 + 4 * y.numel(),
          flops=2 * positions * (27 if desc.ndim == 3 else 9) * xs.c * desc.cout)
    return y, rnorm


_GRAD_SPLIT = [None]       # (data_ptr, numel, SplitVol) of the most recent fused bwd-data result: its single consumer is
#                            the very next backward node (the producer layer's), which takes it instead of re-packing


def _put_grad_split(g, gs):
    _GRAD_SPLIT[0] = (g.data_ptr(), g.numel(), gs)


def _take_grad_split(g):
    rec, _GRAD_SPLIT[0] = _GRAD_SPLIT[0], None
    if rec is not None and rec[0] == g.data_ptr() and rec[1] == g.numel():
        return rec[2]
    return None


def _dz_shape(x, weight, kind, precision):
    """cheap test: would eq_conv run this convolution on the depth-batched kernel?"""
    if kind != KIND_CONV or x.dim() != 5 or weight.dim() != 5 or weight.shape[-1] != 3 or precision not in (1, 2, 3):
        return False
    n, cin, d, h, w = x.shape
    desc = _desc(KIND_CONV, 3, n, d, h, w, cin, weight.shape[0], 3, 1.0, False, 0.0, False, 1 if precision == 3 else precision)
    return _dz_ok(desc)


def _dz_ok(desc):
    return desc.precision in (1, 2) and bool(L.lib().lf_conv3d_dz_supported(ctypes.byref(desc)))


def conv3d_dz(xs, wpk, bias, cout, scale, act, slope, norm, precision, want_dense=True, want_split=False,
              name='lf_conv3d_dz'):
    """one launch of the depth-batched kernel: SplitVol -> (dense fp32 channels-last | None, SplitVol | None, rnorm | None)"""
    desc = _desc(KIND_CONV, 3, xs.n, xs.d, xs.h, xs.w, xs.c, cout, 3, scale, act, slope, norm, precision)
    dev = xs.buf.device
    y = empty_cl((xs.n, cout, xs.d, xs.h, xs.w), dev) if want_dense else None
    ys = SplitVol.empty(xs.n, cout, xs.d, xs.h, xs.w, dev) if want_split else None
    rnorm = torch.empty(xs.n * xs.d * xs.h * xs.w, device=dev, dtype=torch.float32) if norm else None
    positions = xs.n * xs.d * xs.h * xs.w
    _call(name, L.lib().lf_conv3d_dz,
          (ctypes.byref(desc), _p(xs.buf), _p(wpk), _p(bias), _p(y), _p(None if ys is None else ys.buf), _p(rnorm), _stream()),
          nbytes=xs.buf.numel() * 2 + (4 * y.numel() if y is not None else 0) + (ys.buf.numel() * 2 if ys is not None else 0),
          flops=2 * positions * 27 * xs.c * cout)
    return y, ys, rnorm


def conv3d_dw(xs, dus, precision, scale=1.0, ndim=3):
    """weight / bias gradient of a 3x3x3 (ndim 3) or 3x3 (ndim 2: one plane per image) convolution from the
    split-planar twins of its input and of d(loss)/d(pre-activation output):
    -> (grad_w_packed [27 | 9][Cin][Cout], grad_bias [1][Cout]).  lf_conv3d_dw"""
    lib = L.lib()
    desc = _desc(KIND_CONV, ndim, xs.n, xs.d, xs.h, xs.w, xs.c, dus.c, 3, scale, 0, 0.0, 0, precision)
    if not lib.lf_conv3d_dw_supported(ctypes.byref(desc)):
        raise ValueError(f"conv3d_dw: unsupported shape (Cin {xs.c}, Cout {dus.c}, precision {precision})")
    dev = xs.buf.device
    gwp = torch.empty(27 if ndim == 3 else 9, xs.c, dus.c, device=dev, dtype=torch.float32)
    gbp = torch.empty(1, dus.c, device=dev, dtype=torch.float32)
    ws = torch.empty(lib.lf_conv3d_dw_ws(ctypes.byref(desc)), device=dev, dtype=torch.float32)
    _call('lf_conv3d_dw', lib.lf_conv3d_dw,
          (ctypes.byref(desc), _p(xs.buf), _p(dus.buf), _p(ws), _p(gwp), _p(gbp), _stream()), kernels=4,
          nbytes=2 * (xs.buf.numel() + dus.buf.numel()), flops=2 * xs.n * xs.d * xs.h * xs.w * gwp.shape[0] * xs.c * dus.c)
    return gwp, gbp


class _ActRec:
    """What the backward of a fused conv+LeakyReLU+PixelNorm layer needs (its output and norms).  When the ONLY
    consumer of that output is another lfb200 convolution (Block: conv1 -> conv2; Photographer: camera block ->
    depth collapse), the consumer's bwd-data kernel applies this layer's activation/norm backward in its epilogue
    (lf_conv_bwd_data_epi) and sets `pre_applied`, and this layer's own backward then skips lf_actnorm_bwd."""
    __slots__ = ('shape', 'rnorm', 'act', 'slope', 'norm', 'pre_applied', 'train')

    # (holds the norms but NOT the output tensor: the consumer has that tensor saved as its own input, and a
    # reference from here would make an output <-> record cycle that only the garbage collector could free)
    def __init__(self, shape, rnorm, act, slope, norm):
        self.shape, self.rnorm, self.act, self.slope, self.norm, self.pre_applied = shape, rnorm, act, slope, norm, False
        self.train = False      # the layer's weights take gradients (a consumer that fuses this layer's backward then also writes dense du)


def mark_single_consumer(t):
    """Declare that the very next lfb200 convolution is the only consumer of `t` (see _ActRec)."""
    t._lf_single_use = True
    return t


# Measured on B200 (config B): the fused-epilogue bwd-data is SLOWER than bwd-data + the vectorised lf_actnorm_bwd
# (3x3x3 conv 1.02 ms vs 0.75 + 0.15; collapse 0.32 vs 0.15 + 0.15): the 128 epilogue threads each re-read a 128-byte
# row of y (32 lines per load instruction) and the epilogue becomes the critical stage.  Opt-in (LFB200_FUSE_EPI=1)
# until the row is staged through shared memory.
_FUSE_EPI = _os.environ.get('LFB200_FUSE_EPI', '0') == '1'
_EX_OFF = _os.environ.get('LFB200_EX_OFF', '0') == '1'      # A/B: depth-collapse backward on the FFMA expand kernel + lf_actnorm_bwd_split
_WS_2D = _os.environ.get('LFB200_WS_2D', '0') == '1'       # A/B: 2-D 3x3 layers on the weight-streaming kernel even when the per-tap one fits
_DW_FFMA = _os.environ.get('LFB200_DW_FFMA', '0') == '1'     # A/B: weight gradients on the exact FFMA kernel


class _EqConv(torch.autograd.Function):
    """y = PixelNorm(LeakyReLU(conv(x, W) * he + b)) in one kernel.
    Reference: modules/equalized.py:57-64 + blocks.py:152-158 + modules/__init__.py:14-15."""
    last_rec = None        # _ActRec of the most recent forward, picked up by eq_conv() to tag the returned tensor
    last_split = None      # split-planar twin of the most recent forward's output (when asked for), tagged likewise
    last_in_split = None   # split-planar twin of the most recent forward's INPUT when it had to be packed here

    @staticmethod
    def forward(ctx, x, weight, bias, kind, depth, act, slope, norm, precision, fan_in=None, rec_in=None,
                x_split=None, emit_split=False):
        _need_cuda(x, weight, bias)
        x = to_cl(x)
        dev = x.device
        if kind == KIND_CONV:
            nd = x.dim() - 2
            n, cin = x.shape[0], x.shape[1]
            d = x.shape[2] if nd == 3 else 1
            h, w = x.shape[-2], x.shape[-1]
            cout, k = weight.shape[0], weight.shape[-1]
            if weight.shape[1] != cin:
                raise ValueError(f"conv: input has {cin} channels, weight expects {weight.shape[1]}")
            out_shape = (n, cout, d, h, w) if nd == 3 else (n, cout, h, w)
            gcin, gcout, positions = cin, cout, n * d * h * w
        elif kind == KIND_COLLAPSE:
            nd = 3
            n, cin, d, h, w = x.shape
            if d != depth or weight.shape[1] != cin * d:
                raise ValueError("collapse: weight does not match [C*S] input channels")
            cout, k = weight.shape[0], d
            out_shape = (n, cout, h, w)
            gcin, gcout, positions = cin, cout, n * h * w
        else:
            nd = 2
            n, cin, h, w = x.shape
            d = depth
            cout_total = weight.shape[0]
            if cout_total % d != 0 or weight.shape[1] != cin:
                raise ValueError("expand: weight does not match")
            cout, k = cout_total // d, 1
            out_shape = (n, cout, d, h, w)
            gcin, gcout, positions = cin, cout, n * h * w
        if fan_in is None:             # a channel-group slice of a wider layer passes the full layer's fan-in
            fan_in = int(math.prod(weight.shape[1:]))
        scale = math.sqrt(2.0 / fan_in)
        wf, wb = _pack_weight_cached(weight, kind, depth)
        if bias is None:
            bpk = None
        elif kind == KIND_EXPAND:
            bpk = bias.detach().float().reshape(cout, d).t().contiguous()
        else:
            bpk = bias.detach().float().contiguous()
        desc = _desc(kind, nd, n, d, h, w, gcin, gcout, k, scale, act, slope, norm,
                     PRECISION_BF16X3 if precision == PRECISION_MIXED else precision)
        use_dz = kind == KIND_CONV and nd == 3 and k == 3 and _dz_ok(desc)
        # wide layers: 3-D ones the depth-batched kernel cannot hold, 2-D ones the per-tap kernel cannot hold
        use_ws = ((not use_dz) and kind == KIND_CONV and k == 3 and (nd == 3 or _WS_2D or not _tc_ok(desc)) and _ws_ok(desc))
        y = None if (use_dz or use_ws) else empty_cl(out_shape, dev)
        rnorm = torch.empty(positions, device=dev, dtype=torch.float32) if (norm and not (use_dz or use_ws)) else None
        taps = wf.shape[0]
        wkey = (weight, id(weight), weight._version, kind)
        _EqConv.last_split = None
        ctx.xs = None
        if kind == KIND_COLLAPSE and rec_in is not None:
            ctx.xs = x_split                                  # the producer's output twin, for the fused backward
        if use_dz:
            # depth-batched tcgen05 kernel on split-planar activations (one launch for bf16x3); the producer may have
            # left the split-planar form of x next to it (x_split), otherwise it is packed here
            xs = x_split if x_split is not None else split_pack(x)
            _EqConv.last_in_split = xs if x_split is None else None
            ctx.xs = xs if rec_in is not None else None      # the producer layer's output, for the fused backward epilogue
            y, ys, rnorm = conv3d_dz(xs, _dz_pack(wf, wkey + ('dzf',)), bpk, gcout, scale, act, slope, norm, desc.precision,
                                     want_dense=True, want_split=emit_split, name=_conv_name(kind, nd, k, 'fwd'))
            _EqConv.last_split = ys
        elif (kind == KIND_COLLAPSE and x_split is not None and not _EX_OFF and desc.precision in (1, 2)
              and L.lib().lf_collapse_tc_supported(ctypes.byref(desc))):
            # the producer left the split-planar twin of the volume: HBM-bound tensor-core collapse (csrc/collapse_tc.cu)
            _call(_conv_name(kind, nd, k, 'fwd'), L.lib().lf_collapse_tc,
                  (ctypes.byref(desc), _p(x_split.buf), _p(_ct_pack(wf, wkey + ('ct',))), _p(bpk), _p(y), _p(rnorm), _stream()),
                  nbytes=2 * x_split.buf.numel() + 4 * y.numel(), flops=2 * positions * taps * gcin * gcout)
        elif use_ws:
            xs = x_split if x_split is not None else split_pack(x if nd == 3 else x.unsqueeze(2))
            y, rnorm = conv3d_ws(xs, _ws_pack(wf, wkey + ('wsf',)), bpk, desc, name=_conv_name(kind, nd, k, 'fwd'))
            if nd == 2:
                y = y.squeeze(2)
        else:
            if _tc_ok(desc):
                wf_arg = _tc_pack(wf, wkey + ('f',))
            else:                      # shapes the tensor-core kernel does not cover run on the exact fp32 path
                desc.precision = 0
                wf_arg = wf
            _call(_conv_name(kind, nd, k, 'fwd'), L.lib().lf_conv_fwd,
                  (ctypes.byref(desc), _p(x), _p(wf_arg), _p(bpk), _p(y), _p(rnorm), _stream()),
                  kernels=(2 if (norm and (kind == KIND_EXPAND or gcout > 64)) else 1) if desc.precision != 1 else _tc_passes(desc),
                  nbytes=4 * (x.numel() + y.numel()), flops=2 * positions * taps * gcin * gcout)
        ctx.save_for_backward(x, y, rnorm, wb)
        ctx.wkey = wkey
        ctx.rec_in = rec_in
        ctx.rec_out = _ActRec(tuple(y.shape), rnorm, act, slope, norm) if ((act or norm) and kind != KIND_EXPAND) else None
        if ctx.rec_out is not None:
            ctx.rec_out.train = bool(weight.requires_grad)
        _EqConv.last_rec = ctx.rec_out
        ctx.cfg = (kind, depth, act, slope, norm, precision, nd, n, d, h, w, gcin, gcout, k, scale,
                   tuple(weight.shape), bias is not None)
        return y

    @staticmethod
    def backward(ctx, gy):
        x, y, rnorm, wb = ctx.saved_tensors
        _need_cuda(gy, x)
        (kind, depth, act, slope, norm, precision, nd, n, d, h, w, cin, cout, k, scale, wshape, has_bias) = ctx.cfg
        gy = to_cl(gy)
        lib = L.lib()
        if precision == PRECISION_MIXED:
            precision = PRECISION_BF16
        if _bwd_precision_override is not None:
            precision = _bwd_precision_override
        need_w = ctx.needs_input_grad[1] or (has_bias and ctx.needs_input_grad[2])
        gx = gw = gb = None
        du = du_split = None
        bkind = {KIND_CONV: KIND_CONV, KIND_COLLAPSE: KIND_EXPAND, KIND_EXPAND: KIND_COLLAPSE}[kind]
        bnd = {KIND_CONV: nd, KIND_COLLAPSE: 2, KIND_EXPAND: 3}[kind]
        bdesc = _desc(bkind, bnd, n, d, h, w, cout, cin, k, scale, 0, 0.0, 0, precision)
        bflops = 2 * (n * h * w * (d if kind == KIND_CONV else 1)) * wb.shape[0] * cin * cout
        fused_done = False
        rec_out, rec_in = ctx.rec_out, ctx.rec_in
        pre_applied = rec_out is not None and rec_out.pre_applied
        if pre_applied:                   # the consumer's bwd-data epilogue already produced du for this layer
            rec_out.pre_applied = False
        epi = (rec_in is not None and ctx.needs_input_grad[0] and rec_in.shape == tuple(x.shape)
               and bool(lib.lf_conv_bwd_data_epi_supported(ctypes.byref(bdesc))))
        # Measured on B200 (config B 3x3x3): the fused staging makes the producers the bottleneck (0.57 ms) while
        # the vectorised lf_actnorm_bwd (0.13 ms) + plain conv (0.32 ms) is faster, so fusion is opt-in
        # (LFB200_FUSE_BWD=1) until the producer stage is widened.
        if (_FUSE_BWD and not pre_applied and not epi and ctx.needs_input_grad[0] and (act or norm) and not need_w and kind == KIND_CONV and precision == PRECISION_BF16
                and _tc_ok(bdesc) and cout in (16, 32, 64, 128)):
            # pose-loop case: PixelNorm/LeakyReLU backward fused into the tcgen05 kernel's operand staging
            gx = torch.empty_like(x)
            wb_arg = _tc_pack(wb, ctx.wkey + ('b',))
            _call(_conv_name(kind, nd, k, 'bwd_data_fused'), lib.lf_conv_bwd_data_fused,
                  (ctypes.byref(bdesc), _p(gy), _p(y), _p(rnorm), int(act), slope, int(norm), _p(wb_arg), _p(gx),
                   _stream()), kernels=3 if precision == 1 else 1,
                  nbytes=4 * (2 * gy.numel() + gx.numel()), flops=bflops)
            fused_done = True
        wdesc = _desc(kind, nd, n, d, h, w, cin, cout, k, scale, 0, 0.0, 0, 0)
        if need_w and kind == KIND_CONV and nd in (2, 3) and k == 3 and not _DW_FFMA:
            wdesc.precision = {1: 1, 2: 2, 3: 1}.get(precision, 0)
            if not (wdesc.precision and lib.lf_conv3d_dw_supported(ctypes.byref(wdesc))):
                wdesc.precision = 0
        use_dw = wdesc.precision != 0          # weight gradient on the tensor cores, from the split-planar twins
        use_dz_b = ctx.needs_input_grad[0] and kind == KIND_CONV and nd == 3 and k == 3 and _dz_ok(bdesc)
        if use_dz_b and not fused_done:
            # ---- depth-batched path: split-planar du straight out of the activation backward, and (when the producer
            # of x is a Block conv whose only consumer this is) that producer's activation backward in the epilogue
            if (act or norm) and not pre_applied:
                du_split = SplitVol.empty(n, cout, d, h, w, x.device)
                if cout in (16, 32):
                    du = torch.empty_like(gy) if (need_w and not use_dw) else None
                    _call('lf_actnorm_bwd', lib.lf_actnorm_bwd_split,
                          (_p(gy), _p(y), _p(rnorm), _p(du), _p(du_split.buf), n, d, h, w, cout, int(act), slope, int(norm),
                           _stream()), nbytes=4 * 2 * gy.numel() + 2 * du_split.buf.numel())
                else:
                    du = torch.empty_like(gy)
                    _call('lf_actnorm_bwd', lib.lf_actnorm_bwd, (_p(gy), _p(y), _p(rnorm), _p(du), n * d * h * w, 1, 1, cout,
                                                                int(act), slope, int(norm), _stream()), nbytes=4 * 3 * gy.numel())
                    du_split = split_pack(du)
            else:
                du = gy
                du_split = _take_grad_split(gy) or split_pack(gy)
            wpk_b = _dz_pack(wb, ctx.wkey + ('dzb',))
            if rec_in is not None and ctx.xs is not None and rec_in.shape == tuple(x.shape):
                gx = empty_cl(tuple(x.shape), x.device)
                gxs = SplitVol.empty(n, cin, d, h, w, x.device)
                _call(_conv_name(kind, nd, k, 'bwd_data'), lib.lf_conv3d_dz_bwd_epi,
                      (ctypes.byref(bdesc), _p(du_split.buf), _p(wpk_b), _p(ctx.xs.buf), _p(rec_in.rnorm), int(rec_in.act),
                       float(rec_in.slope), int(rec_in.norm), _p(gx), _p(gxs.buf), _stream()),
                      nbytes=2 * du_split.buf.numel() + 2 * ctx.xs.buf.numel() + 4 * gx.numel() + 2 * gxs.buf.numel(), flops=bflops)
                rec_in.pre_applied = True
                _put_grad_split(gx, gxs)
            else:
                gx, _, _ = conv3d_dz(du_split, wpk_b, None, cin, scale, False, 0.0, False, bdesc.precision,
                                     name=_conv_name(kind, nd, k, 'bwd_data'))
            fused_done = True
        if not fused_done:
            if (act or norm) and not pre_applied:
                du = torch.empty_like(gy)
                if kind == KIND_EXPAND:
                    outer, gd, inner = n, d, h * w
                elif kind == KIND_COLLAPSE:
                    outer, gd, inner = n * h * w, 1, 1
                else:
                    outer, gd, inner = n * d * h * w, 1, 1
                _call('lf_actnorm_bwd', lib.lf_actnorm_bwd, (_p(gy), _p(y), _p(rnorm), _p(du), outer, gd, inner, cout,
                                                            int(act), slope, int(norm), _stream()),
                      nbytes=4 * 3 * gy.numel())
            else:
                du = gy
            use_ex = (kind == KIND_COLLAPSE and rec_in is not None and ctx.xs is not None and ctx.needs_input_grad[0]
                      and rec_in.shape == tuple(x.shape) and not _EX_OFF)
            if use_ex:
                fdesc = _desc(KIND_COLLAPSE, 3, n, d, h, w, cin, cout, d, scale, 0, 0.0, 0, 1 if precision == 3 else precision)
                use_ex = _ex_ok(fdesc)
            if use_ex:
                # tensor-core depth expand + the producer layer's PixelNorm/LeakyReLU backward, straight to split-planar du
                wf_c, _ = _pack_weight_cached(ctx.wkey[0], kind, depth)
                du2s = split_pack(du.unsqueeze(2))
                gx = torch.empty_like(x)                      # dense only when the producer's weights train
                gxs = SplitVol.empty(n, cin, d, h, w, x.device)
                _call(_conv_name(kind, nd, k, 'bwd_data'), lib.lf_expand_tc_bwd_epi,
                      (ctypes.byref(fdesc), _p(du2s.buf), _p(_ex_pack(wf_c, ctx.wkey + ('ex',))), _p(ctx.xs.buf), _p(rec_in.rnorm),
                       int(rec_in.act), float(rec_in.slope), int(rec_in.norm), _p(gxs.buf), _p(gx if rec_in.train else None),
                       _stream()), nbytes=2 * (ctx.xs.buf.numel() + gxs.buf.numel()), flops=bflops)
                rec_in.pre_applied = True
                _put_grad_split(gx, gxs)
            elif epi:
                # bwd-data + the producer layer's PixelNorm/LeakyReLU backward in one kernel: returns du of that layer
                gx = torch.empty_like(x)
                w_arg = wb if bkind == KIND_EXPAND else _tc_pack(wb, ctx.wkey + ('b',))
                _call(_conv_name(kind, nd, k, 'bwd_data_epi'), lib.lf_conv_bwd_data_epi,
                      (ctypes.byref(bdesc), _p(du), _p(w_arg), _p(x), _p(rec_in.rnorm), int(rec_in.act),
                       float(rec_in.slope), int(rec_in.norm), _p(gx), _stream()),
                      kernels=1 if bkind == KIND_EXPAND else _tc_passes(bdesc),
                      nbytes=4 * (du.numel() + 2 * gx.numel()), flops=bflops)
                rec_in.pre_applied = True
            elif (ctx.needs_input_grad[0] and kind == KIND_CONV and k == 3 and (nd == 3 or _WS_2D or not _tc_ok(bdesc))
                  and _ws_ok(bdesc)):
                # wide layer: bwd-data = the weight-streaming kernel on the flipped / transposed weights
                gx, _ = conv3d_ws(split_pack(du if nd == 3 else du.unsqueeze(2)), _ws_pack(wb, ctx.wkey + ('wsb',)), None,
                                  bdesc, name=_conv_name(kind, nd, k, 'bwd_data'))
                if nd == 2:
                    gx = gx.squeeze(2)
            elif ctx.needs_input_grad[0]:
                gx = torch.empty_like(x)
                # bwd-data = the same implicit GEMM with flipped/transposed weights, no epilogue
                if _tc_ok(bdesc):
                    wb_arg = _tc_pack(wb, ctx.wkey + ('b',))
                else:
                    bdesc.precision = 0
                    wb_arg = wb
                _call(_conv_name(kind, nd, k, 'bwd_data'), lib.lf_conv_fwd,
                      (ctypes.byref(bdesc), _p(du), _p(wb_arg), None, _p(gx), None, _stream()),
                      kernels=_tc_passes(bdesc) if bdesc.precision == 1 else 1,
                      nbytes=4 * (du.numel() + gx.numel()), flops=bflops)
        if ctx.needs_input_grad[1] or (has_bias and ctx.needs_input_grad[2]):
            taps = wb.shape[0]
            if use_dw:
                # tensor-core weight gradient straight from the split-planar twins of x and du (csrc/conv3d_dw.cu)
                as5 = (lambda t: t) if nd == 3 else (lambda t: t.unsqueeze(2))       # a 2-D map is a one-plane volume
                gwp, gbp = conv3d_dw(ctx.xs if ctx.xs is not None else split_pack(as5(x)),
                                     du_split if du_split is not None else split_pack(as5(du)), wdesc.precision, scale, nd)
            else:
                wdesc.precision = 0
                if du is None:
                    du = du_split.to_dense()
                gwp = torch.zeros(taps, cin, cout, device=x.device, dtype=torch.float32)
                gbp = torch.zeros(d if kind == KIND_EXPAND else 1, cout, device=x.device, dtype=torch.float32)
                _call('lf_conv_bwd_weight', lib.lf_conv_bwd_weight,
                      (ctypes.byref(wdesc), _p(x), _p(du), _p(gwp), _p(gbp), _stream()))
            if ctx.needs_input_grad[1]:
                gw = _unpack_weight_grad(gwp, wshape, kind, depth)
            if has_bias and ctx.needs_input_grad[2]:
                gb = gbp.t().reshape(-1) if kind == KIND_EXPAND else gbp.reshape(-1)
        return gx, gw, gb, None, None, None, None, None, None, None, None, None, None


def _ex_shape(x, weight, kind, depth, precision):
    """would the backward of this depth collapse run on the fused tcgen05 kernel (needs the producer's split-planar twin)?"""
    if kind != KIND_COLLAPSE or _EX_OFF or x.dim() != 5 or precision not in (1, 2, 3) or getattr(x, '_lf_split', None) is None:
        return False
    n, cin, d, h, w = x.shape
    return _ex_ok(_desc(KIND_COLLAPSE, 3, n, d, h, w, cin, weight.shape[0], d, 1.0, False, 0.0, False, 1 if precision == 3 else precision))


def eq_conv(x, weight, bias, act=False, slope=0.2, norm=False, kind=KIND_CONV, depth=0, precision=None, fan_in=None,
            emit_split=False):
    """emit_split: also leave the split-planar twin of the output on the returned tensor (`_lf_split`), for a following
    3x3x3 convolution to stage with TMA instead of re-packing (the epilogue writes it for free: the kernel is
    tensor-bound)."""
    if precision is None:
        precision = _default_precision
    rec_in = None
    if getattr(x, '_lf_single_use', False) and torch.is_grad_enabled() and (
            _FUSE_EPI or _dz_shape(x, weight, kind, precision) or _ex_shape(x, weight, kind, depth, precision)):
        rec_in = getattr(x, '_lf_actnorm', None)
    x_split = getattr(x, '_lf_split', None)
    if x_split is None:
        # inference: a tensor that was packed for one convolution keeps its twin for the next convolution that reads it
        # (the GRU's hidden state feeds two gates); dropped as soon as the tensor is written to
        cached = getattr(x, '_lf_split_cache', None)
        if cached is not None and cached[0] == x._version:
            x_split = cached[1]
    y = _EqConv.apply(x, weight, bias, kind, depth, bool(act), float(slope), bool(norm), int(precision), fan_in, rec_in,
                      x_split, bool(emit_split))
    if _EqConv.last_in_split is not None and not torch.is_grad_enabled():
        x._lf_split_cache = (x._version, _EqConv.last_in_split)
    _EqConv.last_in_split = None
    if y.requires_grad and _EqConv.last_rec is not None:
        y._lf_actnorm = _EqConv.last_rec        # lets a single downstream lfb200 conv fuse this layer's backward
    if _EqConv.last_split is not None:
        y._lf_split = _EqConv.last_split
    _EqConv.last_rec = _EqConv.last_split = None
    return y


# ------------------------------------------------------------------------------------------------
# Interpolate
# ------------------------------------------------------------------------------------------------
class _Interp(torch.autograd.Function):
    """modules/__init__.py:18-33 (F.interpolate, scale 2 or 0.5, nearest / (bi|tri)linear)."""

    @staticmethod
    def forward(ctx, x, mode, factor):
        _need_cuda(x)
        x = to_cl(x)
        nd = x.dim() - 2
        n, c = x.shape[:2]
        d = x.shape[2] if nd == 3 else 1
        h, w = x.shape[-2:]
        f = (lambda s: s * 2) if factor > 0 else (lambda s: s // 2)
        out_shape = (n, c, f(d), f(h), f(w)) if nd == 3 else (n, c, f(h), f(w))
        y = empty_cl(out_shape, x.device)
        _call('lf_interp_fwd', L.lib().lf_interp_fwd, (_p(x), _p(y), nd, n, d, h, w, c, mode, factor, _stream()),
              nbytes=4 * (x.numel() + y.numel()))
        ctx.cfg = (nd, n, d, h, w, c, mode, factor, tuple(x.shape))
        return y

    @staticmethod
    def backward(ctx, gy):
        nd, n, d, h, w, c, mode, factor, xshape = ctx.cfg
        _need_cuda(gy)
        gy = to_cl(gy)
        gx = empty_cl(xshape, gy.device)
        _call('lf_interp_bwd', L.lib().lf_interp_bwd, (_p(gy), _p(gx), nd, n, d, h, w, c, mode, factor, _stream()),
              nbytes=4 * (gy.numel() + gx.numel()))
        return gx, None, None


def interpolate(x, scale_factor, mode):
    if scale_factor == 2.0:
        factor = 2
    elif scale_factor == 0.5:
        factor = -2
    else:
        raise ValueError(f"interpolate: scale_factor {scale_factor} unsupported (2.0 or 0.5)")
    if mode == 'nearest':
        m = 0
    elif mode in ('bilinear', 'trilinear', 'linear'):
        m = 1
    else:
        raise ValueError(f"interpolate: mode {mode!r} unsupported")
    return _Interp.apply(x, m, factor)


# ------------------------------------------------------------------------------------------------
# K4: view-axis pooling + GRU gates
# ------------------------------------------------------------------------------------------------
POOL_KINDS = {'max': 0, 'mean': 1, 'abs_max': 2, 'median': 3}


class _FusePool(torch.autograd.Function):
    """recon/fusion.py:45-57 over dim 1 of [B,V,C,D,H,W]."""

    @staticmethod
    def forward(ctx, z, kind):
        _need_cuda(z)
        B, V = z.shape[:2]
        zf = to_cl(z.reshape(B * V, *z.shape[2:]))
        C = z.shape[2]
        P = int(math.prod(z.shape[3:]))
        out = empty_cl((B, *z.shape[2:]), z.device)
        _call('lf_fuse_pool_fwd', L.lib().lf_fuse_pool_fwd, (_p(zf), _p(out), B, V, P, C, kind, _stream()),
              nbytes=4 * (zf.numel() + out.numel()))
        ctx.save_for_backward(zf)
        ctx.cfg = (B, V, P, C, kind, tuple(z.shape))
        return out.unsqueeze(1)

    @staticmethod
    def backward(ctx, gout):
        (zf,) = ctx.saved_tensors
        _need_cuda(gout, zf)
        B, V, P, C, kind, zshape = ctx.cfg
        g = to_cl(gout.reshape(B, *zshape[2:]))
        gz = torch.empty_like(zf)
        _call('lf_fuse_pool_bwd', L.lib().lf_fuse_pool_bwd, (_p(g), _p(zf), _p(gz), B, V, P, C, kind, _stream()))
        return gz.view(zshape), None


def fuse_pool(z, pool_type):
    if pool_type not in POOL_KINDS:
        raise ValueError(f"Unknown pool_type value {pool_type}")
    return _FusePool.apply(z, POOL_KINDS[pool_type])


class _GruGates1(torch.autograd.Function):
    """update = sigmoid(u_pre); hr = h * sigmoid(r_pre)   (modules/gru.py:38-40)."""

    @staticmethod
    def forward(ctx, u_pre, r_pre, h):
        _need_cuda(u_pre, r_pre, h)
        u_pre, r_pre, h = to_cl(u_pre), to_cl(r_pre), to_cl(h)
        update, hr = torch.empty_like(u_pre), torch.empty_like(h)
        _call('lf_gru_gates1', L.lib().lf_gru_gates1,
              (_p(u_pre), _p(r_pre), _p(h), _p(update), _p(hr), u_pre.numel(), _stream()))
        ctx.save_for_backward(update, r_pre, h)
        return update, hr

    @staticmethod
    def backward(ctx, g_update, g_hr):
        update, r_pre, h = ctx.saved_tensors
        zero = lambda: torch.zeros_like(h)                                    # noqa: E731
        gu = to_cl(g_update.float()) if g_update is not None else zero()
        gh = to_cl(g_hr.float()) if g_hr is not None else zero()
        g_u, g_r, g_h = torch.empty_like(h), torch.empty_like(h), torch.empty_like(h)
        _call('lf_gru_gates1_bwd', L.lib().lf_gru_gates1_bwd,
              (_p(gu), _p(gh), _p(update), _p(r_pre), _p(h), _p(g_u), _p(g_r), _p(g_h), h.numel(), _stream()))
        return g_u, g_r, g_h


class _GruGates2(torch.autograd.Function):
    """h_new = h*(1-update) + o*update   (modules/gru.py:41)."""

    @staticmethod
    def forward(ctx, h, update, o):
        _need_cuda(h, update, o)
        h, update, o = to_cl(h), to_cl(update), to_cl(o)
        out = torch.empty_like(h)
        _call('lf_gru_gates2', L.lib().lf_gru_gates2, (_p(h), _p(update), _p(o), _p(out), h.numel(), _stream()))
        ctx.save_for_backward(h, update, o)
        return out

    @staticmethod
    def backward(ctx, g):
        h, update, o = ctx.saved_tensors
        g = to_cl(g.float())
        g_h, g_u, g_o = torch.empty_like(h), torch.empty_like(h), torch.empty_like(h)
        _call('lf_gru_gates2_bwd', L.lib().lf_gru_gates2_bwd,
              (_p(g), _p(h), _p(update), _p(o), _p(g_h), _p(g_u), _p(g_o), h.numel(), _stream()))
        return g_h, g_u, g_o


def gru_gates1(u_pre, r_pre, h):
    return _GruGates1.apply(u_pre, r_pre, h)


def gru_gates2(h, update, o):
    return _GruGates2.apply(h, update, o)


class _LstmGates(torch.autograd.Function):
    """ConvLSTM gate non-linearities in one pass (modules/lstm.py:41-56); gates [N,4H,...] = (i | f | o | g)."""

    @staticmethod
    def forward(ctx, gates, c_cur):
        _need_cuda(gates, c_cur)
        gates, c_cur = to_cl(gates), to_cl(c_cur)
        hid = c_cur.shape[1]
        pos = c_cur.numel() // hid
        h_next, c_next = torch.empty_like(c_cur), torch.empty_like(c_cur)
        _call('lf_lstm_gates_fwd', L.lib().lf_lstm_gates_fwd, (_p(gates), _p(c_cur), _p(h_next), _p(c_next), pos, hid, _stream()))
        ctx.save_for_backward(gates, c_cur)
        return h_next, c_next

    @staticmethod
    def backward(ctx, g_h, g_c):
        gates, c_cur = ctx.saved_tensors
        hid = c_cur.shape[1]
        pos = c_cur.numel() // hid
        g_h = None if g_h is None else to_cl(g_h.float())
        g_c = None if g_c is None else to_cl(g_c.float())
        g_gates, g_cc = torch.empty_like(gates), torch.empty_like(c_cur)
        _call('lf_lstm_gates_bwd', L.lib().lf_lstm_gates_bwd,
              (_p(g_h), _p(g_c), _p(gates), _p(c_cur), _p(g_gates), _p(g_cc), pos, hid, _stream()))
        return g_gates, g_cc


def lstm_gates(gates, c_cur):
    """-> (h_next, c_next)"""
    return _LstmGates.apply(gates, c_cur)


class _SoftmaxBlend(torch.autograd.Function):
    """w = softmax over axis 1 of scores [B,V,P...]; out = sum_v w * z with z [B,V,P...,C] in memory (channels-last)."""

    @staticmethod
    def forward(ctx, scores, z, B, V, P, C):
        wts = torch.empty(B, V, P, device=z.device)
        out = torch.empty(B, P, C, device=z.device)
        _call('lf_softmax_blend_fwd', L.lib().lf_softmax_blend_fwd, (_p(scores), _p(z), _p(wts), _p(out), B, V, P, C, _stream()),
              nbytes=4 * (z.numel() + out.numel()))
        ctx.save_for_backward(wts, z)
        ctx.dims = (B, V, P, C)
        return out, wts

    @staticmethod
    def backward(ctx, g_out, g_wts):
        wts, z = ctx.saved_tensors
        B, V, P, C = ctx.dims
        g_out = torch.zeros(B, P, C, device=z.device) if g_out is None else g_out.float().contiguous()
        g_wts = None if g_wts is None else g_wts.float().contiguous()
        g_scores = torch.empty(B, V, P, device=z.device)
        g_z = torch.empty_like(z) if ctx.needs_input_grad[1] else None
        _call('lf_softmax_blend_bwd', L.lib().lf_softmax_blend_bwd,
              (_p(g_out), _p(g_wts), _p(wts), _p(z), _p(g_scores), _p(g_z), B, V, P, C, _stream()),
              nbytes=4 * (2 * z.numel() + g_out.numel()))
        return g_scores, g_z, None, None, None, None


def view_softmax_blend(scores, z_obj):
    """BlendFuser (recon/fusion.py:92-96): scores [B,V,1,D,H,W], z_obj [B,V,C,D,H,W] ->
    (sum_v softmax_v(scores) * z_obj  [B,1,C,D,H,W], weights [B,V,1,D,H,W])."""
    _need_cuda(scores, z_obj)
    B, V, C = z_obj.shape[:3]
    sp = tuple(z_obj.shape[3:])
    P = 1
    for e in sp:
        P *= e
    zc = z_obj.float().movedim(2, -1).contiguous()                   # [B,V,D,H,W,C]: a no-op for per-view channels-last cubes
    out, wts = _SoftmaxBlend.apply(scores.float().reshape(B, V, P).contiguous(), zc.view(B, V, P, C), B, V, P, C)
    return out.view(B, *sp, C).movedim(-1, 1).unsqueeze(1), wts.view(B, V, 1, *sp)


class _DepthSum(torch.autograd.Function):
    """projection_type='sum' (recon/models.py:436-437): [N,C,D,H,W] -> [N,C,H,W]"""

    @staticmethod
    def forward(ctx, x):
        _need_cuda(x)
        x = to_cl(x)
        n, c, d, h, w = x.shape
        out = empty_cl((n, c, h, w), x.device)
        _call('lf_depth_sum_fwd', L.lib().lf_depth_sum_fwd, (_p(x), _p(out), n, d, h * w, c, _stream()),
              nbytes=4 * (x.numel() + out.numel()))
        ctx.d = d
        return out

    @staticmethod
    def backward(ctx, g):
        return g.unsqueeze(2).expand(-1, -1, ctx.d, -1, -1)


def depth_sum(x):
    return _DepthSum.apply(x)


# ------------------------------------------------------------------------------------------------
# fused pose-loss head
# ------------------------------------------------------------------------------------------------
def _loss_ws(query, desc, device):
    """device workspace of the pose-loss head (lf_pose_loss_fwd_ws / lf_pose_loss_bwd_ws bytes)"""
    nbytes = query(ctypes.byref(desc))
    if nbytes < 0:
        L.check(int(nbytes), 'pose_loss workspace')
    return torch.empty((nbytes + 3) // 4, device=device)


class _PoseLoss(torch.autograd.Function):
    """interpret_logits + denormalize_depth + uncrop x2 + default_pose_loss terms in two full-frame passes.
    Returns terms [N,4] = (ov_depth, depth, iou, mask); differentiable w.r.t. the two logit maps, the
    viewport and the translation's z."""

    @staticmethod
    def forward(ctx, depth_logits, mask_logits, viewport, tz, target_depth, target_mask, z_span, eps, width, height):
        _need_cuda(depth_logits, mask_logits, viewport, tz, target_depth, target_mask)
        n, p = depth_logits.shape[0], depth_logits.shape[-1]
        dl = depth_logits.detach().float().contiguous().view(n, p, p)
        ml = mask_logits.detach().float().contiguous().view(n, p, p)
        vp = viewport.detach().float().contiguous()
        tzc = tz.detach().float().contiguous()
        td = target_depth.detach().float().contiguous().view(height, width)
        tm = target_mask.detach().float().contiguous().view(height, width)
        desc = L.LossDesc(n, p, width, height, float(z_span), float(eps))
        sums = torch.empty(n, 8, device=dl.device)
        terms = torch.empty(n, 4, device=dl.device)
        ws = _loss_ws(L.lib().lf_pose_loss_fwd_ws, desc, dl.device)
        _call('lf_pose_loss_fwd', L.lib().lf_pose_loss_fwd,
              (ctypes.byref(desc), _p(dl), _p(ml), _p(vp), _p(tzc), _p(td), _p(tm), _p(sums), _p(terms), _p(ws), _stream()),
              kernels=3)
        ctx.save_for_backward(dl, ml, vp, tzc, td, tm, sums)
        ctx.cfg = (n, p, width, height, float(z_span), float(eps), tuple(depth_logits.shape), tuple(mask_logits.shape))
        return terms

    @staticmethod
    def backward(ctx, gterms):
        dl, ml, vp, tzc, td, tm, sums = ctx.saved_tensors
        _need_cuda(gterms, dl)
        n, p, width, height, z_span, eps, dshape, mshape = ctx.cfg
        desc = L.LossDesc(n, p, width, height, z_span, eps)
        g_dl, g_ml = torch.empty_like(dl), torch.empty_like(ml)
        g_vp, g_tz = torch.empty_like(vp), torch.empty_like(tzc)
        gt = gterms.float().contiguous()
        ws = _loss_ws(L.lib().lf_pose_loss_bwd_ws, desc, dl.device)
        _call('lf_pose_loss_bwd', L.lib().lf_pose_loss_bwd,
              (ctypes.byref(desc), _p(dl), _p(ml), _p(vp), _p(tzc), _p(td), _p(tm), _p(sums), _p(gt),
               _p(g_dl), _p(g_ml), _p(g_vp), _p(g_tz), _p(ws), _stream()), kernels=3)
        return g_dl.view(dshape), g_ml.view(mshape), g_vp, g_tz, None, None, None, None, None, None


class _PoseLossPacked(torch.autograd.Function):
    """_PoseLoss on the decoder's own tensors: the channels-last logits [N,2,P,P] of the fused heads (depth = channel 0,
    mask = channel 1) and the translation [N,3], addressed through lf_loss_desc's strides — no de-interleaving copies
    forward, no select/add/copy chain backward."""

    @staticmethod
    def forward(ctx, logits, viewport, translation, target_depth, target_mask, z_span, eps, width, height):
        _need_cuda(logits, viewport, translation, target_depth, target_mask)
        n, hh, p = logits.shape[0], logits.shape[1], logits.shape[-1]
        lg = logits.detach()
        vp = viewport.detach().float().contiguous()
        tr = translation.detach().float().contiguous()
        td = target_depth.detach().float().contiguous().view(height, width)
        tm = target_mask.detach().float().contiguous().view(height, width)
        desc = L.LossDesc(n, p, width, height, float(z_span), float(eps), hh, p * p * hh, 3)
        sums = torch.empty(n, 8, device=lg.device)
        terms = torch.empty(n, 4, device=lg.device)
        base = lg.data_ptr()
        ws = _loss_ws(L.lib().lf_pose_loss_fwd_ws, desc, lg.device)
        _call('lf_pose_loss_fwd', L.lib().lf_pose_loss_fwd,
              (ctypes.byref(desc), base, base + 4, _p(vp), tr.data_ptr() + 8, _p(td), _p(tm), _p(sums), _p(terms), _p(ws),
               _stream()),
              kernels=3)
        ctx.save_for_backward(lg, vp, tr, td, tm, sums)
        ctx.cfg = (n, hh, p, width, height, float(z_span), float(eps))
        return terms

    @staticmethod
    def backward(ctx, gterms):
        lg, vp, tr, td, tm, sums = ctx.saved_tensors
        _need_cuda(gterms, lg)
        n, hh, p, width, height, z_span, eps = ctx.cfg
        desc = L.LossDesc(n, p, width, height, z_span, eps, hh, p * p * hh, 3)
        g_lg = torch.zeros_like(lg)                       # (same channels-last strides)
        g_tr = torch.zeros_like(tr)                       # (the kernel writes its z column only)
        g_vp = torch.empty_like(vp)
        gt = gterms.float().contiguous()
        base, gbase = lg.data_ptr(), g_lg.data_ptr()
        ws = _loss_ws(L.lib().lf_pose_loss_bwd_ws, desc, lg.device)
        _call('lf_pose_loss_bwd', L.lib().lf_pose_loss_bwd,
              (ctypes.byref(desc), base, base + 4, _p(vp), tr.data_ptr() + 8, _p(td), _p(tm), _p(sums), _p(gt),
               gbase, gbase + 4, _p(g_vp), g_tr.data_ptr() + 8, _p(ws), _stream()), kernels=3)
        return g_lg, g_vp, g_tr, None, None, None, None, None, None


def pose_loss_terms_packed(logits, viewport, translation, target_depth, target_mask, z_span, eps=0.01, width=640, height=480):
    """terms [N,4] straight from the decoder's logits [N,2,P,P] (depth, mask heads) and the translation [N,3]; falls back
    to the de-interleaved form when the logits are not the fused heads' channels-last fp32 tensor."""
    n, hh, p = logits.shape[0], logits.shape[1], logits.shape[-1]
    if (logits.dim() == 4 and hh == 2 and logits.dtype == torch.float32 and logits.shape[2] == p
            and logits.stride() == (p * p * hh, 1, p * hh, hh) and translation.dtype == torch.float32):
        return _PoseLossPacked.apply(logits, viewport, translation, target_depth, target_mask, z_span, eps, width, height)
    return _PoseLoss.apply(logits[:, 0], logits[:, 1], viewport, translation[:, 2], target_depth, target_mask, z_span, eps,
                           width, height)


def refine_record_(terms, w_rank, w_opt, lq, tr, rank, gterms, h_rank, h_optim, h_terms, h_lq, h_tr, slot, chunk, step_count):
    """lf_refine_record: ranking / optimisation losses, d mean(optim)/d terms and the chunk-history snapshot in one launch."""
    _need_cuda(terms, w_rank, w_opt, lq, tr, rank, gterms, h_rank, slot)
    n, k = terms.shape
    _call('lf_refine_record', L.lib().lf_refine_record,
          (_p(terms), n, k, _p(w_rank), _p(w_opt), _p(lq), _p(tr), _p(rank), _p(gterms), _p(h_rank), _p(h_optim), _p(h_terms),
           _p(h_lq), _p(h_tr), slot.data_ptr(), int(chunk), _p(step_count) if step_count is not None else None, _stream()))


@torch.no_grad()
def pose_search_terms(depth_logits, mask_logits, viewport, tz, target_depth, target_mask, z_span, eps=0.01,
                      width=640, height=480):
    """forward-only [N,4] (ov_depth, depth, iou, mask) for the coarse search: lf_pose_loss_search_fwd"""
    _need_cuda(depth_logits, mask_logits, viewport, tz, target_depth, target_mask)
    n, p = depth_logits.shape[0], depth_logits.shape[-1]
    dl, ml = depth_logits.float().contiguous().view(n, p, p), mask_logits.float().contiguous().view(n, p, p)
    desc = L.LossDesc(n, p, width, height, float(z_span), float(eps))
    sums, terms = torch.empty(n, 8, device=dl.device), torch.empty(n, 4, device=dl.device)
    ws = _loss_ws(L.lib().lf_pose_loss_fwd_ws, desc, dl.device)
    _call('lf_pose_loss_search_fwd', L.lib().lf_pose_loss_search_fwd,
          (ctypes.byref(desc), _p(dl), _p(ml), _p(viewport.float().contiguous()), _p(tz.float().contiguous()),
           _p(target_depth.float().contiguous().view(height, width)), _p(target_mask.float().contiguous().view(height, width)),
           _p(sums), _p(terms), _p(ws), _stream()), kernels=3)
    return terms


def pose_loss_terms(depth_logits, mask_logits, viewport, tz, target_depth, target_mask, z_span, eps=0.01,
                    width=640, height=480):
    return _PoseLoss.apply(depth_logits, mask_logits, viewport, tz, target_depth, target_mask, z_span, eps, width, height)


# ------------------------------------------------------------------------------------------------
# camera algebra + batched optimiser
# ------------------------------------------------------------------------------------------------
class _CameraO2CBlock(torch.autograd.Function):
    """(log_quaternion, translation, viewport) -> [N, LF_CAM_STRIDE] object->camera block, analytic VJP."""

    @staticmethod
    def forward(ctx, lq, tr, vp, intrinsic, z_span, cube_size):
        _need_cuda(lq, tr, vp, intrinsic)
        n = lq.shape[0]
        lqc, trc, vpc = (t.detach().float().contiguous() for t in (lq, tr, vp))
        kc = intrinsic.detach().float().contiguous()
        block = torch.empty(n, L.CAM_STRIDE, device=lq.device, dtype=torch.float32)
        _call('lf_camera_o2c_fwd', L.lib().lf_camera_o2c_fwd,
              (_p(lqc), _p(trc), _p(vpc), _p(kc), _p(block), n, float(z_span), float(cube_size), _stream()))
        ctx.save_for_backward(lqc, trc)
        return block

    @staticmethod
    def backward(ctx, gblock):
        lqc, trc = ctx.saved_tensors
        _need_cuda(gblock, lqc)
        n = lqc.shape[0]
        gb = gblock.float().contiguous()
        g_lq, g_tr = torch.empty_like(lqc), torch.empty_like(trc)
        g_vp = torch.empty(n, 4, device=lqc.device, dtype=torch.float32)
        _call('lf_camera_o2c_bwd', L.lib().lf_camera_o2c_bwd,
              (_p(lqc), _p(trc), _p(gb), _p(g_lq), _p(g_tr), _p(g_vp), n, _stream()))
        return g_lq, g_tr, g_vp, None, None, None


def camera_o2c_block(log_quaternion, translation, viewport, intrinsic, z_span, cube_size):
    return _CameraO2CBlock.apply(log_quaternion, translation, viewport, intrinsic, z_span, cube_size)


def adam_step_(param, grad, exp_avg, exp_avg_sq, step_count, lr, beta1=0.9, beta2=0.999, eps=1e-8):
    """In-place torch.optim.Adam update of param [N,W] with a per-row learning rate lr [N]."""
    _need_cuda(param, grad, exp_avg, exp_avg_sq, step_count, lr)
    n, width = param.shape
    _call('lf_adam_step', L.lib().lf_adam_step,
          (_p(param), _p(grad.contiguous()), _p(exp_avg), _p(exp_avg_sq), n, width, _p(step_count), _p(lr),
           beta1, beta2, eps, _stream()))


def plateau_step_(rank_loss, lr, best, num_bad, threshold, patience, factor):
    _need_cuda(rank_loss, lr, best, num_bad)
    _call('lf_plateau_step', L.lib().lf_plateau_step,
          (_p(rank_loss.contiguous()), _p(lr), _p(best), _p(num_bad), rank_loss.shape[0], float(threshold),
           float(patience), float(factor), _stream()))


# ------------------------------------------------------------------------------------------------
# fused 1x1 output heads
# ------------------------------------------------------------------------------------------------
class _Heads(torch.autograd.Function):
    """All 1x1 output heads of a decoder in one pass over its feature map (exact fp32).  weight [H, C] is the
    row-stack of the heads' [Cout_i, C, 1, 1] weights; every head has fan-in C, hence one He constant."""

    @staticmethod
    def forward(ctx, x, weight, bias):
        _need_cuda(x, weight, bias)
        x = to_cl(x)
        n, c, hh, ww = x.shape
        h = weight.shape[0]
        scale = math.sqrt(2.0 / c)
        wf = weight.detach().float().contiguous()
        y = empty_cl((n, h, hh, ww), x.device)
        _call('lf_heads_fwd', L.lib().lf_heads_fwd,
              (_p(x), _p(wf), _p(None if bias is None else bias.detach().float().contiguous()), _p(y), n * hh * ww, c, h,
               scale, _stream()), nbytes=4 * (x.numel() + y.numel()), flops=2 * n * hh * ww * c * h)
        ctx.save_for_backward(x, wf)
        ctx.scale = scale
        return y

    @staticmethod
    def backward(ctx, gy):
        x, wf = ctx.saved_tensors
        _need_cuda(gy, x)
        gy = to_cl(gy)
        n, c, hh, ww = x.shape
        h = wf.shape[0]
        gx = gw = gb = None
        if ctx.needs_input_grad[0]:
            gx = torch.empty_like(x)
            _call('lf_heads_bwd', L.lib().lf_heads_bwd, (_p(gy), _p(wf), _p(gx), n * hh * ww, c, h, ctx.scale, _stream()),
                  nbytes=4 * (x.numel() + gy.numel()), flops=2 * n * hh * ww * c * h)
        if ctx.needs_input_grad[1] or ctx.needs_input_grad[2]:       # training: tiny [H, C] reductions in torch
            g2 = gy.permute(0, 2, 3, 1).reshape(-1, h)
            if ctx.needs_input_grad[1]:
                gw = (g2.t() @ x.permute(0, 2, 3, 1).reshape(-1, c)) * ctx.scale
            if ctx.needs_input_grad[2]:
                gb = g2.sum(dim=0)
        return gx, gw, gb


def heads_supported(c, h):
    q4 = c // 4
    return c % 4 == 0 and c >= 4 and (q4 & (q4 - 1)) == 0 and q4 <= 32 and 1 <= h <= 8


def fused_heads(x, weights, biases):
    """x [N,C,H,W]; weights: list of [Cout_i, C, 1, 1]; biases: list of [Cout_i] or None -> [N, sum Cout_i, H, W]."""
    c = x.shape[1]
    w = torch.cat([wi.reshape(wi.shape[0], c) for wi in weights], dim=0)
    if all(b is None for b in biases):
        b = None
    else:
        b = torch.cat([bi if bi is not None else wi.new_zeros(wi.shape[0]) for wi, bi in zip(weights, biases)], dim=0)
    return _Heads.apply(x, w, b)


# ------------------------------------------------------------------------------------------------
# IBR colour branch (forward only)
# ------------------------------------------------------------------------------------------------
IBR_CAM_STRIDE = 48


def _no_grad_path(name, *tensors):
    if torch.is_grad_enabled() and any(t is not None and t.requires_grad for t in tensors):
        raise NotImplementedError(f"{name}: the IBR colour branch is forward-only in lfb200 (it is not on the pose "
                                  f"loop's gradient path); call it under torch.no_grad() or detach its inputs")


def ibr_reproject(image_in, depth_in, depth_out, cam_in_block, cam_out_block):
    """latentfusion/ibr.py:55-93 for one object.  image_in [Vi,C,H,W], depth_in [Vi,1,H,W], depth_out [Vo,1,H,W],
    camera blocks from Camera.ibr_block() -> (image_reproj [Vo,Vi,C,H,W], depth_reproj [Vo,Vi,1,H,W])."""
    _need_cuda(image_in, depth_in, depth_out, cam_in_block, cam_out_block)
    _no_grad_path('ibr_reproject', image_in, depth_in, depth_out, cam_in_block, cam_out_block)
    vi, c, h, w = image_in.shape
    vo = depth_out.shape[0]
    if depth_in.shape[0] != vi or cam_in_block.shape != (vi, IBR_CAM_STRIDE) or cam_out_block.shape != (vo, IBR_CAM_STRIDE):
        raise ValueError("ibr_reproject: view counts of images, depths and cameras do not match")
    if tuple(depth_in.shape[-2:]) != (h, w) or tuple(depth_out.shape[-2:]) != (h, w):
        raise ValueError("ibr_reproject: image and depth sizes must match")
    img = image_in.detach().float().contiguous()
    din = depth_in.detach().float().contiguous()
    dout = depth_out.detach().float().contiguous()
    ci, co = cam_in_block.detach().float().contiguous(), cam_out_block.detach().float().contiguous()
    image_reproj = torch.empty(vo, vi, c, h, w, device=img.device)
    depth_reproj = torch.empty(vo, vi, 1, h, w, device=img.device)
    _call('lf_ibr_reproject_fwd', L.lib().lf_ibr_reproject_fwd,
          (_p(img), _p(din), _p(dout), _p(co), _p(ci), _p(image_reproj), _p(depth_reproj), vo, vi, c, h, w, _stream()),
          nbytes=4 * (image_reproj.numel() + depth_reproj.numel() + img.numel() + din.numel() + dout.numel()))
    return image_reproj, depth_reproj


class _IbrBlend(torch.autograd.Function):
    """out[b,c,p] = sum_i w[b,i,(p)] * img[b,i,c,p]; differentiable w.r.t. the weights (kernel) and the images."""

    @staticmethod
    def forward(ctx, img, wts, per_pixel):
        b, vi, c, h, w = img.shape
        out = torch.empty(b, c, h, w, device=img.device)
        _call('lf_ibr_blend_fwd', L.lib().lf_ibr_blend_fwd, (_p(img), _p(wts), _p(out), b, vi, c, h * w, int(per_pixel), _stream()),
              nbytes=4 * (img.numel() + out.numel()))
        ctx.save_for_backward(img, wts)
        ctx.per_pixel = per_pixel
        return out

    @staticmethod
    def backward(ctx, g):
        img, wts = ctx.saved_tensors
        b, vi, c, h, w = img.shape
        g = g.float().contiguous()
        gw = gi = None
        if ctx.needs_input_grad[1]:
            gw = torch.empty(b, vi, h, w, device=img.device)
            _call('lf_ibr_blend_bwd', L.lib().lf_ibr_blend_bwd, (_p(g), _p(img), _p(gw), b, vi, c, h * w, _stream()),
                  nbytes=4 * (img.numel() + g.numel() + gw.numel()))
            if not ctx.per_pixel:
                gw = gw.sum(dim=(2, 3))
        if ctx.needs_input_grad[0]:
            wv = wts.view(b, vi, 1, h, w) if ctx.per_pixel else wts.view(b, vi, 1, 1, 1)
            gi = g.unsqueeze(1) * wv
        return gi, gw, None


def ibr_blend(image_reproj, weights):
    """sum over views of weights * image_reproj.  image_reproj [B,Vi,C,H,W]; weights [B,Vi] (per view) or
    [B,Vi,H,W] (per pixel).  latentfusion/ibr.py:223-224, :231-234."""
    _need_cuda(image_reproj, weights)
    b, vi, c, h, w = image_reproj.shape
    per_pixel = weights.dim() == 4
    if tuple(weights.shape[:2]) != (b, vi) or (per_pixel and tuple(weights.shape[2:]) != (h, w)) or weights.dim() not in (2, 4):
        raise ValueError("ibr_blend: weights must be [B,Vi] or [B,Vi,H,W]")
    return _IbrBlend.apply(image_reproj.float().contiguous(), weights.float().contiguous(), per_pixel)


class _IbrWarpBlend(torch.autograd.Function):
    """latentfusion/ibr.py:237-249; differentiable w.r.t. the logits (all four outputs)."""

    @staticmethod
    def forward(ctx, lg, img, flow_size):
        b, vi, c, h, w = img.shape
        image = torch.empty(b, c, h, w, device=img.device)
        wts = torch.empty(b, vi, h, w, device=img.device)
        dx, dy = torch.empty_like(wts), torch.empty_like(wts)
        _call('lf_ibr_warp_blend_fwd', L.lib().lf_ibr_warp_blend_fwd,
              (_p(lg), _p(img), float(flow_size), _p(image), _p(wts), _p(dx), _p(dy), b, vi, c, h, w, _stream()),
              nbytes=4 * (lg.numel() + img.numel() + image.numel() + 3 * wts.numel()))
        ctx.save_for_backward(lg, img)
        ctx.flow_size = float(flow_size)
        return image, wts, dx, dy

    @staticmethod
    def backward(ctx, g_image, g_w, g_dx, g_dy):
        lg, img = ctx.saved_tensors
        if ctx.needs_input_grad[1]:
            raise NotImplementedError("ibr_warp_blend: no gradient w.r.t. the reprojected images (the reference trains "
                                      "the generator with the recon networks frozen, train_ibr.py:320)")
        b, vi, c, h, w = img.shape
        prep = lambda t: None if t is None else t.float().contiguous()     # noqa: E731
        g_image = torch.zeros(b, c, h, w, device=img.device) if g_image is None else prep(g_image)
        g_w, g_dx, g_dy = prep(g_w), prep(g_dx), prep(g_dy)
        gl = torch.empty_like(lg)
        _call('lf_ibr_warp_blend_bwd', L.lib().lf_ibr_warp_blend_bwd,
              (_p(lg), _p(img), ctx.flow_size, _p(g_image), _p(g_w), _p(g_dx), _p(g_dy), _p(gl), b, vi, c, h, w, _stream()),
              nbytes=4 * (2 * lg.numel() + img.numel() + g_image.numel()))
        return gl, None, None


def ibr_warp_blend(logits, image_reproj, flow_size):
    """latentfusion/ibr.py:237-249 -> (image [B,C,H,W], blend_weights [B,Vi,1,H,W], flow_dx, flow_dy [B,Vi,H,W])."""
    _need_cuda(logits, image_reproj)
    b, vi, c, h, w = image_reproj.shape
    if tuple(logits.shape) != (b, 3 * vi, h, w):
        raise ValueError(f"ibr_warp_blend: logits must be [B, 3*Vi, H, W] = {(b, 3 * vi, h, w)}, got {tuple(logits.shape)}")
    if c > 8:
        raise ValueError("ibr_warp_blend: at most 8 colour channels")
    image, wts, dx, dy = _IbrWarpBlend.apply(logits.float().contiguous(), image_reproj.float().contiguous(), flow_size)
    return image, wts.unsqueeze(2), dx, dy
