"""The refine iteration's small kernels against float64 restatements of the reference maths.

* the fused pose-loss head (csrc/pose_loss.cu: forward, the search forward, and the gather backward) against an fp64
  restatement of uncrop x2 + default_pose_loss, at viewports across the frame edges, larger than the frame, magnified,
  off-frame and flipped, at odd frame and crop sizes, and on targets with sensor holes, fractional and empty masks;
* the resize (csrc/elementwise.cu interp kernels) against F.interpolate in fp64 under autograd;
* the camera block (csrc/camera.cu) against an fp64 restatement of its chain;
* the batched Adam + ReduceLROnPlateau step against N independent fp64 torch optimisers and schedulers.

The loss head switches discontinuously at nearest-tap ties (and at the bilinear floor and the border clamps), at the
mask gate's logit 0 and at the sign of (rendered - target) depth.  Near such a switch fp32 and fp64 may take different
branches, so the inputs are moved off them (`_clear_switches`) and every comparison first asserts that no pixel lies
within a margin of one.  The exact-tie viewports (integer corners, extent P or 2P) are computed exactly in both
precisions and keep their ties: they are what pins the half-to-even rounding of the nearest tap.
"""
import math

import pytest
import torch
import torch.nn.functional as F

from tests import parity_helpers as ph

Z_SPAN, EPS = 0.5, 0.01
TERMS = ('ov_depth', 'depth', 'iou', 'mask')

# margins to the switches (fp32 errors measured on a B200 are far below them, see the bounds further down)
TIE_MARGIN = 2e-4          # in crop-pixel units of the sample coordinate
GATE_MARGIN = 1e-3         # |mask logit| of every crop texel
SIGN_MARGIN = 1e-5         # relative |rendered - target depth| where the target depth is not 0


@pytest.fixture(scope='module')
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device('cuda:0')


# ---------------------------------------------------------------------------------------------------------------------
# fp64 restatement of interpret_logits -> denormalize_depth -> uncrop x2 -> default_pose_loss
# (pose/estimation.py:61-91, pose/utils.py:56-72, modules/geometry.py:290-302, recon/models.py:280-300)
# ---------------------------------------------------------------------------------------------------------------------
def _grid(vp, width, height):
    n, dt, d = vp.shape[0], vp.dtype, vp.device
    xs = torch.arange(width, dtype=dt, device=d)
    ys = torch.arange(height, dtype=dt, device=d)
    gx = (xs[None, :] - vp[:, 0, None]) / (vp[:, 2] - vp[:, 0])[:, None] * 2 - 1
    gy = (ys[None, :] - vp[:, 1, None]) / (vp[:, 3] - vp[:, 1])[:, None] * 2 - 1
    return torch.stack((gx[:, None, :].expand(n, height, width), gy[:, :, None].expand(n, height, width)), dim=-1)


def _frames(dl, ml, vp, tz, width, height, premask=False):
    """(rendered metric depth x rendered mask, rendered mask logits, rendered mask), each [N,1,H,W]"""
    n = dl.shape[0]
    inside = (torch.sigmoid(ml) > 0.5).to(dl.dtype)
    depth = (torch.tanh(dl) + 1) * inside - 1                                 # interpret_logits(apply_mask=True)
    lo = (tz - Z_SPAN - EPS).view(n, 1, 1)
    hi = (tz + Z_SPAN + EPS).view(n, 1, 1)
    z = (depth / 2.0 + 0.5) * (hi - lo) + lo                                  # Camera.denormalize_depth
    if premask:                                                               # PoseEstimator._render_observation
        z = z * torch.sigmoid(ml)
    grid = _grid(vp, width, height)
    kw = dict(padding_mode='border', align_corners=False)
    frame_depth = F.grid_sample(z[:, None], grid, mode='nearest', **kw)
    frame_logits = F.grid_sample(ml[:, None], grid, mode='bilinear', **kw)
    frame_mask = torch.sigmoid(frame_logits)
    return frame_depth * frame_mask, frame_logits, frame_mask


def loss_head_ref(dl, ml, vp, tz, tdepth, tmask, premask=False):
    """terms [N,4] = (ov_depth, depth, iou, mask) in the dtype of the inputs; tdepth, tmask [H,W]"""
    height, width = tdepth.shape[-2:]
    pd, logits, pm = _frames(dl, ml, vp, tz, width, height, premask)
    td = tdepth.to(dl.dtype).view(1, 1, height, width)
    tm = tmask.to(dl.dtype).view(1, 1, height, width)
    valid = (~((td == 0) & (tm > 0.1))).to(dl.dtype)                          # sensor holes
    err = (pd - td * tm).abs() * valid                                        # Observation.prepare(): depth * mask
    dims = (1, 2, 3)
    ov = (err * pm * tm).sum(dims).clamp(min=1e-5) / (pm * tm).sum(dims).clamp(min=1e-4)
    tmv = tm * valid
    inter = (pm * tmv).sum(dims)
    union = pm.sum(dims) + tmv.sum(dims) - inter
    iou = torch.log(union.clamp(min=1e-4)) - torch.log(inter.clamp(min=1e-4))
    # BCE with logits, written with log1p: ATen's form adds exp(-|x|) to 1 and loses every digit of it below 1e-16, all
    # there is of the term when the rendered mask is off (logits near -30) and the target mask is empty
    bce = (logits.clamp(min=0) - logits * tm + torch.log1p(torch.exp(-logits.abs()))).mean(dims)
    return torch.stack((ov, err.mean(dims), iou, bce), dim=1)


# ---------------------------------------------------------------------------------------------------------------------
# switch margins
# ---------------------------------------------------------------------------------------------------------------------
def _near_tie(v0, v1, P, length):
    """pixels of one axis whose sample coordinate lies within TIE_MARGIN of a multiple of 1/2 inside [0, P-1]: the
    nearest tap, the bilinear floor and the border clamp switch there"""
    x = torch.arange(length, dtype=torch.float64)
    ix = (((x - v0) / (v1 - v0) * 2 - 1 + 1) * P - 1) / 2
    inside = (ix > -TIE_MARGIN) & (ix < P - 1 + TIE_MARGIN)
    return inside & ((2 * ix - torch.round(2 * ix)).abs() < 2 * TIE_MARGIN)


def _tie_rows(vp, P, width, height, exact):
    """rows of vp (fp64 values of the fp32 inputs) with a pixel near a tap switch; exact rows are skipped"""
    bad = []
    for i, r in enumerate(vp.tolist()):
        if not exact[i] and (_near_tie(r[0], r[2], P, width).any() or _near_tie(r[1], r[3], P, height).any()):
            bad.append(i)
    return bad


def _sign_pixels(dl, ml, vp, tz, tdepth, tmask):
    """[N,H,W] pixels where the rendered depth is within SIGN_MARGIN of a non-zero target depth"""
    height, width = tdepth.shape
    with torch.no_grad():
        pd = _frames(dl.double(), ml.double(), vp.double(), tz.double(), width, height)[0][:, 0]
    td = (tdepth * tmask).double()
    valid = ~((tdepth == 0) & (tmask > 0.1))
    return (td != 0) & valid & ((pd - td).abs() < SIGN_MARGIN * td.abs())


def assert_off_switches(dl, ml, vp, tz, tdepth, tmask, exact):
    P = dl.shape[-1]
    height, width = tdepth.shape
    assert float(ml.abs().min()) > GATE_MARGIN, 'a mask logit sits at the gate'
    bad = _tie_rows(vp.double().cpu(), P, width, height, exact)
    assert not bad, f'viewports {bad} put a pixel at a tap switch'
    n = int(_sign_pixels(dl.cpu(), ml.cpu(), vp.cpu(), tz.cpu(), tdepth.cpu(), tmask.cpu()).sum())
    assert n == 0, f'{n} pixels at the sign switch of (rendered - target) depth'


def _clear_switches(dl, ml, vp, tz, tdepth, tmask, exact):
    """move the inputs off the switches: viewports in steps of 1/64 px, target depths by 0.1 %"""
    P = dl.shape[-1]
    height, width = tdepth.shape
    vp, tdepth = vp.clone(), tdepth.clone()
    for _ in range(64):
        bad = _tie_rows(vp.double(), P, width, height, exact)
        if not bad:
            break
        for i in bad:
            vp[i] += torch.tensor([1.0, 1.0, 0.5, 0.5]) / 64
    for _ in range(64):
        near = _sign_pixels(dl, ml, vp, tz, tdepth, tmask).any(0)
        if not near.any():
            break
        tdepth[near] *= 1.001
    return vp, tdepth


# ---------------------------------------------------------------------------------------------------------------------
# loss-head cases (all drawn on the CPU in fp32; the references run on their fp64 values)
# ---------------------------------------------------------------------------------------------------------------------
def _logits(gen, n, P, kind):
    dl = torch.randn(n, P, P, generator=gen) * 1.5
    if kind == 'generic':
        ml = torch.randn(n, P, P, generator=gen) * 3.0
        ml = ml + 0.05 * torch.sign(ml)                     # keep every texel off the gate at logit 0
    elif kind == 'gate_off':                                # all rendered mask logits <= -3: the depth gate is shut
        ml = -3.0 - 3.0 * torch.rand(n, P, P, generator=gen)
    else:                                                   # 'mask_off': also every clamp of the ov/iou sums engages
        ml = -28.0 - 8.0 * torch.rand(n, P, P, generator=gen)
    return dl, ml


def geometry_640(P):
    """(viewports [N,4], per-row logit kinds, exact-tie rows) of the 640x480 cases at crop size P"""
    if P == 128:
        rows = [([251.3, 180.7, 389.9, 319.2], 'generic', False),           # interior
                ([-40.3, -25.6, 90.1, 101.7], 'generic', False),            # across the left / top edges
                ([560.2, 410.9, 700.4, 551.3], 'generic', False),           # across the right / bottom edges
                ([-100.5, -80.25, 760.7, 560.3], 'generic', False),         # larger than the frame: no clamped pixel
                ([300.37, 200.81, 324.59, 224.13], 'generic', False),       # magnified: 24 px for 128 texels
                ([200.0, 150.0, 328.0, 278.0], 'generic', True),            # integer corners, extent P: every pixel a tie
                ([96.0, 41.0, 352.0, 297.0], 'generic', True),              # integer corners, extent 2P
                ([230.6, 170.3, 402.2, 331.9], 'gate_off', False),
                ([180.4, 120.7, 330.1, 280.6], 'mask_off', False)]
    else:
        rows = [([700.0, 500.0, 800.0, 600.0], 'generic', False),           # entirely off-frame: every pixel clamped
                ([410.3, 120.2, 310.7, 250.9], 'generic', False),           # flipped in x: full-scan path
                ([120.3, 330.2, 220.7, 215.9], 'generic', False),           # flipped in y
                ([260.2, 190.6, 350.1, 280.3], 'generic', False)]
    return [r[0] for r in rows], [r[1] for r in rows], [r[2] for r in rows]


def geometry_random(gen, n, width, height):
    """random viewports around a small frame: across edges, off-frame, larger than it, a tenth flipped on one axis"""
    c = torch.rand(n, 2, generator=gen) * 1.6 - 0.3
    e = torch.rand(n, 2, generator=gen) * 1.4 + 0.1
    wh = torch.tensor([width, height], dtype=torch.float32)
    lo, hi = (c - e / 2) * wh, (c + e / 2) * wh
    vp = torch.cat((lo, hi), dim=1)
    flip = torch.rand(n, generator=gen) < 0.1
    axis = torch.rand(n, generator=gen) < 0.5
    for i in range(n):
        if flip[i]:
            a = 0 if axis[i] else 1
            vp[i, a], vp[i, a + 2] = vp[i, a + 2].clone(), vp[i, a].clone()
    kinds = ['generic'] * n
    kinds[3], kinds[7] = 'gate_off', 'mask_off'
    return vp.tolist(), kinds, [False] * n


def make_target(kind, width, height, gen):
    """(depth, mask) [H,W] fp32"""
    yy, xx = torch.meshgrid(torch.arange(height, dtype=torch.float32), torch.arange(width, dtype=torch.float32),
                            indexing='ij')
    cx, cy, r = 0.52 * width, 0.47 * height, 0.3 * min(width, height)
    rr = ((xx - cx) ** 2 + (yy - cy) ** 2).sqrt()
    disc = (rr <= r).float()
    depth = 1.5 + 0.3 * torch.sin(xx / 17.0) * torch.cos(yy / 13.0)
    if kind == 'empty':                                     # nothing claimed by the mask; depth readings everywhere
        return depth.clone(), torch.zeros(height, width)
    mask = disc.clone()
    depth = depth * disc
    if kind == 'rich':
        band = (yy >= int(cy) - 3) & (yy < int(cy) + 3) & (disc > 0)
        depth[band] = 0.0                                   # sensor holes: no depth under the mask
        ring = (rr > r) & (rr <= 1.3 * r)
        frac = torch.tensor([0.05, 0.3, 0.7, 0.95])[((xx + 2 * yy).long() % 4)]
        mask[ring] = frac[ring]
        ring_depth = 1.5 + 0.2 * torch.rand(height, width, generator=gen)
        ring_depth[(xx.long() % 3) == 0] = 0.0              # 0.05 with no depth is valid, 0.3+ with no depth a hole
        depth[ring] = ring_depth[ring]
    return depth, mask


def loss_case(group, target, seed):
    gen = torch.Generator().manual_seed(seed)
    if group in ('640_128', '640_64'):
        width, height, P = 640, 480, int(group.split('_')[1])
        vps, kinds, exact = geometry_640(P)
    else:
        width, height, P = 97, 61, int(group.split('_')[1])
        vps, kinds, exact = geometry_random(gen, 70, width, height)
    n = len(vps)
    dl, ml = torch.empty(n, P, P), torch.empty(n, P, P)
    for i, k in enumerate(kinds):
        dl[i:i + 1], ml[i:i + 1] = _logits(gen, 1, P, k)
    vp = torch.tensor(vps, dtype=torch.float32)
    tz = 1.5 + 0.1 * torch.randn(n, generator=gen)
    tdepth, tmask = make_target(target, width, height, gen)
    vp, tdepth = _clear_switches(dl, ml, vp, tz, tdepth, tmask, exact)
    return dict(dl=dl, ml=ml, vp=vp, tz=tz, tdepth=tdepth, tmask=tmask, exact=exact, width=width, height=height)


def _fp32_yardstick(c, dev):
    """the product's own fp32 composition (interpret_logits, denormalize_depth, default_pose_loss) on the GPU"""
    from latentfusion_b200 import consts
    from latentfusion_b200.modules.geometry import Camera
    from latentfusion_b200.observation import Observation
    from latentfusion_b200.pose import estimation
    n, W, H = c['dl'].shape[0], c['width'], c['height']
    K = torch.tensor(consts.INTRINSIC, device=dev).unsqueeze(0).expand(n, -1, -1).contiguous()
    vp = c['vp'].to(dev).requires_grad_(True)
    tz = c['tz'].to(dev).requires_grad_(True)
    tr = torch.cat((torch.zeros(n, 2, device=dev), tz[:, None]), dim=1)
    cam = Camera(K, None, Z_SPAN, vp, width=W, height=H, log_quaternion=torch.zeros(n, 3, device=dev), translation=tr)
    full = Camera(K[:1], None, Z_SPAN, None, width=W, height=H, log_quaternion=torch.zeros(1, 3, device=dev),
                  translation=tr[:1].detach())
    target = Observation(torch.zeros(1, 3, H, W, device=dev), c['tdepth'].to(dev).view(1, 1, H, W),
                         c['tmask'].to(dev).view(1, 1, H, W), full)
    dl, ml = c['dl'].to(dev)[:, None], c['ml'].to(dev)[:, None]
    depth = (torch.tanh(dl) + 1) * (torch.sigmoid(ml) > 0.5) - 1
    losses = estimation.default_pose_loss(target, cam.denormalize_depth(depth), ml, cam)
    return torch.stack([losses[k] for k in TERMS], dim=1), vp, tz


def _gterms_list(n, dev):
    out = []
    for k in range(4):
        g = torch.zeros(n, 4, device=dev)
        g[:, k] = 1.0
        out.append((TERMS[k], g))
    out.append(('bench weights', torch.tensor([0.3, 1.0, 0.0, 0.0], device=dev).expand(n, 4) / n))
    return out


# Bounds over the measured fp32 errors (B200, 1000 W): terms 1e-4 relative; logit gradients elementwise against each
# hypothesis' max |fp64| gradient, 1e-3 (measured up to 2.7e-4, at P = 2 where a texel sums ~1500 cancelling pixel
# gradients); viewport / tz through assert_grad_close_to_fp64.
TERMS_RTOL = 1e-4
LOGIT_GRAD_TOL = 1e-3


def _close_terms(ours, ref, what):
    err = ((ours.detach().double() - ref).abs() / ref.abs().clamp(min=1e-30)).max()
    assert float(err) <= TERMS_RTOL, f'{what}: terms relative error {float(err):.3g} > {TERMS_RTOL}'


def _close_logit_grads(ours, ref, what):
    scale = ref.abs().flatten(1).max(dim=1).values.view(-1, 1, 1)
    err = (ours.double() - ref).abs()
    # a hypothesis whose fp64 gradient is exactly 0 (e.g. the depth gate shut everywhere) must get exactly 0
    ratio = torch.where(scale > 0, err / scale.clamp(min=1e-300), err * float('inf'))
    ratio = torch.nan_to_num(ratio, nan=0.0)
    worst = float(ratio.max())
    assert worst <= LOGIT_GRAD_TOL, f'{what}: logit gradient error {worst:.3g} of the max |fp64| > {LOGIT_GRAD_TOL}'


LOSS_CASES = [(g, t) for g in ('640_128', '640_64') for t in ('disc', 'rich', 'empty')] + \
             [(g, t) for g in ('97x61_2', '97x61_33', '97x61_97') for t in ('rich', 'empty')]


@pytest.mark.gpu
@pytest.mark.parametrize('group,target', LOSS_CASES)
def test_loss_head_vs_fp64(dev, group, target):
    """ops.pose_loss_terms, ops.pose_loss_terms_packed and ops.pose_search_terms against the fp64 restatement: the
    terms, and per one-hot term (and the bench's weights) the gradients to both logit maps, the viewport and t_z."""
    from latentfusion_b200 import ops
    c = loss_case(group, target, seed=1000 + LOSS_CASES.index((group, target)))
    n, W, H = c['dl'].shape[0], c['width'], c['height']
    assert_off_switches(c['dl'], c['ml'], c['vp'], c['tz'], c['tdepth'], c['tmask'], c['exact'])
    # fp64 reference (on the GPU: same ATen maths, double precision)
    d64 = {k: c[k].to(dev).double().requires_grad_(True) for k in ('dl', 'ml', 'vp', 'tz')}
    td, tm = c['tdepth'].to(dev), c['tmask'].to(dev)
    ref = loss_head_ref(d64['dl'], d64['ml'], d64['vp'], d64['tz'], td, tm)
    with torch.no_grad():
        ref_search = loss_head_ref(*(d64[k].detach() for k in ('dl', 'ml', 'vp', 'tz')), td, tm, premask=True)
    # kernels: plain, packed (channels-last [N,2,P,P] + translation [N,3])
    k32 = {k: c[k].to(dev).requires_grad_(True) for k in ('dl', 'ml', 'vp', 'tz')}
    terms = ops.pose_loss_terms(k32['dl'], k32['ml'], k32['vp'], k32['tz'], td, tm, Z_SPAN, EPS, W, H)
    lg = torch.stack((c['dl'], c['ml']), dim=1).to(dev).contiguous(memory_format=torch.channels_last).requires_grad_(True)
    P = lg.shape[-1]
    assert lg.stride() == (2 * P * P, 1, 2 * P, 2)                   # the layout the packed path reads in place
    pvp = c['vp'].to(dev).requires_grad_(True)
    ptr = torch.cat((0.01 * torch.ones(n, 2), c['tz'][:, None]), dim=1).to(dev).requires_grad_(True)
    pterms = ops.pose_loss_terms_packed(lg, pvp, ptr, td, tm, Z_SPAN, EPS, W, H)
    sterms = ops.pose_search_terms(c['dl'].to(dev), c['ml'].to(dev), c['vp'].to(dev), c['tz'].to(dev), td, tm,
                                   Z_SPAN, EPS, W, H)
    t32, vp32, tz32 = _fp32_yardstick(c, dev)
    _close_terms(terms, ref.detach(), 'pose_loss_terms')
    _close_terms(pterms, ref.detach(), 'pose_loss_terms_packed')
    _close_terms(sterms, ref_search, 'pose_search_terms')
    for name, gt in _gterms_list(n, dev):
        what = f'{group}/{target}/{name}'
        r_dl, r_ml, r_vp, r_tz = torch.autograd.grad(ref, [d64[k] for k in ('dl', 'ml', 'vp', 'tz')], gt.double(),
                                                     retain_graph=True)
        y_vp, y_tz = torch.autograd.grad(t32, [vp32, tz32], gt, retain_graph=True)
        o_dl, o_ml, o_vp, o_tz = torch.autograd.grad(terms, [k32[k] for k in ('dl', 'ml', 'vp', 'tz')], gt,
                                                     retain_graph=True)
        p_lg, p_vp, p_tr = torch.autograd.grad(pterms, [lg, pvp, ptr], gt, retain_graph=True)
        assert torch.count_nonzero(p_tr[:, :2]) == 0
        for tag, g_dl, g_ml, g_vp, g_tz in (('', o_dl, o_ml, o_vp, o_tz),
                                            (' packed', p_lg[:, 0], p_lg[:, 1], p_vp, p_tr[:, 2])):
            _close_logit_grads(g_dl, r_dl, what + tag + ' d/d depth logits')
            _close_logit_grads(g_ml, r_ml, what + tag + ' d/d mask logits')
            ph.assert_grad_close_to_fp64(g_vp, y_vp, r_vp, what + tag + ' d/d viewport')
            ph.assert_grad_close_to_fp64(g_tz, y_tz, r_tz, what + tag + ' d/d t_z')


def test_loss_head_fp64_restatement_reproduces_the_reference_golden(golden):
    """The fp64 restatement on the golden rendered logits, hypothesis cameras and target gives the reference's own
    loss terms (lfsynth_s16_c8.npz, computed by the unmodified reference in fp32)."""
    g = golden
    dl = g['render.depth_logits'][0, :, 0].double()
    ml = g['render.mask_logits'][0, :, 0].double()
    cam = g.cam('hyp_cam')
    terms = loss_head_ref(dl, ml, cam['viewport'].double(), cam['translation'][:, 2].double(),
                          g['target.depth'][0, 0], g['target.mask'][0, 0])
    for i, k in enumerate(TERMS):
        torch.testing.assert_close(terms[:, i], g[f'loss.{k}'].double(), rtol=1e-4, atol=0)


def test_switch_margins_see_the_switches():
    """The margin checks find what they look for: a half-integer sample coordinate, a gate logit of 0 and a rendered
    depth equal to the target depth."""
    assert bool(_near_tie(0.0, 128.0, 128, 16)[1:].all())              # ix = X - 0.5: a tie from X = 1 on
    assert not bool(_near_tie(0.3, 128.3, 128, 16)[1:].any())
    dl = torch.zeros(1, 4, 4)
    ml = torch.full((1, 4, 4), 20.0)
    vp = torch.tensor([[0.0, 0.0, 8.0, 8.0]])
    tz = torch.tensor([1.5])
    z = 1.5 * torch.sigmoid(torch.tensor(20.0, dtype=torch.float64))      # tanh(0) = 0: the middle of the depth range
    tdepth, tmask = torch.full((8, 8), float(z)), torch.ones(8, 8)
    assert bool(_sign_pixels(dl, ml, vp, tz, tdepth, tmask).all())
    vp2, td2 = _clear_switches(dl, ml, vp, tz, tdepth, tmask, [True])
    assert not bool(_sign_pixels(dl, ml, vp2, tz, td2, tmask).any())
    with pytest.raises(AssertionError, match='gate'):
        assert_off_switches(dl, ml * 0.0, vp2, tz, td2, tmask, [True])


# ---------------------------------------------------------------------------------------------------------------------
# resize (Interpolate) vs F.interpolate in fp64
# ---------------------------------------------------------------------------------------------------------------------
RESIZE_EXTENTS = {
    (2, 2.0): [(1, 1), (1, 2), (2, 5), (7, 6)],
    (2, 0.5): [(2, 2), (3, 5), (7, 6), (2, 9)],
    (3, 2.0): [(1, 1, 1), (1, 2, 3), (3, 4, 5), (2, 6, 1)],
    (3, 0.5): [(2, 2, 2), (3, 5, 2), (5, 4, 7), (6, 3, 9)],
}
RESIZE_TOL = dict(atol=1e-5, rtol=1e-5)


@pytest.mark.gpu
@pytest.mark.parametrize('nd,scale', sorted(RESIZE_EXTENTS))
@pytest.mark.parametrize('mode', ['nearest', 'linear'])
def test_resize_vs_fp64_autograd(dev, nd, scale, mode):
    """ops.interpolate forward and backward against F.interpolate(align_corners=False) in fp64: extents 1, 2, odd and
    even, C in {1, 3, 4, 12} (both kernels), N in {1, 3}, inputs that are not contiguous."""
    from latentfusion_b200 import ops
    torch_mode = mode if mode == 'nearest' else ('bilinear' if nd == 2 else 'trilinear')
    gen = torch.Generator().manual_seed(77)
    for si, ext in enumerate(RESIZE_EXTENTS[(nd, scale)]):
        for C in (1, 3, 4, 12):
            for N in (1, 3):
                # a view of every other element of a wider tensor, or a permuted one: never the dense channels-last
                # layout the kernels read, so the op's own re-layout is exercised forward and backward
                if (si + C) % 2:
                    base = torch.randn(N, C, *ext[:-1], 2 * ext[-1], generator=gen)
                    view = lambda t: t[..., ::2]                                            # noqa: E731
                else:
                    base = torch.randn(*ext[::-1], C, N, generator=gen)
                    view = lambda t: t.permute(nd + 1, nd, *range(nd - 1, -1, -1))       # noqa: E731
                b32 = base.to(dev, copy=True).requires_grad_(True)
                b64 = base.to(dev, torch.float64, copy=True).requires_grad_(True)
                kw = {} if mode == 'nearest' else dict(align_corners=False)
                y64 = F.interpolate(view(b64), scale_factor=scale, mode=torch_mode, **kw)
                y32 = ops.interpolate(view(b32), scale, torch_mode)
                what = f'{nd}d x{scale} {mode} ext={ext} C={C} N={N}'
                assert y32.shape == y64.shape, what
                torch.testing.assert_close(y32.double(), y64.detach(), **RESIZE_TOL, msg=lambda m: f'{what}: {m}')
                gy = torch.randn(y64.shape, generator=gen).to(dev)
                y64.backward(gy.double())
                y32.backward(gy)
                torch.testing.assert_close(b32.grad.double(), b64.grad, **RESIZE_TOL, msg=lambda m: f'{what} grad: {m}')


# ---------------------------------------------------------------------------------------------------------------------
# camera block
# ---------------------------------------------------------------------------------------------------------------------
CAM_NORMS = (0.0, 1e-6, 1e-3, 1.0, math.pi - 1e-3, math.pi, 4.0)


def camera_block_ref(lq, tr, vp, K, z_span, cube_size):
    """fp64 restatement of csrc/camera.cu's chain: qexp (1e-8 clamp) -> normalise twice -> R -> R^T [I | -t], the
    viewport, intrinsics and depth entries of the block (include/lfb200.h)"""
    n = lq.shape[0]
    th = torch.linalg.vector_norm(lq, dim=1, keepdim=True)
    q = torch.cat((torch.cos(th), 1.0 / th.clamp(min=1e-8) * torch.sin(th) * lq), dim=1)
    q = F.normalize(F.normalize(q, dim=1, eps=1e-12), dim=1, eps=1e-12)
    w, x, y, z = q.unbind(1)
    R = torch.stack((1 - 2 * (y * y + z * z), 2 * (x * y - z * w), 2 * (x * z + y * w),
                     2 * (x * y + z * w), 1 - 2 * (x * x + z * z), 2 * (y * z - x * w),
                     2 * (x * z - y * w), 2 * (y * z + x * w), 1 - 2 * (x * x + y * y)), dim=1).view(n, 3, 3)
    Rt = R.transpose(1, 2)
    m = torch.cat((Rt, -(Rt @ tr[:, :, None])), dim=2).reshape(n, 12)
    vpe = torch.stack((vp[:, 0], vp[:, 1], vp[:, 2] - vp[:, 0], vp[:, 3] - vp[:, 1]), dim=1)
    ke = torch.stack((K[:, 0, 2], K[:, 1, 2], K[:, 0, 0], K[:, 1, 1]), dim=1)
    const = torch.tensor([z_span, cube_size / 2], dtype=lq.dtype, device=lq.device).expand(n, 2)
    from latentfusion_b200._lib import CAM_STRIDE
    return torch.cat((m, vpe, ke, (tr[:, 2] - z_span)[:, None], const,
                      torch.zeros(n, CAM_STRIDE - 23, dtype=lq.dtype, device=lq.device)), dim=1)


@pytest.mark.gpu
def test_camera_block_vs_fp64(dev):
    """lf_camera_o2c_fwd / _bwd at |log q| in {0, 1e-6, 1e-3, 1, pi-1e-3, pi, 4} in random directions, N = 130 (three
    64-thread blocks), random upstream gradients on block entries 0-15 and 20."""
    from latentfusion_b200 import consts, ops
    from latentfusion_b200.modules.geometry import Camera
    gen = torch.Generator().manual_seed(31)
    n = 130
    u = torch.randn(n, 3, generator=gen)
    u = u / u.norm(dim=1, keepdim=True)
    lq = u * torch.tensor(CAM_NORMS)[torch.arange(n) % len(CAM_NORMS)][:, None]
    tr = torch.randn(n, 3, generator=gen) * 0.2 + torch.tensor([0.0, 0.0, 1.5])
    vp = torch.tensor([200.0, 150.0, 328.0, 278.0]) + torch.randn(n, 4, generator=gen) * 20
    K = torch.tensor(consts.INTRINSIC).unsqueeze(0).repeat(n, 1, 1) + torch.randn(n, 3, 4, generator=gen) * \
        torch.tensor([[5.0, 0, 3.0, 0], [0, 5.0, 3.0, 0], [0, 0, 0, 0]])
    gb = torch.zeros(n, 40)
    gb[:, :16] = torch.randn(n, 16, generator=gen)
    gb[:, 20] = torch.randn(n, generator=gen)
    z_span, cube = 0.5, 1.0

    p64 = [t.double().requires_grad_(True) for t in (lq, tr, vp)]
    b64 = camera_block_ref(*p64, K.double(), z_span, cube)
    g64 = torch.autograd.grad(b64, p64, gb.double())
    # fp32 yardstick: the product's differentiable torch camera algebra on the CPU
    p32 = [t.clone().requires_grad_(True) for t in (lq, tr, vp)]
    cam = Camera(K.clone(), None, z_span, p32[2], log_quaternion=p32[0], translation=p32[1])
    b32 = cam.o2c_block(cube)
    g32 = torch.autograd.grad(b32, p32, gb)
    # the kernels
    pk = [t.to(dev).requires_grad_(True) for t in (lq, tr, vp)]
    bk = ops.camera_o2c_block(*pk, K.to(dev), z_span, cube)
    gk = torch.autograd.grad(bk, pk, gb.to(dev))
    fwd_err = float((bk.cpu().double() - b64.detach()).abs().max())
    fwd_err32 = float((b32.detach().double() - b64.detach()).abs().max())
    assert fwd_err <= max(3 * fwd_err32, 1e-6), f'block |ours - fp64| = {fwd_err:.3g} (fp32 chain {fwd_err32:.3g})'
    for name, o, y, r in zip(('log_quaternion', 'translation', 'viewport'), gk, g32, g64):
        assert torch.isfinite(o).all(), name
        ph.assert_grad_close_to_fp64(o.cpu(), y, r, name)
        # per norm class as well: a wrong branch at |log q| = 0 or pi must not hide behind the other rows' scale
        for j, nrm in enumerate(CAM_NORMS):
            rows = torch.arange(j, n, len(CAM_NORMS))
            ph.assert_grad_close_to_fp64(o.cpu()[rows], y[rows], r[rows], f'{name} at |log q| = {nrm:.6g}')


# ---------------------------------------------------------------------------------------------------------------------
# batched Adam + ReduceLROnPlateau
# ---------------------------------------------------------------------------------------------------------------------
STEPS, ROWS, THRESHOLD, LR0 = 150, 37, 1e-4, 2.0 ** -7      # LR0 exact in fp32, so factor 0.5 keeps it exact


def rank_loss_sequences(gen):
    """[STEPS, ROWS] fp32: improving, flat, oscillating, improving by 10x and by 0.4x the threshold per step (the
    latter counts as better every third step)"""
    k = torch.arange(STEPS, dtype=torch.float64)[:, None]
    r = torch.arange(ROWS, dtype=torch.float64)[None, :]
    kind = torch.arange(ROWS) % 5
    scale = 1.0 + 0.01 * r
    seq = torch.where(kind == 0, scale * 0.97 ** k,
          torch.where(kind == 1, scale.expand(STEPS, ROWS),
          torch.where(kind == 2, scale * (1.0 + 0.3 * torch.sin(0.9 * k + r)),
          torch.where(kind == 3, scale * (1.0 - 10 * THRESHOLD) ** k, scale * (1.0 - 0.4 * THRESHOLD) ** k))))
    return seq.float()


def assert_off_threshold(seq):
    """no step compares within 1e-5 relative of the threshold boundary best * (1 - threshold)"""
    best = torch.full((ROWS,), float('inf'), dtype=torch.float64)
    for m in seq.double():
        bound = best * (1 - THRESHOLD)
        fin = torch.isfinite(best)
        assert bool(((m[fin] - bound[fin]).abs() > 1e-5 * bound[fin]).all()), 'a loss sits at the plateau threshold'
        best = torch.where(m < bound, m, best)


def run_adam_plateau(device, patience, factor, seed):
    from latentfusion_b200.pose.refine_graph import _BatchedAdamPlateau
    gen = torch.Generator().manual_seed(seed)
    p0 = [torch.randn(ROWS, w, generator=gen) for w in (3, 3, 4)]
    grads = [torch.randn(STEPS, ROWS, w, generator=gen) * 0.3 for w in (3, 3, 4)]
    seq = rank_loss_sequences(gen)
    assert_off_threshold(seq)
    # the batched optimiser (device branch on a GPU, torch branch on the CPU)
    params = [p.clone().to(device) for p in p0]
    opt = _BatchedAdamPlateau(params, ROWS, LR0, patience, THRESHOLD, factor)
    lr_hist = []
    for s in range(STEPS):
        for p, g in zip(params, grads):
            p.grad = g[s].to(device)
        opt.step(seq[s].to(device))
        lr_hist.append(opt.lr.view(-1).cpu().double())
    lr_hist = torch.stack(lr_hist)
    # N independent fp64 torch optimisers + schedulers
    ref_lr = torch.empty(STEPS, ROWS, dtype=torch.float64)
    ref_p = []
    for i in range(ROWS):
        ps = [p[i].double().clone().requires_grad_(True) for p in p0]
        adam = torch.optim.Adam(ps, lr=LR0)
        sched = torch.optim.lr_scheduler.ReduceLROnPlateau(adam, mode='min', factor=factor, patience=patience,
                                                           threshold=THRESHOLD, threshold_mode='rel')
        for s in range(STEPS):
            for p, g in zip(ps, grads):
                p.grad = g[s, i].double()
            adam.step()
            sched.step(float(seq[s, i]))
            ref_lr[s, i] = adam.param_groups[0]['lr']
        ref_p.append([p.detach() for p in ps])
    ref_p = [torch.stack([rp[j] for rp in ref_p]) for j in range(3)]
    return [p.detach().cpu().double() for p in params], lr_hist, ref_p, ref_lr


ADAM_PARAM_TOL = dict(atol=2e-5, rtol=1e-5)


def check_adam_plateau(device, patience, factor):
    ours, lr, ref_p, ref_lr = run_adam_plateau(device, patience, factor, seed=int(patience * 10 + factor * 100))
    reductions = (ref_lr[-1] < LR0).sum()
    assert int(reductions) > 0, 'no learning rate was lowered'
    if factor == 0.5:
        assert torch.equal(lr, ref_lr), f'lr differs first at step {int((lr != ref_lr).any(1).nonzero()[0])}'
    else:
        torch.testing.assert_close(lr, ref_lr, atol=0, rtol=1e-6)
    for o, r in zip(ours, ref_p):
        torch.testing.assert_close(o, r, **ADAM_PARAM_TOL)


@pytest.mark.gpu
@pytest.mark.parametrize('patience', [0, 2, 10])
@pytest.mark.parametrize('factor', [0.5, 0.1])
def test_adam_plateau_kernels_vs_fp64_torch(dev, patience, factor):
    """lf_adam_step + lf_plateau_step over 150 steps and 37 rows against 37 fp64 torch.optim.Adam +
    ReduceLROnPlateau pairs: every row's learning rate at every step, and the parameters at the end."""
    check_adam_plateau(dev, patience, factor)


@pytest.mark.parametrize('patience', [0, 2, 10])
@pytest.mark.parametrize('factor', [0.5, 0.1])
def test_adam_plateau_torch_branch_vs_fp64_torch(patience, factor):
    """The same on _BatchedAdamPlateau's CPU (torch) branch."""
    check_adam_plateau(torch.device('cpu'), patience, factor)
