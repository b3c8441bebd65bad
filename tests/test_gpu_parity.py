"""GPU parity tests: the sm_100a path (through the C ABI) vs golden vectors from the unmodified
reference and vs the CPU oracle on seeded inputs.  fp32 tolerances per SURVEY.md §4-4:
outputs atol 1e-4 / rtol 1e-3, camera gradients rtol 2e-3."""
import json

import pytest
import torch

from tests import parity_helpers as ph
from tests.parity_helpers import OUT_TOL, GRAD_TOL

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def g():
    return ph.Golden()


@pytest.fixture(scope='module')
def dev():
    assert torch.cuda.is_available(), "GPU tests need a CUDA device"
    return torch.device('cuda:0')


def test_o2c_resample_vs_golden(g, dev):
    from latentfusion_b200.modules.geometry import ObjectToCameraTransform
    cam = ph.product_camera(g.cam('hyp_cam'), dev, requires_grad=True)
    vol = g['o2c.vol'].to(dev).requires_grad_(True)
    out = ObjectToCameraTransform(1.0)(vol, cam)
    assert out.shape == g['o2c.out'].shape
    torch.testing.assert_close(out.cpu(), g['o2c.out'], **OUT_TOL)
    (out * g['o2c.w'].to(dev)).sum().backward()
    torch.testing.assert_close(vol.grad.cpu(), g['o2c.grad_vol'], **OUT_TOL)
    for k in ('log_quaternion', 'translation', 'viewport'):
        torch.testing.assert_close(getattr(cam, k).grad.cpu(), g[f'o2c.grad_{k}'], atol=1e-3, rtol=2e-3)


def test_c2o_resample_vs_golden(g, dev):
    from latentfusion_b200.modules.geometry import CameraToObjectTransform
    cam = ph.product_camera(g.cam('ref_cam'), dev)
    vol = g['c2o.vol'].to(dev).requires_grad_(True)
    out = CameraToObjectTransform(1.0)(vol, cam)
    torch.testing.assert_close(out.cpu(), g['c2o.out'], **OUT_TOL)
    (out * g['c2o.w'].to(dev)).sum().backward()
    torch.testing.assert_close(vol.grad.cpu(), g['c2o.grad_vol'], **OUT_TOL)


@pytest.mark.parametrize('C,S,N', [(8, 16, 3), (32, 24, 2), (6, 9, 2), (1, 10, 2), (64, 12, 2), (16, 20, 2), (32, 33, 2)])
def test_o2c_vs_oracle_shapes(dev, C, S, N):
    """channel counts hitting the depth-marching kernel (C in 16/32/64, incl. S not a multiple of the tile), the
    brick kernel's float4 path (other C%4==0), its scalar path and multi-chunk groups."""
    from oracle import lf_oracle as O
    from latentfusion_b200.modules.geometry import ObjectToCameraTransform
    cams, _ = ph.synthetic_cameras(N, S, seed=C)
    d = ph.cam_to_dict(cams)
    torch.manual_seed(S)
    vol = torch.randn(1, C, S, S, S)
    w = torch.randn(N, C, S, S, S)

    def oracle_grads(dtype):
        with ph.oracle_dtype(dtype):
            ocam = ph.oracle_camera({k: v.to(dtype) for k, v in d.items()}, requires_grad=True)
            ref = O.object_to_camera(vol.to(dtype), ocam)
            (ref * w.to(dtype)).sum().backward()
            return ref.detach(), torch.cat([ocam.log_quaternion.grad, ocam.translation.grad, ocam.viewport.grad], 1)

    ref32, g32 = oracle_grads(torch.float32)
    _, g64 = oracle_grads(torch.float64)
    cam = ph.product_camera(d, dev, requires_grad=True)
    out = ObjectToCameraTransform(1.0)(vol.to(dev), cam)
    # white-noise volumes are the worst case for coordinate rounding (|d out / d coord| ~ S); the camera
    # sits ~20-30 m away at these tiny S, so 1 ulp of the projected coordinate is ~1e-5 voxel
    torch.testing.assert_close(out.cpu(), ref32, atol=5e-4, rtol=1e-3)
    (out * w.to(dev)).sum().backward()
    ours = torch.cat([cam.log_quaternion.grad, cam.translation.grad, cam.viewport.grad], 1).cpu()
    ph.assert_grad_close_to_fp64(ours, g32, g64, f'o2c camera grads C={C} S={S}')


@pytest.mark.parametrize('C,S,V', [(16, 12, 3), (32, 17, 2), (64, 8, 2)])
def test_c2o_vs_oracle_shapes(dev, C, S, V):
    """camera->object resample on the depth-marching kernel against the oracle (distinct source cube per view)."""
    from oracle import lf_oracle as O
    from latentfusion_b200.modules.geometry import CameraToObjectTransform
    cams, _ = ph.synthetic_cameras(V, S, seed=C + 1, perturb=False)
    d = ph.cam_to_dict(cams)
    torch.manual_seed(S)
    vol = torch.randn(V, C, S, S, S)
    ref = O.camera_to_object(vol, ph.oracle_camera(d))
    out = CameraToObjectTransform(1.0)(vol.to(dev), ph.product_camera(d, dev))
    torch.testing.assert_close(out.cpu(), ref, atol=5e-4, rtol=1e-3)


def test_march_and_brick_resamplers_agree_at_full_size(dev):
    """the two forward kernels (depth-marching with register-resident corners / brick gather) evaluate the same
    weights and corners and differ only in the order of the 8-term sum."""
    import os
    from latentfusion_b200.modules.geometry import ObjectToCameraTransform, CameraToObjectTransform
    S, C, N = 64, 32, 8
    cams, _ = ph.synthetic_cameras(N, S, seed=5)
    cam = cams.to(dev)
    torch.manual_seed(1)
    vol = torch.randn(1, C, S, S, S, device=dev)
    vols = torch.randn(N, C, S, S, S, device=dev)
    march = (ObjectToCameraTransform(1.0)(vol, cam), CameraToObjectTransform(1.0)(vols, cam))
    from latentfusion_b200 import _lib as L
    L.check(L.lib().lf_set_option(b'LFB200_RESAMPLE_BRICK', 1), 'set_option')     # (the env var is only read at load time)
    try:
        brick = (ObjectToCameraTransform(1.0)(vol, cam), CameraToObjectTransform(1.0)(vols, cam))
    finally:
        L.lib().lf_set_option(b'LFB200_RESAMPLE_BRICK', 0)
    for a, b in zip(march, brick):
        torch.testing.assert_close(a, b, atol=2e-6, rtol=1e-5)


def test_march_and_brick_camera_gradients_agree_at_full_size(dev):
    """the two camera-gradient kernels (depth-marching with per-lane column sums / brick gather with per-voxel
    reductions) evaluate the same corners, weights and chain rule and differ only in summation order."""
    from latentfusion_b200 import _lib as L, ops
    S, C, N = 64, 32, 8
    cams, _ = ph.synthetic_cameras(N, S, seed=5)
    blk = cams.to(dev).o2c_block(1.0)
    torch.manual_seed(2)
    # a smooth cube plus noise: the terms of the camera gradient then do not cancel to rounding level
    lin = torch.linspace(-1, 1, S, device=dev)
    vol = (torch.sin(3 * lin)[None, None, :, None, None] * torch.cos(2 * lin)[None, None, None, :, None]
           * lin[None, None, None, None, :] + 0.1 * torch.randn(1, C, S, S, S, device=dev))
    w = torch.randn(N, C, S, S, S, device=dev)
    grads = []
    for opt in (0, 2, 1):
        L.check(L.lib().lf_set_option(b'LFB200_BWDCAM', opt), 'set_option')
        try:
            b = blk.clone().requires_grad_(True)
            (ops.resample_o2c(vol, b) * w).sum().backward()
            grads.append(b.grad.clone())
        finally:
            L.lib().lf_set_option(b'LFB200_BWDCAM', 0)
    scale = grads[2].abs().amax(0, keepdim=True).clamp_min(1e-6)
    for gm in grads[:2]:
        assert ((gm - grads[2]).abs() / scale).max().item() < 2e-4


def test_o2c_bwd_cam_is_deterministic(dev):
    from latentfusion_b200.modules.geometry import ObjectToCameraTransform
    cams, _ = ph.synthetic_cameras(4, 32, seed=1)
    d = ph.cam_to_dict(cams)
    torch.manual_seed(0)
    vol = torch.randn(1, 16, 32, 32, 32, device=dev)
    w = torch.randn(4, 16, 32, 32, 32, device=dev)
    grads = []
    for _ in range(2):
        cam = ph.product_camera(d, dev, requires_grad=True)
        (ObjectToCameraTransform(1.0)(vol, cam) * w).sum().backward()
        grads.append(torch.cat([cam.log_quaternion.grad, cam.translation.grad, cam.viewport.grad], 1))
    assert torch.equal(grads[0], grads[1])


def test_pose_loss_and_resize_backward_are_deterministic(dev):
    """The refine iteration's other reductions add in a fixed order too: the fused pose-loss head (terms, gradients to
    the logits, viewport and translation) and the bilinear resize backward give the same bits on every call."""
    from latentfusion_b200 import ops
    cams, _ = ph.synthetic_cameras(8, 64, seed=3)
    cam = cams.to(dev)
    torch.manual_seed(0)
    logits = torch.randn(8, 128, 128, 2, device=dev)          # channels-last [N,2,P,P] as the fused heads write them
    yy, xx = torch.meshgrid(torch.arange(480.0, device=dev), torch.arange(640.0, device=dev), indexing='ij')
    tmask = (((yy - 251.5) ** 2 + (xx - 315.4) ** 2) <= 45.0 ** 2).float().view(1, 1, 480, 640)
    tdepth = tmask * float(cam.translation[0, 2])
    gterms = torch.rand(8, 4, device=dev)
    x0 = torch.randn(8, 64, 64, 64, device=dev)
    gy = torch.randn(8, 64, 128, 128, device=dev)
    runs = []
    for _ in range(2):
        lg = logits.clone().requires_grad_(True)
        vp = cam.viewport.detach().clone().requires_grad_(True)
        tr = cam.translation.detach().clone().requires_grad_(True)
        terms = ops.pose_loss_terms_packed(lg.permute(0, 3, 1, 2), vp, tr, tdepth, tmask, cam.z_span)
        terms.backward(gterms)
        x = x0.clone().requires_grad_(True)
        ops.interpolate(x, 2.0, 'bilinear').backward(gy)
        runs.append((terms.detach(), lg.grad, vp.grad, tr.grad, x.grad))
    for name, a, b in zip(('terms', 'd/dlogits', 'd/dviewport', 'd/dtranslation', 'resize d/dx'), *runs):
        assert torch.equal(a, b), name


@pytest.mark.parametrize('name,conv,scale,mode', [('blk3d_same', 3, 1.0, 'nearest'), ('blk3d_up', 3, 2.0, 'nearest'),
                                                  ('blk3d_down', 3, 0.5, 'nearest'), ('blk2d_up', 2, 2.0, 'bilinear'),
                                                  ('blk2d_down', 2, 0.5, 'bilinear')])
@pytest.mark.parametrize('precision', [0, 1])
def test_conv_block_vs_golden(g, dev, name, conv, scale, mode, precision, monkeypatch):
    """precision 1 = the tcgen05 bf16x3 kernels where the shape is covered (Cin % 4 == 0), same tolerances."""
    from latentfusion_b200 import ops
    from latentfusion_b200.modules import EqualizedConv2d, EqualizedConv3d
    from latentfusion_b200.modules.blocks import Block
    monkeypatch.setattr(ops, '_default_precision', precision)
    sd = g.state_dict(name)
    cout, cin = sd['conv1.module.weight'].shape[:2]
    blk = Block(cin, cout, conv_module=EqualizedConv3d if conv == 3 else EqualizedConv2d,
                scale_factor=scale, scale_mode=mode)
    blk.load_state_dict(sd, strict=True)
    blk = blk.to(dev)
    x = g[f'{name}.x'].to(dev).requires_grad_(True)
    y = blk(x)
    torch.testing.assert_close(y.cpu(), g[f'{name}.y'], **OUT_TOL)
    (y * g[f'{name}.w'].to(dev)).sum().backward()
    torch.testing.assert_close(x.grad.cpu(), g[f'{name}.grad_x'], atol=2e-4, rtol=2e-3)
    for k, p in blk.named_parameters():
        torch.testing.assert_close(p.grad.cpu(), g[f'{name}.grad/{k}'], atol=2e-3, rtol=2e-3)


def test_sculptor_and_fusers_vs_golden(g, dev):
    from latentfusion_b200.recon import fusion
    sculptor, fuser, _ = ph.build_product_models(g, dev)
    cam = ph.product_camera(g.cam('ref_cam'), dev)
    color, mask = g['color'].to(dev), g['mask'].to(dev)
    with torch.no_grad():
        x = torch.cat((color.flatten(0, 1), mask.flatten(0, 1) * 2 - 1), dim=1)
        z, z_cam_mid, _ = sculptor(x, cam)
        torch.testing.assert_close(*g.sampled('z_views', z.cpu()), **OUT_TOL)
        torch.testing.assert_close(*g.sampled('z_cam_mid0', z_cam_mid[-1].cpu()), **OUT_TOL)
        for kind in ('max', 'mean', 'median', 'abs_max'):
            zp, _ = sculptor.encode(fusion.get_fuser(f'pool:{kind}', g.meta['C'], 1.0), cam, color, mask=mask)
            torch.testing.assert_close(*g.sampled(f'z_obj_pool_{kind}', zp.cpu()), **OUT_TOL)
        zg, _ = sculptor.encode(fuser, cam, color, mask=mask)
        torch.testing.assert_close(zg.cpu(), g['z_obj_gru'], atol=2e-4, rtol=2e-3)


def test_lstm_and_concat_fusers_vs_golden(dev):
    """recon/fusion.py:87-92 (ConcatFuser) and :204-246 (LSTMFuser, ConvLSTMCell) against the unmodified reference:
    reference-format state_dict loads strictly; forward at the exact-fp32 and bf16x3 settings; backward to the
    per-view cubes at exact fp32."""
    import os
    from latentfusion_b200 import ops
    from latentfusion_b200.recon import fusion
    gf = ph.Golden(os.path.join(ph.ROOT, 'tests', 'golden', 'fusers_c8_s10.npz'))
    C = gf.meta['C']
    lstm = fusion.get_fuser('lstm', in_channels=C, cube_size=1.0)
    lstm.load_state_dict(gf.state_dict('lstm'), strict=True)
    lstm = lstm.to(dev)
    z = gf['z_obj'].to(dev)
    old = ops.get_default_precision()
    try:
        for precision in (0, 1):
            ops.set_default_precision(precision)
            with torch.no_grad():
                out, _ = lstm(z, None, None, None)
            torch.testing.assert_close(out.cpu(), gf['fused.lstm'], **OUT_TOL)
        ops.set_default_precision(0)
        zt = z.clone().requires_grad_(True)
        out, _ = lstm(zt, None, None, None)
        (out * gf['lstm.w'].to(dev)).sum().backward()
        torch.testing.assert_close(zt.grad.cpu(), gf['lstm.grad_z'], **GRAD_TOL)
    finally:
        ops.set_default_precision(old)
    cat, _ = fusion.get_fuser('concat', in_channels=C, cube_size=1.0)(z, None, None, None)
    assert torch.equal(cat.cpu(), gf['fused.concat'])


def test_blend_fuser_vs_golden(dev):
    """recon/fusion.py:95-149 (BlendFuser: UNet3d on [z_cam, depth coordinate] -> camera->object resample -> softmax over
    the views -> weighted sum) against the unmodified reference's output; strict state_dict load."""
    import os
    from latentfusion_b200.recon import fusion
    from latentfusion_b200.utils import parse_block_config as pbc
    gf = ph.Golden(os.path.join(ph.ROOT, 'tests', 'golden', 'fusers_c8_s10.npz'))
    blend = fusion.get_fuser('blend', in_channels=gf.meta['C'], cube_size=1.0, block_config=pbc(gf.text('blend.cfg')))
    blend.load_state_dict(gf.state_dict('blend'), strict=True)
    blend = blend.to(dev)
    cam = ph.product_camera(gf.cam('blend.cam'), dev)
    with torch.no_grad():
        fused, extra = blend(gf['blend.z_obj'].to(dev), [gf['blend.z_cam'].to(dev)], None, cam)
    torch.testing.assert_close(extra['blend_weights'].cpu(), gf['blend.weights'], **OUT_TOL)
    torch.testing.assert_close(fused.cpu(), gf['fused.blend'], **OUT_TOL)


def test_render_loss_and_camera_grads_vs_golden(g, dev):
    ph.smoke_check()


def test_gradient_estimator_three_iterations_vs_golden(g, dev):
    """GradientPoseEstimator (adam_quick.toml args) reproduces the reference's camera trajectory."""
    from latentfusion_b200.pose import estimation
    from latentfusion_b200.observation import Observation
    from latentfusion_b200.recon.inference import LatentFusionModel
    sculptor, fuser, photographer = ph.build_product_models(g, dev)
    model = LatentFusionModel(sculptor, fuser, photographer, g.meta['camera_dist'], dev)
    cfg = {'type': 'gradient', 'args': dict(optimizer='adam', num_iters=100, num_samples=8, ranking_size=8,
                                            learning_rate=0.01, lr_reduce_patience=10, lr_reduce_threshold=1e-4,
                                            converge_threshold=1e-6, converge_patience=10),
           'loss_weights': dict(depth=1.0, ov_depth=0.3, iou=0.0, mask=0.0, latent=0.0)}
    N = g.meta['N']
    est = estimation.load_from_config(cfg, model, num_samples=N, ranking_size=N, num_iters=3, track_stats=True,
                                      return_camera_history=True)
    gt = ph.product_camera(g.cam('ref_cam_full'), 'cpu')[0:1]
    target = Observation(torch.zeros(1, 3, 480, 640), g['target.depth'], g['target.mask'], gt)
    init = ph.product_camera(g.cam('est.init_cam'), 'cpu')
    best, stats, history = est.estimate(g['z_obj_gru'].to(dev), target, camera=init)
    torch.testing.assert_close(stats['rank_loss'], g['est.rank_loss'], atol=1e-3, rtol=1e-3)
    for i, (_, cams) in enumerate(history):
        for k in ('log_quaternion', 'translation'):
            torch.testing.assert_close(getattr(cams, k), g[f'est.hist{i}.{k}'], atol=2e-4, rtol=1e-3)
    torch.testing.assert_close(best.translation, g['est.best_cam.translation'], atol=2e-4, rtol=1e-3)


def test_cross_entropy_estimator_runs_on_the_cuda_path(g, dev):
    """Coarse pose search (reference pose/estimation.py:300-470, configs/cross_entropy_latent.toml scaled down):
    GMM proposals on the host, every render + the target's latent code on the lfb200 kernels, forward only."""
    import numpy as np
    from latentfusion_b200 import ops
    from latentfusion_b200.pose import estimation, utils as pu
    from latentfusion_b200.observation import Observation
    from latentfusion_b200.recon.inference import LatentFusionModel
    sculptor, fuser, photographer = ph.build_product_models(g, dev)
    model = LatentFusionModel(sculptor, fuser, photographer, g.meta['camera_dist'], dev)
    cfg = {'type': 'cross_entropy',
           'args': dict(num_samples=8, num_iters=2, ranking_size=4, num_elites=4, num_gmm_components=2,
                        learning_rate=0.3, sample_flipped=True, init_hemisphere=False, init_upright=False),
           'loss_weights': dict(depth=0.0, ov_depth=0.0, iou=0.0, mask=0.0, latent=1.0)}
    est = estimation.load_from_config(cfg, model, return_camera_history=True)
    gt = ph.product_camera(g.cam('ref_cam_full'), 'cpu')[0:1]
    torch.manual_seed(5)
    np.random.seed(5)
    target = Observation(torch.rand(1, 3, 480, 640), g['target.depth'], g['target.mask'], gt)
    cams = pu.sample_cameras_with_estimate(n=16, camera_est=gt)
    ops.KernelTrace.reset(False)
    best, history = est.estimate(g['z_obj_gru'].to(dev), target, cameras=cams)
    assert 1 <= len(best) <= 4
    assert ops.KernelTrace.launches > 40             # the renders + the target autoencode went through the C ABI
    for losses, ranked in history:
        assert torch.isfinite(losses).all()
        assert torch.isfinite(ranked.translation).all() and torch.isfinite(ranked.log_quaternion).all()


@pytest.mark.parametrize('precision', [0, 1])
def test_config_a_render_vs_oracle(dev, precision, monkeypatch):
    """BASELINE config 1 shape (V=4, S=32, C=16, N=2): CUDA path vs the CPU oracle, fwd + camera grads, on the exact
    FFMA kernels (0) and on the tcgen05 bf16x3 kernels (1)."""
    from oracle import lf_oracle as O
    from latentfusion_b200 import ops
    from latentfusion_b200.recon.inference import LatentFusionModel
    monkeypatch.setattr(ops, '_default_precision', precision)
    S, C, V, N = 32, 16, 4, 2
    sculptor, fuser, photographer, arch, sds = ph.random_lfsynth(S, C, seed=3, device=dev)
    ref_cams, dist = ph.synthetic_cameras(V, S, seed=4, perturb=False)
    hyp_cams, _ = ph.synthetic_cameras(N, S, seed=5)
    torch.manual_seed(6)
    color = torch.rand(1, V, 3, 2 * S, 2 * S) * 2 - 1
    mask = (torch.rand(1, V, 1, 2 * S, 2 * S) > 0.3).float()
    model = LatentFusionModel(sculptor, fuser, photographer, dist, dev)
    with torch.no_grad():
        z_obj, _ = sculptor.encode(fuser, ref_cams.to(dev), color.to(dev), mask=mask.to(dev))
        z_ref = O.sculptor_encode(sds['sculptor'], arch['sculptor'], 'gru', sds['fuser'],
                                  ph.oracle_camera(ph.cam_to_dict(ref_cams)), color, mask)
    torch.testing.assert_close(z_obj.cpu(), z_ref, atol=2e-4, rtol=2e-3)
    d = ph.cam_to_dict(hyp_cams)
    cam = ph.product_camera(d, dev, requires_grad=True)
    y, latent = model.render_latent_object(z_obj, cam)
    ocam = ph.oracle_camera(d, requires_grad=True)
    logits, olat = O.photographer_forward(sds['photographer'], arch['photographer'], z_ref[0], ocam)
    torch.testing.assert_close(y['depth_logits'].cpu()[0], logits[:, 0:1].detach(), atol=2e-4, rtol=2e-3)
    torch.testing.assert_close(y['mask_logits'].cpu()[0], logits[:, 1:2].detach(), atol=2e-4, rtol=2e-3)
    torch.testing.assert_close(latent.cpu(), olat.detach(), atol=2e-4, rtol=2e-3)
    torch.manual_seed(7)
    w = torch.randn_like(logits)
    (logits * w).sum().backward()
    g32 = torch.cat([ocam.log_quaternion.grad, ocam.translation.grad, ocam.viewport.grad], 1)
    with ph.oracle_dtype(torch.float64):
        o64 = ph.oracle_camera({k: v.double() for k, v in d.items()}, requires_grad=True)
        sd64 = {k: v.double() for k, v in sds['photographer'].items()}
        l64, _ = O.photographer_forward(sd64, arch['photographer'], z_ref[0].double(), o64)
        (l64 * w.double()).sum().backward()
        g64 = torch.cat([o64.log_quaternion.grad, o64.translation.grad, o64.viewport.grad], 1)
    out = torch.cat((y['depth_logits'][0], y['mask_logits'][0]), dim=1)
    (out * w.to(dev)).sum().backward()
    ours = torch.cat([cam.log_quaternion.grad, cam.translation.grad, cam.viewport.grad], 1).cpu()
    # (two fp32 evaluations of the same cancelling sum: the bf16x3 path measured 3.2x, the exact path 2.1x)
    ph.assert_grad_close_to_fp64(ours, g32, g64, 'config-A camera grads', factor=4.0)


# camera-gradient bound (fraction of the gradient scale, vs the reference's fp64 run) per cube kind: see the docstring
_CFGB_GRAD_BOUND = {'white': 5e-2, 'smooth': 1.5e-2}


@pytest.mark.parametrize('cube', ['smooth', 'white'])
@pytest.mark.parametrize('precision', [1, 0, 2])
def test_config_b_render_loss_grads_vs_reference_golden(dev, precision, cube):
    """The BENCHMARKED configuration (BASELINE configs[1]: S=64, C=32, 128^2) at the BENCHMARKED precision
    (1 = tcgen05 bf16x3; 0 = exact FFMA kernels; 2 = plain bf16 operands) against goldens written by the UNMODIFIED
    reference (oracle/make_golden_configB.py) in fp32 and in fp64, for two object cubes: white noise (worst case) and
    the same noise low-pass filtered (a spatially smooth latent).

    Outputs (logits, projected latent, the four loss terms through the fused loss head): atol 5e-4 / rtol 1e-3 vs the
    fp32 golden (the reference's own fp32-vs-fp64 difference on the logits is 1.1e-4 / 4e-5 abs); precision 2: 5e-2.

    Camera gradients are cancelling sums over 2M trilinear samples whose derivative jumps at every cell boundary, so
    ANY fp32 evaluation carries noise proportional to its ~1e-5-voxel coordinate rounding.  Measured against the
    fp64 golden, as a fraction of the gradient scale (log-quaternion / translation / viewport):
        white :  reference CPU fp32 2.1e-2 / 0.9e-2 / 0.5e-2;  reference algorithm in ATen CUDA fp32 1.9e-2 / 1.8e-2 / 0.9e-2;
                 lfb200 precision 0: 2.5e-2 / 3.9e-2 / 1.4e-2;  precision 1: 2.6e-2 / 3.8e-2 / 1.5e-2
        smooth:  reference CPU fp32 2.2e-3 / 0.7e-3 / 1.6e-3;  ATen CUDA fp32 0.4e-3 / 2.4e-3 / 2.4e-3;
                 lfb200 precision 0: 2.6e-3 / 5.2e-3 / 7.5e-3;  precision 1: 2.1e-3 / 6.4e-3 / 9.8e-3
    (tools/grad_probe*.py; the exact-FFMA and the bf16x3 paths are equally close, i.e. the split-bf16 tensor-core
    arithmetic is not what limits the gradients; half of lfb200's deviation is the camera block being rounded to fp32
    before the resampler differentiates it.)  Bounds asserted: 5e-2 (white), 1.5e-2 (smooth) of the gradient scale."""
    from latentfusion_b200 import ops
    old = ops.get_default_precision()
    ops.set_default_precision(precision)
    try:
        g, model, z_obj, target = ph.config_b_case(dev, smooth=(cube == 'smooth'))
        cam = ph.product_camera(g.cam('hyp_cam'), dev, requires_grad=True)
        ops.KernelTrace.reset(False)
        y, latent = model.render_latent_object(z_obj, cam, return_latent=True, apply_mask=True)
        assert ops.KernelTrace.launches > 10
        tol = dict(atol=5e-4, rtol=1e-3) if precision != 2 else dict(atol=5e-2, rtol=5e-2)
        torch.testing.assert_close(y['depth_logits'].cpu(), g['render.depth_logits'], **tol)
        torch.testing.assert_close(y['mask_logits'].cpu(), g['render.mask_logits'], **tol)
        torch.testing.assert_close(latent.cpu()[..., ::4, ::4], g['render.latent_s4'], **tol)
        terms = ops.pose_loss_terms(y['depth_logits'].squeeze(0)[:, 0], y['mask_logits'].squeeze(0)[:, 0], cam.viewport,
                                    cam.translation[:, 2], target.depth, target.mask, cam.z_span, 0.01, cam.width, cam.height)
        names = ('ov_depth', 'depth', 'iou', 'mask')
        for i, k in enumerate(names):
            torch.testing.assert_close(terms[:, i].cpu(), g[f'loss.{k}'], atol=tol['atol'], rtol=2e-3 if precision != 2 else 5e-2)
        if precision == 2:
            return
        w = g.meta['weights']
        sum(w[k] * terms[:, i] for i, k in enumerate(names)).mean().backward()
        for name in ('log_quaternion', 'translation', 'viewport'):
            ours, g64 = getattr(cam, name).grad.cpu().double(), g[f'grad64.{name}']
            err = float((ours - g64).abs().max() / g64.abs().max())
            assert err <= _CFGB_GRAD_BOUND[cube], f'config-B {cube} cube, precision {precision}: d/d{name} off by {err:.3g} of scale'
    finally:
        ops.set_default_precision(old)


def test_full_size_properties(dev):
    """BASELINE config 2 extents (S=64, C=32, N=8): size-independent properties of the resampler —
    linearity in the volume, constants preserved, adjointness <R v, w> == <v, R^T w>."""
    from latentfusion_b200.modules.geometry import ObjectToCameraTransform
    S, C, N = 64, 32, 8
    cams, _ = ph.synthetic_cameras(N, S, seed=9)
    cam = cams.to(dev)
    T = ObjectToCameraTransform(1.0)
    torch.manual_seed(0)
    a = torch.randn(1, C, S, S, S, device=dev)
    b = torch.randn(1, C, S, S, S, device=dev)
    ra, rb, rab = T(a, cam), T(b, cam), T(2.0 * a - 3.0 * b, cam)
    torch.testing.assert_close(rab, 2.0 * ra - 3.0 * rb, atol=1e-4, rtol=1e-4)
    ones = T(torch.full((1, C, S, S, S), 1.5, device=dev), cam)
    torch.testing.assert_close(ones, torch.full_like(ones, 1.5), atol=1e-5, rtol=1e-5)
    v = a.clone().requires_grad_(True)
    w = torch.randn(N, C, S, S, S, device=dev)
    lhs = (T(v, cam) * w).sum()
    lhs.backward()
    rhs = (v.grad * a).sum()
    torch.testing.assert_close(lhs.detach(), rhs, atol=1e-1, rtol=1e-3)


def test_config2_batch_of_64_hypotheses_matches_single_runs(dev):
    """BASELINE configs[2] extents (adam_quick.toml at num_samples=64: N=64, S=64, C=32 -> 2.1 GB tensors, element
    indices past 2^29).  Hypotheses are independent, so the last hypothesis of the batch must be bit-identical to
    the same hypothesis processed alone: resample forward, resample backward-to-camera, tcgen05 conv, depth collapse."""
    from latentfusion_b200 import ops
    from latentfusion_b200.modules.geometry import ObjectToCameraTransform
    S, C, N = 64, 32, 64
    cams, _ = ph.synthetic_cameras(N, S, seed=21)
    cam = cams.to(dev)
    last = cam[N - 1:N]
    T = ObjectToCameraTransform(1.0)
    torch.manual_seed(2)
    vol = torch.randn(1, C, S, S, S, device=dev)
    full = T(vol, cam)
    one = T(vol, last)
    assert torch.equal(full[N - 1:N], one)
    w = torch.randn(32, C, 3, 3, 3, device=dev)
    b = torch.randn(32, device=dev) * 0.1
    for precision in (1, 2):
        yf = ops.eq_conv(full, w, b, act=True, norm=True, precision=precision)
        yo = ops.eq_conv(one, w, b, act=True, norm=True, precision=precision)
        assert torch.equal(yf[N - 1:N], yo)
    wc = torch.randn(32, C * S, 1, 1, device=dev)
    pf = ops.eq_conv(full, wc, None, kind=ops.KIND_COLLAPSE, depth=S)
    po = ops.eq_conv(one, wc, None, kind=ops.KIND_COLLAPSE, depth=S)
    assert torch.equal(pf[N - 1:N], po)
    del yf, yo, pf, po
    # backward to the cameras: d<full, g>/d(cam block) row N-1 == the single-camera run
    g = torch.randn_like(one)
    blk = cam.o2c_block(1.0).detach().requires_grad_(True)
    out = ops.resample_o2c(vol, blk)
    gfull = torch.zeros_like(out)
    gfull[N - 1:N] = g
    out.backward(gfull)
    blk1 = last.o2c_block(1.0).detach().requires_grad_(True)
    ops.resample_o2c(vol, blk1).backward(g)
    assert torch.equal(blk.grad[N - 1], blk1.grad[0])
    assert torch.count_nonzero(blk.grad[:N - 1]) == 0


def test_fused_pose_loss_head_vs_reference_formulas(g, dev):
    """csrc/pose_loss.cu against the torch composition of the reference ops (interpret_logits ->
    denormalize_depth -> uncrop x2 -> default_pose_loss): terms and all four gradient paths."""
    from latentfusion_b200 import ops
    from latentfusion_b200.pose import estimation
    from latentfusion_b200.observation import Observation
    P = 2 * g.meta['S']
    torch.manual_seed(0)
    logits = (torch.randn(2, 2, P, P, device=dev) * 2.0)
    gt = ph.product_camera(g.cam('ref_cam_full'), dev)[0:1]
    target = Observation(torch.zeros(1, 3, 480, 640, device=dev), g['target.depth'].to(dev), g['target.mask'].to(dev), gt)
    w = torch.tensor([0.3, 1.0, 0.2, 0.1], device=dev)

    def run(fused):
        cam = ph.product_camera(g.cam('hyp_cam'), dev, requires_grad=True)
        lg = logits.clone().requires_grad_(True)
        if fused:
            terms = ops.pose_loss_terms(lg[:, 0], lg[:, 1], cam.viewport, cam.translation[:, 2], target.depth,
                                        target.mask, cam.z_span, 0.01, cam.width, cam.height)
        else:
            depth, mask = torch.tanh(lg[:, 0:1]), torch.sigmoid(lg[:, 1:2])
            depth = (depth + 1) * (mask > 0.5) - 1
            losses = estimation.default_pose_loss(target, cam.denormalize_depth(depth), lg[:, 1:2], cam)
            terms = torch.stack([losses[k] for k in ('ov_depth', 'depth', 'iou', 'mask')], dim=1)
        (terms * w).sum(dim=1).mean().backward()
        return terms.detach(), lg.grad, cam.viewport.grad, cam.translation.grad

    t1, gl1, gv1, gt1 = run(True)
    t0, gl0, gv0, gt0 = run(False)
    torch.testing.assert_close(t1, t0, atol=1e-4, rtol=1e-4)
    torch.testing.assert_close(gl1, gl0, atol=1e-6, rtol=2e-3)
    torch.testing.assert_close(gv1, gv0, atol=1e-5, rtol=2e-3)
    torch.testing.assert_close(gt1, gt0, atol=1e-5, rtol=2e-3)


@pytest.mark.parametrize('precision', [1])
def test_tensor_core_bf16x3_path_meets_fp32_tolerance(g, dev, precision):
    """The tcgen05 bf16x3 convolution path (bench.py's default) against the golden vectors of the unmodified
    reference at the SAME fp32 tolerances as the exact kernels: render logits, losses, camera gradients, and the
    three-iteration estimator trajectory."""
    from latentfusion_b200 import ops
    old = ops.get_default_precision()
    ops.set_default_precision(precision)
    try:
        ph.smoke_check()
        test_gradient_estimator_three_iterations_vs_golden(g, dev)
    finally:
        ops.set_default_precision(old)


def test_bf16_path_stated_tolerance(g, dev):
    """precision 2 (plain bf16 operands, fp32 accumulate) gets its own, looser stated bound: 5e-2 abs on the
    O(1) logits of the golden configuration."""
    from latentfusion_b200 import ops
    from latentfusion_b200.recon.inference import LatentFusionModel
    old = ops.get_default_precision()
    ops.set_default_precision(2)
    try:
        sculptor, fuser, photographer = ph.build_product_models(g, dev)
        model = LatentFusionModel(sculptor, fuser, photographer, g.meta['camera_dist'], dev)
        cam = ph.product_camera(g.cam('hyp_cam'), dev)
        y, _ = model.render_latent_object(g['z_obj_gru'].to(dev), cam)
        torch.testing.assert_close(y['depth_logits'].cpu(), g['render.depth_logits'], atol=5e-2, rtol=5e-2)
        torch.testing.assert_close(y['mask_logits'].cpu(), g['render.mask_logits'], atol=5e-2, rtol=5e-2)
    finally:
        ops.set_default_precision(old)


def test_camera_block_kernel_vs_torch_chain(g, dev):
    """csrc/camera.cu (forward + analytic VJP) against the differentiable torch camera algebra on CPU."""
    d = g.cam('hyp_cam')
    cpu = ph.product_camera(d, 'cpu', requires_grad=True)
    gpu = ph.product_camera(d, dev, requires_grad=True)
    b_cpu, b_gpu = cpu.o2c_block(1.0), gpu.o2c_block(1.0)
    torch.testing.assert_close(b_gpu.cpu(), b_cpu.detach(), atol=1e-5, rtol=1e-5)
    torch.manual_seed(0)
    w = torch.zeros_like(b_cpu)
    w[:, :16] = torch.randn(2, 16)
    w[:, 20] = torch.randn(2)
    (b_cpu * w).sum().backward()
    (b_gpu * w.to(dev)).sum().backward()
    for k in ('log_quaternion', 'translation', 'viewport'):
        torch.testing.assert_close(getattr(gpu, k).grad.cpu(), getattr(cpu, k).grad, atol=1e-4, rtol=1e-4)


def test_mixed_precision_path_stated_tolerance(g, dev):
    """precision 3: bf16x3 forward + single-pass bf16 backward-data.  Forward outputs meet the fp32 tolerance;
    the camera gradients get the looser stated bound of 5e-2 (measured ~3e-2), which is why bench.py's
    fp32-parity default is precision 1, not 3."""
    import json
    from latentfusion_b200 import ops
    from latentfusion_b200.pose import estimation
    from latentfusion_b200.observation import Observation
    from latentfusion_b200.recon.inference import LatentFusionModel
    old = ops.get_default_precision()
    ops.set_default_precision(3)
    try:
        sculptor, fuser, photographer = ph.build_product_models(g, dev)
        model = LatentFusionModel(sculptor, fuser, photographer, g.meta['camera_dist'], dev)
        cam = ph.product_camera(g.cam('hyp_cam'), dev, requires_grad=True)
        y, _ = model.render_latent_object(g['z_obj_gru'].to(dev), cam)
        torch.testing.assert_close(y['depth_logits'].cpu(), g['render.depth_logits'], **OUT_TOL)
        gt = ph.product_camera(g.cam('ref_cam_full'), dev)[0:1]
        target = Observation(torch.zeros(1, 3, 480, 640, device=dev), g['target.depth'].to(dev), g['target.mask'].to(dev), gt)
        losses = estimation.default_pose_loss(target, cam.denormalize_depth(y['depth'].squeeze(0)), y['mask_logits'].squeeze(0), cam)
        w = json.loads(g.text('loss.weights'))
        sum(w[k] * v for k, v in losses.items()).mean().backward()
        for k in ('log_quaternion', 'translation', 'viewport'):
            torch.testing.assert_close(getattr(cam, k).grad.cpu(), g[f'grad.{k}'], atol=5e-2, rtol=5e-2)
    finally:
        ops.set_default_precision(old)


def test_small_fused_kernels_vs_torch_autograd(dev):
    """GRU gate backward, ConvLSTM gates, the BlendFuser's softmax-over-views blend and the 'sum' projection:
    each kernel (forward and backward) against fp64 autograd of the reference expression
    (modules/gru.py:38-41, modules/lstm.py:41-56, recon/fusion.py:92-96, recon/models.py:436-437)."""
    from latentfusion_b200 import ops
    torch.manual_seed(21)
    n, c, d, h, w = 2, 8, 5, 6, 7
    mk = lambda *s: torch.randn(*s, device=dev)                                          # noqa: E731

    def check(outs, refs, ins, rins):
        gs = [torch.randn_like(o) for o in outs]
        sum((o * g).sum() for o, g in zip(outs, gs)).backward()
        sum((o * g.double()).sum() for o, g in zip(refs, gs)).backward()
        for o, r in zip(outs, refs):
            torch.testing.assert_close(o.double(), r, atol=1e-5, rtol=1e-5)
        for a, b in zip(ins, rins):
            torch.testing.assert_close(a.grad.double(), b.grad, atol=2e-5, rtol=1e-4)

    # GRU gates
    u, r, hh = (mk(n, c, d, h, w).requires_grad_(True) for _ in range(3))
    u6, r6, h6 = (t.detach().double().requires_grad_(True) for t in (u, r, hh))
    upd, hr = ops.gru_gates1(u, r, hh)
    check([upd, hr], [torch.sigmoid(u6), h6 * torch.sigmoid(r6)], [u, r, hh], [u6, r6, h6])
    a, b, o = (mk(n, c, d, h, w).requires_grad_(True) for _ in range(3))
    a6, b6, o6 = (t.detach().double().requires_grad_(True) for t in (a, b, o))
    check([ops.gru_gates2(a, b, o)], [a6 * (1 - b6) + o6 * b6], [a, b, o], [a6, b6, o6])
    # LSTM gates
    gates, cc = mk(n, 4 * c, d, h, w).requires_grad_(True), mk(n, c, d, h, w).requires_grad_(True)
    g6, c6 = gates.detach().double().requires_grad_(True), cc.detach().double().requires_grad_(True)
    gi, gf, go, gg = torch.split(g6, c, dim=1)
    cn = torch.sigmoid(gf) * c6 + torch.sigmoid(gi) * torch.tanh(gg)
    check(list(ops.lstm_gates(gates, cc)), [torch.sigmoid(go) * torch.tanh(cn), cn], [gates, cc], [g6, c6])
    # BlendFuser blend
    v = 4
    sc, z = mk(n, v, 1, d, h, w).requires_grad_(True), mk(n, v, c, d, h, w).requires_grad_(True)
    s6, z6 = sc.detach().double().requires_grad_(True), z.detach().double().requires_grad_(True)
    w6 = torch.softmax(s6, dim=1)
    fused, wts = ops.view_softmax_blend(sc, z)
    check([fused, wts], [(z6 * w6).sum(dim=1, keepdim=True), w6], [sc, z], [s6, z6])
    # 'sum' projection
    x = mk(n, c, d, h, w).requires_grad_(True)
    x6 = x.detach().double().requires_grad_(True)
    check([ops.depth_sum(x)], [x6.sum(dim=2)], [x], [x6])


def test_latent_loss_refinement_graphed_equals_eager(g, dev):
    """configs/adam_latent.toml (latent = 0.2; reference estimation.py:605-609): the captured-graph refiner — fused loss
    head + latent cosine against a target code recomputed through the hypothesis cameras every iteration — follows the
    same trajectory as the eager loop (per-hypothesis torch optimisers, default_pose_loss on uncropped frames)."""
    from latentfusion_b200.pose import estimation
    from latentfusion_b200.observation import Observation
    from latentfusion_b200.recon.inference import LatentFusionModel
    sculptor, fuser, photographer = ph.build_product_models(g, dev)
    model = LatentFusionModel(sculptor, fuser, photographer, g.meta['camera_dist'], dev)
    cfg = {'type': 'gradient', 'args': dict(optimizer='adam', num_iters=3, num_samples=g.meta['N'], ranking_size=g.meta['N'],
                                            learning_rate=0.01, lr_reduce_patience=10, lr_reduce_threshold=1e-4,
                                            converge_threshold=1e-6, converge_patience=10),
           'loss_weights': dict(depth=1.0, ov_depth=0.3, iou=0.0, mask=0.0, latent=0.2)}
    gt = ph.product_camera(g.cam('ref_cam_full'), 'cpu')[0:1]
    torch.manual_seed(5)
    target = Observation(torch.rand(1, 3, 480, 640), g['target.depth'], g['target.mask'], gt)
    init = ph.product_camera(g.cam('est.init_cam'), 'cpu')
    runs = {}
    for graphed in (True, False):
        est = estimation.load_from_config(cfg, model, track_stats=True, return_camera_history=True)
        est.cuda_graph = graphed
        best, stats, history = est.estimate(g['z_obj_gru'].to(dev), target, camera=init)
        assert (getattr(est, '_refiner', None) is not None) == graphed
        runs[graphed] = (best, stats, history)
    a, b = runs[True], runs[False]
    assert float(a[1]['latent_loss'].abs().max()) > 1e-3                       # the term is really there
    torch.testing.assert_close(a[1]['latent_loss'], b[1]['latent_loss'], atol=2e-4, rtol=2e-3)
    torch.testing.assert_close(a[1]['rank_loss'], b[1]['rank_loss'], atol=1e-3, rtol=2e-3)
    for (_, ca), (_, cb) in zip(a[2], b[2]):
        torch.testing.assert_close(ca.translation, cb.translation, atol=3e-4, rtol=1e-3)
        torch.testing.assert_close(ca.log_quaternion, cb.log_quaternion, atol=3e-4, rtol=1e-3)


def test_packed_loss_head_record_kernel_and_block_gradient_match_the_unfused_forms(dev):
    """the graph path's glue-free forms: (a) the loss head on the decoder's channels-last logits / translation through
    lf_loss_desc strides == the de-interleaved call, values and all four gradient paths; (b) lf_refine_record == the
    torch expressions it replaces; (c) lf_resample_o2c_bwd_cam_block == the 17-term gradient re-laid out."""
    from latentfusion_b200 import _lib as L, ops
    torch.manual_seed(3)
    N, P, H, W = 5, 32, 48, 64
    logits = torch.randn(N, 2, P, P, device=dev).contiguous(memory_format=torch.channels_last)
    vp = torch.tensor([[10., 8., 50., 40.]], device=dev).repeat(N, 1) + torch.rand(N, 4, device=dev)
    tr = torch.randn(N, 3, device=dev) * 0.1 + torch.tensor([0., 0., 1.5], device=dev)
    td = (torch.rand(H, W, device=dev) > 0.3).float() * (1.4 + 0.2 * torch.rand(H, W, device=dev))
    tm = (torch.rand(H, W, device=dev) > 0.5).float()
    gt = torch.randn(N, 4, device=dev)
    outs = []
    for packed in (True, False):
        lg, v, t = (x.clone().requires_grad_(True) for x in (logits, vp, tr))
        if packed:
            assert lg.stride() == (2 * P * P, 1, 2 * P, 2)
            terms = ops.pose_loss_terms_packed(lg, v, t, td, tm, 0.5, 0.01, W, H)
        else:
            terms = ops.pose_loss_terms(lg[:, 0], lg[:, 1], v, t[:, 2], td, tm, 0.5, 0.01, W, H)
        terms.backward(gt)
        outs.append((terms.detach(), lg.grad, v.grad, t.grad))
    for a, b in zip(*outs):
        # same kernels, same per-pixel arithmetic; only the float atomics' arrival order differs
        torch.testing.assert_close(a, b, atol=1e-5, rtol=1e-4)
    # (b)
    chunk, K = 4, 4
    terms = torch.rand(N, K, device=dev)
    w_rank = torch.tensor([1.0, 0.5, 0.25, 2.0], device=dev)
    w_opt = torch.tensor([1.0, 0.0, 0.25, 3.0], device=dev)
    lq, trn = torch.randn(N, 3, device=dev), torch.randn(N, 3, device=dev)
    rank, gterms = torch.zeros(N, device=dev), torch.zeros(N, K, device=dev)
    h_rank, h_opt = torch.zeros(chunk, N, device=dev), torch.zeros(chunk, N, device=dev)
    h_terms = torch.zeros(chunk, K, N, device=dev)
    h_lq, h_tr = torch.zeros(chunk, N, 3, device=dev), torch.zeros(chunk, N, 3, device=dev)
    slot = torch.full((1,), 3, dtype=torch.long, device=dev)
    steps = torch.zeros(1, device=dev)
    ops.refine_record_(terms, w_rank, w_opt, lq, trn, rank, gterms, h_rank, h_opt, h_terms, h_lq, h_tr, slot, chunk, steps)
    t_req = terms.clone().requires_grad_(True)
    r_ref = sum(float(w_rank[k]) * t_req[:, k] for k in range(K))
    o_ref = sum(float(w_opt[k]) * t_req[:, k] for k in range(K))
    o_ref.mean().backward()
    assert torch.equal(rank, r_ref.detach()) and torch.equal(h_rank[3], r_ref.detach()) and torch.equal(h_opt[3], o_ref.detach())
    assert torch.equal(gterms, t_req.grad)
    assert torch.equal(h_terms[3], terms.t()) and torch.equal(h_lq[3], lq) and torch.equal(h_tr[3], trn)
    assert int(slot) == 0 and float(steps) == 1.0 and float(h_rank[:3].abs().sum()) == 0.0
    # (c)
    S, C, Nc = 16, 16, 3
    cams, _ = ph.synthetic_cameras(Nc, S, seed=4)
    blk = cams.to(dev).o2c_block(1.0).detach().contiguous()
    vol = ops.to_cl(torch.randn(1, C, S, S, S, device=dev))
    g = ops.to_cl(torch.randn(Nc, C, S, S, S, device=dev))
    ws = torch.empty(L.lib().lf_resample_o2c_bwd_cam_ws(Nc, S), device=dev)
    g17 = torch.empty(Nc, L.CAMGRAD_STRIDE, device=dev)
    gblk = torch.full((Nc, L.CAM_STRIDE), float('nan'), device=dev)
    st = torch.cuda.current_stream().cuda_stream
    L.check(L.lib().lf_resample_o2c_bwd_cam(ops._p(g), ops._p(vol), ops._p(blk), ops._p(g17), ops._p(ws), 1, Nc, C, S, st), 'bwd_cam')
    L.check(L.lib().lf_resample_o2c_bwd_cam_block(ops._p(g), ops._p(vol), ops._p(blk), ops._p(gblk), ops._p(ws), 1, Nc, C, S, st), 'bwd_cam_block')
    ref = torch.zeros(Nc, L.CAM_STRIDE, device=dev)
    ref[:, :16] = g17[:, :16]
    ref[:, 20] = g17[:, 16]
    assert torch.equal(gblk, ref)


@pytest.mark.parametrize('C,S,N', [(32, 24, 3), (16, 17, 2), (64, 8, 2)])
def test_o2c_resample_straight_into_split_planar_layout(dev, C, S, N):
    """K1 writing the consumer's split-planar layout (hi | lo bf16 planes with a zero halo) == lf_split_pack of its dense
    fp32 output, bit for bit (same fp32 values, same rounding split), into a buffer that starts as garbage."""
    from latentfusion_b200 import _lib as L, ops
    cams, _ = ph.synthetic_cameras(N, S, seed=C + S)
    blk = cams.to(dev).o2c_block(1.0).detach().contiguous()
    torch.manual_seed(S)
    vol = ops.to_cl(torch.randn(1, C, S, S, S, device=dev))
    dense = ops.resample_o2c(vol, blk)
    want = ops.split_pack(dense)
    assert L.lib().lf_resample_o2c_fwd_split_supported(C, S)
    got = ops.SplitVol.empty(N, C, S, S, S, dev)
    got.buf.fill_(0x7fc1)                                        # NaN bit patterns: every element must be overwritten
    L.check(L.lib().lf_resample_o2c_fwd_split(ops._p(vol), ops._p(blk), ops._p(got.buf), 1, N, C, S,
                                              torch.cuda.current_stream().cuda_stream), 'o2c_fwd_split')
    assert torch.equal(got.buf, want.buf)
    # and through the public op: the twin rides on the returned tensor
    out = ops.resample_o2c(vol, blk, split_only=True)
    assert torch.equal(out._lf_split.buf, want.buf)
    torch.testing.assert_close(out._lf_split.to_dense(), dense, atol=0, rtol=2 ** -15)
