"""TEST INFRASTRUCTURE — generates tests/golden/*.npz by running the UNMODIFIED reference.

Run in the authoring container (needs /root/reference; the GPU box never runs this):

    python oracle/make_golden.py

It imports the reference through ``oracle/ref_import.py`` (5 import stubs + 1 scheduler shim,
SURVEY.md §8c), builds the synthetic "LF-synth(S, C)" networks of SURVEY.md §8(d) at a tiny size,
and dumps inputs, the reference-format state_dicts and every intermediate/result the parity tests
check.  The reference ships no tests or golden vectors of its own (SURVEY.md §4); these files are
the pin for ``oracle/lf_oracle.py`` and, through it, for the CUDA path.
"""
import json
import math
import os
import sys
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
warnings.filterwarnings('ignore')

from oracle import ref_import  # noqa: E402
from tests import parity_helpers as ph  # noqa: E402

ref_import.install()

import torch  # noqa: E402

torch.set_num_threads(1)        # fixed reduction order for the fixtures
torch.backends.cudnn.allow_tf32 = False
torch.backends.cuda.matmul.allow_tf32 = False

from latentfusion import consts, three  # noqa: E402
from latentfusion.modules import blocks as ref_blocks  # noqa: E402
from latentfusion.modules import EqualizedConv2d, EqualizedConv3d  # noqa: E402
from latentfusion.modules.geometry import (Camera, CameraToObjectTransform,  # noqa: E402
                                           ObjectToCameraTransform)
from latentfusion.observation import Observation  # noqa: E402
from latentfusion.pose import estimation as ref_estimation  # noqa: E402
from latentfusion.pose import utils as ref_pu  # noqa: E402
from latentfusion.recon import fusion as ref_fusion  # noqa: E402
from latentfusion.recon import models as ref_models  # noqa: E402
from latentfusion.recon.inference import LatentFusionModel  # noqa: E402
from latentfusion.recon.utils import optimal_camera_dist  # noqa: E402
from latentfusion.utils import parse_block_config as pbc  # noqa: E402

OUT = os.path.join(os.path.dirname(HERE), 'tests', 'golden')


def npy(t):
    return t.detach().cpu().numpy()


def cam_dict(prefix, cam):
    return {f'{prefix}.intrinsic': npy(cam.intrinsic), f'{prefix}.log_quaternion': npy(cam.log_quaternion),
            f'{prefix}.translation': npy(cam.translation), f'{prefix}.viewport': npy(cam.viewport)}


def sd_dict(prefix, module):
    return {f'{prefix}/{k}': npy(v) for k, v in module.state_dict().items()}


def lf_synth(S, C):
    """SURVEY.md §8(d) "LF-synth(S, C)"."""
    arch_s = dict(in_size=2 * S, image_config=pbc(f"{C},D,{2*C}:{2*C},{2*C}"),
                  camera_config=pbc(f"{C},{C}"), object_config=pbc(f"{C},{C}"),
                  projection_type='factor', input_color=True, input_depth=False, input_mask=True,
                  scale_mode='nearest')
    arch_p = dict(in_size=S, image_config=pbc(f"{C},D,{2*C}:{2*C},U,{2*C},U,{C}"),
                  camera_config=pbc(f"{C},{C}"), object_config=[], projection_type='factor',
                  predict_depth=True, predict_mask=True, predict_color=False, scale_mode='nearest')
    sculptor = ref_models.Sculptor(**arch_s)
    fuser = ref_fusion.get_fuser('gru', in_channels=C, cube_size=1.0)
    photographer = ref_models.Photographer(**arch_p)
    # Non-zero biases so the bias path is exercised (the reference initialises them to 0).
    for m in (sculptor, fuser, photographer):
        for k, p in m.named_parameters():
            if k.endswith('bias'):
                p.data.normal_(0, 0.1)
    return sculptor, fuser, photographer, arch_s, arch_p


def reference_cameras(V, in_size, camera_dist, seed):
    torch.manual_seed(seed)
    K = torch.tensor(consts.INTRINSIC).unsqueeze(0).expand(V, -1, -1).contiguous()
    quats = three.orientation.evenly_distributed_quats(V)
    trans = torch.tensor([[0.0, 0.0, camera_dist]]).expand(V, -1).contiguous()
    extr = three.to_extrinsic_matrix(trans, quats)
    cam = Camera(K, extr, z_span=0.5, width=640, height=480)
    return cam


def disc(size, radius, center=None):
    yy, xx = torch.meshgrid(torch.arange(size[0], dtype=torch.float32),
                            torch.arange(size[1], dtype=torch.float32), indexing='ij')
    cy, cx = center if center is not None else ((size[0] - 1) / 2.0, (size[1] - 1) / 2.0)
    return (((yy - cy) ** 2 + (xx - cx) ** 2) <= radius ** 2).float()


def main():
    os.makedirs(OUT, exist_ok=True)
    S, C, V, N = 16, 8, 3, 2
    torch.manual_seed(0)
    sculptor, fuser, photographer, arch_s, arch_p = lf_synth(S, C)
    camera_dist = optimal_camera_dist(615.4991, 2 * S, 0.5, slack=128 / (2 * S))
    model = LatentFusionModel(sculptor, fuser, photographer, camera_dist, 'cpu')

    g = {}
    g['meta'] = np.array(json.dumps(dict(S=S, C=C, V=V, N=N, camera_dist=camera_dist,
                                         arch_sculptor=arch_s, arch_photographer=arch_p,
                                         torch=torch.__version__)))
    g.update(sd_dict('sculptor', sculptor))
    g.update(sd_dict('fuser', fuser))
    g.update(sd_dict('photographer', photographer))

    # ---------------- reference views -> z_obj (Sculptor.encode + fusers) ----------------
    ref_cam_full = reference_cameras(V, 2 * S, camera_dist, seed=10)
    ref_cam = ref_cam_full.zoom(None, 2 * S, camera_dist)
    torch.manual_seed(11)
    color = torch.rand(1, V, 3, 2 * S, 2 * S) * 2 - 1
    mask = disc((2 * S, 2 * S), 0.4 * 2 * S).view(1, 1, 1, 2 * S, 2 * S).expand(1, V, -1, -1, -1).contiguous()
    g.update(cam_dict('ref_cam_full', ref_cam_full))
    g.update(cam_dict('ref_cam', ref_cam))
    g['color'], g['mask'] = npy(color), npy(mask)
    with torch.no_grad():
        x = torch.cat((color.flatten(0, 1), mask.flatten(0, 1) * 2 - 1), dim=1)
        z_views, z_cam_mid, z_obj_mid = sculptor(x, ref_cam)
        g['z_views'] = npy(z_views)
        g['z_cam_mid0'] = npy(z_cam_mid[0])
        z_obj, _ = sculptor.encode(fuser, ref_cam, color, mask=mask)
        g['z_obj_gru'] = npy(z_obj)
        for kind in ('max', 'mean', 'median', 'abs_max'):
            zp, _ = sculptor.encode(ref_fusion.get_fuser(f'pool:{kind}', C, 1.0), ref_cam, color, mask=mask)
            g[f'z_obj_pool_{kind}'] = npy(zp)

    # ---------------- hypothesis cameras: render + loss + grads ----------------
    torch.manual_seed(12)
    gt_full = ref_cam_full[0:1]
    hyp = Camera.cat([ref_pu.perturb_camera(gt_full, 0.01, 10.0 / 180.0 * math.pi) for _ in range(N)])
    hyp = hyp.zoom(None, 2 * S, camera_dist)
    hyp_p = ref_pu.parameterize_camera(hyp, optimize_viewport=True)
    g.update(cam_dict('hyp_cam', hyp))
    y, z_lat = model.render_latent_object(z_obj, hyp_p, return_latent=True, apply_mask=True)
    g['render.depth'] = npy(y['depth'])
    g['render.mask'] = npy(y['mask'])
    g['render.depth_logits'] = npy(y['depth_logits'])
    g['render.mask_logits'] = npy(y['mask_logits'])
    g['render.latent'] = npy(z_lat)

    # target observation: disc at camera_dist (SURVEY §8d), full frame 640x480
    tmask = disc((480, 640), 60.0, center=(251.5, 315.4)).view(1, 1, 480, 640)
    tdepth = tmask * camera_dist
    tdepth[0, 0, 250:254, 300:330] = 0.0           # sensor holes -> exercises invalid_mask
    tcolor = torch.zeros(1, 3, 480, 640)
    target = Observation(tcolor, tdepth, tmask, gt_full)
    g['target.depth'], g['target.mask'] = npy(tdepth), npy(tmask)

    z_depth = hyp_p.denormalize_depth(y['depth'].squeeze(0))
    loss_dict = ref_estimation.default_pose_loss(target, z_depth, y['mask_logits'].squeeze(0), hyp_p)
    weights = dict(depth=1.0, ov_depth=0.3, iou=0.2, mask=0.1)
    total = sum(weights[k] * v for k, v in loss_dict.items())
    total.mean().backward()
    for k, v in loss_dict.items():
        g[f'loss.{k}'] = npy(v)
    g['loss.weights'] = np.array(json.dumps(weights))
    g['grad.log_quaternion'] = npy(hyp_p.log_quaternion.grad)
    g['grad.translation'] = npy(hyp_p.translation.grad)
    g['grad.viewport'] = npy(hyp_p.viewport.grad)

    # ---------------- op-level: the two resamplers with grads to volume and camera ---------
    torch.manual_seed(13)
    vol = torch.randn(1, 5, 12, 12, 12, requires_grad=True)        # odd channel count on purpose
    cam_o = ref_pu.parameterize_camera(hyp, optimize_viewport=True)
    out = ObjectToCameraTransform(1.0)(vol, cam_o)
    w = torch.randn_like(out)
    (out * w).sum().backward()
    g['o2c.vol'], g['o2c.out'], g['o2c.w'] = npy(vol), npy(out), npy(w)
    g['o2c.grad_vol'] = npy(vol.grad)
    g['o2c.grad_log_quaternion'] = npy(cam_o.log_quaternion.grad)
    g['o2c.grad_translation'] = npy(cam_o.translation.grad)
    g['o2c.grad_viewport'] = npy(cam_o.viewport.grad)

    cvol = torch.randn(V, 5, 12, 12, 12, requires_grad=True)
    # NB: the reference's camera->object grid is built with an in-place divide
    # (geometry.py:637), so it is NOT differentiable w.r.t. the camera; only d/d(volume) exists.
    out = CameraToObjectTransform(1.0)(cvol, ref_cam)
    w = torch.randn_like(out)
    (out * w).sum().backward()
    g['c2o.vol'], g['c2o.out'], g['c2o.w'] = npy(cvol), npy(out), npy(w)
    g['c2o.grad_vol'] = npy(cvol.grad)

    # ---------------- op-level: conv blocks (3D nearest up/down, 2D bilinear up/down) -------
    torch.manual_seed(14)
    for name, conv, dims, cin, cout, scale, mode in (
            ('blk3d_same', EqualizedConv3d, (2, 6, 6, 6, 6), 6, 10, 1.0, 'nearest'),
            ('blk3d_up', EqualizedConv3d, (1, 4, 5, 5, 5), 4, 8, 2.0, 'nearest'),
            ('blk3d_down', EqualizedConv3d, (1, 4, 6, 6, 6), 4, 8, 0.5, 'nearest'),
            ('blk2d_up', EqualizedConv2d, (2, 6, 9, 9), 6, 8, 2.0, 'bilinear'),
            ('blk2d_down', EqualizedConv2d, (2, 6, 10, 10), 6, 12, 0.5, 'bilinear')):
        blk = ref_blocks.Block(cin, cout, conv_module=conv, scale_factor=scale, scale_mode=mode)
        for k, p in blk.named_parameters():
            if k.endswith('bias'):
                p.data.normal_(0, 0.1)
        xin = torch.randn(*dims, requires_grad=True)
        yout = blk(xin)
        wq = torch.randn_like(yout)
        (yout * wq).sum().backward()
        g.update(sd_dict(name, blk))
        g[f'{name}.x'], g[f'{name}.y'], g[f'{name}.w'] = npy(xin), npy(yout), npy(wq)
        g[f'{name}.grad_x'] = npy(xin.grad)
        for k, p in blk.named_parameters():
            g[f'{name}.grad/{k}'] = npy(p.grad)

    # ---------------- estimator: 3 iterations of GradientPoseEstimator (adam_quick.toml) ----
    torch.manual_seed(15)
    est = ref_estimation.load_from_config(
        os.path.join(ref_import.REFERENCE_ROOT, 'configs', 'adam_quick.toml'), model,
        num_samples=N, ranking_size=N, num_iters=3, track_stats=True, return_camera_history=True)
    hyp_full = Camera.cat([ref_pu.perturb_camera(gt_full, 0.01, 10.0 / 180.0 * math.pi) for _ in range(N)])
    g.update(cam_dict('est.init_cam', hyp_full))
    best, stats, history = est.estimate(z_obj, target, camera=hyp_full)
    g.update(cam_dict('est.best_cam', best))
    g['est.rank_loss'] = npy(stats['rank_loss'])
    g['est.depth_loss'] = npy(stats['depth_loss'])
    g['est.ov_depth_loss'] = npy(stats['ov_depth_loss'])
    for i, (loss, cams) in enumerate(history):
        g.update(cam_dict(f'est.hist{i}', cams))

    # Keep the file small: the networks' weights and the seeded inputs are drawn again by the tests
    # (tests/parity_helpers.py, recipe 'lfsynth'), which check them against these digests; the encoder's
    # largest outputs are stored as a fixed sample.
    regen = [k for k in g if k.split('/')[0] in ('sculptor', 'fuser', 'photographer')
             or k in ('color', 'o2c.vol', 'o2c.w', 'c2o.vol', 'c2o.w')]
    g['regenerated'] = np.array(json.dumps(dict(recipe='lfsynth', digests={k: ph.digest(g.pop(k)) for k in regen})))
    for k in ('z_views', 'z_cam_mid0', 'z_obj_pool_max', 'z_obj_pool_mean', 'z_obj_pool_median', 'z_obj_pool_abs_max'):
        full = g.pop(k)
        g[f'{k}.shape'], g[f'{k}.sample'] = np.array(full.shape), ph.sample(full)

    path = os.path.join(OUT, 'lfsynth_s16_c8.npz')
    np.savez_compressed(path, **g)
    print('wrote', path, f'{os.path.getsize(path) / 1e6:.2f} MB', len(g), 'arrays')


if __name__ == '__main__':
    main()
