"""CPU: pins oracle/lf_oracle.py (the PyTorch restatement) against golden vectors produced by the
UNMODIFIED reference (oracle/make_golden.py).  Tolerances are fp32 reassociation noise only."""
import json

import pytest
import torch

from oracle import lf_oracle as O

TOL = dict(atol=2e-5, rtol=1e-4)


def ocam(d):
    return O.Cam(d['intrinsic'], d['log_quaternion'], d['translation'], d['viewport'])


def arch_of(meta, which):
    a = dict(meta[f'arch_{which}'])
    a.setdefault('cube_size', 1.0)
    a['num_heads'] = 2
    return a


def test_zoom_viewport(golden):
    full = ocam(golden.cam('ref_cam_full'))
    z = full.zoom(2 * golden.meta['S'], golden.meta['camera_dist'])
    torch.testing.assert_close(z.viewport, golden['ref_cam.viewport'], atol=1e-3, rtol=1e-5)


def test_o2c_resample_and_grads(golden):
    d = golden.cam('hyp_cam')
    cam = ocam({k: v.clone().requires_grad_(k != 'intrinsic') for k, v in d.items()})
    vol = golden['o2c.vol'].clone().requires_grad_(True)
    out = O.object_to_camera(vol, cam)
    torch.testing.assert_close(out, golden['o2c.out'], **TOL)
    (out * golden['o2c.w']).sum().backward()
    torch.testing.assert_close(vol.grad, golden['o2c.grad_vol'], **TOL)
    for k in ('log_quaternion', 'translation', 'viewport'):
        torch.testing.assert_close(getattr(cam, k).grad, golden[f'o2c.grad_{k}'], atol=1e-3, rtol=2e-3)


def test_c2o_resample_and_grad(golden):
    cam = ocam(golden.cam('ref_cam'))
    vol = golden['c2o.vol'].clone().requires_grad_(True)
    out = O.camera_to_object(vol, cam)
    torch.testing.assert_close(out, golden['c2o.out'], **TOL)
    (out * golden['c2o.w']).sum().backward()
    torch.testing.assert_close(vol.grad, golden['c2o.grad_vol'], **TOL)


@pytest.mark.parametrize('name,scale,mode', [('blk3d_same', 1.0, 'nearest'), ('blk3d_up', 2.0, 'nearest'),
                                             ('blk3d_down', 0.5, 'nearest'), ('blk2d_up', 2.0, 'bilinear'),
                                             ('blk2d_down', 0.5, 'bilinear')])
def test_conv_block(golden, name, scale, mode):
    sd = {f'b.{k}': v.clone().requires_grad_(True) for k, v in golden.state_dict(name).items()}
    x = golden[f'{name}.x'].clone().requires_grad_(True)
    y = O.conv_block(x, sd, 'b', scale, mode)
    torch.testing.assert_close(y, golden[f'{name}.y'], **TOL)
    (y * golden[f'{name}.w']).sum().backward()
    torch.testing.assert_close(x.grad, golden[f'{name}.grad_x'], atol=1e-4, rtol=1e-3)
    for k, v in sd.items():
        torch.testing.assert_close(v.grad, golden[f'{name}.grad/{k[2:]}'], atol=1e-3, rtol=1e-3)


def test_sculptor_and_fusers(golden):
    arch = arch_of(golden.meta, 'sculptor')
    sd = golden.state_dict('sculptor')
    cam = ocam(golden.cam('ref_cam'))
    color, mask = golden['color'], golden['mask']
    with torch.no_grad():
        x = torch.cat((color.flatten(0, 1), mask.flatten(0, 1) * 2 - 1), dim=1)
        z, z_cam_mid, _ = O.sculptor_forward(sd, arch, x, cam)
        torch.testing.assert_close(*golden.sampled('z_views', z), **TOL)
        torch.testing.assert_close(*golden.sampled('z_cam_mid0', z_cam_mid[0]), **TOL)
        zv = z.view(1, -1, *z.shape[1:])
        for kind in ('max', 'mean', 'median', 'abs_max'):
            torch.testing.assert_close(*golden.sampled(f'z_obj_pool_{kind}', O.fuse(f'pool:{kind}', zv)), **TOL)
        zg = O.sculptor_encode(sd, arch, 'gru', golden.state_dict('fuser'), cam, color, mask)
        torch.testing.assert_close(zg, golden['z_obj_gru'], atol=1e-4, rtol=1e-3)


def test_render_loss_and_camera_grads(golden):
    arch = arch_of(golden.meta, 'photographer')
    sd = golden.state_dict('photographer')
    d = golden.cam('hyp_cam')
    cam = ocam({k: v.clone().requires_grad_(k != 'intrinsic') for k, v in d.items()})
    z_obj = golden['z_obj_gru'][0]            # [1,C,S,S,S]
    weights = json.loads(str(golden._z['loss.weights']))
    total, losses, y, latent = O.refine_iteration(sd, arch, z_obj, cam, golden['target.depth'],
                                                  golden['target.mask'], weights)
    torch.testing.assert_close(y['depth_logits'], golden['render.depth_logits'][0], **TOL)
    torch.testing.assert_close(y['mask_logits'], golden['render.mask_logits'][0], **TOL)
    torch.testing.assert_close(y['depth'], golden['render.depth'][0], **TOL)
    torch.testing.assert_close(latent, golden['render.latent'], **TOL)
    for k, v in losses.items():
        torch.testing.assert_close(v, golden[f'loss.{k}'], atol=1e-4, rtol=1e-4)
    total.mean().backward()
    for k in ('log_quaternion', 'translation', 'viewport'):
        torch.testing.assert_close(getattr(cam, k).grad, golden[f'grad.{k}'], atol=1e-4, rtol=2e-3)
