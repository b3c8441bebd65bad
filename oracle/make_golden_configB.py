"""TEST INFRASTRUCTURE — golden vectors of the UNMODIFIED reference at the BENCHMARKED configuration.

BASELINE configs[1] ("config B", SURVEY.md §8d): LF-synth(S=64, C=32), 128^2 render, the estimator's own
perturbation model for the hypothesis cameras.  N=2 hypotheses (the cost of the reference is linear in N and the
hypotheses are independent, so two pin the composition as well as eight).

    python oracle/make_golden_configB.py        # authoring container only (needs /root/reference)

Writes tests/golden/configB_s64_c32.npz:
  * digests of the reference-format Photographer state_dict (random N(0,1) weights, seed 0; 278k floats), which
    the tests draw again rather than read,
  * the hypothesis cameras, the target observation's generator parameters,
  * depth/mask logits, a strided sample of the projected latent, the four pose-loss terms,
  * camera gradients of (1.0*depth + 0.3*ov_depth) [configs/adam_quick.toml] in fp32 — the reference as shipped —
    and in fp64 (the same reference modules cast to double, with the one fp32 cast in
    modules/geometry.py:16-17 lifted), which is the conditioning yardstick for the gradient tolerances.

The object cube is NOT stored (33 MB): it is `torch.manual_seed(5); torch.randn(1,32,64,64,64) * 0.5`, regenerated
by the test (same torch build on the GPU box); its checksum is stored to catch generator drift.
"""
import json
import math
import os
import sys
import time
import warnings

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
warnings.filterwarnings('ignore')

from oracle import ref_import  # noqa: E402
from tests import parity_helpers as ph  # noqa: E402

ref_import.install()

import torch  # noqa: E402
import torch.nn.functional as F  # noqa: E402

from latentfusion import consts, three  # noqa: E402
from latentfusion.modules import geometry as ref_geometry  # noqa: E402
from latentfusion.modules.geometry import Camera  # noqa: E402
from latentfusion.observation import Observation  # noqa: E402
from latentfusion.pose import estimation as ref_estimation  # noqa: E402
from latentfusion.pose import utils as ref_pu  # noqa: E402
from latentfusion.recon import fusion as ref_fusion  # noqa: E402
from latentfusion.recon import models as ref_models  # noqa: E402
from latentfusion.recon.inference import LatentFusionModel  # noqa: E402
from latentfusion.recon.utils import optimal_camera_dist  # noqa: E402
from latentfusion.utils import parse_block_config as pbc  # noqa: E402

SMOOTH = '--smooth' in sys.argv
OUT = os.path.join(os.path.dirname(HERE), 'tests', 'golden',
                   'configB_s64_c32_smooth.npz' if SMOOTH else 'configB_s64_c32.npz')
S, C, N = 64, 32, 2
WEIGHTS = dict(depth=1.0, ov_depth=0.3, iou=0.0, mask=0.0)          # configs/adam_quick.toml


def npy(t):
    return t.detach().cpu().numpy()


def disc(h, w, cy, cx, radius):
    yy, xx = torch.meshgrid(torch.arange(h, dtype=torch.float32), torch.arange(w, dtype=torch.float32), indexing='ij')
    return (((yy - cy) ** 2 + (xx - cx) ** 2) <= radius ** 2).float()


def make_cube(smooth):
    """white noise (worst case: d sample / d coordinate jumps at every cell boundary), or the same noise low-pass
    filtered with a 5^3 box and rescaled to std 0.5 (a spatially smooth latent, like a Sculptor output)."""
    torch.manual_seed(5)
    z = torch.randn(1, C, S, S, S)
    if smooth:
        z = F.avg_pool3d(F.pad(z, (2, 2, 2, 2, 2, 2), mode='replicate'), 5, stride=1)
        z = z / z.std()
    return z * 0.5


def run(model, z_obj, hyp, target, dtype):
    cam = ref_pu.parameterize_camera(hyp.clone() if hasattr(hyp, 'clone') else hyp, optimize_viewport=True)
    if dtype == torch.float64:
        for name in ('log_quaternion', 'translation', 'viewport'):
            p = getattr(cam, name)
            p.data = p.data.double()
        cam.intrinsic = cam.intrinsic.double()
    y, latent = model.render_latent_object(z_obj.to(dtype), cam, return_latent=True, apply_mask=True)
    z_depth = cam.denormalize_depth(y['depth'].squeeze(0))
    losses = ref_estimation.default_pose_loss(target, z_depth, y['mask_logits'].squeeze(0), cam)
    total = sum(WEIGHTS[k] * v for k, v in losses.items())
    total.mean().backward()
    grads = {k: getattr(cam, k).grad.clone() for k in ('log_quaternion', 'translation', 'viewport')}
    return y, latent, losses, grads


def main():
    torch.set_num_threads(os.cpu_count() or 1)
    torch.manual_seed(0)
    arch_p = dict(in_size=S, image_config=pbc(f"{C},D,{2*C}:{2*C},U,{2*C},U,{C}"),
                  camera_config=pbc(f"{C},{C}"), object_config=[], projection_type='factor',
                  predict_depth=True, predict_mask=True, predict_color=False, scale_mode='nearest')
    arch_s = dict(in_size=2 * S, image_config=pbc(f"{C},D,{2*C}:{2*C},{2*C}"), camera_config=pbc(f"{C},{C}"),
                  object_config=pbc(f"{C},{C}"), projection_type='factor', input_color=True, input_depth=False,
                  input_mask=True, scale_mode='nearest')
    photographer = ref_models.Photographer(**arch_p)
    for k, p in photographer.named_parameters():
        if k.endswith('bias'):
            p.data.normal_(0, 0.1)
    sculptor = ref_models.Sculptor(**arch_s)          # only to satisfy the façade's constructor
    fuser = ref_fusion.get_fuser('pool:mean', C, 1.0)
    camera_dist = optimal_camera_dist(615.4991, 2 * S, 0.5, slack=128 / (2 * S))
    model = LatentFusionModel(sculptor, fuser, photographer, camera_dist, 'cpu')

    # cameras: the estimator's own perturbation of a ground-truth view (estimation.py:23-24)
    torch.manual_seed(2)
    K = torch.tensor(consts.INTRINSIC).unsqueeze(0)
    quats = three.orientation.evenly_distributed_quats(1)
    trans = torch.tensor([[0.0, 0.0, camera_dist]])
    gt_full = Camera(K, three.to_extrinsic_matrix(trans, quats), z_span=0.5, width=640, height=480)
    torch.manual_seed(7)
    hyp_full = Camera.cat([ref_pu.perturb_camera(gt_full, 0.01, 10.0 / 180.0 * math.pi) for _ in range(N)])
    hyp = hyp_full.zoom(None, 2 * S, camera_dist)

    tmask = disc(480, 640, 251.5, 315.4, 45.0).view(1, 1, 480, 640)
    tdepth = tmask * camera_dist
    target = Observation(torch.zeros(1, 3, 480, 640), tdepth, tmask, gt_full)

    z_obj = make_cube(SMOOTH).unsqueeze(0)                             # [B=1, 1, C, S, S, S]

    g = {}
    g['meta'] = np.array(json.dumps(dict(S=S, C=C, N=N, camera_dist=camera_dist, arch_photographer=arch_p,
                                         weights=WEIGHTS, z_obj='make_cube(smooth)', smooth=SMOOTH,
                                         target=dict(cy=251.5, cx=315.4, radius=45.0), torch=torch.__version__)))
    # the weights are drawn again by the tests (tests/parity_helpers.py, recipe 'configB'), checked against these digests
    g['regenerated'] = np.array(json.dumps(dict(recipe='configB', digests={
        f'photographer/{k}': ph.digest(npy(v)) for k, v in photographer.state_dict().items()})))
    for k in ('intrinsic', 'log_quaternion', 'translation', 'viewport'):
        g[f'hyp_cam.{k}'] = npy(getattr(hyp, k))
        g[f'gt_cam.{k}'] = npy(getattr(gt_full, k))
    g['z_obj.checksum'] = np.array([float(z_obj.double().sum()), float(z_obj.double().abs().sum())])

    t0 = time.time()
    y, latent, losses, grads = run(model, z_obj, hyp, target, torch.float32)
    print(f'fp32 reference: {time.time() - t0:.1f} s')
    g['render.depth_logits'] = npy(y['depth_logits'])
    g['render.mask_logits'] = npy(y['mask_logits'])
    g['render.latent_s4'] = npy(latent[..., ::4, ::4])
    for k, v in losses.items():
        g[f'loss.{k}'] = npy(v)
    for k, v in grads.items():
        g[f'grad.{k}'] = npy(v)

    # fp64 yardstick: same modules in double; the single hard fp32 cast of the reference is lifted
    ref_geometry._grid_sample = lambda tensor, grid, **kw: F.grid_sample(tensor, grid, **kw)
    model.photographer.double()
    target64 = Observation(torch.zeros(1, 3, 480, 640).double(), tdepth.double(), tmask.double(), gt_full)
    t0 = time.time()
    try:
        torch.set_default_dtype(torch.float64)
        y64, _, losses64, grads64 = run(model, z_obj, hyp, target64, torch.float64)
    finally:
        torch.set_default_dtype(torch.float32)
    print(f'fp64 reference: {time.time() - t0:.1f} s')
    g['render64.depth_logits'] = npy(y64['depth_logits'])
    g['render64.mask_logits'] = npy(y64['mask_logits'])
    for k, v in losses64.items():
        g[f'loss64.{k}'] = npy(v)
    for k, v in grads64.items():
        g[f'grad64.{k}'] = npy(v)
    for k in grads:
        e = (grads[k].double() - grads64[k]).abs().max() / grads64[k].abs().max()
        print(f'  reference fp32 vs fp64 grad.{k}: rel {float(e):.3e}')
    e = (y['depth_logits'].double() - y64['depth_logits']).abs().max()
    print(f'  reference fp32 vs fp64 depth logits: abs {float(e):.3e}')

    np.savez_compressed(OUT, **g)
    print('wrote', OUT, f'{os.path.getsize(OUT) / 1e6:.2f} MB', len(g), 'arrays')


if __name__ == '__main__':
    main()
