"""Shared helpers for the parity tests and ``__graft_entry__.smoke()`` (test infrastructure)."""
import hashlib
import json
import os

import numpy as np
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLDEN = os.path.join(ROOT, 'tests', 'golden', 'lfsynth_s16_c8.npz')

# fp32 parity tolerances (SURVEY.md §4-4): outputs atol 1e-4 / rtol 1e-3, camera grads rtol 2e-3
OUT_TOL = dict(atol=1e-4, rtol=1e-3)
GRAD_TOL = dict(atol=2e-4, rtol=2e-3)

# A golden output too large to store whole keeps every SAMPLE_STRIDE-th element of its flattened values.  The stride
# is prime, so it is coprime with every extent and the sample covers all positions along each axis.
SAMPLE_STRIDE = 7


def sample(a):
    """The stored sample of a large output (numpy array or tensor)."""
    return a.reshape(-1)[::SAMPLE_STRIDE]


def digest(a):
    """Short SHA-256 of an array's dtype, shape and bytes: pins the arrays a golden file regenerates instead of
    storing."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(f'{a.dtype.str}{a.shape}'.encode())
    h.update(a.tobytes())
    return h.hexdigest()[:16]


def reference_init(nets, seed):
    """Draw the weights of product networks exactly as the reference's constructors draw the same architectures after
    torch.manual_seed(seed), then the non-zero biases the golden scripts draw.  Each reference equalised convolution
    wraps an nn.ConvNd, whose own init (kaiming_uniform_: one uniform draw per weight) is overwritten by N(0, 1); the
    biases are then drawn N(0, 0.1), network by network."""
    from latentfusion_b200.modules.equalized import Equalized
    torch.manual_seed(seed)
    with torch.no_grad():
        for net in nets:
            for m in net.modules():
                if isinstance(m, Equalized):
                    w = m.module.weight
                    torch.empty_like(w).uniform_()
                    w.normal_(0, 1)
        for net in nets:
            for k, p in net.named_parameters():
                if k.endswith('bias'):
                    p.normal_(0, 0.1)


def _regenerate_lfsynth(meta):
    """oracle/make_golden.py's networks (seed 0), reference views (seed 11) and resampler inputs (seed 13)."""
    from latentfusion_b200.recon import fusion, models
    S, C, V, N = meta['S'], meta['C'], meta['V'], meta['N']
    nets = {'sculptor': models.Sculptor(**meta['arch_sculptor']),
            'fuser': fusion.get_fuser('gru', in_channels=C, cube_size=1.0),
            'photographer': models.Photographer(**meta['arch_photographer'])}
    reference_init(nets.values(), seed=0)
    out = {f'{name}/{k}': v.numpy() for name, net in nets.items() for k, v in net.state_dict().items()}
    torch.manual_seed(11)
    out['color'] = (torch.rand(1, V, 3, 2 * S, 2 * S) * 2 - 1).numpy()
    torch.manual_seed(13)
    for k, n in (('o2c.vol', 1), ('o2c.w', N), ('c2o.vol', V), ('c2o.w', V)):
        out[k] = torch.randn(n, 5, 12, 12, 12).numpy()
    return out


def _regenerate_config_b(meta):
    """oracle/make_golden_configB.py's Photographer (seed 0)."""
    from latentfusion_b200.recon import models
    photographer = models.Photographer(**meta['arch_photographer'])
    reference_init([photographer], seed=0)
    return {f'photographer/{k}': v.numpy() for k, v in photographer.state_dict().items()}


_REGENERATE = {'lfsynth': _regenerate_lfsynth, 'configB': _regenerate_config_b}


class Golden:
    """Read-only view of a tests/golden/*.npz file.  Seeded inputs and weights that a file lists under `regenerated`
    are drawn again here and must match the digests of what the reference was run with; outputs stored as a sample
    are compared through `sampled`."""

    def __init__(self, path=GOLDEN):
        self._z = np.load(path)
        self.meta = json.loads(str(self._z['meta']))
        self._regen = {}
        if 'regenerated' in self._z.files:
            spec = json.loads(str(self._z['regenerated']))
            self._regen = _REGENERATE[spec['recipe']](self.meta)
            assert set(self._regen) == set(spec['digests']), \
                f'{path}: regenerated keys differ: {sorted(set(self._regen) ^ set(spec["digests"]))}'
            bad = [k for k, d in spec['digests'].items() if digest(self._regen[k]) != d]
            assert not bad, f'{path}: regenerated arrays differ from the ones the reference was run with: {bad}'

    def __getitem__(self, key):
        if key in self._regen:
            return torch.from_numpy(self._regen[key].copy())
        return torch.from_numpy(np.array(self._z[key]))

    def text(self, key):
        return str(self._z[key])

    def state_dict(self, prefix):
        p = prefix + '/'
        return {k[len(p):]: self[k] for k in (*self._z.files, *self._regen) if k.startswith(p)}

    def sampled(self, key, ours):
        """(ours, golden) on the stored sample of output `key`, after checking that `ours` has the full shape."""
        shape = tuple(int(n) for n in self._z[f'{key}.shape'])
        assert tuple(ours.shape) == shape, f'{key}: shape {tuple(ours.shape)} != {shape}'
        return sample(ours), self[f'{key}.sample']

    def cam(self, prefix):
        return {k: self[f'{prefix}.{k}'] for k in ('intrinsic', 'log_quaternion', 'translation', 'viewport')}


def product_camera(d, device, requires_grad=False):
    from latentfusion_b200.modules.geometry import Camera
    from latentfusion_b200.pose import utils as pu
    cam = Camera(d['intrinsic'].clone(), None, 0.5, d['viewport'].clone(), width=640, height=480,
                 log_quaternion=d['log_quaternion'].clone(), translation=d['translation'].clone()).to(device)
    if requires_grad:
        cam = pu.parameterize_camera(cam, optimize_viewport=True)
    return cam


def oracle_camera(d, requires_grad=False):
    from oracle import lf_oracle as O
    t = {k: v.clone() for k, v in d.items()}
    if requires_grad:
        for k in ('log_quaternion', 'translation', 'viewport'):
            t[k].requires_grad_(True)
    return O.Cam(t['intrinsic'], t['log_quaternion'], t['translation'], t['viewport'])


def build_product_models(g, device):
    """Instantiate the product networks from the reference-format args + state_dicts in the golden
    file (strict load => identical key names and shapes)."""
    from latentfusion_b200.recon import models, fusion
    a_s, a_p = g.meta['arch_sculptor'], g.meta['arch_photographer']
    sculptor = models.Sculptor(**a_s)
    sculptor.load_state_dict(g.state_dict('sculptor'), strict=True)
    photographer = models.Photographer(**a_p)
    photographer.load_state_dict(g.state_dict('photographer'), strict=True)
    fuser = fusion.get_fuser('gru', in_channels=g.meta['C'], cube_size=1.0)
    fuser.load_state_dict(g.state_dict('fuser'), strict=True)
    return sculptor.to(device), fuser.to(device), photographer.to(device)


def oracle_arch(meta, which):
    a = dict(meta[f'arch_{which}'])
    a.setdefault('cube_size', 1.0)
    a['num_heads'] = 2
    return a


def random_lfsynth(S, C, seed, device):
    """Random LF-synth(S, C) product networks + their state_dicts (for oracle-vs-CUDA at sizes that
    have no committed golden)."""
    from latentfusion_b200.recon import models, fusion
    from latentfusion_b200.utils import parse_block_config as pbc
    torch.manual_seed(seed)
    a_s = dict(in_size=2 * S, image_config=pbc(f"{C},D,{2*C}:{2*C},{2*C}"), camera_config=pbc(f"{C},{C}"),
               object_config=pbc(f"{C},{C}"), projection_type='factor', input_color=True, input_depth=False,
               input_mask=True, scale_mode='nearest')
    a_p = dict(in_size=S, image_config=pbc(f"{C},D,{2*C}:{2*C},U,{2*C},U,{C}"), camera_config=pbc(f"{C},{C}"),
               object_config=[], projection_type='factor', predict_depth=True, predict_mask=True,
               predict_color=False, scale_mode='nearest')
    sculptor, photographer = models.Sculptor(**a_s), models.Photographer(**a_p)
    fuser = fusion.get_fuser('gru', in_channels=C, cube_size=1.0)
    for m in (sculptor, photographer, fuser):
        for k, p in m.named_parameters():
            if k.endswith('bias'):
                p.data.normal_(0, 0.1)
    arch = {'sculptor': {**a_s, 'cube_size': 1.0, 'num_heads': 2}, 'photographer': {**a_p, 'cube_size': 1.0, 'num_heads': 2}}
    sds = {'sculptor': {k: v.detach().clone() for k, v in sculptor.state_dict().items()},
           'photographer': {k: v.detach().clone() for k, v in photographer.state_dict().items()},
           'fuser': {k: v.detach().clone() for k, v in fuser.state_dict().items()}}
    return sculptor.to(device), fuser.to(device), photographer.to(device), arch, sds


def synthetic_cameras(n, S, seed, perturb=True):
    """Zoomed cameras around the object drawn the way the reference draws them (SURVEY §8d)."""
    from latentfusion_b200 import consts, three
    from latentfusion_b200.modules.geometry import Camera
    from latentfusion_b200.recon.utils import optimal_camera_dist
    from latentfusion_b200.pose import utils as pu
    import math
    torch.manual_seed(seed)
    dist = optimal_camera_dist(615.4991, 2 * S, 0.5, slack=128 / (2 * S))
    K = torch.tensor(consts.INTRINSIC).unsqueeze(0).expand(n, -1, -1).contiguous()
    quats = three.orientation.evenly_distributed_quats(n)
    trans = torch.tensor([[0.0, 0.0, dist]]).expand(n, -1).contiguous()
    cam = Camera(K, three.to_extrinsic_matrix(trans, quats), z_span=0.5, width=640, height=480)
    if perturb:
        cam = pu.perturb_camera(cam, 0.01, 10.0 / 180.0 * math.pi)
    return cam.zoom(None, 2 * S, dist), dist


def cam_to_dict(cam):
    return {k: getattr(cam, k).detach().cpu().clone() for k in ('intrinsic', 'log_quaternion', 'translation', 'viewport')}


def smoke_check(precision=None):
    """Tiny render fwd + loss + bwd-to-camera on cuda:0 against (a) the golden vectors produced by the
    unmodified reference and (b) the CPU oracle.  `precision` selects the convolution path for the duration of the
    check (1 = the tcgen05 bf16x3 kernels bench.py times; None = leave the process default alone)."""
    from latentfusion_b200 import ops
    if precision is not None:
        old = ops.get_default_precision()
        ops.set_default_precision(precision)
        try:
            return smoke_check(None)
        finally:
            ops.set_default_precision(old)
    from oracle import lf_oracle as O
    from latentfusion_b200.pose import estimation
    from latentfusion_b200.observation import Observation
    from latentfusion_b200.recon.inference import LatentFusionModel
    g = Golden()
    dev = torch.device('cuda:0')
    sculptor, fuser, photographer = build_product_models(g, dev)
    model = LatentFusionModel(sculptor, fuser, photographer, g.meta['camera_dist'], dev)
    cam = product_camera(g.cam('hyp_cam'), dev, requires_grad=True)
    z_obj = g['z_obj_gru'].to(dev)
    y, latent = model.render_latent_object(z_obj, cam, return_latent=True, apply_mask=True)
    torch.testing.assert_close(y['depth_logits'].cpu(), g['render.depth_logits'], **OUT_TOL)
    torch.testing.assert_close(y['mask_logits'].cpu(), g['render.mask_logits'], **OUT_TOL)
    gt = product_camera(g.cam('ref_cam_full'), dev)[0:1]
    target = Observation(torch.zeros(1, 3, 480, 640, device=dev), g['target.depth'].to(dev),
                         g['target.mask'].to(dev), gt)
    z_depth = cam.denormalize_depth(y['depth'].squeeze(0))
    losses = estimation.default_pose_loss(target, z_depth, y['mask_logits'].squeeze(0), cam)
    w = json.loads(g.text('loss.weights'))
    sum(w[k] * v for k, v in losses.items()).mean().backward()
    for k in ('log_quaternion', 'translation', 'viewport'):
        torch.testing.assert_close(getattr(cam, k).grad.cpu(), g[f'grad.{k}'], **GRAD_TOL)
    # oracle leg
    ocam = oracle_camera(g.cam('hyp_cam'))
    logits, _ = O.photographer_forward(g.state_dict('photographer'), oracle_arch(g.meta, 'photographer'),
                                       g['z_obj_gru'][0], ocam)
    torch.testing.assert_close(y['depth_logits'].detach().cpu()[0], logits[:, 0:1], **OUT_TOL)
    torch.cuda.synchronize()


class oracle_dtype:
    """Run the PyTorch oracle in another floating type (fp64 = ground truth for conditioning checks)."""

    def __init__(self, dtype):
        self.dtype = dtype

    def __enter__(self):
        import torch.nn.functional as F
        from oracle import lf_oracle as O
        self._O, self._old_resample, self._old_default = O, O.resample, torch.get_default_dtype()
        dt = self.dtype
        O.resample = lambda vol, grid: F.grid_sample(vol.to(dt), grid.to(dt), padding_mode='border', align_corners=False)
        torch.set_default_dtype(dt)
        return self

    def __exit__(self, *exc):
        self._O.resample = self._old_resample
        torch.set_default_dtype(self._old_default)


def assert_grad_close_to_fp64(ours, g32, g64, what='', factor=3.0):
    """Camera gradients are cancelling sums (lever arm ~ camera distance): the reference's own fp32 arithmetic
    deviates from fp64 by err32.  Ours must be as good as that up to a factor, or within 2e-3 of the gradient's
    scale."""
    scale = g64.abs().max()
    err32 = (g32.double() - g64).abs().max()
    err = (ours.double() - g64).abs().max()
    bound = max(factor * float(err32), 2e-3 * float(scale))
    assert float(err) <= bound, f'{what}: |ours - fp64| = {float(err):.4g} > {bound:.4g} (fp32 reference error {float(err32):.4g}, scale {float(scale):.4g})'


GOLDEN_B = os.path.join(ROOT, 'tests', 'golden', 'configB_s64_c32.npz')


GOLDEN_B_SMOOTH = os.path.join(ROOT, 'tests', 'golden', 'configB_s64_c32_smooth.npz')


def config_b_cube(C, S, smooth):
    """oracle/make_golden_configB.py:make_cube — white noise, or the same noise low-pass filtered (5^3 box)."""
    import torch.nn.functional as F
    torch.manual_seed(5)
    z = torch.randn(1, C, S, S, S)
    if smooth:
        z = F.avg_pool3d(F.pad(z, (2, 2, 2, 2, 2, 2), mode='replicate'), 5, stride=1)
        z = z / z.std()
    return z * 0.5


def config_b_case(dev, smooth=False):
    """The benchmarked configuration (BASELINE configs[1]: LF-synth(64, 32), 128^2 render) as pinned by
    oracle/make_golden_configB.py from the unmodified reference: (golden, model, z_obj, target observation)."""
    from latentfusion_b200.observation import Observation
    from latentfusion_b200.recon import fusion, models
    from latentfusion_b200.recon.inference import LatentFusionModel
    from latentfusion_b200.utils import parse_block_config as pbc
    g = Golden(GOLDEN_B_SMOOTH if smooth else GOLDEN_B)
    S, C = g.meta['S'], g.meta['C']
    photographer = models.Photographer(**g.meta['arch_photographer'])
    photographer.load_state_dict(g.state_dict('photographer'), strict=True)
    sculptor = models.Sculptor(in_size=2 * S, image_config=pbc(f"{C},D,{2*C}:{2*C},{2*C}"), camera_config=pbc(f"{C},{C}"),
                               object_config=pbc(f"{C},{C}"), projection_type='factor', input_color=True,
                               input_depth=False, input_mask=True, scale_mode='nearest')
    fuser = fusion.get_fuser('pool:mean', C, 1.0)
    model = LatentFusionModel(sculptor.to(dev), fuser.to(dev), photographer.to(dev), g.meta['camera_dist'], dev)
    z_obj = config_b_cube(C, S, smooth).unsqueeze(0)
    chk = g['z_obj.checksum']
    assert abs(float(z_obj.double().sum()) - float(chk[0])) < 1e-6 * float(chk[1]), 'torch CPU generator drifted'
    t = g.meta['target']
    yy, xx = torch.meshgrid(torch.arange(480, dtype=torch.float32), torch.arange(640, dtype=torch.float32), indexing='ij')
    tmask = (((yy - t['cy']) ** 2 + (xx - t['cx']) ** 2) <= t['radius'] ** 2).float().view(1, 1, 480, 640)
    gt = product_camera(g.cam('gt_cam'), dev)
    target = Observation(torch.zeros(1, 3, 480, 640, device=dev), (tmask * g.meta['camera_dist']).to(dev), tmask.to(dev), gt)
    return g, model, z_obj.to(dev), target
