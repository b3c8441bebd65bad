#!/usr/bin/env python
"""Per-kernel micro-benchmark at BASELINE config-2 extents (dev tool; numbers quoted in profiles/ come
from bench.py's live trace, this is for iterating on one kernel and for ncu captures).

  python tools/kbench.py [--only resample|conv|ibr|loss|all] [--iters 20] [--precision 0|1|2]
"""
import argparse
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
import torch  # noqa: E402

from latentfusion_b200 import ops  # noqa: E402
from latentfusion_b200.modules.geometry import ObjectToCameraTransform  # noqa: E402
from tests import parity_helpers as ph  # noqa: E402


def timeit(fn, iters, flush, reps=8):
    """Median over `iters` of (reps back-to-back launches)/reps: the launches queue up behind an L2-evicting
    fill so host launch latency is hidden and the first launch starts cold; every input/output here is
    larger than L2, so the following ones stream from HBM as well."""
    ms = []
    for _ in range(3):
        fn()
    torch.cuda.synchronize()
    for _ in range(iters):
        flush.fill_(1.0)          # evict L2 (buffer > 126 MB); also keeps the GPU busy while we enqueue
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1) / reps)
    ms.sort()
    return ms[len(ms) // 2], ms[0]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--only', default='all')
    ap.add_argument('--iters', type=int, default=20)
    ap.add_argument('--precision', type=int, default=0)
    ap.add_argument('-S', type=int, default=64)
    ap.add_argument('-C', type=int, default=32)
    ap.add_argument('-N', type=int, default=8)
    a = ap.parse_args()
    S, C, N = a.S, a.C, a.N
    dev = torch.device('cuda:0')
    flush = torch.empty(64 * 1024 * 1024, device=dev)     # 256 MB
    peaks = json.load(open(os.path.join(ROOT, 'MEASURED_PEAKS.json'))) if os.path.exists(os.path.join(ROOT, 'MEASURED_PEAKS.json')) else {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0}
    out = {}
    cams, _ = ph.synthetic_cameras(N, S, seed=9)
    cam = cams.to(dev)
    torch.manual_seed(0)
    vol = ops.to_cl(torch.randn(1, C, S, S, S, device=dev))
    if a.only in ('all', 'resample'):
        T = ObjectToCameraTransform(1.0)
        blk = cam.o2c_block(1.0)
        nbytes = 4 * C * S ** 3 * (1 + N)
        med, best = timeit(lambda: ops.resample_o2c(vol, blk), a.iters, flush)
        out['o2c_fwd'] = dict(ms=med, best_ms=best, GBs=nbytes / med / 1e6, frac=nbytes / med / 1e6 / peaks['hbm_gbs'])
        w = ops.to_cl(torch.randn(N, C, S, S, S, device=dev))
        blk_g = blk.clone().requires_grad_(True)

        def bwd():
            o = ops.resample_o2c(vol, blk_g)
            o.backward(w)
        med2, best2 = timeit(bwd, a.iters, flush)
        out['o2c_fwd+bwd_cam'] = dict(ms=med2, bwd_only_ms=med2 - med, GBs_bwd=nbytes / (med2 - med) / 1e6)
    if a.only in ('all', 'resample', 'bwdcam'):
        # camera gradient alone, straight through the C ABI, per kernel variant (LFB200_BWDCAM)
        import ctypes
        from latentfusion_b200 import _lib as L
        blk = cam.o2c_block(1.0).detach().contiguous()
        w = ops.to_cl(torch.randn(N, C, S, S, S, device=dev))
        ws = torch.empty(L.lib().lf_resample_o2c_bwd_cam_ws(N, S), device=dev)
        gc = torch.empty(N, L.CAMGRAD_STRIDE, device=dev)
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        nbytes = 4 * C * S ** 3 * (1 + N)
        for opt, name in ((0, 'march_4w5_d2'), (2, 'march_8w2_d4'), (1, 'brick')):
            L.check(L.lib().lf_set_option(b'LFB200_BWDCAM', opt), 'opt')
            med, best = timeit(lambda: L.check(L.lib().lf_resample_o2c_bwd_cam(
                ops._p(w), ops._p(vol), ops._p(blk), ops._p(gc), ops._p(ws), 1, N, C, S, st), 'bwd_cam'), a.iters, flush)
            out[f'o2c_bwd_cam[{name}]'] = dict(ms=med, best_ms=best, GBs=nbytes / med / 1e6,
                                              frac=nbytes / med / 1e6 / peaks['hbm_gbs'])
        L.lib().lf_set_option(b'LFB200_BWDCAM', 0)
    if a.only in ('all', 'conv'):
        x = ops.to_cl(torch.randn(N, C, S, S, S, device=dev))
        wgt = torch.randn(C, C, 3, 3, 3, device=dev)
        b = torch.randn(C, device=dev)
        flops = 2 * N * S ** 3 * 27 * C * C
        # straight through the C ABI (weights pre-packed once) so the number is the kernel, not the Python wrapper
        import ctypes, math
        from latentfusion_b200 import _lib as L
        wf, _ = ops._pack_weight(wgt, ops.KIND_CONV, 0)
        desc = ops._desc(ops.KIND_CONV, 3, N, S, S, S, C, C, 3, math.sqrt(2.0 / (27 * C)), True, 0.2, True, a.precision)
        warg = ops._tc_pack(wf, (wgt, id(wgt), wgt._version, 0, 'f')) if a.precision else wf
        y = torch.empty_like(x)
        rn = torch.empty(N * S ** 3, device=dev)
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        args = (ctypes.byref(desc), ops._p(x), ops._p(warg), ops._p(b), ops._p(y), ops._p(rn), st)
        med, best = timeit(lambda: L.check(L.lib().lf_conv_fwd(*args), 'conv'), a.iters, flush)
        out[f'conv3d_block_fwd[p{a.precision}]'] = dict(ms=med, best_ms=best, TFs=flops / med / 1e9,
                                                     GBs=8 * x.numel() / med / 1e6)
        x2 = ops.to_cl(torch.randn(N, C, S, S, S, device=dev))
        w2 = torch.randn(C, C * S, 1, 1, device=dev)
        med, best = timeit(lambda: ops.eq_conv(x2, w2, b, act=True, norm=True, kind=ops.KIND_COLLAPSE, depth=S,
                                               precision=0), a.iters, flush)
        out['collapse_fwd'] = dict(ms=med, GBs=4 * x2.numel() / med / 1e6)
    if a.only in ('all', 'ibr'):
        # IBR colour branch at the configs[1] extents: 16 reference views -> N output views at (2S)^2
        import torch.nn.functional as F
        from latentfusion_b200 import ibr
        P, VI, VO = 2 * S, 16, N
        cin = ph.synthetic_cameras(VI, S, seed=41, perturb=False)[0].to(dev)
        cout = ph.synthetic_cameras(VO, S, seed=42)[0].to(dev)
        image = torch.rand(VI, 3, P, P, device=dev) * 2 - 1
        din = (torch.rand(VI, 1, P, P, device=dev) - 0.5)
        dout = (torch.rand(VO, 1, P, P, device=dev) - 0.5)
        bi, bo = cin.ibr_block(), cout.ibr_block()
        nbytes = 4 * (VO * VI * 4 * P * P + VI * 4 * P * P + VO * P * P)
        with torch.no_grad():
            med, best = timeit(lambda: ops.ibr_reproject(image, din, dout, bi, bo), a.iters, flush)

            def torch_ops():          # the reference's formulation on the device: warp field + two grid_sample calls
                grid = ibr.depth_to_warp_field(cin, cout, dout).reshape(VO * VI, P, P, 2)
                return F.grid_sample(image[None].expand(VO, -1, -1, -1, -1).reshape(VO * VI, 3, P, P), grid,
                                     mode='bilinear', align_corners=False)
            med_t, _ = timeit(torch_ops, max(3, a.iters // 4), flush)
        out['ibr_reproject'] = dict(ms=med, best_ms=best, GBs=nbytes / med / 1e6, frac=nbytes / med / 1e6 / peaks['hbm_gbs'],
                                    torch_ops_colour_only_ms=med_t)
    if os.environ.get('LFB200_TC_DEBUG') and int(os.environ['LFB200_TC_DEBUG']) & 8:
        import ctypes, numpy as np
        from latentfusion_b200 import _lib as L
        buf = np.zeros((3, 64, 2), dtype=np.int64)
        torch.cuda.synchronize()
        L.lib()._handle if False else None
        fn = ctypes.CDLL(L.LIB_PATH).lf_debug_tc_timeline
        fn(buf.ctypes.data_as(ctypes.c_void_p))
        t0 = buf[buf > 0].min()
        for role, name in enumerate(('producer(plane)', 'mma(step)', 'epilogue(step)')):
            rows = [(i, int(buf[role, i, 0] - t0), int(buf[role, i, 1] - t0)) for i in range(40) if buf[role, i, 0] > 0]
            print(name, ' '.join(f'{i}:[{a},{b}]' for i, a, b in rows[:20]))
    if a.only in ('all', 'loss'):
        # the fused pose-loss head at the refine shapes (N hypotheses, 2S x 2S crop, 640 x 480 frame), and the 2-D resize
        # backward at the decoder's / encoder's shapes for N refine views and for the training step's 64 / 128 views
        import ctypes
        from latentfusion_b200 import _lib as L
        P = 2 * S
        torch.manual_seed(1)
        base = torch.randn(N, P, P, 2, device=dev)              # the fused heads' channels-last logits [N,2,P,P]
        vp0, tr0 = cam.viewport.detach().clone(), cam.translation.detach().clone()
        yy, xx = torch.meshgrid(torch.arange(480.0, device=dev), torch.arange(640.0, device=dev), indexing='ij')
        tm = (((yy - 251.5) ** 2 + (xx - 315.4) ** 2) <= 45.0 ** 2).float().view(1, 1, 480, 640)
        td = tm * float(tr0[0, 2])
        med, best = timeit(lambda: ops.pose_loss_terms_packed(base.permute(0, 3, 1, 2), vp0, tr0, td, tm, cam.z_span),
                           a.iters, flush)
        out['pose_loss_fwd'] = dict(ms=med, best_ms=best)
        lg, vp, tr = base.clone().requires_grad_(True), vp0.clone().requires_grad_(True), tr0.clone().requires_grad_(True)
        gt = torch.ones(N, 4, device=dev)

        def loss_fwd_bwd():
            ops.pose_loss_terms_packed(lg.permute(0, 3, 1, 2), vp, tr, td, tm, cam.z_span).backward(gt)
        med2, best2 = timeit(loss_fwd_bwd, a.iters, flush)
        out['pose_loss_fwd+bwd'] = dict(ms=med2, best_ms=best2, bwd_only_ms=med2 - med)
        st = ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)
        for name, n, hw, c, factor in (('up_32to64', N, 32, 64, 2), ('up_64to128', N, 64, 64, 2), ('down_128to64', N, 128, 32, -2),
                                       ('train_up_32to64', 64, 32, 64, 2), ('train_up_64to128', 64, 64, 64, 2),
                                       ('train_down_128to64', 128, 128, 32, -2)):
            ohw = hw * 2 if factor > 0 else hw // 2
            gy = torch.randn(n, ohw, ohw, c, device=dev)
            gx = torch.empty(n, hw, hw, c, device=dev)
            med, best = timeit(lambda: L.check(L.lib().lf_interp_bwd(ops._p(gy), ops._p(gx), 2, n, 1, hw, hw, c, 1, factor, st),
                                               'interp_bwd'), a.iters, flush)
            out[f'interp_bwd_bilinear[{name}]'] = dict(ms=med, best_ms=best, GBs=4 * (gy.numel() + gx.numel()) / med / 1e6)
    print(json.dumps(out, indent=1))


if __name__ == '__main__':
    main()
