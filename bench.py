#!/usr/bin/env python
"""bench.py — pose-refine render iters/sec (16 ref views, 64^3 latent, 128^2 render) on N B200s.

One *step* = one body of GradientPoseEstimator._optimize_camera (reference
pose/estimation.py:601-677) over 8 pose hypotheses per GPU: camera assembly -> render_latent_object
forward -> default_pose_loss -> backward to the 10 camera floats -> per-hypothesis Adam + plateau
scheduler step -> ranking.  Workload = BASELINE.json configs[1]: LF-synth(S=64, C=32), V=16, N=8,
fp32 (SURVEY.md §8d), synthetic ShapeNet-shaped inputs, random-init weights.

  python bench.py [--gpus N] [--steps K] [--warmup W]            our arm (torchrun for N>1)
  python bench.py --impl reference [...]                         the reference algorithm's CPU path
                                                                 (oracle port: plain PyTorch ops on host cores)
Prints ONE JSON line (rank 0).
"""
import argparse
import json
import math
import os
import statistics
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

S, C, V, N_HYP = 64, 32, 16, 8
METRIC = "pose-refine render iters/sec (16-view, 64^3 latent, 128^2 out)"
LOSS_WEIGHTS = dict(depth=1.0, ov_depth=0.3, iou=0.0, mask=0.0, latent=0.0)        # configs/adam_quick.toml
EST_ARGS = dict(optimizer='adam', num_samples=N_HYP, ranking_size=N_HYP, learning_rate=0.01,
                lr_reduce_patience=10, lr_reduce_threshold=1e-4, converge_threshold=1e-6,
                converge_patience=10 ** 9)                                          # never stop early in a timed run


def measured_peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        p = json.load(open(path))
        return dict(hbm_gbs=p['hbm_gbs'], bf16_tflops=p['bf16_tflops'], bf16_tflops_sustained=p['bf16_tflops_sustained'],
                    source='measured (MEASURED_PEAKS.json)')
    return dict(hbm_gbs=6650.0, bf16_tflops=1590.0, bf16_tflops_sustained=1400.0, source='fallback (B200_PROFILING.md)')


class ClockSampler:
    """SM clock / throttle-reason sampler for the timed region.  The region is short (K x ~2.7 ms), so the `nvidia-smi`
    loop (the recipe's clocks line, 20 ms period) is armed BEFORE the warm-up — its start-up takes longer than the whole
    region — and only the rows that arrive between start() and stop() count; the same NVML counters are also read
    in-process every ~2 ms (pynvml) so that the window always holds samples."""
    Q = ('clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,'
         'clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,'
         'clocks_event_reasons.sw_power_cap')

    def __init__(self, index):
        self.index, self.rows, self.proc = index, [], None
        self.t0 = self.t1 = None
        self.nvml_rows, self.nvml_thread, self.nvml_stop = [], None, threading.Event()

    def arm(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', '-i', str(self.index), f'--query-gpu={self.Q}',
                                          '--format=csv,noheader,nounits', '-lms', '20'],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
            import atexit
            atexit.register(lambda p=self.proc: p.poll() is None and p.kill())     # never leave the loop running behind us
        except Exception:
            self.proc = None
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nvml = pynvml
            self.handle = pynvml.nvmlDeviceGetHandleByIndex(self.index)
            self.nvml_thread = threading.Thread(target=self._poll_nvml, daemon=True)
            self.nvml_thread.start()
        except Exception:
            self.nvml_thread = None

    def _pump(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [c.strip() for c in line.split(',')]))

    def _poll_nvml(self):
        n = self.nvml
        while not self.nvml_stop.is_set():
            try:
                self.nvml_rows.append((time.time(), n.nvmlDeviceGetClockInfo(self.handle, n.NVML_CLOCK_SM),
                                       n.nvmlDeviceGetCurrentClocksEventReasons(self.handle)))
            except Exception:
                return
            time.sleep(0.002)

    def start(self):
        if self.proc is None and self.nvml_thread is None:
            self.arm()
        self.t0 = time.time()

    def stop(self):
        self.t1 = time.time()
        self.nvml_stop.set()
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=5)
            except Exception:
                self.proc.kill()
        if self.proc is None and self.nvml_thread is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"], "samples": 0}
        inside = lambda t: self.t0 <= t <= self.t1 + 0.02
        rows = [r for t, r in self.rows if inside(t) and len(r) >= 7]
        clocks = [float(r[0]) for r in rows if r[0].replace('.', '').isdigit()]
        reasons = set()
        for r in rows:
            for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                if v.lower().startswith('active'):
                    reasons.add(name)
        smax = next((float(r[1]) for _, r in self.rows if len(r) >= 7 and r[1].replace('.', '').isdigit()), None)
        n_smi = len(clocks)
        nv = [(c, m) for t, c, m in self.nvml_rows if inside(t)]
        if nv:
            n = self.nvml
            clocks += [float(c) for c, _ in nv]
            bits = (('hw_slowdown', 'nvmlClocksEventReasonHwSlowdown'), ('hw_thermal_slowdown', 'nvmlClocksEventReasonHwThermalSlowdown'),
                    ('sw_thermal_slowdown', 'nvmlClocksEventReasonSwThermalSlowdown'), ('sw_power_cap', 'nvmlClocksEventReasonSwPowerCap'))
            for name, attr in bits:
                bit = getattr(n, attr, None)
                if bit is not None and any(m & bit for _, m in nv):
                    reasons.add(name)
            if smax is None:
                try:
                    smax = float(n.nvmlDeviceGetMaxClockInfo(self.handle, n.NVML_CLOCK_SM))
                except Exception:
                    pass
        return {"sm_mhz": statistics.median(clocks) if clocks else None, "sm_max_mhz": smax,
                "reasons": sorted(reasons), "samples": len(clocks), "samples_nvidia_smi": n_smi, "samples_nvml": len(nv),
                "window_ms": round(1000.0 * (self.t1 - self.t0), 1)}


# ------------------------------------------------------------------------------------------------
# workload construction (identical seeds on both arms)
# ------------------------------------------------------------------------------------------------
def synthetic_inputs(seed=0):
    """Reference views + masks, reference cameras, hypothesis cameras, target observation — all HOST tensors."""
    from tests import parity_helpers as ph
    ref_cams, dist = ph.synthetic_cameras(V, S, seed=seed + 1, perturb=False)
    gt, _ = ph.synthetic_cameras(1, S, seed=seed + 2, perturb=False)
    torch.manual_seed(seed + 3)
    color = torch.rand(1, V, 3, 2 * S, 2 * S) * 2 - 1
    yy, xx = torch.meshgrid(torch.arange(2 * S, dtype=torch.float32), torch.arange(2 * S, dtype=torch.float32), indexing='ij')
    disc = (((yy - S + 0.5) ** 2 + (xx - S + 0.5) ** 2) <= (0.4 * 2 * S) ** 2).float()
    mask = disc.view(1, 1, 1, 2 * S, 2 * S).expand(1, V, -1, -1, -1).contiguous()
    yy, xx = torch.meshgrid(torch.arange(480, dtype=torch.float32), torch.arange(640, dtype=torch.float32), indexing='ij')
    tmask = (((yy - 251.5) ** 2 + (xx - 315.4) ** 2) <= 45.0 ** 2).float().view(1, 1, 480, 640)
    tdepth = tmask * dist
    return dict(ref_cams=ref_cams, gt=gt, dist=dist, color=color, mask=mask, tmask=tmask, tdepth=tdepth)


def hypothesis_cameras(gt_full, n, seed):
    from latentfusion_b200.modules.geometry import Camera
    from latentfusion_b200.pose import utils as pu
    torch.manual_seed(seed)
    return Camera.cat([pu.perturb_camera(gt_full, 0.01, 10.0 / 180.0 * math.pi) for _ in range(n)])


# ------------------------------------------------------------------------------------------------
# reference arm: the reference algorithm on host cores (oracle port, test infrastructure)
# ------------------------------------------------------------------------------------------------
def reference_iteration(O, sds, arch, z_obj, cam_dict, tdepth, tmask, n_hyp):
    """Forward + backward of one refine iteration for n_hyp hypotheses with plain PyTorch CPU ops —
    op for op what the reference executes (F.grid_sample, F.conv3d, ... see oracle/lf_oracle.py)."""
    cam = O.Cam(cam_dict['intrinsic'][:n_hyp], cam_dict['log_quaternion'][:n_hyp].clone().requires_grad_(True),
                cam_dict['translation'][:n_hyp].clone().requires_grad_(True),
                cam_dict['viewport'][:n_hyp].clone().requires_grad_(True))
    # the reference also back-propagates into the (frozen) network weights: keep requires_grad on them
    total, losses, _, _ = O.refine_iteration(sds['photographer'], arch['photographer'], z_obj, cam, tdepth, tmask,
                                             LOSS_WEIGHTS)
    total.mean().backward()
    return total.detach()


def pick_threads(O, sds, arch, z_obj, cam_dict, tdepth, tmask):
    """PyTorch's CPU ops do not scale to every core of a large host (oversubscription makes them slower):
    time one 1-hypothesis iteration at a few thread counts and keep the fastest — the baseline gets the
    best configuration it can use; `cores` in the JSON is the count actually used."""
    cores = os.cpu_count() or 1
    best, best_t = cores, float('inf')
    for nt in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
        torch.set_num_threads(nt)
        reference_iteration(O, sds, arch, z_obj, cam_dict, tdepth, tmask, 1)      # warm
        t0 = time.perf_counter()
        reference_iteration(O, sds, arch, z_obj, cam_dict, tdepth, tmask, 1)
        dt = time.perf_counter() - t0
        if dt < best_t:
            best, best_t = nt, dt
    torch.set_num_threads(best)
    return best


def run_reference(args):
    """Reference arm: the reference's OWN estimator loop (GradientPoseEstimator.estimate, adam_quick.toml) on the host
    cores — the unmodified reference staged under oracle/_ref (kind "reference"), or, when that copy is absent, the
    oracle port of the render+loss+backward part (kind "port").  One step = one full iteration over all N hypotheses
    (render fwd, loss, backward, N Adam + plateau steps, ranking); no extrapolation."""
    rank = int(os.environ.get('RANK', '0'))
    if rank != 0:
        return
    import warnings
    warnings.filterwarnings('ignore')
    os.environ.setdefault('TQDM_DISABLE', '1')
    from oracle import ref_bench
    device = torch.device(args.ref_device)
    cores = os.cpu_count() or 1
    if ref_bench.available():
        kind = 'reference'
        threads = cores
        if device.type == 'cpu':
            # PyTorch CPU ops do not scale to every core of a large host: keep the fastest of a few thread counts
            best = float('inf')
            for nt in sorted({cores, min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
                dt = ref_bench.time_iterations('cpu', 2, 0, 1, threads=nt)
                if dt < best:
                    best, threads = dt, nt
        sec_per_iter = ref_bench.time_iterations(str(device), N_HYP, args.warmup, args.steps, tf32=False,
                                                 threads=threads if device.type == 'cpu' else None)
        sample = (f"{args.steps} full iterations of the unmodified reference's GradientPoseEstimator.estimate() "
                  f"(adam_quick.toml) over all {N_HYP} hypotheses after {args.warmup} warm-up iterations; "
                  f"{'host CPU, ' + str(threads) + ' threads' if device.type == 'cpu' else 'stock PyTorch CUDA ops, TF32 off'}")
        cores_used = threads
    else:
        kind = 'port'
        sec_per_iter, cores_used, sample = _reference_port(args, device)
    value = 1.0 / sec_per_iter
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": "iters/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": sec_per_iter * 1e3, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"configs[1]: LF-synth(S={S},C={C}), V={V}, N={N_HYP} hypotheses, 128^2 render, fp32",
                       "device": str(device)},
            "cpu_baseline": {"value": value, "unit": "iters/s", "cores": cores_used if device.type == 'cpu' else 0,
                             "kind": kind, "sample": sample},
            "e2e": {"value": value, "unit": "iters/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line), flush=True)


def _reference_port(args, device):
    """fallback when oracle/_ref is absent: the oracle port (plain PyTorch ops restating the reference), full N"""
    from oracle import lf_oracle as O
    from tests import parity_helpers as ph
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    cores = os.cpu_count() or 1
    torch.set_num_threads(cores)
    inp = synthetic_inputs()
    torch.manual_seed(0)
    _, _, _, arch, sds = ph.random_lfsynth(S, C, seed=0, device='cpu')
    for k in sds['photographer']:
        sds['photographer'][k] = sds['photographer'][k].to(device).requires_grad_(True)
    torch.manual_seed(5)
    z_obj = torch.randn(1, C, S, S, S, device=device) * 0.5
    hyp = hypothesis_cameras(inp['gt'].uncrop(), N_HYP, seed=7).zoom(None, 2 * S, inp['dist'])
    cam_dict = {k: v.to(device) for k, v in ph.cam_to_dict(hyp).items()}
    tdepth, tmask = inp['tdepth'].to(device), inp['tmask'].to(device)
    if device.type == 'cpu':
        cores = pick_threads(O, sds, arch, z_obj, cam_dict, tdepth, tmask)

    def one():
        if device.type == 'cuda':
            torch.cuda.synchronize()
        t0 = time.perf_counter()
        reference_iteration(_dev(O, device), sds, arch, z_obj, cam_dict, tdepth, tmask, N_HYP)
        if device.type == 'cuda':
            torch.cuda.synchronize()
        return time.perf_counter() - t0

    for _ in range(args.warmup):
        one()
    times = [one() for _ in range(args.steps)]
    return statistics.mean(times), cores, (f"fwd+bwd of all {N_HYP} hypotheses per step; oracle port (plain PyTorch "
                                           f"{device.type} ops restating the reference), no optimiser step")


def _dev(O, device):
    """The oracle builds a few constant tensors on the default device; route them for the cuda context run."""
    if device.type == 'cuda':
        torch.set_default_device(device)
    return O


# ------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------
def run_ours(args):
    import torch.distributed as dist
    from tests import parity_helpers as ph
    from latentfusion_b200 import ops
    from latentfusion_b200.observation import Observation
    from latentfusion_b200.pose import estimation
    from latentfusion_b200.recon.inference import LatentFusionModel

    world = int(os.environ.get('WORLD_SIZE', '1'))
    rank = int(os.environ.get('RANK', '0'))
    local = int(os.environ.get('LOCAL_RANK', '0'))
    if not torch.cuda.is_available():
        raise RuntimeError("bench.py (our arm) needs a CUDA device; there is no CPU fallback")
    torch.cuda.set_device(local)
    dev = torch.device('cuda', local)
    if world > 1:
        os.environ.setdefault('NCCL_DEBUG', 'WARN')      # (NCCL's one-line version banner precedes the JSON line on stdout, as in round 1)
        dist.init_process_group('nccl', device_id=dev)
    ops.set_default_precision(args.precision)

    inp = synthetic_inputs()
    sculptor, fuser, photographer, arch, sds = ph.random_lfsynth(S, C, seed=0, device=dev)
    model = LatentFusionModel(sculptor, fuser, photographer, inp['dist'], dev)

    # ---- reconstruction (once per object, untimed here; reported separately): views shard over ranks,
    # per-view cubes are all-gathered (NCCL), the GRU recurrence runs replicated (SURVEY §8e).
    from latentfusion_b200 import dist as lfdist
    recon_times = []
    for _ in range(3):                      # first call is cold (allocator, weight packing); report the last
        t0 = torch.cuda.Event(enable_timing=True); t1 = torch.cuda.Event(enable_timing=True)
        torch.cuda.synchronize(); t0.record()
        with torch.no_grad():
            z_obj = lfdist.build_latent_object_sharded(model, inp['ref_cams'], inp['color'], inp['mask'], rank, world)
        t1.record(); torch.cuda.synchronize()
        recon_times.append(t0.elapsed_time(t1))
    recon_ms = recon_times[-1]

    # ---- per-rank hypotheses (weak scaling: N_HYP per GPU, independent -> no per-iteration collective)
    hyp_full = hypothesis_cameras(inp['gt'].uncrop(), N_HYP, seed=7 + rank)
    gt_full = inp['gt'].uncrop()
    target_host = Observation(torch.zeros(1, 3, 480, 640).pin_memory(), inp['tdepth'].pin_memory(),
                              inp['tmask'].pin_memory(), gt_full)
    target_dev = target_host.to(dev)
    cfg = {'type': 'gradient', 'args': dict(EST_ARGS, num_iters=args.steps), 'loss_weights': LOSS_WEIGHTS}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(ms):
        if world > 1:
            t = torch.tensor([ms], device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            return t.item()
        return ms

    # L2 hygiene: the per-step working set (8 cubes x 268 MB activations) is >> 126 MB L2, so every
    # iteration streams from HBM; no explicit flush is needed (stated in config.l2).
    # ---------------- device-resident number ("value") ----------------
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.arm()                                             # (nvidia-smi needs longer to start than the region lasts)
    est = estimation.load_from_config(cfg, model, num_iters=args.warmup)
    est.estimate(z_obj, target_dev, camera=hyp_full.to(dev))      # W warm-up iterations (captures the loop body once)
    est.num_iters = args.steps
    barrier()
    if rank == 0:
        sampler.start()
    ops.KernelTrace.reset(enabled=False)
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    timed_best = est.estimate(z_obj, target_dev, camera=hyp_full.to(dev))
    e1.record()
    barrier()
    outputs = timed_outputs(timed_best, getattr(est, '_refiner', None)) if args.dump_outputs else None
    ms_total = max_over_ranks(e0.elapsed_time(e1))
    launches = ops.KernelTrace.launches
    ms_per_step = ms_total / args.steps
    # Per-kernel durations: the timed region above replays a CUDA graph (no events can sit between its
    # nodes), so the same loop body is run eagerly right after it — same stream, same tensors, same kernels —
    # with a CUDA event pair around every C-ABI call, while the clock sampler is still running.
    ktrace, trace_iters = {}, 4
    if not args.no_kernel_events and getattr(est, '_refiner', None) is not None:
        est._refiner._iteration()                                    # settle allocator after the graph run
        torch.cuda.synchronize()
        ops.KernelTrace.reset(enabled=True)
        for _ in range(trace_iters):
            est._refiner._iteration()
        torch.cuda.synchronize()
        ktrace = ops.KernelTrace.summary()
    ops.KernelTrace.reset(False)
    clocks = sampler.stop() if rank == 0 else None
    value = world * 1000.0 / ms_per_step

    # ---------------- strong scaling of configs[2] (64 hypotheses in total, split over the ranks) ----------------
    strong = None
    if not args.no_strong and N_HYP == 8 and 64 % world == 0:
        n_loc = 64 // world
        cfg_s = {'type': 'gradient', 'args': dict(EST_ARGS, num_iters=3, num_samples=n_loc, ranking_size=n_loc),
                 'loss_weights': LOSS_WEIGHTS}
        est_s = estimation.load_from_config(cfg_s, model)
        hyp_s = hypothesis_cameras(gt_full, 64, seed=11)[rank * n_loc:(rank + 1) * n_loc].to(dev)
        est_s.estimate(z_obj, target_dev, camera=hyp_s)          # warm-up (captures this shape's graph)
        est_s.num_iters = 5
        barrier()
        e0.record()
        est_s.estimate(z_obj, target_dev, camera=hyp_s)
        e1.record()
        barrier()
        ms_s = max_over_ranks(e0.elapsed_time(e1)) / 5
        strong = {"workload": "configs[2]: adam_quick.toml at num_samples=64 (64 hypotheses in total, strong scaling)",
                  "hypotheses_total": 64, "hypotheses_per_gpu": n_loc, "ms_per_step": ms_s, "iters_per_s": 1000.0 / ms_s,
                  "hypothesis_renders_per_s": 64 * 1000.0 / ms_s, "steps": 5}
        del est_s

    # ---------------- configs[3]: one reconstruction training iteration, views sharded over the ranks ----------------
    train = None
    if not args.no_train:
        train = train_block(args, dev, rank, world, barrier, max_over_ranks)
    # ---------------- configs[4]: cross-entropy coarse search on the latent loss, 128^3 cube, samples sharded --------
    search = None
    if not args.no_search:
        search = search_block(args, dev, rank, world, barrier, max_over_ranks)

    # ---------------- end-to-end through the public API with HOST buffers ----------------
    # One user-level call: estimator.estimate(z_obj, HOST target observation, HOST hypothesis cameras) for K
    # iterations.  Inside the timed region: the H2D copy of the target (colour+depth+mask, pinned) and of the
    # camera parameters, K replays of the captured loop body, and the D2H drain of every iteration's
    # ranking losses / loss terms / camera snapshots (what the reference reads back per iteration).
    hyp_host = hypothesis_cameras(gt_full, N_HYP, seed=7 + rank)
    for t in (hyp_host.intrinsic, hyp_host.log_quaternion, hyp_host.translation, hyp_host.viewport):
        t.data = t.data.pin_memory()
    h2d_total = sum(t.numel() * 4 for t in (target_host.color, target_host.depth, target_host.mask, hyp_host.intrinsic,
                                            hyp_host.log_quaternion, hyp_host.translation, hyp_host.viewport))
    d2h_per_iter = N_HYP * 4 * (1 + 1 + 4 + 3 + 3)       # rank, optim, 4 terms, log-quaternion, translation
    est_e = est
    barrier()
    e0.record()
    best = est_e.estimate(z_obj, target_host, camera=hyp_host)
    _ = best.translation.sum().item()
    e1.record()
    barrier()
    e2e_ms = max_over_ranks(e0.elapsed_time(e1)) / args.steps
    e2e_value = world * 1000.0 / e2e_ms
    h2d = h2d_total // args.steps
    d2h = d2h_per_iter

    if world > 1:
        dist.destroy_process_group()
    if rank != 0:
        return
    if outputs is not None:
        os.makedirs(args.dump_outputs, exist_ok=True)
        for name, a in outputs.items():
            np.save(os.path.join(args.dump_outputs, f'{name}.npy'), a)

    # ---------------- roofline of the dominant kernel + per-kernel table ----------------
    peaks = measured_peaks()
    kernels = {}
    for name, d in ktrace.items():
        gbs = d['bytes'] / d['calls'] / (d['ms_avg'] * 1e-3) / 1e9 if d['bytes'] else None
        tfs = d['flops'] / d['calls'] / (d['ms_avg'] * 1e-3) / 1e12 if d['flops'] else None
        kernels[name] = {"calls_per_step": d['calls'] / trace_iters, "ms_avg": round(d['ms_avg'], 4),
                         "share_of_step": round(d['ms_total'] / trace_iters / ms_per_step, 4),
                         "achieved_GBs": None if gbs is None else round(gbs, 1),
                         "achieved_TFs": None if tfs is None else round(tfs, 2)}
    traffic = {}
    tpath = os.path.join(ROOT, 'profiles', 'r02_traffic.json')
    if os.path.exists(tpath):
        traffic = json.load(open(tpath))        # dram bytes per launch from the committed ncu --set full captures
    roof = None
    if ktrace:
        top = max(ktrace.items(), key=lambda kv: kv[1]['ms_total'])
        name, d = top
        conv_like = d['flops'] > 0 and (d['flops'] / max(d['bytes'], 1)) > 50
        if conv_like:
            peak = peaks['bf16_tflops_sustained']
            ach = d['flops'] / d['calls'] / (d['ms_avg'] * 1e-3) / 1e12
            tr = traffic.get('conv3d_dz_kernel') if (args.precision and 'conv3d' in name) else None
            roof = {"kernel": name, "bound": "tensor", "achieved": round(ach, 2), "peak": peak, "unit": "TFLOP/s",
                    "frac": round(ach / peak, 4), "traffic": tr,
                    "products_per_mac": 3 if args.precision in (1, 3) else 1,
                    "issued_TFs": round(ach * (3 if args.precision in (1, 3) else 1), 1),
                    "issued_frac": round(ach * (3 if args.precision in (1, 3) else 1) / peak, 4),
                    "peak_source": peaks['source'] + ' bf16 sustained',
                    "note": ("algorithmic flops 2*27*Cin*Cout*positions counted ONCE; precision 1 (bf16x3) issues 3 tensor-core "
                             "products per tap in one kernel pass (depth-batched N=3*Cout MMAs): the tensor-pipe rate is issued_TFs = 3 x achieved, "
                             "and frac is capped at 1/3 for this fp32-parity arithmetic")
                            if args.precision in (1, 3) else "algorithmic flops 2*27*Cin*Cout*positions"}
        else:
            peak = peaks['hbm_gbs']
            ach = d['bytes'] / d['calls'] / (d['ms_avg'] * 1e-3) / 1e9
            roof = {"kernel": name, "bound": "hbm", "achieved": round(ach, 1), "peak": peak, "unit": "GB/s",
                    "frac": round(ach / peak, 4), "traffic": None, "peak_source": peaks['source']}
    res = kernels.get('lf_resample_o2c_fwd')
    resample_roof = None
    if res and res['achieved_GBs']:
        resample_roof = {"kernel": "lf_resample_o2c_fwd", "bound": "hbm", "achieved": res['achieved_GBs'],
                         "peak": peaks['hbm_gbs'], "unit": "GB/s", "frac": round(res['achieved_GBs'] / peaks['hbm_gbs'], 4),
                         "algorithmic_bytes": 4 * C * S ** 3 * (1 + N_HYP), "traffic": traffic.get('resample_fwd_kernel'),
                         "peak_source": peaks['source']}

    # ---------------- CPU baseline (bounded sample, rank 0, N=1 only) + the stock-PyTorch-CUDA context number ----------
    cpu = None
    ref_cuda = None
    if world == 1 and not args.no_cpu_baseline:
        del est, est_e
        torch.cuda.empty_cache()
        cpu = cpu_baseline(sds, arch, inp)
        ref_cuda = reference_cuda_block(dev)

    line = {"metric": METRIC, "value": value, "unit": "iters/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f32" if args.precision == 0 else ("bf16x3" if args.precision == 1 else "bf16"),
            "data": "synthetic",
            "config": {"workload": f"configs[{1 if N_HYP == 8 else 2}]: LF-synth(S={S},C={C}), V={V} ref views, N={N_HYP} hypotheses/GPU, "
                                   f"128^2 render, fp32 storage; 1 iter = render fwd + pose loss + bwd to cameras + Adam",
                       "hypotheses_per_gpu": N_HYP, "hypothesis_renders_per_s": value * N_HYP,
                       "parallelism": f"hypotheses sharded x{world}, z_obj replicated",
                       "l2": "per-step working set (>2 GB of activations) exceeds the 126 MB L2; no flush needed",
                       "precision": args.precision, "recon_ms_once_per_object": round(recon_ms, 2),
                       "recon_ms_first_call": round(recon_times[0], 2)},
            "e2e": {"value": e2e_value, "unit": "iters/s", "ms_per_step": e2e_ms, "h2d_bytes_per_step": h2d,
                    "d2h_bytes_per_step": d2h,
                    "note": "one estimator.estimate(z_obj, host target obs, host cameras) call of K iterations / K: includes H2D of target+cameras (graph captured once, during warm-up), per-iteration D2H of losses and camera snapshots"},
            "gpu_launches": launches, "clocks": clocks, "roofline": roof, "roofline_resample": resample_roof,
            "kernels": kernels, "cpu_baseline": cpu, "reference_cuda": ref_cuda, "strong_scaling": strong,
            "train_step": train, "coarse_search": search,
            "recon": {"ms": round(recon_ms, 2), "ms_first_call": round(recon_times[0], 2), "views": V,
                      "views_per_gpu": (V + world - 1) // world, "fuser": "gru",
                      "note": "LatentFusionModel.build_latent_object, views sharded over the ranks (dist.py), max over ranks"}}
    print(json.dumps(line), flush=True)


def timed_outputs(best, refiner):
    """Host float32 copies of what the timed estimate() call computed: the ranked cameras it returns and, from its
    last iteration, every hypothesis' rank loss, loss terms and updated camera parameters (this rank's hypotheses).
    Every reduction on this path adds in a fixed order, so runs with the same arguments write the same bits."""
    out = {'best_translation': best.translation, 'best_log_quaternion': best.log_quaternion}
    if refiner is not None:
        last = (int(refiner.slot) - 1) % refiner.chunk  # the slot advances after every replayed iteration
        out.update(last_rank_loss=refiner.h_rank[last], last_loss_terms=refiner.h_terms[last],
                   hyp_log_quaternion=refiner.lq, hyp_translation=refiner.tr, hyp_viewport=refiner.vp)
    return {k: v.detach().float().cpu().numpy() for k, v in out.items()}


def train_block(args, dev, rank, world, barrier, max_over_ranks, B=8, vin=16, vout=8):
    """BASELINE configs[3]: ReconTrainer.run_iteration (generator half, released recipe) on B objects x vin input views,
    vout reconstruction views, LF-synth(64, 32).  The views of every object shard over the ranks (each rank encodes
    vin/world views, decodes vout/world), per-view cubes are all-gathered with a differentiable collective, weight
    gradients all-reduced in one flat bucket (latentfusion_b200/train.py)."""
    from tests import parity_helpers as ph
    from latentfusion_b200 import ops
    from latentfusion_b200.train import ReconTrainStep
    torch.cuda.reset_peak_memory_stats()
    if vin % world or vout % world:
        return {"skipped": f"views ({vin} in / {vout} out) do not divide over {world} ranks"}
    import torch.distributed as dist
    sculptor, fuser, photographer, _, _ = ph.random_lfsynth(S, C, seed=0, device=dev)
    step = ReconTrainStep(sculptor, fuser, photographer, depth_k=4096, group=(dist.group.WORLD if world > 1 else None))
    P, vi, vo = 2 * S, vin // world, vout // world
    cin, _ = ph.synthetic_cameras(B * vin, S, seed=21, perturb=False)
    cout, _ = ph.synthetic_cameras(B * vout, S, seed=22, perturb=False)
    pick = lambda cams, v, vl: cams[[b * v + rank * vl + j for b in range(B) for j in range(vl)]]    # noqa: E731
    # the same global batch at every world size (each rank keeps its view slice): the reported loss is then comparable
    # across N (equal up to fp32 reassociation of the sharded sums)
    g = torch.Generator().manual_seed(23)
    cut = lambda t, vl: t[:, rank * vl:(rank + 1) * vl].contiguous().pin_memory()                 # noqa: E731
    host = {'image': cut(torch.rand(B, vin, 3, P, P, generator=g) * 2 - 1, vi),
            'mask': cut((torch.rand(B, vin, 1, P, P, generator=g) > 0.4).float(), vi),
            'depth': cut(torch.rand(B, vout, 1, P, P, generator=g) * 2 - 1, vo),
            'gmask': cut((torch.rand(B, vout, 1, P, P, generator=g) > 0.5).float(), vo)}

    def one():
        batch = {'in': {'camera': pick(cin, vin, vi).to(dev), 'image': host['image'].to(dev, non_blocking=True),
                        'mask': host['mask'].to(dev, non_blocking=True)},
                 'out_gt': {'camera': pick(cout, vout, vo).to(dev), 'depth': host['depth'].to(dev, non_blocking=True),
                            'mask': host['gmask'].to(dev, non_blocking=True)}}
        return float(step.run_iteration(batch)['total'])          # D2H of the loss: the step's result
    one()
    ops.KernelTrace.reset(False)
    barrier()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    e0.record()
    steps = 2
    for _ in range(steps):
        loss = one()
    e1.record()
    barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / steps
    launches = ops.KernelTrace.launches // steps
    mem = torch.cuda.max_memory_allocated() / 2 ** 30
    del step, sculptor, fuser, photographer
    torch.cuda.empty_cache()
    return {"workload": f"configs[3]: {B} objects x {vin} input + {vout} reconstruction views, LF-synth({S},{C}), "
                        f"hard smooth-L1 depth + BCE mask, Adam(0, 0.99); views sharded x{world}",
            "ms_per_step": round(ms, 2), "object_views_per_s": round(B * (vin + vout) * 1000.0 / ms, 2), "steps": steps,
            "loss": loss, "lfb200_launches_per_step": launches, "peak_mem_gb": round(mem, 1),
            "h2d_bytes_per_step": sum(t.numel() * 4 for t in host.values()), "precision": args.precision,
            "note": "e2e: pinned host batch -> device inside the timed region, loss read back every step; 3x3x3 weight "
                    "gradients on the tensor cores (lf_conv3d_dw), the 2-D / projection ones on lf_conv_bwd_weight"}


def search_block(args, dev, rank, world, barrier, max_over_ranks, S4=128, C4=16, gens=2):
    """BASELINE configs[4]: CrossEntropyPoseEstimator with configs/cross_entropy_latent.toml (latent = 1.0, 96 samples x
    flips per generation) on a 128^3 latent cube: reconstruction of 16 views sharded over the ranks (NCCL all-gather of
    the per-view cubes), then `gens` timed generations whose samples shard over the ranks (scores all-gathered)."""
    import torch.distributed as dist
    from tests import parity_helpers as ph
    from latentfusion_b200 import dist as lfdist
    from latentfusion_b200.observation import Observation
    from latentfusion_b200.pose import estimation
    from latentfusion_b200.recon.inference import LatentFusionModel
    torch.cuda.reset_peak_memory_stats()
    sculptor, fuser, photographer, _, _ = ph.random_lfsynth(S4, C4, seed=0, device=dev)
    ref_cams, dist_ = ph.synthetic_cameras(V, S4, seed=31, perturb=False)
    gt, _ = ph.synthetic_cameras(1, S4, seed=32, perturb=False)
    model = LatentFusionModel(sculptor, fuser, photographer, dist_, dev)
    P = 2 * S4
    g = torch.Generator().manual_seed(33)
    color = torch.rand(1, V, 3, P, P, generator=g) * 2 - 1
    mask = (torch.rand(1, V, 1, P, P, generator=g) > 0.3).float()
    e0 = torch.cuda.Event(enable_timing=True); e1 = torch.cuda.Event(enable_timing=True)
    recon = []
    for _ in range(3):                      # cold, allocator settling, steady
        barrier(); e0.record()
        with torch.no_grad():
            z_obj = lfdist.build_latent_object_sharded(model, ref_cams, color, mask, rank, world)
        e1.record(); barrier()
        recon.append(max_over_ranks(e0.elapsed_time(e1)))
    yy, xx = torch.meshgrid(torch.arange(480, dtype=torch.float32), torch.arange(640, dtype=torch.float32), indexing='ij')
    tmask = (((yy - 251.5) ** 2 + (xx - 315.4) ** 2) <= 45.0 ** 2).float().view(1, 1, 480, 640)
    gt_full = gt.uncrop()
    # (a sloped disc: the reference's initial-pose estimate rejects outliers by MAD, which is 0 on a constant depth)
    tdepth = tmask * (dist_ + 0.05 * ((xx - 315.4) / 45.0).view(1, 1, 480, 640))
    target = Observation(torch.rand(1, 3, 480, 640, generator=g), tdepth, tmask, gt_full).to(dev)
    cfg = {'type': 'cross_entropy',
           'args': dict(num_samples=96, num_iters=30, ranking_size=16, num_elites=48, num_gmm_components=6,
                        learning_rate=0.3, sample_flipped=True, init_hemisphere=False, init_upright=False),
           'loss_weights': dict(depth=0.0, ov_depth=0.0, iou=0.0, mask=0.0, latent=1.0)}
    est = estimation.load_from_config(cfg, model)
    est.verbose = False
    est.num_iters = 1                         # (the elite schedule keeps the config's 30-generation horizon)
    group = dist.group.WORLD if world > 1 else None
    torch.manual_seed(5)                      # every rank draws the same population
    np.random.seed(5)
    est.estimate(z_obj, target, group=group)                      # warm-up generation
    est.num_iters = gens
    barrier(); e0.record()
    est.estimate(z_obj, target, group=group)
    e1.record(); barrier()
    ms = max_over_ranks(e0.elapsed_time(e1)) / gens
    renders = getattr(est, 'last_renders_per_generation', None) or 96
    mem = torch.cuda.max_memory_allocated() / 2 ** 30
    del est, model
    torch.cuda.empty_cache()
    return {"workload": f"configs[4]: cross_entropy_latent.toml (latent=1.0), LF-synth({S4},{C4}), 16 ref views; "
                        f"samples sharded x{world}", "ms_per_generation": round(ms, 2), "renders_per_generation": renders,
            "renders_per_s": round(renders * 1000.0 / ms, 1), "generations": gens,
            "recon_ms": round(recon[-1], 2), "recon_ms_first_call": round(recon[0], 2), "peak_mem_gb": round(mem, 1),
            "note": "generation = sample (GMM, host) -> zoom -> Photographer.decode forward -> fused forward-only loss head + latent "
                    "cosine -> all-gather scores -> refit GMM on elites (host, sklearn)"}


def cpu_baseline(sds, arch, inp):
    """The reference timed beside the GPU number, on the box's host cores, bounded (one warm + two timed full
    iterations over all N hypotheses): the unmodified reference's estimator when oracle/_ref is staged, else the port."""
    import warnings
    warnings.filterwarnings('ignore')
    os.environ.setdefault('TQDM_DISABLE', '1')
    from oracle import ref_bench
    cores = os.cpu_count() or 1
    if ref_bench.available():
        best, threads = float('inf'), cores
        for nt in sorted({min(cores, 64), min(cores, 32), min(cores, 16), min(cores, 8)}, reverse=True):
            dt = ref_bench.time_iterations('cpu', 2, 0, 1, threads=nt)
            if dt < best:
                best, threads = dt, nt
        sec = ref_bench.time_iterations('cpu', N_HYP, 1, 2, threads=threads)
        return {"value": 1.0 / sec, "unit": "iters/s", "cores": threads, "kind": "reference",
                "sample": f"2 full iterations (after 1 warm-up) of the unmodified reference's GradientPoseEstimator over all "
                          f"{N_HYP} hypotheses, host CPU, {threads} threads (fastest of 64/32/16/8)"}
    from oracle import lf_oracle as O
    from tests import parity_helpers as ph
    torch.set_num_threads(cores)
    sd = {k: v.detach().cpu().clone().requires_grad_(True) for k, v in sds['photographer'].items()}
    torch.manual_seed(5)
    z_obj = torch.randn(1, C, S, S, S) * 0.5
    hyp = hypothesis_cameras(inp['gt'].uncrop(), N_HYP, seed=7).zoom(None, 2 * S, inp['dist'])
    cam_dict = ph.cam_to_dict(hyp)
    cores = pick_threads(O, {'photographer': sd}, arch, z_obj, cam_dict, inp['tdepth'], inp['tmask'])
    t0 = time.perf_counter()
    reps = 2
    for _ in range(reps):
        reference_iteration(O, {'photographer': sd}, arch, z_obj, cam_dict, inp['tdepth'], inp['tmask'], N_HYP)
    sec = (time.perf_counter() - t0) / reps
    return {"value": 1.0 / sec, "unit": "iters/s", "cores": cores, "kind": "port",
            "sample": f"{reps} x (fwd+bwd of all {N_HYP} hypotheses); plain PyTorch CPU ops restating the reference "
                      f"(oracle/lf_oracle.py), {cores} threads"}


def reference_cuda_block(dev):
    """Context (north_star's ">= 10x the reference PyTorch render loop"): the unmodified reference's estimator on this
    same GPU through stock PyTorch CUDA ops, TF32 off (the fp32-parity setting) and on (PyTorch's cuDNN default)."""
    from oracle import ref_bench
    if not ref_bench.available():
        return None
    out = {"kind": "reference", "steps": 20, "warmup": 2, "unit": "iters/s"}
    for name, tf32 in (("tf32_off", False), ("tf32_on", True)):
        sec = ref_bench.time_iterations(str(dev), N_HYP, 2, 20, tf32=tf32)
        out[name] = 1.0 / sec
        torch.cuda.empty_cache()
    torch.backends.cudnn.allow_tf32 = False
    torch.backends.cuda.matmul.allow_tf32 = False
    return out


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=20)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--precision', type=int, default=int(os.environ.get('LFB200_PRECISION', '1')),
                    help='0 exact fp32 FFMA convs; 1 tcgen05 bf16x3 split (fp32-parity grade, default); 2 tcgen05 bf16')
    ap.add_argument('--ref-device', default='cpu', help='reference arm device (cpu = the baseline; cuda = context)')
    ap.add_argument('--ref-hyp', type=int, default=2, help='hypotheses per reference step (bounded sample)')
    ap.add_argument('--hypotheses', type=int, default=N_HYP,
                    help='hypotheses per GPU (default 8 = BASELINE configs[1]; 64 = configs[2], adam_quick.toml at num_samples=64)')
    ap.add_argument('--no-kernel-events', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-strong', action='store_true', help='skip the configs[2] strong-scaling extra')
    ap.add_argument('--no-train', action='store_true', help='skip the configs[3] training-iteration extra')
    ap.add_argument('--no-search', action='store_true', help='skip the configs[4] coarse-search extra')
    ap.add_argument('--dump-outputs', metavar='DIR',
                    help='write what the timed path computed in its last step as DIR/<name>.npy (float32; with --gpus '
                         '> 1, rank 0\'s hypotheses and the merged ranking); the inputs are seeded, so runs with the same '
                         'arguments can be compared output for output')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl != 'ours':
        ap.error('--dump-outputs applies to --impl ours')
    args.warmup = max(args.warmup, 0)
    if args.hypotheses != N_HYP:
        globals()['N_HYP'] = args.hypotheses
        EST_ARGS.update(num_samples=args.hypotheses, ranking_size=args.hypotheses)
    if args.impl == 'reference':
        run_reference(args)
    else:
        args.warmup = max(args.warmup, 3)
        run_ours(args)


if __name__ == '__main__':
    main()
