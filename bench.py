#!/usr/bin/env python3
# -*- coding: utf-8 -*-
"""Benchmark of the Stereo2Voxel forward hot path (BASELINE.json: "stereo pairs/sec Stereo2Voxel fwd").

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path, one rank per GPU
    python bench.py --impl reference --gpus N --steps K ...  # CPU oracle (north_star restatement) on host cores

A "step" is one Stereo2Voxel forward over one batch of synthetic stereo pairs (config.py default
size, random-init weights): BASELINE configs[1] (batch 64 per GPU, bf16 unless --precision).  With
N GPUs every rank runs its own batch of 64 (weak scaling: 64*N pairs per step = configs[2]'s 512 at
N=8) and the per-shard IoU counts are summed with one NCCL all-reduce per step.

Prints ONE JSON line (rank 0).  `value` = pairs/s with inputs resident in HBM; `e2e` = the same through
the public nn.Module call with pinned HOST inputs (decoded 8-bit HWC images -- the reference's inputs are PNG renders,
README.md:73-74 -- H2D inside the timed region, voxels + IoU read back).

--dump-outputs DIR writes what the last timed step of the resident loop returned (disp_left, disp_right, voxels, iou_counts)
as DIR/<name>.npy, after that loop and outside every timed region.  Inputs and weights are seeded, so two builds run with the
same arguments can be compared output for output.

The same line carries the other BASELINE configs as extra keys, each measured briefly in the same run (N = 1):
  fp32_mode              configs[1] "fp32": the fast tensor-core mode that meets the 1e-3 tolerance ('bf16x3'), with its error
  latency                B = 1 / 8 through the CUDA-graph replay
  stereo2point_chamfer   configs[3]: Stereo2Point forward + chamfer_dist at B = 32, 2048 vs 16384 points
  costvolume_sweep       configs[4]: D in {32,64,128} x C in {32,64} at 1/4 resolution, HBM fraction per point
  gpu_stock_baseline     the oracle module on the SAME GPU through stock torch + cuDNN (the on-box bar, SURVEY.md 8(d))
  peaks_measured         TF32 matmul and fp32 FMA issue peaks measured in this run
and, at N > 1, `strong_512`: configs[2] as written (global batch 512 sharded over the N GPUs).  --no-extras skips them.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)


def parse():
    p = argparse.ArgumentParser()
    p.add_argument('--gpus', type=int, default=1)
    p.add_argument('--steps', type=int, default=10)
    p.add_argument('--warmup', type=int, default=3)
    p.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    p.add_argument('--batch', type=int, default=None, help='pairs per GPU per step (default cfg.CONST.BATCH_SIZE = 64)')
    p.add_argument('--precision', default='bf16', choices=['bf16', 'bf16x3', 'tf32', 'tf32x3', 'fp32'])
    p.add_argument('--no-cpu-baseline', action='store_true')
    p.add_argument('--no-extras', action='store_true', help='only the headline measurement (no secondary configs)')
    p.add_argument('--dump-outputs', metavar='DIR', default=None,
                   help='write the outputs of the last timed step of the headline loop (rank 0) as DIR/<name>.npy')
    return p.parse_args()


def peaks():
    path = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(path):
        d = json.load(open(path))
        return {'hbm_gbs': d['hbm_gbs'], 'bf16_tflops': d['bf16_tflops'], 'bf16_tflops_sustained': d['bf16_tflops_sustained'],
                'source': 'measured'}
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0, 'source': 'fallback'}


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""

    def __init__(self, index=0):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._index = index
        self._t = threading.Thread(target=self._run, daemon=True)

    def _run(self):
        # NVML in-process (a query takes ~0.1 ms, so even a 150 ms timed region gets dozens of samples);
        # nvidia-smi subprocesses (~80 ms each) only as a fallback
        try:
            import pynvml as nv
            nv.nvmlInit()
            h = nv.nvmlDeviceGetHandleByIndex(self._index)
            self.max_mhz = float(nv.nvmlDeviceGetMaxClockInfo(h, nv.NVML_CLOCK_SM))
            bits = {'hw_slowdown': 0x8, 'hw_thermal_slowdown': 0x40, 'sw_thermal_slowdown': 0x20, 'sw_power_cap': 0x4}
            get_reasons = getattr(nv, 'nvmlDeviceGetCurrentClocksEventReasons', None) or \
                getattr(nv, 'nvmlDeviceGetCurrentClocksThrottleReasons')
            while not self._stop.is_set():
                self.samples.append(float(nv.nvmlDeviceGetClockInfo(h, nv.NVML_CLOCK_SM)))
                r = get_reasons(h)
                for n, b in bits.items():
                    if r & b:
                        self.reasons.add(n)
                self._stop.wait(0.004)
            return
        except Exception:
            pass
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        while not self._stop.is_set():
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self._index), '--query-gpu=' + q, '--format=csv,noheader,nounits'],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(',')
                self.samples.append(float(out[0]))
                self.max_mhz = float(out[1])
                for n, v in zip(names, out[2:]):
                    if v.strip().lower().startswith('active'):
                        self.reasons.add(n)
            except Exception:
                pass
            self._stop.wait(0.1)

    def __enter__(self):
        self._t.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        self._t.join(2)

    def summary(self):
        s = sorted(self.samples)
        return {'sm_mhz': s[len(s) // 2] if s else None, 'sm_max_mhz': self.max_mhz, 'reasons': sorted(self.reasons),
                'samples': len(s)}


def cpu_oracle_run(cfg, sample_pairs, steps, warmup, threads):
    """Times the oracle (stock torch.nn restatement of the north_star) on the host cores."""
    import torch
    from oracle import models as O
    from stereo_3d_reconstruction_b200.utils import synthetic
    torch.set_num_threads(threads)
    m = O.make_model('Stereo2Voxel', cfg, seed=cfg.CONST.SEED)
    left, right, _ = synthetic.stereo_pair(sample_pairs, cfg.CONST.IMG_H, cfg.CONST.IMG_W, 2 * cfg.NETWORK.MAX_DISP, seed=0)
    with torch.no_grad():
        for _ in range(warmup):
            m(left, right)
        t0 = time.perf_counter()
        for _ in range(steps):
            m(left, right)
        dt = time.perf_counter() - t0
    return sample_pairs * steps / dt, dt / steps


def run_reference(args):
    """--impl reference: the reference's own implementation of the path cannot be run (its source is
    not on disk: /root/reference = README.md + requirements.txt), so this arm times the oracle port on
    all host cores, on a bounded sample of the same workload."""
    rank = int(os.environ.get('RANK', 0))
    if rank != 0:
        return
    from config import cfg
    cores = os.cpu_count() or 1
    sample = 8
    value, sec = cpu_oracle_run(cfg, sample, max(1, args.steps), max(1, min(args.warmup, 2)), cores)
    B = args.batch or cfg.CONST.BATCH_SIZE
    line = {
        'impl': 'reference', 'metric': 'stereo pairs/sec Stereo2Voxel fwd', 'value': value, 'unit': 'pairs/s',
        'n_gpus': args.gpus, 'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': sec * 1e3,
        'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': 'Stereo2Voxel forward, batch %d per GPU, %dx%d, D=%d (CPU arm: bounded sample of %d pairs per step)'
                   % (B, cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.NETWORK.MAX_DISP, sample)},
        'cpu_baseline': {'value': value, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port',
                         'sample': '%d pairs per step, %d steps, fp32 torch.nn oracle (north_star restatement; reference source not on disk)'
                                   % (sample, args.steps)},
        'e2e': {'value': value, 'unit': 'pairs/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
    }
    print(json.dumps(line))



# ---------------------------------------------------------------------------------------------------------------------
# Secondary BASELINE configs, measured briefly on rank 0 at N = 1 and reported as extra keys of the same JSON line.
# Every timing: >= 3 warm-ups, CUDA events on the launching stream, inputs larger than L2 or an explicit L2 flush.
# ---------------------------------------------------------------------------------------------------------------------
def _events_ms(fn, iters, warm=3, flush=None):
    """Median ms of `fn` over `iters` single launches, each preceded by an L2 flush when `flush` is given."""
    import torch
    for _ in range(warm):
        fn()
    ts = []
    for _ in range(iters):
        if flush is not None:
            flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); fn(); e1.record()
        torch.cuda.synchronize()
        ts.append(e0.elapsed_time(e1))
    ts.sort()
    return ts[len(ts) // 2]


def _rotating_ms(make_fn, inputs, rounds=4, warm=1):
    """Mean ms per launch of back-to-back launches cycling over `inputs` -- distinct copies of the operand whose total size
    exceeds L2 (126 MB), so every launch reads cold data without an L2 flush in between; launch latency and event overhead
    (~10 us per isolated launch, as much as a 10-20 us kernel itself) are amortised over rounds * len(inputs) launches."""
    import torch
    fns = [make_fn(x) for x in inputs]
    for _ in range(warm):
        for f in fns:
            f()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(rounds):
        for f in fns:
            f()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / (rounds * len(fns))


def _loop_ms(fn, iters, warm=3):
    """Mean ms per call of `iters` back-to-back calls (for steps that stream far more than L2 per call)."""
    import torch
    for _ in range(warm):
        fn()
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        fn()
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def extra_fp32_mode(cfg0, B, dev, steps):
    """configs[1] 'fp32': 'bf16x3' (bf16 hi/lo pairs, three MMAs per product) -- throughput at batch B and the error
    against the CPU oracle on 1 pair of the same default config (tolerance the north_star states for fp32: 1e-3)."""
    import torch
    from oracle import models as O
    from stereo_3d_reconstruction_b200 import models
    from stereo_3d_reconstruction_b200.utils import synthetic
    cfg = cfg0.clone()
    cfg.NETWORK.PRECISION = 'bf16x3'
    cfg.CONST.MICRO_BATCH = max(B, cfg.CONST.MICRO_BATCH)
    H, W, D = cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.NETWORK.MAX_DISP
    model = models.build_model('Stereo2Voxel', cfg, seed=cfg.CONST.SEED).to(dev).pack()
    sets = [tuple(t.to(dev) for t in synthetic.stereo_pair(B, H, W, 2 * D, seed=77 + i)[:2]) for i in range(2)]
    it = [0]

    def step():
        l, r = sets[it[0] & 1]; it[0] += 1
        model(l, r)
    ms = _loop_ms(step, max(3, min(steps, 5)))
    oracle = O.make_model('Stereo2Voxel', cfg, seed=cfg.CONST.SEED)
    l1, r1, _ = synthetic.stereo_pair(1, H, W, 2 * D, seed=99)
    with torch.no_grad():
        rdl, rdr, rvox = oracle(l1, r1)
        dl, dr, vox = model(l1.to(dev), r1.to(dev))
    dmax = max(rdl.abs().max().item(), rdr.abs().max().item())
    e_d = max((dl.cpu() - rdl).abs().max().item(), (dr.cpu() - rdr).abs().max().item()) / dmax
    e_v = (vox.cpu() - rvox).abs().max().item()
    del model
    torch.cuda.empty_cache()
    return {'precision': 'bf16x3', 'what': 'bf16 hi/lo operand pairs, hi*hi + lo*hi + hi*lo per product on kind::f16 MMAs, fp32 accumulate',
            'value': B / ms * 1e3, 'unit': 'pairs/s', 'ms_per_step': ms, 'batch': B,
            'disparity_rel_err_vs_oracle': e_d, 'occupancy_abs_err_vs_oracle': e_v, 'tolerance': 1e-3,
            'within_tolerance': bool(e_d <= 1e-3 and e_v <= 1e-3)}


def extra_latency(model, cfg, dev):
    """Small-batch latency through the CUDA-graph replay (one graph launch per forward)."""
    import torch
    from stereo_3d_reconstruction_b200.utils import synthetic
    out = {}
    for b in (1, 8):
        l, r, _ = synthetic.stereo_pair(b, cfg.CONST.IMG_H, cfg.CONST.IMG_W, 2 * cfg.NETWORK.MAX_DISP, seed=300 + b)
        l, r = l.to(dev), r.to(dev)
        with torch.no_grad():
            ms = _loop_ms(lambda: model.graphed(l, r), 30, warm=5)
        out['b%d_ms' % b] = ms
        out['b%d_pairs_per_s' % b] = b / ms * 1e3
    out['how'] = 'model.graphed(): CUDA-graph replay, inputs resident, bf16'
    return out


def extra_stereo2point(cfg0, dev, fma_peak):
    """configs[3]: Stereo2Point forward + chamfer_dist, batch 32, 2048 predicted vs 16384 GT points."""
    import torch
    from stereo_3d_reconstruction_b200 import models, ops
    from stereo_3d_reconstruction_b200.extensions.chamfer_dist import chamfer_per_sample
    from stereo_3d_reconstruction_b200.utils import synthetic
    cfg = cfg0.clone()
    cfg.NETWORK.PRECISION = 'bf16'
    B, N, M = 32, cfg.CONST.N_POINTS, cfg.CONST.N_GT_POINTS
    model = models.build_model('Stereo2Point', cfg, seed=cfg.CONST.SEED).to(dev).pack()
    sets = [tuple(t.to(dev) for t in synthetic.stereo_pair(B, cfg.CONST.IMG_H, cfg.CONST.IMG_W, 2 * cfg.NETWORK.MAX_DISP, seed=400 + i)[:2])
            for i in range(4)]                                   # 4 x 2 x 25 MB of images > L2
    gt = synthetic.point_clouds(B, 1, M, seed=3)[1].to(dev)
    it = [0]

    def step():
        l, r = sets[it[0] % 4]; it[0] += 1
        with torch.no_grad():
            _, _, pts = model(l, r)
            return chamfer_per_sample(pts.contiguous(), gt)
    ms = _loop_ms(step, 8)
    pts = torch.rand(B, N, 3, device=dev) - 0.5
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    from stereo_3d_reconstruction_b200 import lib as _l
    ms_ch = _events_ms(lambda: ops.chamfer_forward(pts, gt), 10, flush=flush)
    _l.set_knob('chamfer_sym', -1)                                # A/B: one search per direction (the no-workspace entry point)
    ms_two = _events_ms(lambda: ops.chamfer_forward(pts, gt), 10, flush=flush)
    _l.set_knob('chamfer_sym', 0)
    # Symmetric one-pass kernel: every unordered pair (i, j) is evaluated once and serves both directions.  Its exact
    # arithmetic is 8 fp32 operations per pair on the FMA pipe (3 sub, 3 mul, 2 add as packed FADD2 / FMUL2 / FFMA2 = two
    # lane-operations each); minima, shuffles and loads run beside it on the other pipes (SASS: 96 + 96 + 64 packed
    # instructions + 56 FMNMX3 + 18 SHFL/FMNMX + 6 LDS.128 per 64 pairs).
    pairs = 1.0 * B * N * M
    lane_ops = 8
    res = {'value': B / ms * 1e3, 'unit': 'pairs/s', 'ms_per_step': ms, 'batch': B, 'n_pred': N, 'n_gt': M, 'precision': 'bf16',
           'chamfer_ms': ms_ch, 'chamfer_kernel': 'chamfer_sym_kernel + chamfer_sym_finish_kernel (one pass for both directions)',
           'chamfer_two_pass_ms': ms_two, 'chamfer_pair_evals_per_s': 2.0 * pairs / ms_ch * 1e3,
           'chamfer_unordered_pairs_per_s': pairs / ms_ch * 1e3, 'chamfer_fp32_lane_ops_per_pair': lane_ops,
           'chamfer_bytes': B * (N + M) * 20}
    if fma_peak:
        res['chamfer_frac_of_measured_fp32_issue_peak'] = pairs * lane_ops / (ms_ch / 1e3) / fma_peak
    del model
    torch.cuda.empty_cache()
    return res


def extra_costvolume_sweep(dev, hbm_gbs):
    """configs[4]: cost-volume + soft-argmin sweep at 1/4 resolution (64x64), batch 64, bf16 features.  Algorithmic bytes
    (SURVEY.md 8(d)): every unique input read once + every output written once."""
    import torch
    from stereo_3d_reconstruction_b200 import ops
    B, h, w = 64, 64, 64
    flush = torch.empty(256 * 2 ** 20, dtype=torch.uint8, device=dev)
    pts = []
    for C in (32, 64):
        feat = torch.randn(2 * B, 1, h, w, C, device=dev).to(torch.bfloat16)
        for D in (32, 64, 128):
            rec = {'C': C, 'D': D}
            vol = torch.empty(2 * B, D, h, w, 2 * C, device=dev, dtype=torch.bfloat16)
            ms = _events_ms(lambda: ops.cost_volume_concat(feat, B, D, out=vol), 5, flush=flush)
            by = 2 * B * C * h * w * 2 + vol.numel() * 2
            rec.update(concat_ms=ms, concat_frac_hbm=by / ms / 1e6 / hbm_gbs)
            del vol
            disp = torch.empty(2 * B, h, w, device=dev)
            ms = _events_ms(lambda: ops.corr_soft_argmin(feat, B, D, out=disp), 10, flush=flush)
            by = 2 * B * C * h * w * 2 + 2 * B * h * w * 4
            rec.update(corr_ms=ms, corr_frac_hbm=by / ms / 1e6 / hbm_gbs, corr_tensor_tflops=2.0 * 2 * B * C * w * h * w / ms / 1e9)
            # the same kernel in a back-to-back stream over operand copies that exceed L2 together (no launch latency in the number)
            nrot = -(-320 * 2 ** 20 // (feat.numel() * 2))
            feats = [feat] + [feat.clone() for _ in range(nrot - 1)]
            ms = _rotating_ms(lambda f: (lambda: ops.corr_soft_argmin(f, B, D, out=disp)), feats)
            rec.update(corr_stream_ms=ms, corr_stream_frac_hbm=by / ms / 1e6 / hbm_gbs)
            del feats
            if C == 32:
                cost = torch.randn(2 * B, D, h, w, device=dev)
                ms = _events_ms(lambda: ops.soft_argmin(cost, -1.0, out=disp), 10, flush=flush)
                by = cost.numel() * 4 + disp.numel() * 4
                rec.update(softargmin_ms=ms, softargmin_frac_hbm=by / ms / 1e6 / hbm_gbs)
                nrot = max(2, -(-320 * 2 ** 20 // (cost.numel() * 4)))
                costs = [cost] + [cost.clone() for _ in range(nrot - 1)]
                ms = _rotating_ms(lambda c: (lambda: ops.soft_argmin(c, -1.0, out=disp)), costs)
                rec.update(softargmin_stream_ms=ms, softargmin_stream_frac_hbm=by / ms / 1e6 / hbm_gbs)
                del cost, costs
            pts.append(rec)
    return {'batch': B, 'hw': [h, w], 'dtype': 'bf16', 'peak_hbm_gbs': hbm_gbs,
            'l2': 'flushed (256 MB write) before every single timed launch; *_stream_*: back-to-back launches over operand copies that '
                  'total > 320 MB (> 126 MB L2), i.e. the kernel without the ~10 us of launch + event latency of an isolated launch',
            'points': pts}


def extra_gpu_stock_baseline(cfg0, B, dev):
    """The oracle module (stock torch.nn -> cuDNN / cuBLAS) on the same GPU: the on-box bar of SURVEY.md 8(d).  Same
    default config, batch B, inputs resident, CUDA events.  Not the product path (it is cuDNN) -- a baseline beside it."""
    import torch
    from oracle import models as O
    from stereo_3d_reconstruction_b200.utils import synthetic
    H, W, D = cfg0.CONST.IMG_H, cfg0.CONST.IMG_W, cfg0.NETWORK.MAX_DISP
    oracle = O.make_model('Stereo2Voxel', cfg0, seed=cfg0.CONST.SEED).to(dev)
    l, r, _ = synthetic.stereo_pair(B, H, W, 2 * D, seed=500)
    l, r = l.to(dev), r.to(dev)
    out = {'batch': B, 'what': 'oracle/models.py (torch.nn) through stock torch %s + cuDNN %s on this GPU' %
           (torch.__version__, torch.backends.cudnn.version())}
    old = (torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark)
    torch.backends.cudnn.benchmark = True
    try:
        for name, tf32, ac in (('fp32', False, None), ('tf32', True, None), ('bf16_autocast', True, torch.bfloat16)):
            torch.backends.cudnn.allow_tf32 = tf32
            torch.backends.cuda.matmul.allow_tf32 = tf32
            try:
                def step():
                    with torch.no_grad():
                        if ac is None:
                            oracle(l, r)
                        else:
                            with torch.autocast('cuda', dtype=ac):
                                oracle(l, r)
                ms = _loop_ms(step, 3, warm=3)
                out[name] = {'value': B / ms * 1e3, 'unit': 'pairs/s', 'ms_per_step': ms}
            except Exception as e:                      # e.g. an op without a bf16 kernel: report, do not fail the bench
                out[name] = {'unavailable': '%s: %s' % (type(e).__name__, str(e)[:120])}
            torch.cuda.empty_cache()
    finally:
        torch.backends.cudnn.allow_tf32, torch.backends.cuda.matmul.allow_tf32, torch.backends.cudnn.benchmark = old
    del oracle
    torch.cuda.empty_cache()
    return out


def extra_peaks(dev):
    """TF32 matmul (cuBLAS, 8192^3) and fp32 FMA issue peaks, measured here the way MEASURED_PEAKS.json measures bf16."""
    import ctypes
    import torch
    from stereo_3d_reconstruction_b200 import lib
    out = {}
    n = 8192
    a = torch.randn(n, n, device=dev)
    b = torch.randn(n, n, device=dev)
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = True
    try:
        ms = _events_ms(lambda: torch.matmul(a, b), 10)
        out['tf32_matmul_tflops'] = 2.0 * n ** 3 / ms / 1e9
    finally:
        torch.backends.cuda.matmul.allow_tf32 = old
    del a, b
    sink = torch.zeros(4, device=dev)
    cnt = ctypes.c_int64(0)
    L = lib.load()
    st = torch.cuda.current_stream().cuda_stream
    ms = _events_ms(lambda: lib.check(L.s3d_fma_probe(sink.data_ptr(), 4096, ctypes.byref(cnt), st), 's3d_fma_probe'), 10)
    out['fp32_fma_per_s'] = cnt.value / (ms / 1e3)
    out['fp32_fma_tflops'] = 2.0 * cnt.value / ms / 1e9
    out['how'] = 'torch.matmul fp32 with allow_tf32 (8192^3, median of 10); s3d_fma_probe: 8 independent FFMA chains per thread, 8 CTAs x 256 threads per SM'
    torch.cuda.empty_cache()
    return out


def dump_outputs(outdir, outputs, limit=64 * 2 ** 20):
    """Writes `outputs` (name -> tensor, batch first) as outdir/<name>.npy: float tensors as float32, integer counts as
    float64 (exact).  Above `limit` bytes in all, every array keeps the same seeded sample of batch entries, so two builds
    run with the same arguments are compared pair for pair."""
    import numpy as np
    import torch
    host = {k: (v.float() if v.is_floating_point() else v.double()).cpu().numpy() for k, v in outputs.items()}
    B = next(iter(host.values())).shape[0]
    keep = max(1, limit // sum(v[:1].nbytes for v in host.values()))
    if keep < B:
        idx = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:keep].sort().values.numpy()
        host = {k: v[idx] for k, v in host.items()}
    os.makedirs(outdir, exist_ok=True)
    for k, v in host.items():
        np.save(os.path.join(outdir, k + '.npy'), v)


def run_ours(args):
    import torch
    import torch.distributed as dist
    from config import cfg
    from stereo_3d_reconstruction_b200 import lib, models
    from stereo_3d_reconstruction_b200.utils import synthetic

    rank, world = int(os.environ.get('RANK', 0)), int(os.environ.get('WORLD_SIZE', 1))
    local = int(os.environ.get('LOCAL_RANK', 0))
    if not torch.cuda.is_available():
        sys.exit('bench.py needs a CUDA device: the product path has no CPU fallback (use --impl reference for the CPU arm)')
    torch.cuda.set_device(local)
    lib.check(lib.load().s3d_device_check(local), 's3d_device_check')
    if world > 1:
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
    dev = torch.device('cuda', local)

    cfg.NETWORK.PRECISION = args.precision
    B = args.batch or cfg.CONST.BATCH_SIZE
    cfg.CONST.MICRO_BATCH = max(B, cfg.CONST.MICRO_BATCH)
    H, W, D = cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.NETWORK.MAX_DISP
    model = models.build_model('Stereo2Voxel', cfg, seed=cfg.CONST.SEED).to(dev).pack()

    # rotating input sets: 4 x (left,right) batches > 126 MB L2 (and each step streams >10 GB of activations)
    n_sets = 4
    host_sets, dev_sets = [], []
    for i in range(n_sets):
        l, r, _ = synthetic.stereo_pair(B, H, W, 2 * D, seed=1000 * rank + i)
        g = synthetic.gt_volume(B, cfg.CONST.N_VOX, seed=5000 * rank + i)
        # the end-to-end path feeds DECODED 8-bit images, HWC (what a PNG loader hands over, README.md:73-74): 4x fewer H2D bytes
        # than fp32 NCHW; the first layer reads them directly (csrc/conv_first.cu)
        l8 = (l.clamp(0, 1) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous()
        r8 = (r.clamp(0, 1) * 255).round().to(torch.uint8).permute(0, 2, 3, 1).contiguous()
        host_sets.append((l8.pin_memory(), r8.pin_memory(), g.pin_memory()))
        dev_sets.append((l.to(dev), r.to(dev), g.to(dev)))
    T = len(cfg.TEST.VOXEL_THRESH)
    stats = torch.zeros(2 * T + 1, dtype=torch.int64, device=dev)
    last_out = []            # outputs of the latest resident step: views of the model's workspace, valid until its next forward

    def step_resident(i):
        l, r, g = dev_sets[i % n_sets]
        last_out[:] = model(l, r, g)
        _, _, vox, iou = last_out
        stats[:T] = iou[:, :, 0].sum(0)
        stats[T:2 * T] = iou[:, :, 1].sum(0)
        stats[2 * T] = B
        if world > 1:
            dist.all_reduce(stats)
        return vox

    # ---- end-to-end path: pinned host inputs -> H2D -> forward -> D2H, every step inside the timed region.
    # Double-buffered device inputs + a copy stream, so the H2D of step i+1 overlaps the compute of step i
    # (what a serving loop does); all copies of the K timed steps are still issued and finished inside the region.
    nv = cfg.CONST.N_VOX
    h_vox = [torch.empty((B, nv, nv, nv), dtype=torch.float32).pin_memory() for _ in range(2)]
    h_stats = [torch.empty(2 * T + 1, dtype=torch.int64).pin_memory() for _ in range(2)]
    d_vox = [torch.empty((B, nv, nv, nv), dtype=torch.float32, device=dev) for _ in range(2)]
    d_stats = [torch.empty(2 * T + 1, dtype=torch.int64, device=dev) for _ in range(2)]
    out_stream = torch.cuda.Stream(device=dev)
    out_ready = [torch.cuda.Event() for _ in range(2)]
    out_done = [torch.cuda.Event() for _ in range(2)]
    d_in = [(torch.empty((B, H, W, 3), dtype=torch.uint8, device=dev), torch.empty((B, H, W, 3), dtype=torch.uint8, device=dev),
             torch.empty((B, nv, nv, nv), dtype=torch.uint8, device=dev)) for _ in range(2)]
    copy_stream = torch.cuda.Stream(device=dev)
    in_ready = [torch.cuda.Event() for _ in range(2)]
    in_free = [torch.cuda.Event() for _ in range(2)]
    e2e_state = {'primed': -1, 'first_timed': -1}

    # the public call of the end-to-end loop: the forward replayed from a CUDA graph (model.graphed: one graph launch instead of
    # 36 kernel launches, ~1 % at batch 64); the resident-input loop above stays eager because its per-kernel CUDA events
    # (roofline) need the individual launches
    e2e_forward = model.graphed if hasattr(model, 'graphed') and not os.environ.get('S3D_BENCH_E2E_EAGER') else model

    def stage_inputs(i):
        hl, hr, hg = host_sets[i % n_sets]
        slot = i & 1
        with torch.cuda.stream(copy_stream):
            copy_stream.wait_event(in_free[slot])             # the forward that last read this slot has finished
            d_in[slot][0].copy_(hl, non_blocking=True)
            d_in[slot][1].copy_(hr, non_blocking=True)
            d_in[slot][2].copy_(hg, non_blocking=True)
            in_ready[slot].record(copy_stream)

    def step_e2e(i):
        cur = torch.cuda.current_stream()
        if e2e_state['primed'] != i or i == e2e_state['first_timed']:
            stage_inputs(i)      # first step of the timed region copies its own inputs INSIDE the region (no head start)
        slot = i & 1
        cur.wait_event(in_ready[slot])
        stage_inputs(i + 1); e2e_state['primed'] = i + 1      # prefetch the next step's inputs
        dl_, dr_, dg_ = d_in[slot]
        _, _, vox, iou = e2e_forward(dl_, dr_, dg_)
        in_free[slot].record(cur)
        stats[:T] = iou[:, :, 0].sum(0)
        stats[T:2 * T] = iou[:, :, 1].sum(0)
        stats[2 * T] = B
        if world > 1:
            dist.all_reduce(stats)
        # results leave through a device staging slot and a second stream, so the D2H of step i overlaps the compute of
        # step i+1 (the model's output buffer is reused by the next forward); e2e_finish() joins the last copies
        cur.wait_event(out_done[slot])
        d_vox[slot].copy_(vox, non_blocking=True)
        d_stats[slot].copy_(stats, non_blocking=True)
        out_ready[slot].record(cur)
        with torch.cuda.stream(out_stream):
            out_stream.wait_event(out_ready[slot])
            h_vox[slot].copy_(d_vox[slot], non_blocking=True)
            h_stats[slot].copy_(d_stats[slot], non_blocking=True)
            out_done[slot].record(out_stream)

    def e2e_finish():
        cur = torch.cuda.current_stream()
        for ev in out_done:
            cur.wait_event(ev)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup, finish=None):
        for i in range(warmup):
            fn(i)
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for i in range(steps):
            fn(warmup + i)
        if finish is not None:
            finish()                 # the timed region ends only when every step's results are on the host
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = t.item()
        return ms

    # ---- dominant-kernel timing hooks (CUDA events on the launching stream, inside the timed region) ----
    dom_layers = ('dres0b', 'dres1a', 'cls_a')          # launches of the plain 64->64 3x3x3 kernel (cls_a only on the A/B path)
    agg_other = ('dres0a', 'dres1b', 'cls_chain')       # + reference-once first layer, residual layer, cls_a + classifier chain
    dom_events = []
    agg_events = {k: [] for k in agg_other}
    orig_conv = model._conv

    def hooked(name, x, **kw):
        if name in dom_layers or name in agg_other:
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            out = orig_conv(name, x, **kw)
            b.record()
            (dom_events if name in dom_layers else agg_events[name]).append((a, b))
            return out
        return orig_conv(name, x, **kw)

    model._conv = hooked
    # the HBM-bound kernel the north_star names (classifier conv + soft-argmin over the volume), timed the same way
    from stereo_3d_reconstruction_b200 import ops as _ops
    cls_events = []
    orig_cls = _ops.cls_soft_argmin

    def hooked_cls(x, w_taps, sign=-1.0, out=None):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = orig_cls(x, w_taps, sign, out=out)
        b.record()
        cls_events.append((a, b, x.numel() * x.element_size() + r.numel() * 4))
        return r

    _ops.cls_soft_argmin = hooked_cls
    orig_ccv = _ops.conv_concat_volume               # the fused cost volume + first aggregation layer (dres0a)

    def hooked_ccv(*a_, **kw):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = orig_ccv(*a_, **kw)
        b.record()
        agg_events['dres0a'].append((a, b))
        return r

    _ops.conv_concat_volume = hooked_ccv
    orig_ccs = _ops.conv_concat_volume_sheared       # the same layer in sheared form: 4 map convolutions + the streaming pass

    def hooked_ccs(*a_, **kw):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = orig_ccs(*a_, **kw)
        b.record()
        agg_events['dres0a'].append((a, b))
        return r

    _ops.conv_concat_volume_sheared = hooked_ccs
    # the streaming pass of that form (gonce_assemble_kernel) is the forward's HBM-bound kernel: it reads the fp32 maps once and
    # writes the bf16 volume.  Timed through the library handle, on the launching stream, inside the steps.
    L_ = lib.load()
    orig_asm = L_.s3d_concat_gonce_assemble
    asm_events = []

    def hooked_asm(ml, mr, el, er, bias, out, B_, D_, h_, w_, mw_, odt, st):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        rc = orig_asm(ml, mr, el, er, bias, out, B_, D_, h_, w_, mw_, odt, st)
        b.record()
        asm_events.append((a, b, 2 * B_ * D_ * h_ * w_ * 64 * 2 + 2 * B_ * h_ * (mw_ * 384 + D_ * 256) * 4))
        return rc

    L_.s3d_concat_gonce_assemble = hooked_asm
    orig_chain = _ops.conv_cls_soft_argmin           # cls_a + classifier + soft-argmin (two launches: the march, the combine)

    def hooked_chain(*a_, **kw):
        a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a.record()
        r = orig_chain(*a_, **kw)
        b.record()
        agg_events['cls_chain'].append((a, b))
        return r

    _ops.conv_cls_soft_argmin = hooked_chain
    n0 = lib.launches()
    with ClockSampler(local) as clk:
        ms = timed(step_resident, args.steps, args.warmup)
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, dict(zip(('disp_left', 'disp_right', 'voxels', 'iou_counts'), last_out)))
    launches = (lib.launches() - n0) // (args.steps + args.warmup)        # kernels of this library per step
    n_dom = len(dom_events) // (args.steps + args.warmup)                 # plain aggregation launches per step
    dom_ms = [a.elapsed_time(b) for a, b in dom_events[n_dom * args.warmup:]]
    _ops.conv_concat_volume = orig_ccv
    _ops.conv_concat_volume_sheared = orig_ccs
    L_.s3d_concat_gonce_assemble = orig_asm
    _ops.conv_cls_soft_argmin = orig_chain
    asm_t = [(a.elapsed_time(b), nb) for a, b, nb in asm_events[args.warmup:]]
    # The shipped forward no longer has an HBM-bound classifier kernel (csrc/conv_scatter_cls.cu never writes the volume it would
    # read).  The stand-alone one-pass classifier + soft-argmin (cls_fused_kernel) is still the path of other layer shapes: time
    # it the same way, inside steps of the A/B forward that writes cls_a's output and reads it back.
    if not cls_events and args.precision == 'bf16':
        lib.set_knob('no_cls_chain', 1)
        for i in range(6):
            step_resident(i)
        torch.cuda.synchronize()
        lib.set_knob('no_cls_chain', 0)
        cls_events = cls_events[3:] + cls_events[:0]
        cls_ab = True
    else:
        cls_ab = False
    model._conv = orig_conv
    _ops.cls_soft_argmin = orig_cls
    agg_ms = {k: [a.elapsed_time(b) for a, b in v[args.warmup:]] for k, v in agg_events.items()}
    agg_ms = {k: sum(v) / len(v) for k, v in agg_ms.items() if v}
    cls_t = [(a.elapsed_time(b), nb) for a, b, nb in (cls_events if cls_ab else cls_events[args.warmup:])]
    warm_e2e = min(args.warmup, 2) or 1
    e2e_state['first_timed'] = warm_e2e
    ms_e2e = timed(step_e2e, args.steps, warm_e2e, e2e_finish)
    # The resident-input loop once more, right AFTER the end-to-end one: on a fresh box the first second of work runs ~3 % faster
    # than what follows (power-cap clocks settle), so `value` (measured first) and `e2e` (second) differ by that drift plus the
    # real cost of the copies; this second reading separates the two.
    ms_after = timed(step_resident, max(4, args.steps // 2), 1)

    # ---- configs[2] as written: global batch 512 sharded over the N GPUs (strong scaling; the headline above is weak) ----
    strong = None
    if world > 1 and not args.no_extras and 512 % world == 0:
        per = 512 // world
        sl, sr, _ = synthetic.stereo_pair(per, H, W, 2 * D, seed=7000 + rank)
        sg = synthetic.gt_volume(per, cfg.CONST.N_VOX, seed=8000 + rank)
        sl, sr, sg = sl.to(dev), sr.to(dev), sg.to(dev)
        cfg.CONST.MICRO_BATCH = 64

        def step_strong(i):
            _, _, _, iou = model(sl, sr, sg)
            stats[:T] = iou[:, :, 0].sum(0)
            stats[T:2 * T] = iou[:, :, 1].sum(0)
            stats[2 * T] = per
            dist.all_reduce(stats)
        k = max(2, args.steps // 3)
        ms_s = timed(step_strong, k, 3)
        strong = {'value': 512 * k / (ms_s / 1e3), 'unit': 'pairs/s', 'global_batch': 512, 'per_gpu': per, 'steps': k,
                  'ms_per_step': ms_s / k, 'micro_batch': 64, 'scaling': 'strong',
                  'note': 'BASELINE configs[2]: batch 512 sharded across %d GPUs, IoU stats reduced with one NCCL all-reduce per step' % world}
        del sl, sr, sg

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    pk = peaks()
    value = B * world * args.steps / (ms / 1e3)
    e2e = B * world * args.steps / (ms_e2e / 1e3)
    pc = model._packed['dres0b']
    h, w = -(-H // 4), -(-W // 4)
    flops = pc.flops(2 * B, D, h, w)                  # algorithmic FLOPs of one launch (2B volumes)
    dom = sum(dom_ms) / max(len(dom_ms), 1)
    achieved = flops / (dom / 1e3) / 1e12
    peak = pk['bf16_tflops_sustained']
    total_flops = sum(model._packed[k].flops(*shape) for k, shape in model_flop_shapes(cfg, B).items()
                      if k in model._packed)     # dec_out is fused into dec3's epilogue when it fits
    line = {
        'metric': 'stereo pairs/sec Stereo2Voxel fwd', 'value': value, 'unit': 'pairs/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True,
        'scaling': 'weak', 'vs_baseline': None, 'dtype': args.precision, 'data': 'synthetic',
        'config': {'workload': 'Stereo2Voxel forward, batch %d per GPU (BASELINE configs[1]; x%d GPUs = configs[2] sharding), '
                               '%dx%d input, D=%d planes at 1/4 res, random-init weights' % (B, world, H, W, D),
                   'global_batch': B * world, 'cost_volume': cfg.NETWORK.COST_VOLUME,
                   'l2': 'inputs rotate over %d batches (%d MB > 126 MB L2); each step streams >10 GB of activations'
                         % (n_sets, n_sets * 2 * B * 3 * H * W * 4 // 2 ** 20)},
        'e2e': {'value': e2e, 'unit': 'pairs/s', 'ms_per_step': ms_e2e / args.steps,
                'h2d_bytes_per_step': 2 * B * 3 * H * W + B * cfg.CONST.N_VOX ** 3,
                'inputs': 'uint8 HWC [B,H,W,3] left/right + uint8 GT volume from pinned host memory (decoded-PNG layout)',
                'forward': 'model.graphed(left, right, gt): CUDA-graph replay of the same kernels' if e2e_forward is not model else 'model(left, right, gt), eager',
                'd2h_bytes_per_step': B * cfg.CONST.N_VOX ** 3 * 4 + (2 * T + 1) * 8,
                'resident_loop_after_e2e_ms_per_step': ms_after / max(4, args.steps // 2),
                'e2e_over_resident_after': (ms_after / max(4, args.steps // 2)) / (ms_e2e / args.steps)},
        'gpu_launches': launches * args.steps,          # kernels of this library launched inside the timed region
        'gpu_launches_per_step': launches,
        'clocks': clk.summary(),
        'roofline': {'bound': 'tensor', 'kernel': 'conv_scatter_kernel (3x3x3 64->64 cost aggregation: dres0b, dres1a -- the plain kernel; '
                                                 'the other three aggregation launches are its fused variants, timed below)',
                     'achieved': achieved, 'peak': peak, 'unit': 'TFLOP/s', 'frac': achieved / peak,
                     'peak_source': '%s bf16_tflops_sustained (kernel timed inside a long step)' % pk['source'],
                     # the same against the BURST cuBLAS figure: the kernel runs at the tensor pipe's ceiling for the clock the
                     # power cap allows (ncu: 96.7 % tensor-pipe active) and draws less than cuBLAS, hence frac > 1 above
                     'peak_burst': pk['bf16_tflops'], 'frac_of_burst': achieved / pk['bf16_tflops'],
                     'ms_per_launch': dom, 'flops_per_launch': flops, 'share_of_step': dom * n_dom / (ms / args.steps),
                     # the other aggregation launches: dres0a = cost volume + first layer in sheared form (four 2-D map convolutions,
                     # csrc/map_conv.cu, + the streaming pass csrc/concat_gonce.cu: five launches; knob no_sheared: the reference-once
                     # tensor-core kernel, csrc/conv_scatter_concat.cu), dres1b = the residual layer (residual added as an identity tap on
                     # the tensor core, +6 % MMAs, csrc/conv_scatter_rm.cu), cls_chain = cls_a + classifier + soft-argmin with the
                     # projections on the tensor core (+4.6 % MMAs, its output volume never written; csrc/conv_scatter_cls.cu,
                     # both of its launches); share of all five layers in the step
                     'other_aggregation_ms': agg_ms,
                     'aggregation_share_of_step': (dom * n_dom + sum(agg_ms.values())) / (ms / args.steps),
                     # not measured in this run (needs ncu): one `ncu --set full` capture of this kernel at this shape read
                     # dram__bytes_read.sum + dram__bytes_write.sum = 4.281e9 against 4.295e9 algorithmic bytes (profiles/r1_ncu_summary.md)
                     'traffic': None, 'traffic_source': 'profiles/r1_ncu_summary.md (ncu capture, not live)',
                     'algorithmic_bytes_per_launch': 2 * (2 * B) * D * h * w * pc.cin * 2},
        # the forward's own HBM-bound kernel: the streaming pass of the sheared first aggregation layer (csrc/concat_gonce.cu),
        # measured in the steps; algorithmic bytes = the bf16 volume written + the fp32 maps read once
        'roofline_hbm': None if not asm_t else {
            'bound': 'hbm', 'kernel': 'gonce_assemble_kernel (cost volume + first aggregation layer, sheared form: adds two maps per '
                                      'output element, ReLU, writes the bf16 volume)',
            'achieved': asm_t[0][1] / (sum(t for t, _ in asm_t) / len(asm_t) / 1e3) / 1e9, 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
            'frac': asm_t[0][1] / (sum(t for t, _ in asm_t) / len(asm_t) / 1e3) / 1e9 / pk['hbm_gbs'],
            'ms_per_launch': sum(t for t, _ in asm_t) / len(asm_t), 'bytes_per_launch': asm_t[0][1]},
        'roofline_hbm_cls_fused_ab': None if not cls_t else {
            'bound': 'hbm', 'kernel': 'cls_fused_kernel (Cout=1 3x3x3 classifier + soft-argmin, one pass over the aggregated volume)'
                                      + (' -- measured inside steps of the A/B forward (knob no_cls_chain): the shipped forward fuses the '
                                         'classifier into cls_a and has no kernel that reads the volume' if cls_ab else ''),
            'achieved': cls_t[0][1] / (sum(t for t, _ in cls_t) / len(cls_t) / 1e3) / 1e9, 'peak': pk['hbm_gbs'], 'unit': 'GB/s',
            'frac': cls_t[0][1] / (sum(t for t, _ in cls_t) / len(cls_t) / 1e3) / 1e9 / pk['hbm_gbs'],
            'ms_per_launch': sum(t for t, _ in cls_t) / len(cls_t), 'bytes_per_launch': cls_t[0][1]},
        'model_tflops_per_step': total_flops / 1e12,
        'model_tflops_achieved': total_flops / (ms / args.steps / 1e3) / 1e12,
    }
    if strong is not None:
        line['strong_512'] = strong
    if not args.no_cpu_baseline and world == 1:
        cores = os.cpu_count() or 1
        v, sec = cpu_oracle_run(cfg, 1, 5, 1, cores)
        line['cpu_baseline'] = {'value': v, 'unit': 'pairs/s', 'cores': cores, 'kind': 'port',
                                'sample': 'batch 1 (BASELINE configs[0]), 5 forwards, fp32 torch.nn oracle on %d threads' % cores}
    if world == 1 and not args.no_extras:
        # the other BASELINE configs, each measured briefly (see the module docstring); a failure is reported, not fatal
        def guarded(fn, *a):
            try:
                return fn(*a)
            except Exception as e:
                return {'failed': '%s: %s' % (type(e).__name__, str(e)[:200])}
        base_cfg = cfg.clone()
        base_cfg.NETWORK.PRECISION = 'bf16'
        line['latency'] = guarded(extra_latency, model, cfg, dev) if args.precision == 'bf16' else None
        del model
        dev_sets.clear()
        torch.cuda.empty_cache()
        pm = guarded(extra_peaks, dev)
        line['peaks_measured'] = pm
        line['fp32_mode'] = guarded(extra_fp32_mode, base_cfg, B, dev, args.steps)
        line['stereo2point_chamfer'] = guarded(extra_stereo2point, base_cfg, dev, pm.get('fp32_fma_per_s'))
        line['costvolume_sweep'] = guarded(extra_costvolume_sweep, dev, pk['hbm_gbs'])
        # stand-alone HBM-bound ops of configs[4] at the default point (C = 32, D = 32, batch 64), measured live above with L2 flushed
        sw = line['costvolume_sweep']
        if isinstance(sw, dict) and sw.get('points'):
            p0 = sw['points'][0]
            by = 2 * sw['batch'] * p0['C'] * sw['hw'][0] * sw['hw'][1] * 2 * (1 + 2 * p0['D'])
            line['roofline_hbm_standalone'] = {
                'bound': 'hbm', 'kernel': 'concat_volume_kernel (cost-volume build, C=%d, D=%d, batch %d, %dx%d; stand-alone op of '
                                          'configs[4] -- the forward never materialises the volume)' % (p0['C'], p0['D'], sw['batch'], sw['hw'][0], sw['hw'][1]),
                'achieved': by / p0['concat_ms'] / 1e6, 'peak': pk['hbm_gbs'], 'unit': 'GB/s', 'frac': by / p0['concat_ms'] / 1e6 / pk['hbm_gbs'],
                'ms_per_launch': p0['concat_ms'], 'bytes_per_launch': by,
                'soft_argmin_frac_isolated_launch': p0.get('softargmin_frac_hbm'),
                'soft_argmin_frac_back_to_back': p0.get('softargmin_stream_frac_hbm')}
        line['gpu_stock_baseline'] = guarded(extra_gpu_stock_baseline, base_cfg, B, dev)
        if isinstance(line['gpu_stock_baseline'].get('bf16_autocast'), dict) and 'value' in line['gpu_stock_baseline']['bf16_autocast']:
            line['gpu_stock_baseline']['ours_over_stock_bf16'] = value / line['gpu_stock_baseline']['bf16_autocast']['value']
    print(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def model_flop_shapes(cfg, B):
    """(N, D, H, W) input shape of every packed conv layer of the Stereo2Voxel forward at batch B."""
    H, W, D = cfg.CONST.IMG_H, cfg.CONST.IMG_W, cfg.NETWORK.MAX_DISP
    h2, w2, h4, w4 = -(-H // 2), -(-W // 2), -(-H // 4), -(-W // 4)
    s = {'enc0': (2 * B, 1, H, W), 'enc1': (2 * B, 1, h2, w2), 'enc2': (2 * B, 1, h2, w2)}
    for k in ('enc3', 'enc4', 'enc5'):
        s[k] = (2 * B, 1, h4, w4)
    if cfg.NETWORK.COST_VOLUME == 'concat':
        for k in ('dres0a', 'dres0b', 'dres1a', 'dres1b', 'cls_a', 'cls_b'):
            s[k] = (2 * B, D, h4, w4)
    hh, ww = H, W
    for i in range(len(cfg.NETWORK.REC_CHANNELS)):
        s['rec%d' % i] = (2 * B, 1, hh, ww)
        hh, ww = -(-hh // 2), -(-ww // 2)
    v = 2
    for i in range(len(cfg.NETWORK.DEC_CHANNELS) - 1):
        s['dec%d' % i] = (2 * B, v, v, v)
        v *= 2
    s['dec_out'] = (2 * B, v, v, v)
    for i in range(len(cfg.NETWORK.MERGER_CHANNELS) - 1):
        s['mrg%d' % i] = (2 * B, v, v, v)
    return s


if __name__ == '__main__':
    a = parse()
    if a.impl == 'reference':
        run_reference(a)
    else:
        run_ours(a)
