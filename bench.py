#!/usr/bin/env python
"""bench.py -- contract benchmark of the 4K-NeRF ray-march hot path on B200.

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--dump-outputs DIR]
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N ... bench.py --gpus N ...

Metric (BASELINE.json): rays/s of march + interp + MLP + composite.
Workload: the north-star target -- BASELINE.json configs[1]'s model (DirectVoxGO fine stage,
160^3 density + 12-ch feature grid, rgbnet 39->128->128->3, stepsize 0.5; configs/default.py:107-119)
marched at 4K, 4032x3024 = 12.19 M rays per step, synthetic random-weight scene in the dense "FOG"
regime (every in-box sample is interpolated, shaded and composited; SURVEY.md section 8d).  One
"step" = one fused launch over one full frame; successive steps use different camera poses.  The
same model at configs[1]'s nominal 1008x756 and the sparse "SHELL" regime are reported in `extra`.

N > 1: one process per GPU, the frame's rows are sharded into N bands (k4nerf/dist.py), each
rank marches its band and the packed bands are all-gathered with NCCL ("scaling": "strong").

Timing: CUDA events on the launching stream around exactly K steps, barrier + synchronize on both
sides, max over ranks.  Inputs per step (439 MB of rays + 213 MB of grids) exceed the 126 MB L2.

`--dump-outputs DIR`: after the timed steps, the per-ray results of the last one (rgb_marched, depth,
alphainv_last: what render_rays hands its caller) at a fixed, seeded sample of 2^20 rays, and the
sampled ray indices, as DIR/<name>.npy (28 MB in all).  The scene and the rays are seeded, so two
builds run with the same arguments can be compared output for output.  Geometry (depth, alphainv_last)
repeats bit for bit from run to run; rgb_marched may differ in the last bit (1.8e-7 measured on a B200 at its 1000 W power limit).

`--impl reference`: the reference has NO CPU implementation of this path (every op is CUDA-only,
lib/cuda/render_utils.cpp:46-48) and cannot be imported here, so the arm times the oracle port
(oracle/pipeline.py: the reference's forward restated op-by-op on torch-CPU + C) on the host
cores, each step a bounded 16384-ray sample of the same frame.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, '4k-nerf_b200'))

import torch  # noqa: E402
import torch.distributed as dist  # noqa: E402

H4K, W4K = 3024, 4032
HLR, WLR = 756, 1008
GRID_RES = 160
POSES = [(30.0, -30.0), (75.0, -20.0), (140.0, -35.0), (215.0, -25.0), (290.0, -30.0)]
HBM_FALLBACK_GBS = 6650.0     # /opt/skills/guides/B200_PROFILING.md fallback


_STDOUT_FD = None


def emit(text):
    """Write the result line to the real stdout (see the fd juggling in main for N > 1)."""
    sys.stdout.flush()
    if _STDOUT_FD is not None:
        os.write(_STDOUT_FD, (text + '\n').encode())
    else:
        print(text, flush=True)


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--mlp-mode', default=None, help='tc | f16 | f16x3 | fp32 (default: auto = fastest built for the shape)')
    ap.add_argument('--regime', default='fog', choices=['fog', 'shell'])
    ap.add_argument('--no-extra', action='store_true', help='skip the secondary measurements')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write the last timed step\'s per-ray results (seeded sample of rays) as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    return args


# ------------------------------------------------------------------------------------------------
# scene / rays (synthetic, seeded; built through the oracle's scene helpers = test infrastructure
# used only to CREATE inputs; nothing of the oracle is on the timed path of the `ours` arm)
# ------------------------------------------------------------------------------------------------
def build_scene(regime):
    sys.path.insert(0, os.path.join(ROOT, 'tests'))
    from helpers import make_state, model_from_state
    st = make_state('cfgA', res=GRID_RES, regime=regime)
    return st, model_from_state


def frame_rays_device(H, W, pose, dev):
    """Pixel-centre rays of one view generated on the device (k4_make_rays)."""
    import k4nerf
    from oracle import scenes
    K, c2w = scenes.blender_camera(H, W, theta=pose[0], phi=pose[1])
    ro, rd, vd = k4nerf.get_rays_of_a_view(H, W, K, c2w.to(dev), ndc=False, inverse_y=False, flip_x=False, flip_y=False)
    return ro.view(-1, 3), rd.view(-1, 3), vd.view(-1, 3)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ('index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,'
         'clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
         'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')

    def __init__(self, gpu_index=0):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(['nvidia-smi', f'--query-gpu={self.Q}', '--format=csv,noheader,nounits',
                                          '-lms', '100', '-i', str(self.gpu_index)],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), line.strip()))

    def stop(self):
        if self.proc is not None:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, mx, reasons = [], [], set()
        for ts, line in self.rows:
            if ts < t0 or ts > t1 + 0.2:
                continue
            f = [x.strip() for x in line.split(',')]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1])); mx.append(float(f[2]))
            except ValueError:
                continue
            for name, val in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), f[5:9]):
                if val.lower().startswith('active'):
                    reasons.add(name)
        if not sm:
            return {'sm_mhz': None, 'sm_max_mhz': None, 'reasons': [], 'samples': 0}
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2], 'sm_max_mhz': max(mx), 'reasons': sorted(reasons), 'samples': len(sm)}


def hbm_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['hbm_gbs']), 'measured (MEASURED_PEAKS.json hbm_gbs)'
        except Exception:
            pass
    return HBM_FALLBACK_GBS, 'fallback (B200_PROFILING.md 6.65 TB/s)'


def tensor_peak():
    p = os.path.join(ROOT, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        try:
            return float(json.load(open(p))['bf16_tflops_sustained']), 'measured (MEASURED_PEAKS.json bf16_tflops_sustained)'
        except Exception:
            pass
    return 1400.0, 'fallback (B200_PROFILING.md: ~1.4 PFLOP/s sustained)'


def algorithmic_bytes(n_rays, S_m, S_d, S_c, C=12):
    """SURVEY.md section 8(d): B = 68 N + S_m + 32 S_d + 32 C S_c (fp32 grids, no reuse credit)."""
    return 68 * n_rays + S_m + 32 * S_d + 32 * C * S_c


# ------------------------------------------------------------------------------------------------
# CPU arm: the oracle port on the host cores
# ------------------------------------------------------------------------------------------------
def cpu_sample_rays(H, W, pose, n_chunks, chunk=8192):
    """A bounded sample of the frame: `n_chunks` runs of `chunk` consecutive rays (the reference's
    chunk size, run_sr.py:121-124) spread evenly over the image."""
    from oracle import scenes
    ro, rd, vd = scenes.blender_rays(H, W, theta=pose[0], phi=pose[1])
    n = ro.shape[0]
    outs = []
    for c in range(n_chunks):
        s = int((c + 0.5) * n / n_chunks) - chunk // 2
        s = max(0, min(s, n - chunk))
        outs.append((ro[s:s + chunk], rd[s:s + chunk], vd[s:s + chunk]))
    return outs


def cpu_time_step(st, chunks):
    from oracle import ops, pipeline, scenes
    t0 = time.perf_counter()
    n = 0
    for ro, rd, vd in chunks:
        pipeline.forward(st, ro, rd, vd, ops.CpuOps, **scenes.RENDER_KW_DVGO)
        n += ro.shape[0]
    return n, time.perf_counter() - t0


def cpu_threads():
    """Threads of the CPU arm.  One pool size for torch's intra-op pool AND the C oracle's OpenMP team
    (oracle/ops.set_num_threads): the arm's ops are a few MB each, so more than ~32 threads only adds
    fork/join and cache-line traffic -- 128 torch x 128 OpenMP threads made the round-1 number swing 4x
    between boxes."""
    return max(1, min(32, os.cpu_count() or 1))


def run_reference_arm(args, rank):
    """`--impl reference`: rank 0 alone runs; the other ranks exit 0 without work."""
    if rank != 0:
        return
    from oracle import ops
    cores = cpu_threads()
    ops.set_num_threads(cores)
    try:
        torch.set_num_interop_threads(1)
    except RuntimeError:
        pass
    st, _ = build_scene(args.regime)
    n_chunks = 1
    for w in range(args.warmup):
        cpu_time_step(st, cpu_sample_rays(H4K, W4K, POSES[w % len(POSES)], n_chunks))
    tot_n, tot_t = 0, 0.0
    for k in range(args.steps):
        n, t = cpu_time_step(st, cpu_sample_rays(H4K, W4K, POSES[k % len(POSES)], n_chunks))
        tot_n += n; tot_t += t
    v = tot_n / tot_t
    line = {
        'impl': 'reference', 'metric': 'rays_per_s', 'value': v, 'unit': 'rays/s', 'n_gpus': args.gpus,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': 1e3 * tot_t / max(args.steps, 1),
        'higher_is_better': True, 'scaling': 'strong', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': workload_config(args, 1),
        'cpu_baseline': {'value': v, 'unit': 'rays/s', 'cores': cores, 'kind': 'port',
                         'sample': f'{n_chunks} x 8192-ray chunk of the 4032x3024 frame per step (oracle/pipeline.py on torch-CPU + C, '
                                   f'{cores} threads of {os.cpu_count()} logical cores)'},
        'e2e': {'value': v, 'unit': 'rays/s', 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0},
        'gpu_launches': 0,
        'note': 'the reference ships no CPU path for this op chain; this is the oracle port of it on the host cores',
    }
    print(json.dumps(line), flush=True)


def dump_outputs(out, n_rays, path, n_sample=1 << 20):
    """`--dump-outputs`: the frame's per-ray results at a fixed, seeded sample of rays, as float32 / float64 .npy."""
    import numpy as np
    os.makedirs(path, exist_ok=True)
    idx = torch.randperm(n_rays, generator=torch.Generator().manual_seed(0))[:n_sample].sort().values
    np.save(os.path.join(path, 'ray_index.npy'), idx.double().numpy())
    for k in ('rgb_marched', 'depth', 'alphainv_last'):
        np.save(os.path.join(path, k + '.npy'), out[k][idx.to(out[k].device)].float().cpu().numpy())


def workload_config(args, n_gpus):
    return {
        'workload': 'north-star target: BASELINE configs[1] model (DirectVoxGO 160^3, k0 12 ch, rgbnet 39-128-128-3, '
                    'stepsize 0.5) marched at 4032x3024 rays/step',
        'regime': args.regime, 'rays_per_step': H4K * W4K, 'grid': [GRID_RES] * 3, 'k0_dim': 12,
        'mlp': [39, 128, 128, 3],
        'parallelism': f'8-row blocks dealt round-robin over {n_gpus} rank(s)' + (
            '; exchange: in-kernel NVLink stores into every rank\'s peer-mapped frame + 1-element all-reduce as barrier '
            '(nccl all_gather + transpose when peer mapping is unavailable; see "exchange")' if n_gpus > 1 else ''),
        'l2_policy': 'inputs larger than L2 (439 MB rays + 213 MB grids per step), pose changes every step',
    }


# ------------------------------------------------------------------------------------------------
# GPU arm
# ------------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    rank = int(os.environ.get('RANK', '0'))
    local_rank = int(os.environ.get('LOCAL_RANK', '0'))
    world = int(os.environ.get('WORLD_SIZE', '1'))

    if args.impl == 'reference':
        run_reference_arm(args, rank)
        return

    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device -- the k4nerf hot path has no CPU fallback')
    import k4nerf
    from k4nerf import dist as kdist
    torch.cuda.set_device(local_rank)
    dev = torch.device('cuda', local_rank)
    if world > 1:
        os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
        os.environ.setdefault('NCCL_DEBUG_FILE', '/dev/stderr')
        # keep stdout = the one JSON line: NCCL prints its version banner with printf on fd 1, so fd 1 points at stderr
        # for the whole run and the JSON line goes to the saved descriptor
        global _STDOUT_FD
        sys.stdout.flush()
        _STDOUT_FD = os.dup(1)
        os.dup2(2, 1)
        dist.init_process_group('nccl', device_id=dev)

    st, model_from_state = build_scene(args.regime)
    model = model_from_state(st, dev)
    mode = model.resolve_mlp_mode(args.mlp_mode or model.mlp_mode)
    kw = dict(near=2.0, far=6.0, bg=1, stepsize=0.5, inverse_y=False, flip_x=False, flip_y=False, render_depth=True)

    # inputs resident in HBM before the timed region: one ray set per pose, this rank's rows only
    # (8-row blocks dealt round-robin over the ranks: every rank gets the same mix of long and short rays;
    # only the rank's rows are generated -- k4_make_rays_rows)
    H, W = H4K, W4K
    frame = kdist.CyclicFrame(H, W, dev)              # row list + peer-mapped frames (or packed send / gather buffers)
    n_rows = frame.k
    r0, r1 = 0, n_rows                                   # local image = this rank's rows, in order
    from oracle import scenes as _scenes
    bands = []
    for pose in POSES:
        K, c2w = _scenes.blender_camera(H, W, theta=pose[0], phi=pose[1])
        ro, rd, vd = k4nerf.get_rays_of_a_view(H, W, K, c2w, False, False, False, False,
                                               rows=frame.rows if world > 1 else None, device=dev)
        bands.append((ro.view(-1, 3), rd.view(-1, 3), vd.view(-1, 3)))
    n_band = n_rows * W

    def step(i):
        """One step = one fused launch over this rank's rows and, for N > 1, the exchange that leaves the whole frame,
        in image order, on every rank: NVLink stores into every rank's frame from inside the kernel + a one-element
        all-reduce as the barrier (k4nerf.dist.CyclicFrame, peer mode), or -- K4_PEER=0 / no peer mapping -- the packed
        band buffer, ONE all-gather and the image-order transpose."""
        ro, rd, vd = bands[i % len(bands)]
        model.render_rays(ro, rd, vd, kw, image_hw=(r1 - r0, W), mlp_mode=mode, out=frame.target())
        return frame.finish() if world > 1 else frame.out

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # algorithmic sample counts of EVERY pose (device counters; equal to the oracle's counts, tests): the poses differ
    # in how much of the volume their rays cross, so the per-step bytes are averaged over exactly the steps that are timed
    pose_counters = []
    for b in bands:
        dbg = model.render_rays(*b, kw, image_hw=(r1 - r0, W), mlp_mode=mode, debug=True)
        c = dbg['counters'].clone()
        if world > 1:
            dist.all_reduce(c)
        pose_counters.append([int(x) for x in c.cpu().tolist()])
        del dbg
    timed = [pose_counters[i % len(bands)] for i in range(args.steps)]
    S_m, S_d, S_c, n_batches = [sum(t[j] for t in timed) / max(len(timed), 1) for j in range(4)]     # mean per timed step

    for i in range(max(args.warmup, 3)):
        step(i)
    gather_ms = None
    if world > 1:
        # NCCL sets up its channels lazily: a few more exchanges before the clock starts, and their time on its own
        # (peer mode: the barrier only -- the data moved inside the kernel; gather mode: all-gather + transpose)
        exch = frame.peers.sync if frame.peers is not None else frame.gather
        for _ in range(5):
            exch()
        barrier()
        g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        g0.record()
        for _ in range(5):
            exch()
        g1.record()
        torch.cuda.synchronize()
        gather_ms = g0.elapsed_time(g1) / 5
    barrier()
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()
        time.sleep(0.3)
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    # per-launch kernel time of the dominant kernel, measured live on the launching stream
    k_events = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(args.steps)]
    t_wall0 = time.time()
    e0.record()
    for i in range(args.steps):
        ro, rd, vd = bands[i % len(bands)]
        k_events[i][0].record()
        model.render_rays(ro, rd, vd, kw, image_hw=(r1 - r0, W), mlp_mode=mode, out=frame.target())
        k_events[i][1].record()
        if world > 1:
            full = frame.finish()                        # every rank now holds the frame in image order
    e1.record()
    barrier()
    t_wall1 = time.time()
    ms_total = e0.elapsed_time(e1)
    kernel_ms = sum(a.elapsed_time(b) for a, b in k_events) / max(args.steps, 1)
    t = torch.tensor([ms_total, kernel_ms], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_total, kernel_ms = t.cpu().tolist()
    if rank == 0:
        time.sleep(0.2)
        sampler.stop()
    clocks = sampler.summary(t_wall0, t_wall1) if rank == 0 else None
    ms_per_step = ms_total / max(args.steps, 1)
    value = (H * W) / (ms_per_step * 1e-3)
    if args.dump_outputs and rank == 0:
        dump_outputs(full if world > 1 else frame.out, H * W, args.dump_outputs)

    # ---- e2e: the public API with HOST buffers (pinned rays in, host results out), every step ----
    e2e = None
    hb = [tuple(x.cpu().pin_memory() for x in bands[i]) for i in range(min(2, len(bands)))]
    h_out = torch.empty(5 * n_band, dtype=torch.float32).pin_memory()

    e2e_buf = torch.zeros(5 * n_band, device=dev, dtype=torch.float32)
    e2e_out = kdist.packed_band_views(e2e_buf, n_band, n_band)

    def e2e_step(i):
        ro, rd, vd = [x.to(dev, non_blocking=True) for x in hb[i % len(hb)]]
        if world > 1 and frame.peers is not None:
            # peer mode: the kernel stores into every rank's frame; each rank copies ITS 1/world share of the frame back
            model.render_rays(ro, rd, vd, kw, image_hw=(r1 - r0, W), mlp_mode=mode, out=frame.target())
            par = frame.step & 1
            frame.finish()
            share = (5 * frame.n_full) // world
            n = min(share, h_out.numel())
            h_out[:n].copy_(frame.peers.local[par][rank * share:rank * share + n], non_blocking=True)
            return
        model.render_rays(ro, rd, vd, kw, image_hw=(r1 - r0, W), mlp_mode=mode, out=e2e_out)
        if world > 1:
            frame.buf[:3 * n_band].copy_(e2e_buf[:3 * n_band])
            frame.buf[3 * frame.n_pad:3 * frame.n_pad + n_band].copy_(e2e_buf[3 * n_band:4 * n_band])
            frame.buf[4 * frame.n_pad:4 * frame.n_pad + n_band].copy_(e2e_buf[4 * n_band:])
            frame.gather()
        h_out.copy_(e2e_buf, non_blocking=True)

    e2e_steps = max(2, min(args.steps, 3))
    e2e_step(0)
    barrier()
    e0.record()
    for i in range(e2e_steps):
        e2e_step(i)
    e1.record()
    barrier()
    t = torch.tensor([e0.elapsed_time(e1)], device=dev, dtype=torch.float64)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_ms = t.item() / e2e_steps
    e2e = {'value': (H * W) / (e2e_ms * 1e-3), 'unit': 'rays/s',
           'h2d_bytes_per_step': int(3 * 12 * H * W), 'd2h_bytes_per_step': int(20 * H * W),
           'ms_per_step': e2e_ms, 'api': 'DirectVoxGO.render_rays on pinned host ray buffers, packed result copied back to pinned host memory'}
    del hb, e2e_buf, e2e_out

    # ---- secondary measurements (rank 0 semantics, all ranks participate where collective) ----
    extra = {}
    if not args.no_extra and world == 1:
        extra = secondary(model, st, model_from_state, kw, dev, mode, args)
    elif not args.no_extra:
        extra = secondary_sharded(model, kw, dev, world)

    if rank == 0:
        peak, peak_src = hbm_peak()
        alg_bytes = algorithmic_bytes(H * W, S_m, S_d, S_c)      # whole frame (all ranks)
        achieved = alg_bytes / world / (kernel_ms * 1e-3) / 1e9   # per-launch bytes / per-launch time, GB/s
        kernel_name = {'tc': 'k4_march_tc_kernel', 'ws': 'k4_march_ws_kernel'}.get(mode, 'k4_march_kernel')
        traffic, ncu_pct = None, {}
        tp = os.path.join(ROOT, 'profiles', 'traffic.json')
        if os.path.exists(tp) and world == 1:
            try:
                tj = json.load(open(tp))
                traffic = tj.get(f'{kernel_name}_4032x3024_{args.regime}_dram_bytes_per_launch')   # ncu dram__bytes_read+write.sum of THIS launch
                ncu_pct = tj.get(f'{kernel_name}_ncu_pct', {})
            except Exception:
                traffic = None
        # the resource that actually binds the FOG launch: the rgbnet contraction on the tensor pipe
        mlp_mac = 39 * 128 + 128 * 128 + 128 * 3                  # SURVEY.md 8(a): 21,760 MAC / shaded sample
        tp_peak, tp_src = tensor_peak()
        mlp_tflops = 2.0 * mlp_mac * (S_c / world) / (kernel_ms * 1e-3) / 1e12
        line = {
            'metric': 'rays_per_s', 'value': value, 'unit': 'rays/s', 'n_gpus': world, 'steps': args.steps,
            'warmup': max(args.warmup, 3), 'ms_per_step': ms_per_step, 'higher_is_better': True,
            'scaling': 'strong', 'vs_baseline': None,
            'dtype': {'fp32': 'f32', 'f16': 'f16 operands, f32 accumulate (mma.sync)', 'f16x3': 'f16x3 split (f32-equivalent)',
                      'tc': 'f32 geometry/interpolation/compositing; rgbnet f16 operands, f32 accumulate (tcgen05)',
                      'ws': 'f32 geometry/interpolation/compositing; rgbnet f16 operands, f32 accumulate (tcgen05)'}[mode],
            'data': 'synthetic', 'config': workload_config(args, world), 'mlp_mode': mode,
            'e2e': e2e, 'gpu_launches': args.steps, 'clocks': clocks,
            **({'exchange': 'peer_stores' if frame.peers is not None else 'all_gather',
                'exchange_alone_ms_rank0': gather_ms} if gather_ms is not None else {}),
            'roofline': {'bound': 'hbm', 'achieved': achieved, 'peak': peak, 'unit': 'GB/s', 'frac': achieved / peak,
                         'traffic': traffic, 'peak_source': peak_src,
                         'kernel': kernel_name,
                         'kernel_ms_per_launch': kernel_ms,
                         'algorithmic_bytes_per_ray': alg_bytes / (H * W),
                         'samples_per_ray': {'S_m': S_m / (H * W), 'S_d': S_d / (H * W), 'S_c': S_c / (H * W)},
                         'samples_per_ray_by_pose': [round(pc[2] / (H * W), 2) for pc in pose_counters],
                         'accounting': 'bytes and samples are the mean over the timed steps (each step renders one of 5 poses; round 1 used the counts of pose 0 for every step)',
                         'note': 'logical bytes (no reuse credit): the 213 MB scene is L2/L1 resident, so DRAM traffic is far below this'},
            'roofline_tensor': {'bound': 'tensor', 'achieved': mlp_tflops, 'peak': tp_peak, 'unit': 'TFLOP/s', 'frac': mlp_tflops / tp_peak,
                                'peak_source': tp_src, 'flops': 'useful rgbnet MACs only: 2 x 21,760 x S_c (padding K 39->48, N 3->16 and bias MMAs not counted)',
                                'ncu_pct_of_peak': ncu_pct},
        }
        if extra:
            line['extra'] = extra
        if not args.no_cpu_baseline and world == 1:
            line['cpu_baseline'] = cpu_baseline(st)
        emit(json.dumps(line))
    if world > 1:
        dist.destroy_process_group()


def time_mode(model, rays, kw, hw, mode, iters=3):
    for _ in range(2):
        model.render_rays(*rays, kw, image_hw=hw, mlp_mode=mode)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(iters):
        model.render_rays(*rays, kw, image_hw=hw, mlp_mode=mode)
    e1.record()
    torch.cuda.synchronize()
    return e0.elapsed_time(e1) / iters


def secondary(model, st, model_from_state, kw, dev, mode, args):
    """Same kernels on the other BASELINE.json configs: configs[1] at its nominal 1008x756, the sparse
    SHELL regime at 4K, configs[2] (LLFF MPI model, lib/dmpigo) and configs[3]'s VC-Decoder."""
    import k4nerf
    from helpers import make_state
    from oracle import scenes, sftnet
    out = {}
    peak, _ = hbm_peak()
    rays = frame_rays_device(HLR, WLR, POSES[0], dev)
    ms = time_mode(model, rays, kw, (HLR, WLR), mode)
    out['configs[1]_1008x756_' + args.regime] = {'rays_per_s': HLR * WLR / (ms * 1e-3), 'ms_per_frame': ms}
    other = 'shell' if args.regime == 'fog' else 'fog'
    st2 = make_state('cfgA', res=GRID_RES, regime=other)
    m2 = model_from_state(st2, dev)
    rays4k = frame_rays_device(H4K, W4K, POSES[0], dev)
    dbg = m2.render_rays(*rays4k, kw, image_hw=(H4K, W4K), mlp_mode=mode, debug=True)
    c = [int(x) for x in dbg['counters'].cpu().tolist()]
    ms = time_mode(m2, rays4k, kw, (H4K, W4K), mode)
    n = H4K * W4K
    b = algorithmic_bytes(n, c[0], c[1], c[2])
    out['4032x3024_' + other] = {'rays_per_s': n / (ms * 1e-3), 'ms_per_frame': ms,
                                 'algorithmic_bytes_per_ray': b / n, 'roofline_frac': b / (ms * 1e-3) / 1e9 / peak,
                                 'samples_per_ray': {'S_m': c[0] / n, 'S_d': c[1] / n, 'S_c': c[2] / n}}
    del m2, st2, rays4k, dbg
    torch.cuda.empty_cache()
    # BASELINE.md section 4 "second baseline": the reference's OWN CUDA kernels (oracle/_ref/render_utils_cuda.so, compiled
    # from /root/reference) + ATen fp32 in the reference's forward structure and 8192-ray chunks (run_sr.py:121-124) on this
    # same B200 -- the only like-for-like "vs reference" figure (the reference has no CPU path).  Bounded sample.
    try:
        out['reference_kernels_gpu'] = reference_kernels_gpu(st, dev, args.regime, out_headline_mode=mode)
    except Exception as e:
        out['reference_kernels_gpu'] = {'unavailable': repr(e)}
    # configs[2]: LLFF MPI model [384,384,256], k0 9 ch, rgbnet 15-64-64-3, 256 samples/ray, NDC rays
    try:
      for regime3, sizes in (('shell', ((HLR, WLR), (H4K, W4K))), ('fog', ((H4K, W4K),))):
        st3 = make_state('cfgB', xy=384, depth=256, regime=regime3)
        m3 = model_from_state(st3, dev)
        kw3 = dict(scenes.RENDER_KW_MPI)
        mode3 = m3.resolve_mlp_mode('auto')
        for (H, W) in sizes:
            K, c2w = scenes.llff_camera(H, W, (0.05, -0.03, 0.0))
            ro, rd, vd = k4nerf.get_rays_of_a_view(H, W, K, c2w.to(dev), True, False, False, False)
            r3 = (ro.view(-1, 3), rd.view(-1, 3), vd.view(-1, 3))
            dbg = m3.render_rays(*r3, kw3, image_hw=(H, W), mlp_mode=mode3, debug=True)
            c = [int(x) for x in dbg['counters'].cpu().tolist()]
            ms = time_mode(m3, r3, kw3, (H, W), mode3, iters=2)
            n = H * W
            b = 68 * n + c[0] + 40 * c[1] + 32 * 9 * c[2]
            out[f'configs[2]_llff_mpi_{W}x{H}_{regime3}'] = {
                'rays_per_s': n / (ms * 1e-3), 'ms_per_frame': ms, 'mlp_mode': mode3,
                'algorithmic_bytes_per_ray': b / n, 'roofline_frac': b / (ms * 1e-3) / 1e9 / peak,
                'samples_per_ray': {'S_m': c[0] / n, 'S_d': c[1] / n, 'S_c': c[2] / n}}
            del ro, rd, vd, r3, dbg
        del m3, st3
        torch.cuda.empty_cache()
    except Exception as e:           # never lose the headline line to a secondary measurement
        out['configs[2]_error'] = repr(e)
    # configs[3]: VC-Decoder, 1008x756 -> 4032x3024, tile 510 / pad 10 (run_sr.py --test_tile 510)
    try:
        net = k4nerf.SFTNet(3, 4, 64, 5, 32, 1)
        net.load_state_dict(sftnet.random_state_dict(seed=3, scale=1.0))
        net = net.to(dev)
        g = torch.Generator().manual_seed(1)
        img = torch.rand(1, 3, HLR, WLR, generator=g).to(dev)
        cond = torch.rand(1, HLR, WLR, generator=g).to(dev)
        net.tile_process(img, cond, 510, to_cpu=False)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(3):
            net.tile_process(img, cond, 510, to_cpu=False)
        e1.record()
        torch.cuda.synchronize()
        ms_sr = e0.elapsed_time(e1) / 3
        flop = 2 * 5188864 * sum((p[1] - p[0]) * (p[3] - p[2]) for p in sftnet.tile_plan(HLR, WLR, 510, 10))
        lr = out['configs[1]_1008x756_' + args.regime]['ms_per_frame']
        out['configs[3]_vc_decoder_1008x756_to_4032x3024'] = {
            'ms_per_frame': ms_sr, 'tflops': flop / ms_sr / 1e9, 'algorithmic_tflop_per_frame': flop / 1e12,
            'full_4k_nerf_frame_ms (march 1008x756 ' + args.regime + ' + decode)': lr + ms_sr}
    except Exception as e:
        out['configs[3]_error'] = repr(e)
    return out


def reference_kernels_gpu(st, dev, regime, out_headline_mode, n_chunks=32, chunk=8192):
    from oracle import ops as oops, pipeline, scenes
    if not os.path.exists(oops.ref_ext_path()):
        return {'unavailable': 'oracle/_ref/render_utils_cuda.so not built (needs /root/reference at build time)'}
    ref_ops = oops.RefExtOps()
    old = torch.backends.cuda.matmul.allow_tf32
    torch.backends.cuda.matmul.allow_tf32 = False                 # fp32 Linear, as the parity tests
    st_dev = pipeline.state_to(st, dev)
    chunks = [tuple(t.to(dev) for t in c) for c in cpu_sample_rays(H4K, W4K, POSES[0], n_chunks, chunk)]
    kw = dict(scenes.RENDER_KW_DVGO)
    for c in chunks[:3]:
        pipeline.forward(st_dev, *c, ref_ops, **kw)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    t0 = time.perf_counter()
    e0.record()
    for c in chunks:
        pipeline.forward(st_dev, *c, ref_ops, **kw)
    e1.record()
    torch.cuda.synchronize()
    wall = time.perf_counter() - t0
    torch.backends.cuda.matmul.allow_tf32 = old
    ms = e0.elapsed_time(e1)
    n = n_chunks * chunk
    return {'rays_per_s': n / (ms * 1e-3), 'ms_per_8192_ray_chunk': ms / n_chunks, 'wall_s': wall,
            'sample': f'{n_chunks} x {chunk}-ray chunks spread over the 4032x3024 {regime} frame',
            'what': 'oracle/pipeline.py (the reference forward structure: flat lists, 3 compactions, grid_sample, Linear, index_add) '
                    'on the reference kernels compiled from /root/reference + ATen fp32, device timed incl. its host syncs'}


def secondary_sharded(model, kw, dev, world):
    """configs[4] (N>1): the whole 4K-NeRF frame across the ranks -- 1008x756 marcher (8-row blocks,
    one all-gather) + VC-Decoder x4 sharded by reference tile / tile row-parts (one all-gather).
    Device timed, max over ranks."""
    import k4nerf
    from k4nerf import render as krender
    from k4nerf import dist as krender_dist
    from oracle import scenes, sftnet
    out = {}
    try:
        net = k4nerf.SFTNet(3, 4, 64, 5, 32, 1)
        net.load_state_dict(sftnet.random_state_dict(seed=3, scale=1.0))
        net = net.to(dev)
        K, c2w = scenes.blender_camera(HLR, WLR, *POSES[0])
        run = lambda: krender.render_frame_4k_sharded(model, net, HLR, WLR, K, c2w, False, kw, test_tile=510)
        n_warm, n_timed = 4, 10          # the frame is ~6-15 ms: three frames after two warm-ups measured the clock ramp
        for _ in range(n_warm):
            run()
        torch.cuda.synchronize()
        dist.barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(n_timed):
            sr, _ = run()
        e1.record()
        torch.cuda.synchronize()
        t = torch.tensor([e0.elapsed_time(e1) / n_timed], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        out['configs[4]_full_frame_1008x756_to_4032x3024_sharded'] = {
            'ms_per_frame': t.item(), 'frames_per_s': 1e3 / t.item(), 'n_gpus': world,
            'decoder_units': len(krender_dist.sr_units(HLR, WLR, 510, 10, world, net.receptive_halo())),
            'sr_mean': float(sr.mean())}
    except Exception as e:
        out['configs[4]_error'] = repr(e)
    return out


def cpu_baseline(st):
    """The oracle port timed on the host cores, bounded sample (rank 0, N=1 only)."""
    from oracle import ops
    cores = cpu_threads()
    ops.set_num_threads(cores)
    chunks = cpu_sample_rays(H4K, W4K, POSES[0], 2)
    cpu_time_step(st, chunks[:1])                 # warm-up
    n, t = cpu_time_step(st, chunks)
    return {'value': n / t, 'unit': 'rays/s', 'cores': cores, 'kind': 'port',
            'sample': f'2 x 8192-ray chunks of the 4032x3024 frame ({t:.1f} s; oracle/pipeline.py, torch-CPU + C, {cores} threads)'}


if __name__ == '__main__':
    main()
