#!/usr/bin/env python
"""Benchmark of the shapegan hot path on B200 (contract: see the task statement / DESIGN.md "Measurement").

    python bench.py --gpus N --steps K --warmup W [--impl reference] [--workload wgan_gp|wgan|gan|hybrid|autodecoder]
                    [--dump-outputs DIR]

One "step" of the default workload = BASELINE.json configs[1]: the 3D-CNN WGAN-GP G+D step on 32^3 voxels, batch 64 per GPU,
bf16 -- train_wgan.py:62-71 (critic update: fake B + real B, RMSprop) with the gradient penalty of
train_hybrid_progressive_gan.py:102-111 in place of the weight clip (SURVEY D1; north_star: "the 32^3 WGAN-GP config")
+ train_wgan.py:75-84 (generator update).  metric = voxels/s = n_gpus * B * 32^3 / step time.  Prints ONE JSON line on rank 0.

  value     : step timed with inputs resident in HBM (CUDA events per iteration, L2 flushed between iterations, max over ranks)
  e2e       : same step through the public step object with the batch + latents (+ alpha) copied from pinned host memory and the
              loss scalars read back, every step, inside the timed region
  roofline  : the dominant kernel (tcgen05 implicit GEMM, Conv3d 64->128 forward at B=64) timed alone with CUDA events
              against MEASURED_PEAKS.json (bf16 burst TFLOP/s)
  configs   : the other BASELINE configs / variants, each measured the same way (value + e2e + necessary-FLOP fraction):
              wgan_clip (train_wgan.py as written), wgan_gp_fp32x (the 1e-3 parity mode), gan_b32 (configs[3]: train_gan.py:58-86 at
              32 samples/GPU = global 256 on 8 GPUs), hybrid_it3 (configs[4]: train_hybrid_progressive_gan.py:134-166, 64^3)
  sdfnet    : SDFNet Mpoints/s (fused forward, configs[2] autodecoder step)
  cpu_baseline : the oracle port of the same step (oracle/ref_steps.py, torch CPU fp32 = what the reference runs on a CPU host)
              timed on this box's cores

--dump-outputs DIR writes what the timed step returned in its last timed iteration -- its loss scalars and the updated parameters
and buffers of the models it trains -- as DIR/<name>.npy (float32).  The inputs and initial weights are seeded, so two builds run
with the same arguments can be compared output for output.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import torch

REPO = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, REPO)

VOX = 32 ** 3
FLOPS_D2_FWD = 2 * 17179.9e6          # Conv3d(64->128,k4,s2,p1) forward at B=64: SURVEY.md App. A.2 (dense MACs x 2)
# SURVEY.md 8d, dense MACs per SAMPLE (x2 = FLOP): G fwd 421.5 M, D fwd 419.4 M (first layer 16.8 M), bwd-data = bwd-weight = fwd
G_MAC, D_MAC, D1_MAC, G1_MAC = 421.527552e6, 419.446784e6, 16.777216e6, 2.097152e6
PD3_MAC = 1008.73024e6               # progressive discriminator it=3, per 64^3 sample
SDF_MAC = 460544.0                   # SDFNet forward per point


def gflop_per_sample(workload):
    """(necessary, as written) GFLOP per sample of one step; necessary = without gradients nobody reads (SURVEY 8d)."""
    crit = G_MAC + 2 * D_MAC + 2 * (2 * D_MAC - D1_MAC)                 # fake + real through D, dgrad (not into the input) + wgrad
    gen_nec = G_MAC + D_MAC + D_MAC + (G_MAC - G1_MAC) + G_MAC          # G fwd, D fwd, D dgrad (all layers), G dgrad + wgrad
    gen_written = gen_nec + D_MAC                                       # + the critic wgrad that zero_grad() discards
    gp = 4 * D_MAC                                                      # GP: 4 passes of D (SURVEY H3)
    if workload == 'wgan':
        return 2e-9 * (crit + gen_nec), 2e-9 * (crit + gen_written)
    if workload == 'wgan_gp':
        return 2e-9 * (crit + gp + gen_nec), 2e-9 * (crit + gp + gen_written)
    if workload == 'gan':                                               # train_gan.py:58-86: G step, D-fake step, D-real step
        dfake = G_MAC + D_MAC + (D_MAC - D1_MAC) + D_MAC
        dreal = D_MAC + (D_MAC - D1_MAC) + D_MAC
        return 2e-9 * (gen_nec + dfake + dreal), 2e-9 * (gen_written + dfake + dreal)
    raise ValueError(workload)


def hybrid_gflop_per_sample(r=64):
    """train_hybrid_progressive_gan.py it=3: (D update, G update) necessary GFLOP per sample."""
    pts = r ** 3
    d_up = pts * SDF_MAC + 2 * PD3_MAC + 2 * (2 * PD3_MAC) + 4 * PD3_MAC            # G fwd (no grad needed) + fake/valid fwd+bwd + GP
    g_up = 3 * pts * SDF_MAC + 2 * PD3_MAC                                            # SDFNet fwd + dgrad + wgrad, D fwd + dgrad
    return 2e-9 * d_up, 2e-9 * g_up


WORKLOAD_NAMES = {
    'wgan_gp': 'configs[1]: 3D-CNN WGAN-GP G+D step 32^3, batch %d/GPU (train_wgan.py:62-71 with the GP of train_hybrid_progressive_gan.py:102-111, + :75-84)',
    'wgan': 'configs[1] (clip variant): 3D-CNN WGAN G+D step 32^3, batch %d/GPU (train_wgan.py:62-71 + :75-84 as written)',
    'gan': 'configs[3]: voxel GAN iteration 32^3, batch %d/GPU (train_gan.py:58-86: G step, D-fake step, D-real step)',
    'hybrid': 'configs[4]: hybrid progressive GAN it=3 (64^3 CNN critic + SDFNet generator), batch %d/GPU (train_hybrid_progressive_gan.py:134-166)',
    'autodecoder': 'configs[2]: DeepSDF autodecoder 16384 pts x %d shapes/step (train_sdf_autodecoder.py:84-91)',
}


def workload_name(wl, b):
    return WORKLOAD_NAMES[wl] % b


def peaks():
    p = os.path.join(REPO, 'MEASURED_PEAKS.json')
    if os.path.exists(p):
        d = json.load(open(p))
        return d, 'measured (MEASURED_PEAKS.json)'
    return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0, 'bf16_tflops_sustained': 1400.0}, 'fallback (B200_PROFILING.md)'


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe).  Started before the warm-up (the
    tool needs a few hundred ms to produce its first row); only rows stamped inside [mark_begin, mark_end] are reported."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, False, []
        q = 'clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,' \
            'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap'
        self.cmd = ['nvidia-smi', '-i', str(index), '--query-gpu=' + q, '--format=csv,noheader,nounits', '-lms', '20']
        self.proc = None
        self.t0 = self.t1 = None

    def run(self):
        try:
            self.proc = subprocess.Popen(self.cmd, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            for line in self.proc.stdout:
                if self.stop_flag:
                    break
                self.rows.append((time.perf_counter(), [c.strip() for c in line.split(',')]))
        except Exception:
            pass

    def wait_first(self, timeout=3.0):
        t = time.perf_counter()
        while not self.rows and time.perf_counter() - t < timeout:
            time.sleep(0.01)

    def mark_begin(self):
        self.t0 = time.perf_counter()

    def mark_end(self):
        self.t1 = time.perf_counter()

    def finish(self):
        self.stop_flag = True
        if self.proc is not None:
            self.proc.terminate()
        sm, mx, reasons = [], 0.0, set()
        for ts, r in self.rows:
            if self.t0 is not None and not (self.t0 <= ts <= (self.t1 or ts) + 0.05):
                continue
            try:
                sm.append(float(r[0])); mx = max(mx, float(r[1]))
                for name, v in zip(('hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap'), r[3:7]):
                    if v.lower().startswith('active'):
                        reasons.add(name)
            except Exception:
                continue
        sm.sort()
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': mx or None, 'reasons': sorted(reasons), 'samples': len(sm)}


def synth_voxels(b, seed, r=32):
    g = torch.Generator().manual_seed(seed)
    return torch.clamp(torch.randn((b, r, r, r), generator=g) * 0.05, -0.1, 0.1) / 0.1      # SURVEY 8d / datasets.py:20-22


_JSON_OUT = None      # rank 0's real stdout once file descriptor 1 has been pointed at stderr (multi-rank runs)


def emit(line):
    """the ONE JSON line of this run, on the process's original stdout"""
    if _JSON_OUT is not None:
        _JSON_OUT.write(line + '\n')
        _JSON_OUT.flush()
    else:
        print(line, flush=True)


def dist_setup(n):
    global _JSON_OUT
    world = int(os.environ.get('WORLD_SIZE', '1'))
    if world > 1:
        # rank 0 prints exactly one JSON line on stdout, and NCCL writes its version banner / INFO log (ring, tree, NVLS, nranks) to
        # file descriptor 1 whatever NCCL_DEBUG_FILE says: keep a private handle on the real stdout for the JSON line and point fd 1 at
        # stderr for everything else, so the log is visible instead of silenced
        sys.stdout.flush()
        _JSON_OUT = os.fdopen(os.dup(1), 'w')
        os.dup2(2, 1)
        if os.environ.get('SG_B200_QUIET_NCCL') != '1':      # the GPU boxes preset NCCL_DEBUG=VERSION: ask for the init log explicitly
            os.environ['NCCL_DEBUG'] = 'INFO'
            os.environ.setdefault('NCCL_DEBUG_SUBSYS', 'INIT,ENV')
        import torch.distributed as dist
        local = int(os.environ.get('LOCAL_RANK', '0'))
        torch.cuda.set_device(local)
        dist.init_process_group('nccl', device_id=torch.device('cuda', local))
        return dist.get_rank(), world, local
    return 0, 1, 0


def max_over_ranks(ms, world):
    if world == 1:
        return ms
    import torch.distributed as dist
    t = torch.tensor([ms], dtype=torch.float64, device='cuda')
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    return float(t.item())


def barrier(world):
    if world > 1:
        import torch.distributed as dist
        dist.barrier()
    torch.cuda.synchronize()


# --------------------------------------------------------------------------------------------------------- CPU arms (oracle port)
def usable_cpus():
    try:
        n = len(os.sched_getaffinity(0))
    except Exception:
        n = os.cpu_count() or 1
    try:                                    # cgroup v2 quota of the container, if any
        q, per = open('/sys/fs/cgroup/cpu.max').read().split()
        if q != 'max':
            n = max(1, min(n, int(float(q) / float(per) + 0.5)))
    except Exception:
        pass
    return n


def pick_cpu_threads(run):
    """torch CPU thread count that runs the reference step fastest on this host: os.cpu_count() threads oversubscribe
    the GPU boxes badly (128 logical CPUs, 22.9 s/step at 128 threads vs 1.5 s), so time one step at a few counts."""
    avail = usable_cpus()
    cands = sorted({c for c in (8, 16, 32, 64, avail) if c <= avail} | {min(avail, 8)})
    torch.set_num_threads(cands[0])
    run()                                   # warm-up (primitive caches, allocator)
    best, log = None, []
    for c in cands:
        torch.set_num_threads(c)
        t0 = time.perf_counter()
        run()
        dt = time.perf_counter() - t0
        log.append('%d:%.2fs' % (c, dt))
        if best is None or dt < best[1]:
            best = (c, dt)
    torch.set_num_threads(best[0])
    return best[0], best[1], '{' + ' '.join(log) + '}'


def cpu_step(workload, b, ad_shapes=8):
    """(run, units, unit, metric, sample) of the oracle port of one step of `workload` at the GPU arm's per-GPU batch."""
    from oracle import ref_steps as S
    from oracle import shapes as TS
    if workload in ('wgan', 'wgan_gp'):
        step = S.WGANStepCPU(S.make_params(TS.gen_shapes(), 601), S.make_params(TS.disc_shapes(), 602), gp=(workload == 'wgan_gp'))
        real = synth_voxels(b, 605)
        z1 = torch.randn((b, 128), generator=torch.Generator().manual_seed(1))
        z2 = torch.randn((b, 128), generator=torch.Generator().manual_seed(2))
        alpha = torch.rand((b, 1, 1, 1), generator=torch.Generator().manual_seed(3))
        return (lambda: step(real, z1, z2, alpha)), b * VOX, 'voxels/s', 'wgan_gd_step_voxels_per_s', 'the full B=%d step, fp32, torch CPU' % b
    if workload == 'gan':
        step = S.GANStepCPU(S.make_params(TS.gen_shapes(), 601), S.make_params(TS.disc_shapes(), 602))
        real = synth_voxels(b, 605)
        z1 = torch.randn((b, 128), generator=torch.Generator().manual_seed(1))
        z2 = torch.randn((b, 128), generator=torch.Generator().manual_seed(2))
        return (lambda: step(real, z1, z2)), b * VOX, 'voxels/s', 'gan_iteration_voxels_per_s', 'the full B=%d iteration, fp32, torch CPU' % b
    if workload == 'hybrid':
        bb = min(b, 2)
        gsd, dsd = S.make_params(TS.sdf_shapes(), 41), S.make_params(TS.prog_shapes(), 42)
        step = S.HybridProgressiveStepCPU(gsd, dsd, 3)
        valid = synth_voxels(bb, 10, 64) * 0.1
        z = torch.randn((bb, 128), generator=torch.Generator().manual_seed(1))
        alpha = torch.rand((bb, 1, 1, 1), generator=torch.Generator().manual_seed(3))
        return (lambda: step.discriminator_update(valid, z, alpha)), bb * 64 ** 3, 'voxels/s', 'hybrid_it3_d_update_voxels_per_s', \
            'critic update at B=%d (of %d), 64^3, fp32, torch CPU' % (bb, b)
    n, shapes = 16384 * ad_shapes, ad_shapes
    sd = S.make_params(TS.sdf_shapes(), 101)
    g = torch.Generator().manual_seed(5)
    pts = torch.rand((n, 3), generator=g) * 2 - 1
    table = torch.randn((shapes, 128), generator=g) * 0.01
    idx = torch.arange(n) // 16384
    sdf = torch.clamp(pts.norm(dim=1) - 0.5, -0.1, 0.1)
    step = S.AutodecoderStepCPU(sd, table)
    return (lambda: step(pts, sdf, idx)), n, 'points/s', 'sdfnet_autodecoder_step_points_per_s', \
        '16384 points x %d shapes of the 16384x512 step, fp32, torch CPU' % shapes


def run_reference(args, rank, world):
    """The reference's own CPU implementation of the step (oracle port), on the host threads that run it fastest, at the GPU arm's
    config (same per-GPU batch; exactly --steps timed steps)."""
    if rank != 0:
        return
    run, units, unit, metric, sample = cpu_step(args.workload, args.batch)
    cores, t_one, calib = pick_cpu_threads(run)
    steps = args.steps
    warm = max(0, min(args.warmup, int(30.0 / max(t_one, 1e-3))))
    for _ in range(warm):
        run()
    t0 = time.perf_counter()
    for _ in range(steps):
        run()
    dt = (time.perf_counter() - t0) / steps
    v = units / dt
    sample += '; %d timed steps; threads picked by a one-step sweep %s' % (steps, calib)
    print(json.dumps({
        'impl': 'reference', 'metric': metric, 'value': v, 'unit': unit, 'n_gpus': args.gpus, 'steps': steps, 'warmup': args.warmup,
        'ms_per_step': dt * 1e3, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f32', 'data': 'synthetic',
        'config': {'workload': workload_name(args.workload, args.batch if args.workload != 'autodecoder' else args.ad_shapes),
                   'global_batch': args.gpus * args.batch, 'parallelism': 'dp%d' % args.gpus,
                   'note': 'oracle port of the reference step (oracle/ref_steps.py = the reference modules\' torch-CPU fp32 path, pinned to the '
                           'unmodified reference by tests/test_ref_steps_golden.py) on host cores: one replica\'s batch; the reference is pure '
                           'PyTorch and /root/reference cannot travel to the GPU box'},
        'cpu_baseline': {'value': v, 'unit': unit, 'cores': cores, 'kind': 'port', 'sample': sample},
        'e2e': {'value': v, 'unit': unit, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}))


def cpu_baseline(workload, b):
    run, units, unit, _, sample = cpu_step(workload, b)
    cores, t_one, calib = pick_cpu_threads(run)
    n = max(1, min(5, int(20.0 / max(t_one, 1e-3))))
    t0 = time.perf_counter()
    for _ in range(n):
        run()
    dt = (time.perf_counter() - t0) / n
    return {'value': units / dt, 'unit': unit, 'cores': cores, 'kind': 'port',
            'sample': '%d steps of %s (oracle/ref_steps.py, %d threads picked by a one-step sweep %s)' % (n, sample, cores, calib)}


# --------------------------------------------------------------------------------------------------------- roofline probe
def roofline_probe(flush):
    """Time the dominant kernel alone: sg_igemm (MODE_CONV, halo-reuse variant) for Conv3d(64->128) at B=64, bf16."""
    from shapegan_b200 import _lib as L
    from shapegan_b200 import raw
    b, r, cin, cout = 64, 16, 64, 128
    x = torch.randn((1, b, r, r, r, cin), device='cuda').to(torch.bfloat16)
    w = torch.randn((cout, cin, 4, 4, 4), device='cuda') * 0.05
    img = raw.pack_conv_fwd(w, 1)
    y = torch.empty((1, b, r // 2, r // 2, r // 2, cout), dtype=torch.bfloat16, device='cuda')
    rows = b * (r // 2) ** 3

    def launch():
        raw.igemm(L.MODE_CONV, 1, x, (b, r, r, r, cin), rows, 64 * cin, img, cout, y, cout, act=L.ACT_LRELU)
    for _ in range(3):
        launch()
    torch.cuda.synchronize()
    ms = []
    for _ in range(20):
        flush.zero_()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); launch(); e1.record()
        torch.cuda.synchronize()
        ms.append(e0.elapsed_time(e1))
    ms.sort()
    avg = sum(ms[2:-2]) / len(ms[2:-2])
    # the same launch at the batched critic's size (3 x 64 samples: three work items per CTA, epilogues overlapped) and back to back with
    # L2-resident inputs (how it runs inside the step, right behind its producer): supplementary, the judged figure is the flushed B = 64 one
    extra = {}
    try:
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(20):
            launch()
        e1.record(); torch.cuda.synchronize()
        warm = e0.elapsed_time(e1) / 20
        extra['l2_resident_back_to_back'] = {'launch_ms': warm, 'tflops': FLOPS_D2_FWD / (warm * 1e-3) / 1e12}
        b3 = 3 * b
        x3 = torch.randn((1, b3, r, r, r, cin), device='cuda').to(torch.bfloat16)
        y3 = torch.empty((1, b3, r // 2, r // 2, r // 2, cout), dtype=torch.bfloat16, device='cuda')
        t3 = []
        for i in range(10):
            flush.zero_()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e0.record(); raw.igemm(L.MODE_CONV, 1, x3, (b3, r, r, r, cin), 3 * rows, 64 * cin, img, cout, y3, cout, act=L.ACT_LRELU); e1.record()
            torch.cuda.synchronize()
            if i >= 2:
                t3.append(e0.elapsed_time(e1))
        m3 = sum(t3) / len(t3)
        extra['batched_critic_B192_flushed'] = {'launch_ms': m3, 'tflops': 3 * FLOPS_D2_FWD / (m3 * 1e-3) / 1e12}
        del x3, y3
    except Exception as e:                       # supplementary only
        extra['error'] = str(e).split('\n')[0][:100]
    pk, src = peaks()
    for v in extra.values():
        if isinstance(v, dict):
            v['frac'] = v['tflops'] / pk['bf16_tflops']
    achieved = FLOPS_D2_FWD / (avg * 1e-3) / 1e12
    traffic, tsrc = None, 'no ncu capture of this build committed yet'
    tj = os.path.join(REPO, 'profiles', 'roofline_traffic.json')       # written by tools/make_profiles.py from the ncu --set full capture
    if os.path.exists(tj):
        try:
            d = json.load(open(tj))
            traffic, tsrc = d.get('conv_probe_dram_bytes'), d.get('source')
        except Exception:
            pass
    return {'bound': 'tensor', 'achieved': achieved, 'peak': pk['bf16_tflops'], 'unit': 'TFLOP/s', 'frac': achieved / pk['bf16_tflops'],
            'traffic': traffic, 'traffic_source': '%s; algorithmic DRAM bytes 33.6 MB input + 1.0 MB weights (the 8.4 MB output stays in L2)' % tsrc,
            'kernel': 'sg_igemm_halo2_kernel (CTA pairs, tcgen05.mma.cta_group::2) MODE_CONV Conv3d(64->128,k4,s2,p1) fwd B=64 (34.36 GFLOP/launch), '
                      'L2 flushed before every launch',
            'launch_ms': avg, 'peak_source': src + ', burst (kernel timed alone)', 'same_kernel_other_conditions': extra}


def sdfnet_probe(dev, world):
    """SDFNet Mpoints/s (BASELINE.json metric, second half): fused forward at the north_star's 250k-point batch and at configs[2]'s
    8.39 M points, plus the configs[2] autodecoder step.  Inputs exceed L2 at the large size; CUDA events, 3 warm-ups."""
    from model.sdf_net import SDFNet
    from shapegan_b200 import train
    torch.manual_seed(0)
    net = SDFNet()
    pk, src = peaks()
    out = {}

    def timed(fn, reps):
        for _ in range(3):
            fn()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(reps):
            fn()
        e1.record()
        torch.cuda.synchronize()
        return e0.elapsed_time(e1) / reps

    for tag, n, reps in (('fwd_250k_points', 250000, 20), ('fwd_8388608_points', 512 * 16384, 5)):
        pts = torch.rand((n, 3), device=dev) * 2 - 1
        table = torch.randn((512, 128), device=dev) * 0.1
        idx = ((torch.arange(n, device=dev) * 512) // n).to(torch.int32)
        with torch.no_grad():
            ms = timed(lambda: net(pts, table, idx), reps)
        tf = 0.921e6 * n / (ms * 1e-3) / 1e12
        out[tag] = {'mpoints_per_s': n / ms / 1e3, 'ms': ms, 'tflops': tf, 'frac_of_burst_peak': tf / pk['bf16_tflops']}
    n = 512 * 16384
    pts = torch.rand((n, 3), device=dev) * 2 - 1
    sdf = torch.clamp(pts.norm(dim=1) - 0.5, -0.1, 0.1)
    idx = (torch.arange(n, device=dev) // 16384).to(torch.int32)
    step = train.AutodecoderStep(net, torch.randn((512, 128), device=dev) * 0.01, world_size=1, points_per_shape=16384)
    ms = timed(lambda: step(pts, sdf, idx), 5)
    tf = 2.763e6 * n / (ms * 1e-3) / 1e12
    out['autodecoder_step_512x16384'] = {'mpoints_per_s': n / ms / 1e3, 'ms': ms, 'tflops': tf, 'frac_of_sustained_peak': tf / pk['bf16_tflops_sustained']}
    big = out['fwd_8388608_points']
    out['roofline'] = {'bound': 'tensor', 'achieved': big['tflops'], 'peak': pk['bf16_tflops'], 'unit': 'TFLOP/s', 'frac': big['frac_of_burst_peak'],
                       'traffic': None, 'kernel': 'sg_sdfnet_fwd_kernel, 0.921 MFLOP/point (SURVEY 8d); algorithmic 16 B/point', 'peak_source': src + ', burst'}
    del step
    torch.cuda.empty_cache()
    return out


# --------------------------------------------------------------------------------------------------------- workloads (GPU arm)
class Workload:
    """One timed step: `body()` runs it on the device inputs and leaves the loss scalars in `d_loss`; `host`/`dev` are the matching
    pinned-host / device input tensors the e2e leg copies every step."""

    def __init__(self, name, body, host, dev, d_loss, units, nec_gflop, written_gflop=None, note=''):
        self.name, self.body, self.host, self.dev, self.d_loss = name, body, host, dev, d_loss
        self.units, self.nec_gflop, self.written_gflop, self.note = units, nec_gflop, written_gflop, note
        self.h_loss = torch.zeros(d_loss.numel()).pin_memory()


def model_state(prefix, module):
    """{prefix.name: tensor} of the parameters and floating-point buffers of a module (aliased parameters once)"""
    out = {'%s.%s' % (prefix, k): v for k, v in module.named_parameters()}
    out.update({'%s.%s' % (prefix, k): v for k, v in module.named_buffers() if v.is_floating_point()})
    return out


def named_losses(d_loss, names):
    return {n: d_loss[i] for i, n in enumerate(names)}


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, arrays):
    """--dump-outputs: every array as out_dir/<name>.npy in float32"""
    import numpy as np
    total = sum(t.numel() * 4 for t in arrays.values())
    if total > DUMP_LIMIT:
        raise SystemExit('bench.py: --dump-outputs would write %d bytes (limit %d)' % (total, DUMP_LIMIT))
    os.makedirs(out_dir, exist_ok=True)
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.detach().float().cpu().numpy())


def make_cnn_workload(kind, b, rank, world, dev, gp_fused=True):
    """wgan / wgan_gp / gan on gan.Generator + gan.Discriminator (random-init weights of the reference architecture)."""
    from model.gan import Discriminator, Generator
    from shapegan_b200 import train
    torch.manual_seed(0)
    gen, dis = Generator(), Discriminator()
    host = [synth_voxels(b, 605 + rank).pin_memory(),
            torch.randn((b, 128), generator=torch.Generator().manual_seed(11 + rank)).pin_memory(),
            torch.randn((b, 128), generator=torch.Generator().manual_seed(23 + rank)).pin_memory()]
    if kind == 'wgan_gp':
        host.append(torch.rand((b, 1, 1, 1), generator=torch.Generator().manual_seed(37 + rank)).pin_memory())
    devt = [t.to(dev) for t in host]
    if kind == 'gan':
        step = train.GANStep(gen, dis, world_size=world)
        d_loss = torch.zeros(3, device=dev)

        def body():
            a, c, d = step(devt[0], devt[1], devt[2])
            d_loss[0].copy_(a); d_loss[1].copy_(c); d_loss[2].copy_(d)
    else:
        step = train.WGANStep(gen, dis, gp=(kind == 'wgan_gp'), world_size=world)
        d_loss = torch.zeros(2, device=dev)

        def body():
            cl, gl = step(devt[0], devt[1], devt[2], devt[3] if kind == 'wgan_gp' else None)
            d_loss[0].copy_(cl); d_loss[1].copy_(gl)
    nec, written = gflop_per_sample(kind)
    w = Workload(kind, body, host, devt, d_loss, b * VOX, nec * b, written * b)
    w.keep = (gen, dis, step)
    losses = ('generator_loss', 'fake_loss', 'valid_loss') if kind == 'gan' else ('critic_loss', 'generator_loss')
    w.outputs = {**named_losses(d_loss, losses), **model_state('generator', gen), **model_state('critic', dis)}
    w.dp_note = (step.copt if kind != 'gan' else step.dopt).dp_note
    return w


def make_hybrid_workloads(b, rank, world, dev):
    """configs[4]: (critic update, generator update) of train_hybrid_progressive_gan.py at it=3 (64^3)."""
    from model.progressive_gan import Discriminator
    from model.sdf_net import SDFNet
    from shapegan_b200 import train
    torch.manual_seed(0)
    gen, dis = SDFNet(), Discriminator().to(dev)
    step = train.HybridProgressiveStep(gen, dis, 3, world_size=world)
    host = [(synth_voxels(b, 705 + rank, 64) * 0.1).pin_memory(),
            torch.randn((b, 128), generator=torch.Generator().manual_seed(41 + rank)).pin_memory(),
            torch.rand((b, 1, 1, 1), generator=torch.Generator().manual_seed(43 + rank)).pin_memory()]
    devt = [t.to(dev) for t in host]
    dl, gl = torch.zeros(2, device=dev), torch.zeros(1, device=dev)

    def d_body():
        loss, gp = step.discriminator_update(devt[0], devt[1], devt[2])
        dl[0].copy_(loss); dl[1].copy_(gp)

    def g_body():
        gl[0].copy_(step.generator_update(devt[1]))
    d_nec, g_nec = hybrid_gflop_per_sample(64)
    wd = Workload('hybrid_d_update', d_body, host, devt, dl, b * 64 ** 3, d_nec * b)
    wg = Workload('hybrid_g_update', g_body, [host[1]], [devt[1]], gl, b * 64 ** 3, g_nec * b)
    wd.keep = wg.keep = (gen, dis, step)
    wd.outputs = {**named_losses(dl, ('critic_loss', 'gradient_penalty')), **named_losses(gl, ('generator_loss',)),
                  **model_state('generator', gen), **model_state('critic', dis)}
    wd.dp_note = wg.dp_note = step.dopt.dp_note
    return wd, wg


def capture(body, no_graph):
    """Whole step (fwd + bwd + all-reduce + optimizer) in one CUDA graph when it captures; eager otherwise (same kernels)."""
    if no_graph:
        return body, 'eager'
    try:
        s = torch.cuda.Stream()
        s.wait_stream(torch.cuda.current_stream())
        with torch.cuda.stream(s):
            body()
        torch.cuda.current_stream().wait_stream(s)
        graph = torch.cuda.CUDAGraph()
        with torch.cuda.graph(graph):
            body()
        for _ in range(2):
            graph.replay()
        torch.cuda.synchronize()
        return graph.replay, 'cuda_graph(whole step: fwd+bwd+allreduce+optimizer)'
    except Exception as e:
        torch.cuda.synchronize()
        return body, 'eager (graph capture failed: %s)' % str(e).split('\n')[0][:120]


def measure(w, steps, warmup, world, flush, lib, no_graph=False, sampler=None):
    """value leg (inputs resident) and e2e leg (H2D of the inputs + D2H of the losses every step) of one workload; ms = max over ranks."""
    l0 = lib.sg_launch_count()
    for _ in range(warmup):
        w.body()
    torch.cuda.synchronize()
    launches = (lib.sg_launch_count() - l0) // max(warmup, 1)
    run, note = capture(w.body, no_graph)
    if sampler is not None:
        sampler.wait_first()
    barrier(world)
    if sampler is not None:
        sampler.mark_begin()
    # per-iteration CUDA events, ONE host synchronisation at the end: the device queue stays full (no host jitter between iterations,
    # which at N > 1 every collective would turn into a wait for the slowest rank); the L2 flush sits between the event pairs
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for e0, e1 in evs:
        flush.zero_()
        e0.record(); run(); e1.record()
    torch.cuda.synchronize()
    total = sum(e0.elapsed_time(e1) for e0, e1 in evs)
    barrier(world)
    ms = max_over_ranks(total / steps, world)
    barrier(world)
    evs = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(steps)]
    for e0, e1 in evs:
        flush.zero_()
        e0.record()
        for d, h in zip(w.dev, w.host):
            d.copy_(h, non_blocking=True)
        run()
        w.h_loss.copy_(w.d_loss, non_blocking=True)
        e1.record()
    torch.cuda.synchronize()
    e2e = sum(e0.elapsed_time(e1) for e0, e1 in evs)
    barrier(world)
    if sampler is not None:
        sampler.mark_end()
    e2e_ms = max_over_ranks(e2e / steps, world)
    pk, _ = peaks()
    sus = pk.get('bf16_tflops_sustained', 1400.0)
    return {'ms_per_step': ms, 'value': world * w.units / (ms * 1e-3),
            'e2e': {'value': world * w.units / (e2e_ms * 1e-3), 'ms_per_step': e2e_ms,
                    'h2d_bytes_per_step': int(sum(h.numel() * h.element_size() for h in w.host)), 'd2h_bytes_per_step': int(w.h_loss.numel() * 4)},
            'launch': note, 'gpu_launches_per_step': int(launches), 'steps': steps, 'data_parallel': getattr(w, 'dp_note', 'single'),
            'step_gflop_necessary': w.nec_gflop, 'step_gflop_as_written': w.written_gflop,
            'step_tflops': w.nec_gflop / ms, 'step_frac_of_sustained_peak': w.nec_gflop / ms / sus,
            'losses': [float(x) for x in w.h_loss]}


def extra_configs(args, rank, world, dev, flush, lib):
    """The other BASELINE configs / variants as sub-blocks of the same JSON line (all ranks take part: the steps all-reduce)."""
    from shapegan_b200 import config
    out = {}
    steps = args.extra_steps

    def guarded(tag, fn):
        try:
            out[tag] = fn()
        except Exception as e:                      # secondary numbers must never cost the headline line
            out[tag] = {'error': str(e).split('\n')[0][:200]}
        torch.cuda.empty_cache()

    def cnn(kind, b, precision='bf16'):
        def run():
            config.set_precision(precision)
            try:
                w = make_cnn_workload(kind, b, rank, world, dev)
                r = measure(w, steps, 3, world, flush, lib, args.no_graph)
            finally:
                config.set_precision(args.precision)
            r.update({'workload': workload_name(kind, b), 'unit': 'voxels/s', 'global_batch': world * b,
                      'dtype': 'bf16' if precision == 'bf16' else 'bf16x3(fp32x)'})
            return r
        return run

    if args.workload != 'wgan':
        guarded('wgan_clip', cnn('wgan', args.batch))
    if args.workload != 'wgan_gp':
        guarded('wgan_gp', cnn('wgan_gp', args.batch))
    guarded('wgan_gp_fp32x', cnn('wgan_gp', args.batch, 'fp32x'))
    guarded('gan_b32', cnn('gan', 32))               # configs[3]: global 256 on 8 GPUs = 32 per GPU

    def hybrid(b):
        def run():
            wd, wg = make_hybrid_workloads(b, rank, world, dev)
            rd = measure(wd, max(3, steps // 2), 3, world, flush, lib, args.no_graph)
            rg = measure(wg, max(3, steps // 2), 3, world, flush, lib, args.no_graph)
            sched = rd['ms_per_step'] + rg['ms_per_step'] / 5.0       # the generator is updated every 5th batch (:136)
            return {'workload': workload_name('hybrid', b), 'unit': 'voxels/s', 'global_batch': world * b, 'dtype': 'bf16',
                    'd_update': rd, 'g_update': rg, 'ms_per_batch_5to1_schedule': sched,
                    'value': world * b * 64 ** 3 / (sched * 1e-3),
                    'sdfnet_points_per_step': b * 64 ** 3}
        return run
    guarded('hybrid_it3_b2', hybrid(2))              # configs[4]: global 16 on 8 GPUs = 2 per GPU
    if world == 1:
        guarded('hybrid_it3_b16', hybrid(16))        # the reference's whole batch (BATCH_SIZE = 16, :37) on one GPU
    return out


# --------------------------------------------------------------------------------------------------------- main arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=50)
    ap.add_argument('--warmup', type=int, default=5)
    ap.add_argument('--impl', default='b200')
    ap.add_argument('--workload', default='wgan_gp', choices=['wgan_gp', 'wgan', 'gan', 'hybrid', 'autodecoder'])
    ap.add_argument('--batch', type=int, default=None)
    ap.add_argument('--precision', default='bf16', choices=['bf16', 'fp32x'])
    ap.add_argument('--no-graph', action='store_true')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-sdfnet', action='store_true', help='skip the secondary SDFNet Mpoints/s block')
    ap.add_argument('--no-extra', action='store_true', help='skip the sub-blocks of the other BASELINE configs')
    ap.add_argument('--extra-steps', type=int, default=10)
    ap.add_argument('--ad-shapes', type=int, default=512, help='autodecoder workload: number of shapes (16384 points each)')
    ap.add_argument('--dump-outputs', metavar='DIR', help='write the outputs of the last timed step as DIR/<name>.npy')
    args = ap.parse_args()
    if args.steps < 1:
        ap.error('--steps must be at least 1')
    if args.dump_outputs and args.impl == 'reference':
        ap.error('--dump-outputs applies to the B200 arm')
    if args.batch is None:
        args.batch = {'gan': 32, 'hybrid': 2}.get(args.workload, 64)
    if args.impl == 'reference':
        rank = int(os.environ.get('RANK', '0'))
        run_reference(args, rank, int(os.environ.get('WORLD_SIZE', '1')))
        return
    if not torch.cuda.is_available():
        raise SystemExit('bench.py: no CUDA device (the B200 path has no CPU fallback; use --impl reference for the CPU arm)')
    args.warmup = max(args.warmup, 3)
    rank, world, local = dist_setup(args.gpus)
    dev = torch.device('cuda', local)
    from shapegan_b200 import _lib as L
    from shapegan_b200 import config
    config.set_precision(args.precision)
    lib = L.lib()

    if args.workload == 'autodecoder':
        return bench_autodecoder(args, rank, world, dev, lib)

    sampler = ClockSampler(local) if rank == 0 else None
    if sampler is not None:
        sampler.start()
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)          # > 126 MB L2
    b = args.batch
    if args.workload == 'hybrid':
        wd, wg = make_hybrid_workloads(b, rank, world, dev)
        res = measure(wd, args.steps, args.warmup, world, flush, lib, args.no_graph, sampler)
        res_g = measure(wg, max(3, args.steps // 5), 3, world, flush, lib, args.no_graph)
        metric = 'hybrid_it3_d_update_voxels_per_s'
        w = wd
    else:
        w = make_cnn_workload(args.workload, b, rank, world, dev)
        res = measure(w, args.steps, args.warmup, world, flush, lib, args.no_graph, sampler)
        res_g = None
        metric = 'wgan_gd_step_voxels_per_s' if args.workload.startswith('wgan') else 'gan_iteration_voxels_per_s'
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, w.outputs)
    clocks = sampler.finish() if sampler is not None else None
    extras = None if args.no_extra else extra_configs(args, rank, world, dev, flush, lib)
    err = lib.sg_check_device_error()
    if rank != 0:
        return
    roof = roofline_probe(flush)
    out = {
        'metric': metric, 'value': res['value'], 'unit': 'voxels/s', 'n_gpus': world,
        'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': res['ms_per_step'], 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'bf16' if args.precision == 'bf16' else 'bf16x3(fp32x)', 'data': 'synthetic',
        'config': {'workload': workload_name(args.workload, b),
                   'global_batch': world * b, 'parallelism': 'dp%d' % world, 'launch': res['launch'], 'data_parallel': res['data_parallel'],
                   'l2': 'flushed (256 MiB memset) between timed iterations',
                   'step_gflop_necessary': res['step_gflop_necessary'], 'step_gflop_as_written': res['step_gflop_as_written'],
                   'step_tflops': res['step_tflops'], 'step_frac_of_sustained_peak': res['step_frac_of_sustained_peak'],
                   'flop_convention': 'necessary dense FLOPs (SURVEY 8d: gradients nobody reads are not counted) / measured time'},
        'e2e': dict(res['e2e'], unit='voxels/s'),
        'gpu_launches': int(res['gpu_launches_per_step'] * args.steps * 2),
        'gpu_launches_per_step': res['gpu_launches_per_step'],
        'roofline': roof, 'clocks': clocks, 'device_error_word': err,
        'losses': res['losses'],
    }
    if res_g is not None:
        out['g_update'] = res_g
    if extras is not None:
        out['configs'] = extras
    if not args.no_sdfnet:
        try:
            out['sdfnet'] = sdfnet_probe(dev, world)
        except Exception as e:            # secondary numbers must never cost the headline line
            out['sdfnet'] = {'error': str(e).split('\n')[0][:200]}
    if not args.no_cpu_baseline:
        out['cpu_baseline'] = cpu_baseline(args.workload, b)
    emit(json.dumps(out))


def bench_autodecoder(args, rank, world, dev, lib):
    """BASELINE.json configs[2]: DeepSDF autodecoder 16384 pts x 512 shapes / step (train_sdf_autodecoder.py:84-91)."""
    from model.sdf_net import SDFNet
    from shapegan_b200 import train
    torch.manual_seed(0)
    shapes, per = args.ad_shapes, 16384
    n = shapes * per
    net = SDFNet()
    g = torch.Generator().manual_seed(5 + rank)
    pts = (torch.rand((n, 3), generator=g) * 2 - 1).to(dev)
    sdf = torch.clamp(pts.norm(dim=1) - 0.5, -0.1, 0.1)
    idx = (torch.arange(n, device=dev) // per).to(torch.int32)
    table = torch.randn((shapes, 128), generator=g).to(dev) * 0.01
    step = train.AutodecoderStep(net, table, world_size=world, points_per_shape=per)
    for _ in range(max(args.warmup, 3)):
        step(pts, sdf, idx)
    torch.cuda.synchronize()
    barrier(world)
    total = 0.0
    steps = args.steps
    for _ in range(steps):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); loss = step(pts, sdf, idx); e1.record()
        torch.cuda.synchronize()
        total += e0.elapsed_time(e1)
    ms = max_over_ranks(total / steps, world)
    if rank != 0:
        return
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, {'loss': loss, 'latent_table': step.table, **model_state('sdf_net', net)})
    pk, src = peaks()
    tflops = 2.763e6 * n / (ms * 1e-3) / 1e12
    emit(json.dumps({
        'metric': 'sdfnet_autodecoder_step_points_per_s', 'value': world * n / (ms * 1e-3), 'unit': 'points/s', 'n_gpus': world, 'steps': steps,
        'warmup': args.warmup, 'ms_per_step': ms, 'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'bf16', 'data': 'synthetic',
        'config': {'workload': workload_name('autodecoder', shapes), 'points_per_gpu': n,
                   'l2': 'inputs (%.1f GB) exceed L2' % (n * 20 / 1e9), 'parallelism': 'dp%d' % world},
        'gpu_launches': int(lib.sg_launch_count()),
        'roofline': {'bound': 'tensor', 'achieved': tflops, 'peak': pk['bf16_tflops_sustained'], 'unit': 'TFLOP/s', 'frac': tflops / pk['bf16_tflops_sustained'],
                     'traffic': None, 'note': 'whole step, 2.763 MFLOP/point fwd+bwd (SURVEY 8d); peak = ' + src + ' sustained'},
        'loss': float(loss)}))


if __name__ == '__main__':
    try:
        main()
    finally:
        try:
            import torch.distributed as _dist
            if _dist.is_available() and _dist.is_initialized():
                _dist.destroy_process_group()
        except Exception:
            pass
