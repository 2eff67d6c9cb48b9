#!/usr/bin/env python
"""Benchmark of the differentiable stepping hot path: world-steps/s, forward + backward.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--worlds 4096] [--sim-steps 30]
                    [--dump-outputs DIR]
    torchrun --nnodes=1 --nproc-per-node N ... bench.py --gpus N --steps K --warmup W

Workload (BASELINE.json configs[1], "system_identification shape"): W independent worlds per GPU, each a 1x1x1
SDFBox (726 verts / 1200 faces) resting 2*eps above a pinned 20x1x20 floor slab (89 646 verts / 176 000 faces,
shared mesh), gravity + a constant push, per-world mass / friction / push; one bench step = one optimisation
iteration = `sim_steps` calls of World3D.step(fixed_dt=True) (with all their sub-steps) + loss.backward(),
loss = sum ||pos||^2, gradients w.r.t. the per-world mass, friction and push.

One JSON line on stdout (rank 0).  See the task contract for the keys; `roofline` describes the dominant kernel
by measured time, `cpu_baseline` the oracle port timed on this host.
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

import torch  # noqa: E402

METRIC = 'world-steps/sec fwd+bwd'
UNIT = 'world-steps/s'


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument('--gpus', type=int, default=1)
    ap.add_argument('--steps', type=int, default=5)
    ap.add_argument('--warmup', type=int, default=3)
    ap.add_argument('--impl', default='ours', choices=['ours', 'reference'])
    ap.add_argument('--worlds', type=int, default=4096, help='worlds per GPU')
    ap.add_argument('--sim-steps', type=int, default=30)
    ap.add_argument('--cpu-worlds', type=int, default=0, help='worlds of the bounded CPU sample (0 = two per core)')
    ap.add_argument('--cpu-sim-steps', type=int, default=0, help='0 = --sim-steps')
    ap.add_argument('--no-cpu-baseline', action='store_true')
    ap.add_argument('--no-sdf-query', action='store_true', help='skip the SDF-query HBM-roofline microbenchmark')
    ap.add_argument('--no-secondary', action='store_true', help='skip the config-3 / 4 / 5 secondary workloads')
    ap.add_argument('--strong-total', type=int, default=65536,
                    help='total worlds of the strong-scaling pass (config 5; 0 = skip)')
    ap.add_argument('--dump-outputs', metavar='DIR', default=None,
                    help='write what the last timed step returned (loss, gradients, final poses and velocities) as '
                         'DIR/<name>.npy, to compare two builds output for output')
    return ap.parse_args()


def measured_peaks():
    try:
        with open(os.path.join(ROOT, 'MEASURED_PEAKS.json')) as fh:
            return json.load(fh), 'measured'
    except Exception:
        return {'hbm_gbs': 6650.0, 'bf16_tflops': 1590.0}, 'fallback'


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index=0):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag, self.t_keep = index, [], False, None
        self.period = float(os.environ.get('BENCH_SMI_PERIOD', 0.5))   # every nvidia-smi call can stall launches for ms: sample sparsely

    def run(self):
        q = ('clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,'
             'clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap')
        while not self.stop_flag:
            try:
                out = subprocess.run(['nvidia-smi', '-i', str(self.index), '--query-gpu=' + q,
                                      '--format=csv,noheader,nounits'], capture_output=True, text=True, timeout=5).stdout
                if self.t_keep is not None and time.time() >= self.t_keep:      # samples of the timed regions only
                    self.rows.append([c.strip() for c in out.strip().split(',')])
            except Exception:
                pass
            time.sleep(self.period)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ['hw_slowdown', 'hw_thermal_slowdown', 'sw_thermal_slowdown', 'sw_power_cap']
        reasons = sorted({n for r in self.rows if len(r) >= 6 for n, v in zip(names, r[2:6]) if v.lower().startswith('active')})
        return {'sm_mhz': sm[len(sm) // 2] if sm else None, 'sm_max_mhz': max(mx) if mx else None, 'reasons': reasons,
                'samples': len(sm)}


def make_params(W, device, seed):
    """Per-world parameters in PINNED host memory (the optimisation variables of the sysid experiment)."""
    g = torch.Generator().manual_seed(seed)
    host = {'mass': 0.9 + 0.2 * torch.rand(W, generator=g, dtype=torch.float64),
            'fric_coeff': 0.01 + 0.24 * torch.rand(W, generator=g, dtype=torch.float64),
            'push': 2.0 + 3.0 * torch.rand(W, 2, generator=g, dtype=torch.float64)}
    if device.type == 'cuda':
        host = {k: v.pin_memory() for k, v in host.items()}
    return host


def gpu_iteration(spec, params_dev, sim_steps, device):
    """One optimisation iteration through the public API: build the world, roll out, backward."""
    from diffsdfsim_b200 import scenes
    leaves = {k: v.detach().requires_grad_(True) for k, v in params_dev.items()}
    world = scenes.build_world(spec, device=device, params=leaves)
    loss = 0.
    for _ in range(sim_steps):
        world.step(fixed_dt=True)
        loss = loss + (world.bodies[-1].pos ** 2).sum()
    loss.backward()
    return loss.detach(), {k: v.grad for k, v in leaves.items()}, world


DUMP_LIMIT = 64 << 20


def dump_outputs(out_dir, loss, grads, world):
    """What one optimisation iteration hands its caller -- the loss, the per-world gradients and the final poses and
    velocities of every body -- as float64 `out_dir/<name>.npy`.  Above DUMP_LIMIT bytes in all, a fixed seeded
    sample of the worlds is written instead; `world_index.npy` names the worlds written."""
    import numpy as np
    per_world = {'grad_' + k: g.detach() for k, g in grads.items()}
    per_world['final_p'] = world.get_p().detach().reshape(world.W, -1)
    per_world['final_v'] = world.get_v().detach().reshape(world.W, -1)
    row_bytes = 8 * (1 + sum(t.numel() // world.W for t in per_world.values()))
    keep = min(world.W, (DUMP_LIMIT - 8) // row_bytes)
    idx = torch.arange(world.W)
    if keep < world.W:
        idx = torch.randperm(world.W, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    os.makedirs(out_dir, exist_ok=True)
    arrays = {'loss': loss.detach().reshape(1), 'world_index': idx}
    arrays.update({k: t[idx.to(t.device)] for k, t in per_world.items()})
    for name, t in arrays.items():
        np.save(os.path.join(out_dir, name + '.npy'), t.cpu().numpy().astype(np.float64))


def run_ours(args):
    import torch.distributed as dist
    from diffsdfsim_b200 import _lib, scenes, distributed as D
    rank, local, world_size = D.env_rank()
    assert torch.cuda.is_available(), 'bench.py --impl ours needs a CUDA device (no CPU fallback)'
    torch.cuda.set_device(local)
    device = torch.device('cuda', local)
    D.init(device)
    _lib.lib()
    W = args.worlds
    spec = scenes.box_on_plane(steps=args.sim_steps)
    host = make_params(W, device, seed=rank)
    dev = {k: v.to(device) for k, v in host.items()}
    h2d = sum(v.numel() * v.element_size() for v in host.values())
    out_host = {k: torch.empty_like(v).pin_memory() for k, v in host.items()}
    loss_host = torch.empty(1, dtype=torch.float64).pin_memory()
    d2h = h2d + 8

    def allreduce(loss, grads):
        # shared-parameter reduction of batched system identification: loss and the summed gradients (ONE all-reduce)
        return D.reduce_loss_and_shared_grads(loss, [g.sum(0) for g in grads.values()])[0]

    def barrier():
        if world_size > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # the clock sampler starts before the warm-up: the first nvidia-smi invocation (NVML start-up, driver locks) stalls
    # kernel launches for tens of ms; only samples taken inside the timed regions are kept
    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    barrier()               # the first NCCL barrier sets up its own resources lazily: keep that out of the timed steps
    for _ in range(args.warmup):
        loss, grads, world = gpu_iteration(spec, dev, args.sim_steps, device)
        allreduce(loss, grads)
    # ---- device-resident timing ("value"): parameters already in HBM, no per-call profiling
    barrier()
    sampler.t_keep = time.time()
    _lib.reset_counters(profile=False)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    dbg = []
    for _ in range(args.steps):
        loss, grads, world = gpu_iteration(spec, dev, args.sim_steps, device)
        allreduce(loss, grads)
        if os.environ.get('BENCH_DEBUG'):
            torch.cuda.synchronize(); dbg.append(time.time())
    e1.record()
    barrier()
    last = (loss, grads, world)
    ms = e0.elapsed_time(e1)
    if dbg:
        print('rank', rank, 'value-loop step end times (s):', [round(t - dbg[0], 3) for t in dbg], 'total ms', ms, file=sys.stderr)
    launches = _lib.kernel_launches()
    syncs_per_step = sum(world.stats.get('syncs', [0])) / max(len(world.stats.get('syncs', [0])), 1)
    attempts = float(world.stats['attempts'].double().mean()) / args.sim_steps
    # ---- end-to-end timing: pinned host -> device inputs, device -> host loss and gradients, every step
    _lib.reset_counters(profile=False)
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record()
    for _ in range(args.steps):
        devp = {k: v.to(device, non_blocking=True) for k, v in host.items()}
        loss, grads, _ = gpu_iteration(spec, devp, args.sim_steps, device)
        loss = allreduce(loss, grads)
        loss_host.copy_(loss.reshape(1), non_blocking=True)
        for k in grads:
            out_host[k].copy_(grads[k], non_blocking=True)
        torch.cuda.synchronize()
    e3.record()
    barrier()
    ms_e2e = e2.elapsed_time(e3)
    sampler.stop_flag = True
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, *last)
    # ---- separate profiling pass (NOT part of any reported throughput): per-kernel device time of one iteration
    prof = kernel_profile(spec, dev, args.sim_steps, device) if rank == 0 else {}
    final_pos = world.bodies[-1].pos.detach().cpu()
    final_grads = {k: v.detach().cpu() for k, v in grads.items()}
    rounds_last = float(sum(world.stats['rounds']))
    per_rank = None
    if world_size > 1:
        mine = torch.tensor([ms / args.steps, ms_e2e / args.steps, rounds_last], dtype=torch.float64, device=device)
        allr = [torch.empty_like(mine) for _ in range(world_size)]
        dist.all_gather(allr, mine)
        per_rank = [[round(float(x), 2) for x in r] for r in allr]
    ms, ms_e2e = D.max_over_ranks([ms, ms_e2e], device)
    strong = None
    if args.strong_total > 0:
        strong = strong_scaling_pass(args, spec, device, rank, world_size, barrier, allreduce)
    sdfq = None
    if rank == 0 and not args.no_sdf_query:
        sdfq = sdf_query_roofline(device)
    secondary = None
    if rank == 0 and not args.no_secondary:
        secondary = secondary_workloads(device)
    units = W * args.sim_steps * args.steps * world_size
    if rank != 0:
        return None
    peaks, which = measured_peaks()
    # dominant entry point by measured device time
    top = max(prof.items(), key=lambda kv: kv[1][1]) if prof else ('none', (1, 0.0))
    roof = roofline(top[0], top[1], W, spec, peaks, which, attempts)
    fma = fma_peaks(device)
    busy_ms = sum(v[1] for v in prof.values())
    line = {
        'metric': METRIC, 'value': units / (ms / 1e3), 'unit': UNIT, 'n_gpus': world_size, 'steps': args.steps,
        'warmup': args.warmup, 'ms_per_step': ms / args.steps, 'higher_is_better': True, 'scaling': 'weak',
        'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
        'config': {'workload': 'box_on_plane sysid: %d worlds/GPU x %d World3D.step + backward; floor 176000 faces '
                               '(shared), box 1200 faces; grads wrt per-world mass, friction, push' % (W, args.sim_steps),
                   'worlds_per_gpu': W, 'sim_steps': args.sim_steps, 'attempts_per_world_step': attempts,
                   'l2_policy': 'every iteration rebuilds the world and writes / re-reads its per-round saved state '
                                '(contact sets, poses, multipliers: %.1f GB peak) -- larger than the 126 MB L2; the shared '
                                'meshes (4.4 MB) are L2-resident by design' % (torch.cuda.max_memory_allocated(device) / 1e9)},
        'e2e': {'value': units / (ms_e2e / 1e3), 'unit': UNIT, 'h2d_bytes_per_step': h2d, 'd2h_bytes_per_step': d2h},
        'gpu_launches': launches,
        'clocks': sampler.summary(),
        'roofline': roof,
        'kernel_ms_per_step': {k: round(v[1], 3) for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])},
        'kernel_launches_per_step': {k: v[0] for k, v in sorted(prof.items(), key=lambda kv: -kv[1][1])},
        'profile_note': 'kernel_ms_per_step / kernel_launches_per_step come from ONE extra iteration run after the timed '
                        'regions with CUDA events around every launch (on the launching stream); value and e2e are timed '
                        'without them.  library_kernel_ms / ms_per_step = %.2f' % (busy_ms / (ms / args.steps)),
        'host_syncs_per_world_step_call': syncs_per_step,
        'fma_peaks': fma,
    }
    if per_rank is not None:
        line['per_rank'] = {'columns': ['ms_per_step', 'ms_per_step_e2e', 'rounds_per_iteration'], 'rows': per_rank,
                            'note': 'ranks step DIFFERENT worlds (seed = rank); the job time is the slowest rank'}
    if strong is not None:
        line['strong_scaling'] = strong
    if sdfq is not None:
        line['sdf_query'] = sdfq
    if secondary is not None:
        line['secondary'] = secondary
    line['_final'] = (final_pos, final_grads)
    return line


def strong_scaling_pass(args, spec, device, rank, world_size, barrier, allreduce):
    """BASELINE config 5 as written: a FIXED total of `--strong-total` box-on-plane worlds sharded over the ranks (each rank
    owns total / N worlds), one optimisation iteration (30 World3D.step + backward + the one NCCL all-reduce of loss and
    shared-parameter gradients), device-timed, max over ranks.  Reported next to the weak-scaling headline so that both
    curves can be read from the N = 1, 2, 4, 8 lines."""
    import gc
    from diffsdfsim_b200 import distributed as D, stepper
    total = args.strong_total
    lo, hi = D.shard_range(total, rank, world_size)
    # memory: the tape of a rollout is ~1 MB per world (measured on the headline workload); keep one rollout resident
    gc.collect()
    stepper.clear_slot_pool()
    torch.cuda.empty_cache()
    free = torch.cuda.mem_get_info(device)[0]
    per_world = 1.2e6 * args.sim_steps / 30
    if (hi - lo) * per_world > 0.8 * free:
        return {'worlds_total': total, 'skipped': 'needs ~%.0f GB per GPU, %.0f GB free' % ((hi - lo) * per_world / 1e9, free / 1e9)}
    host = make_params(total, torch.device('cpu'), seed=12345)
    dev = {k: v[lo:hi].to(device) for k, v in host.items()}
    # two untimed iterations at this batch size: the first sizes the tape slots (they start small and grow while the worlds
    # pause), the second allocates them at their final size; from the third on a rollout re-uses the pooled slots (steady
    # state of an optimisation loop, which repeats the rollout every iteration).  One rollout resident at a time.
    for _ in range(2):
        loss, grads, w0 = gpu_iteration(spec, dev, args.sim_steps, device)
        allreduce(loss, grads)
        del w0, loss, grads
        gc.collect()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    loss, grads, w1 = gpu_iteration(spec, dev, args.sim_steps, device)
    allreduce(loss, grads)
    e1.record()
    barrier()
    peak = torch.cuda.max_memory_allocated(device) / 1e9
    del w1, loss, grads
    gc.collect()
    stepper.clear_slot_pool()
    torch.cuda.empty_cache()
    ms = D.max_over_ranks([e0.elapsed_time(e1)], device)[0]
    return {'worlds_total': total, 'worlds_per_gpu': hi - lo, 'n_gpus': world_size, 'ms_per_iteration': ms,
            'value': total * args.sim_steps / (ms / 1e3), 'unit': UNIT, 'scaling': 'strong', 'peak_mem_gb': peak,
            'workload': 'config 5: %d box-on-plane worlds in total, sharded over %d GPU(s), fwd+bwd + NCCL all-reduce; '
                        'third rollout at this batch size (tape slots pooled: steady state of an optimisation loop)'
                        % (total, world_size)}


def kernel_profile(spec, params_dev, sim_steps, device):
    """name -> (launches, total ms) of one optimisation iteration: the round kernels from the library's own event timing
    (dsdf_step_profile), the reverse-sweep / set-up entry points from events around the ctypes calls."""
    import ctypes
    from diffsdfsim_b200 import _lib
    lib = _lib.lib()
    _lib.reset_counters(profile=True)
    lib.dsdf_step_profile(1)
    gpu_iteration(spec, params_dev, sim_steps, device)
    prof = {k: v for k, v in _lib.profile_summary().items() if k not in ('dsdf_step_rounds',)}
    ms, n = (ctypes.c_double * 5)(), (ctypes.c_int32 * 5)()
    lib.dsdf_step_profile_read(ms, n)
    lib.dsdf_step_profile(0)
    _lib.reset_counters(profile=False)
    for name, t, k in zip(['step_prep_kernel', 'dyn_forward_kernel', 'step_integrate_kernel', 'contacts_kernel',
                           'step_commit_kernel'], ms, n):
        prof[name] = (int(k), float(t))
    return prof


def fma_peaks(device):
    """Measured FP64 / FP32 FMA rate of this GPU (dsdf_fma_peaks: dependent-chain microbenchmark)."""
    import ctypes
    from diffsdfsim_b200 import _lib
    scratch = torch.empty(4 << 20, dtype=torch.uint8, device=device)
    d, f = ctypes.c_double(0), ctypes.c_double(0)
    rc = _lib.lib().dsdf_fma_peaks(1 << 14, scratch.data_ptr(), ctypes.byref(d), ctypes.byref(f),
                                   torch.cuda.current_stream().cuda_stream)
    return {'fp64_tflops': d.value, 'fp32_tflops': f.value, 'how': 'dsdf_fma_peaks: 8 independent FMA chains / thread, '
            '8 CTAs x 256 threads per SM, CUDA events'} if rc == 0 else None


def secondary_workloads(device, reps=2):
    """world-steps/s (forward + backward, device-resident parameters, CUDA-event timed, best of `reps`) of the other
    BASELINE configurations at their named sizes: config 4 (256 worlds, per-world IGR-decoder grids and meshes, 33 steps),
    config 3 (1024 worlds x 16 mixed primitives, 200 steps) and config 5's per-GPU share of the inertia-fitting scene
    (8192 worlds, box under X/Y/Z constraints spun up by a torque, no contacts, 60 steps)."""
    import numpy as np
    from diffsdfsim_b200 import meshes, scenes
    F64 = torch.float64
    out = {}

    stalled = [0]

    def timed(build, steps, leaf_key, reps=reps):
        best = None
        for _ in range(reps):
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            torch.cuda.synchronize()
            e0.record()
            params, world = build()
            loss = 0.
            for _ in range(steps):
                world.step(fixed_dt=True)
                loss = loss + (world.bodies[-1].pos ** 2).sum() + (world.bodies[-1].v ** 2).sum()
            loss.backward()
            e1.record()
            torch.cuda.synchronize()
            dt = e0.elapsed_time(e1) / 1e3
            assert torch.isfinite(params[leaf_key].grad).all()
            best = dt if best is None else min(best, dt)
        stalled[0] = int(world.stats.get('stalled', 0))
        return world.W * steps / best, best

    g = torch.Generator().manual_seed(0)
    # ---- config 4 as named: 256 worlds, each with its own 64^3 grid baked from its own random-init IGR-style decoder and
    # its own iso-surface mesh; pinned 50x1x50 floor (1.04 M faces, shared), pinned pole, scale 2, drop from y = 6, 33 steps
    W, R = 256, 64
    pw = scenes.per_world_grid_bodies(W, res=R, seed0=1000, scale=2.0, device=device)
    spec4 = scenes.cow_on_pole(grid=pw['grid'][0].cpu().numpy(), steps=33)
    pos = torch.tensor([0.0, 6.0, 0.0], dtype=F64, device=device).expand(W, 3).contiguous()

    def build4():
        params = dict(pos=pos.detach().clone().requires_grad_(True), **pw)
        # not strict: among 256 random shapes a few reach states the reference itself would halve on for ever (world.py:344-348)
        return params, scenes.build_world(spec4, device=device, params=params, strict_no_penetration=False)
    v, secs = timed(build4, 33, 'pos')
    out['cow_on_pole'] = {'value': v, 'unit': UNIT, 'worlds': W, 'steps': 33, 'seconds': secs,
                          'workload': 'config 4 as named (demos/demo_meshsdf.py:121-142): per-world 64^3 f64 grids baked from '
                                      'random-init IGR-style decoders (8x128, skip_in [4], softplus beta 100) + per-world '
                                      'iso-surface meshes (%d..%d faces), scale 2, pinned pole + 50x1x50 floor (1 040 000 faces), '
                                      '33 steps, fwd+bwd' % (int(pw['nfaces'].min()), int(pw['nfaces'].max())),
                          'stalled_steps': stalled[0],
                          'contacts_kernel_ncu': {
                              'dram_bytes_per_launch': ncu_traffic('contacts_kernel@config4'),
                              'upper_bound_bytes': int(W * (R ** 3 * 8 + (int(pw['nverts'].max()) * 24 + int(pw['nfaces'].max()) * 12))),
                              'source': 'committed ncu capture of the heaviest contacts_kernel launch of profiles/tools/c4prof.py (256 '
                                        'worlds, same per-world grids and meshes; profiles/r2_ncu_summary.md), not measured in this '
                                        'run; upper_bound = every voxel of every 64^3 f64 grid + every vertex and face of every '
                                        'per-world mesh -- the kernel reads a fraction of it (dram_bytes / upper_bound): only the cells of the body mesh near the '
                                        'pole / floor and the voxels under the pole and floor faces it tests'},
                          'note': 'strict_no_penetration=False; stalled_steps = steps in which some world exhausted the 64 '
                                  'sub-step tape (it keeps giving up at dt/2^10, the reference would sub-step ~1000 times)'}
    # ---- config 3: 1024 worlds x 16 mixed primitives (120 body pairs), 200 steps, gradients w.r.t. every body's initial
    # velocity and mass
    W3, S3 = 1024, 200
    spec3 = scenes.mixed16(seed=0, steps=S3, spacing=1.05, speed=2.0)
    vel0 = torch.tensor([b['vel'] for b in spec3['bodies']], dtype=F64)
    mass0 = torch.tensor([b['mass'] for b in spec3['bodies']], dtype=F64)
    vel3 = (vel0[None] + 0.2 * torch.randn(W3, 16, 6, generator=g, dtype=F64) * (vel0[None] != 0)).to(device)
    mass3 = (mass0[None] * (0.9 + 0.2 * torch.rand(W3, 16, generator=g, dtype=F64))).to(device)

    def build3():
        params = dict(vel_all=vel3.detach().clone().requires_grad_(True), mass_all=mass3.detach().clone().requires_grad_(True))
        return params, scenes.build_world(spec3, device=device, params=params, strict_no_penetration=False)
    v, secs = timed(build3, S3, 'vel_all', reps=1)
    out['mixed16'] = {'value': v, 'unit': UNIT, 'worlds': W3, 'steps': S3, 'seconds': secs,
                      'workload': 'config 3: 16 mixed primitives (spheres / boxes / cylinders) per world, free-floating with '
                                  'random velocities (SURVEY s8d C3, no-gravity variant), all 120 pairs searched, 200-step '
                                  'rollout + backward to every initial velocity and mass', 'stalled_steps': stalled[0]}
    W5 = 8192
    mass = (0.5 + torch.rand(W5, generator=g, dtype=F64)).to(device)
    spec5 = scenes.inertia_fitting(steps=60)

    def build5():
        params = dict(mass=mass.detach().requires_grad_(True))
        return params, scenes.build_world(spec5, device=device, params=params)
    v, secs = timed(build5, 60, 'mass')
    out['inertia_fitting'] = {'value': v, 'unit': UNIT, 'worlds': W5, 'steps': 60, 'seconds': secs,
                              'workload': "config 5's per-GPU share: 8192 worlds, box under X/Y/Z constraints, torque "
                                          'until t = 0.3, no contacts'}
    return out


def sdf_query_roofline(device, W=256, R=64, N=1 << 17, reps=5):
    """HBM roofline of the stand-alone SDF query operator (dsdf_sdf_query) on config-4 shaped data: W per-world R^3 f64
    grids (W*R^3*8 = 512 MiB, larger than the 126 MB L2) and N surface-ordered query points per world with value +
    direction out.  Algorithmic bytes per launch = W * (N * (24 in + 8 + 24 out) + R^3 * 8 grid, every voxel touched)."""
    from diffsdfsim_b200 import ops
    peaks, which = measured_peaks()
    g = torch.Generator(device='cpu').manual_seed(0)
    t = torch.linspace(-1, 1, R, dtype=torch.float64)
    X, Y, Z = torch.meshgrid(t, t, t, indexing='ij')
    base = (X * X + Y * Y + Z * Z).sqrt() - 0.6
    grid = (base[None] + 0.01 * torch.rand(W, 1, 1, 1, generator=g, dtype=torch.float64)).to(device).contiguous()
    # points: a jittered lattice in scan order (coherent like mesh vertices emitted by marching cubes)
    n1 = int(round(N ** (1 / 3)))
    while n1 ** 3 < N:
        n1 += 1
    u = torch.linspace(-0.98, 0.98, n1, dtype=torch.float64)
    P = torch.stack(torch.meshgrid(u, u, u, indexing='ij'), -1).reshape(-1, 3)[:N]
    pts = (P[None] + 0.005 * torch.rand(W, N, 3, generator=g, dtype=torch.float64)).to(device).contiguous()
    shape = torch.tensor([0.0, 0.0, 0.0, 1.0], dtype=torch.float64, device=device).expand(W, 4).contiguous()
    def run(want_dir):
        with torch.no_grad():
            for _ in range(3):
                ops.sdf_query('grid', shape, pts, grid=grid, want_dir=want_dir)
            torch.cuda.synchronize()
            ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(reps)]
            for a, b in ev:
                a.record()
                ops.sdf_query('grid', shape, pts, grid=grid, want_dir=want_dir)
                b.record()
            torch.cuda.synchronize()
        return sum(a.elapsed_time(b) for a, b in ev) / reps

    ms = run(True)
    alg = W * (N * 56 + R ** 3 * 8)
    ach = alg / 1e9 / (ms / 1e3)
    ms_v = run(False)                       # value only: 24 B in + 8 B out per point, 8 voxel reads, ~60 FP64 ops
    alg_v = W * (N * 32 + R ** 3 * 8)
    ach_v = alg_v / 1e9 / (ms_v / 1e3)
    return {'kernel': 'dsdf_sdf_query (grid, per-world %d^3 f64 grids, W=%d, N=%d pts/world, value+direction)' % (R, W, N),
            'bound': 'hbm', 'achieved': ach, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s', 'frac': ach / peaks['hbm_gbs'],
            'peak_source': which, 'avg_launch_ms': ms, 'algorithmic_bytes_per_launch': alg,
            'l2_policy': 'inputs (%.2f GB) larger than L2' % (alg / 1e9), 'traffic': ncu_traffic('sdf_query_grid_kernel<1>'),
            'traffic_source': 'committed ncu capture (profiles/ncu_traffic.json), not measured in this run',
            'note': 'value + direction: DRAM traffic equals the algorithmic bytes; the remaining gap is on-chip: 35 eight-byte '
                    'gathers per point (L1/TEX 74 % of peak in ncu) and ~200 FP64 instr/point (FP64 pipe 38 %); occupancy '
                    'does not move it.  value_only = the same query without the direction (its own kernel instantiation: '
                    '8 gathers per point, HBM-bound), see DESIGN.md s5',
            'value_only': {'achieved': ach_v, 'frac': ach_v / peaks['hbm_gbs'], 'avg_launch_ms': ms_v,
                           'algorithmic_bytes_per_launch': alg_v, 'traffic': ncu_traffic('sdf_query_grid_kernel<0>')}}


def ncu_counters(kernel):
    """Selected ncu counters of `kernel` from the committed capture (profiles/ncu_counters.json), for context."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'ncu_counters.json')) as fh:
            c = json.load(fh).get(kernel, {})
        keep = ('achieved occupancy %', 'issue slots busy %', 'FP64 pipe active %', 'DRAM throughput %', 'regs/thread')
        return {k: c[k] for k in keep if k in c}
    except Exception:
        return None


def ncu_traffic(kernel):
    """dram bytes (read + write) per launch of `kernel` from the committed ncu capture (profiles/ncu_traffic.json)."""
    try:
        with open(os.path.join(ROOT, 'profiles', 'ncu_traffic.json')) as fh:
            d = json.load(fh)
        return d.get(kernel, d.get('void ' + kernel))
    except Exception:
        return None


def roofline(name, stat, W, spec, peaks, which, attempts):
    """Algorithmic bytes per launch of the dominant entry point / its measured average duration (DESIGN.md s5)."""
    calls, total_ms = stat
    avg_ms = total_ms / max(calls, 1)
    nb, maxc, fd = 2, 16, 8
    nz, ni = 6 * nb, maxc * (2 + fd)
    if name.startswith('dsdf_lcp'):
        # compulsory: read Q, p, G, h, A, F rows of the ACTIVE problem (~10 contacts) + write x, lam, s
        nia = 100
        per_world = 8 * (nz * nz + nz + nia * nz + nia + 6 * nz + nia * nia + nz + 2 * nia)
    elif name in ('dsdf_contacts_detect', 'contacts_kernel'):
        # per world and search direction: poses + the candidate/contact lists; shared meshes count once per launch
        per_world = 2 * 7 * 8 * 2 + 300 * 4 * 2 + 16 * (4 + 8 + 24 + 80)
        shared = 176000 * 12 + 89646 * 24 + 1200 * 12 + 726 * 24
        alg = per_world * W + shared
        return {'kernel': name, 'bound': 'hbm', 'achieved': alg / 1e9 / (avg_ms / 1e3), 'peak': peaks['hbm_gbs'],
                'unit': 'GB/s', 'frac': alg / 1e9 / (avg_ms / 1e3) / peaks['hbm_gbs'], 'traffic': ncu_traffic('contacts_kernel'),
                'peak_source': which, 'avg_launch_ms': avg_ms, 'algorithmic_bytes_per_launch': alg,
                'traffic_source': 'committed ncu capture (profiles/ncu_traffic.json), not measured in this run',
                'note': 'shared L2-resident meshes: not an HBM-bound kernel on this workload; its limits are latency, '
                        'barriers and FP64 issue (DESIGN.md s4); avg_launch_ms averages full-width and nearly empty rounds',
                'ncu': ncu_counters('contacts_kernel')}
    else:
        per_world = 8 * (nz * nz + ni * nz)
    alg = per_world * W
    ach = alg / 1e9 / (avg_ms / 1e3)
    return {'kernel': name, 'bound': 'hbm', 'achieved': ach, 'peak': peaks['hbm_gbs'], 'unit': 'GB/s',
            'frac': ach / peaks['hbm_gbs'], 'traffic': None, 'peak_source': which, 'avg_launch_ms': avg_ms,
            'algorithmic_bytes_per_launch': alg}


def _cpu_world(job):
    """One world of the bounded CPU sample: the oracle port (oracle/, CPU float64) -- `sim_steps` World.step + backward."""
    w, sim_steps, seed, n_total = job
    import warnings
    warnings.filterwarnings('ignore')
    torch.set_num_threads(1)
    from oracle.scenes import build as build_oracle
    from diffsdfsim_b200 import scenes
    spec = scenes.box_on_plane(steps=sim_steps)
    host = make_params(n_total, torch.device('cpu'), seed)     # world w of the SAME parameter draw the GPU arm uses
    t0 = time.time()
    leaves = dict(mass=host['mass'][w].clone().requires_grad_(True),
                  fric_coeff=host['fric_coeff'][w].clone().requires_grad_(True),
                  push=host['push'][w].clone().requires_grad_(True))
    ow = build_oracle(spec, leaves)
    loss = 0.
    for _ in range(sim_steps):
        ow.step()
        loss = loss + (ow.bodies[-1].pos ** 2).sum()
    loss.backward()
    return (time.time() - t0, ow.bodies[-1].pos.detach().tolist(), float(leaves['mass'].grad),
            float(leaves['fric_coeff'].grad), leaves['push'].grad.tolist())


_POOL = None


def cpu_pool():
    """One worker process per host core (worlds are independent: this is all the parallelism the CPU path has)."""
    global _POOL
    if _POOL is None:
        import multiprocessing as mp
        _POOL = mp.get_context('spawn').Pool(os.cpu_count() or 1)
        _POOL.map(_cpu_world, [(0, 1, 0, 1)] * (os.cpu_count() or 1))      # import + warm every worker
    return _POOL


def cpu_sample(n_worlds, sim_steps, seed=0, n_total=None, results=None):
    """world-steps/s of the CPU path on `n_worlds` worlds spread over all host cores, and the wall seconds it took.
    The worlds are the first `n_worlds` of the `n_total`-world parameter draw; `results` (a list) receives each
    world's (seconds, final position, d loss / d mass, d loss / d friction, d loss / d push)."""
    pool = cpu_pool()
    t0 = time.time()
    out = pool.map(_cpu_world, [(w, sim_steps, seed, n_total or n_worlds) for w in range(n_worlds)], chunksize=1)
    dt = time.time() - t0
    if results is not None:
        results.extend(out)
    return n_worlds * sim_steps / dt, dt


def cpu_sizes(args):
    cores = os.cpu_count() or 1
    return (args.cpu_worlds or 2 * cores), (args.cpu_sim_steps or args.sim_steps), cores


def run_reference(args):
    """The reference's CPU implementation of the path: here the oracle port (the reference is pure Python/torch with
    un-vendored dependencies and cannot travel to the GPU box; see DESIGN.md s2), one world per host core at a time."""
    from diffsdfsim_b200 import distributed as D
    rank, _, _ = D.env_rank()
    if rank != 0:
        return None
    nw, ns, cores = cpu_sizes(args)
    cpu_pool()
    for _ in range(args.warmup):
        cpu_sample(cores, 1)
    t0 = time.time()
    for k in range(args.steps):
        cpu_sample(nw, ns, seed=k)
    total = time.time() - t0
    units = nw * ns * args.steps
    value = units / total
    sample = ('%d worlds x %d World.step + backward per bench step (same scene, meshes and parameters '
              'distribution as the 4096-world workload), one world per process on %d cores' % (nw, ns, cores))
    return {'impl': 'reference', 'metric': METRIC, 'value': value, 'unit': UNIT, 'n_gpus': args.gpus,
            'steps': args.steps, 'warmup': args.warmup, 'ms_per_step': total / args.steps * 1e3,
            'higher_is_better': True, 'scaling': 'weak', 'vs_baseline': None, 'dtype': 'f64', 'data': 'synthetic',
            'config': {'workload': 'box_on_plane sysid (bounded CPU sample of the %d-world workload)' % args.worlds,
                       'worlds_per_gpu': args.worlds, 'sim_steps': args.sim_steps},
            'cpu_baseline': {'value': value, 'unit': UNIT, 'cores': cores, 'kind': 'port', 'sample': sample},
            'e2e': {'value': value, 'unit': UNIT, 'h2d_bytes_per_step': 0, 'd2h_bytes_per_step': 0}}


def close_pool():
    global _POOL
    if _POOL is not None:
        _POOL.close()
        _POOL.join()
        _POOL = None


def main():
    import atexit
    atexit.register(close_pool)
    args = parse()
    # stdout carries exactly ONE JSON line: anything libraries print to file descriptor 1 while the benchmark runs
    # (e.g. NCCL's version banner) is sent to stderr instead
    sys.stdout.flush()
    real_stdout = os.dup(1)
    os.dup2(2, 1)

    def emit(line):
        sys.stdout.flush()
        os.dup2(real_stdout, 1)
        print(json.dumps(line), flush=True)
    if args.impl == 'reference':
        line = run_reference(args)
        if line is not None:
            emit(line)
        return
    line = run_ours(args)
    if line is None:
        return
    if args.gpus == 1 and not args.no_cpu_baseline:
        nw, ns, cores = cpu_sizes(args)
        res = []
        v, secs = cpu_sample(nw, ns, seed=0, n_total=args.worlds, results=res)
        line['cpu_baseline'] = {'value': v, 'unit': UNIT, 'cores': cores, 'kind': 'port',
                                'sample': '%d worlds x %d World.step + backward, one world per process on %d cores, '
                                          '%.1f s wall' % (nw, ns, cores, secs)}
        if ns == args.sim_steps and '_final' in line:
            # the CPU sample re-simulated worlds 0..nw-1 of the GPU batch: report the end-of-rollout drift
            import numpy as np
            pos, gr = line['_final']
            ref_pos = np.array([r[1] for r in res])
            dpos = float(np.abs(pos[:nw].numpy() - ref_pos).max())

            def rel(a, b):
                a, b = np.asarray(a, dtype=np.float64), np.asarray(b, dtype=np.float64)
                return float(np.abs(a - b).max() / max(np.abs(b).max(), 1e-30))
            line['parity'] = {'worlds': nw, 'rollout_steps': ns,
                              'max_abs_pos_drift_vs_oracle': dpos,
                              'max_rel_grad_err': {'mass': rel(gr['mass'][:nw], [r[2] for r in res]),
                                                   'fric_coeff': rel(gr['fric_coeff'][:nw], [r[3] for r in res]),
                                                   'push': rel(gr['push'][:nw], [r[4] for r in res])},
                              'note': 'GPU worlds 0..%d of the timed batch vs the CPU oracle on the same parameters, '
                                      'after the full %d-step rollout (normalised by the largest reference gradient)'
                                      % (nw - 1, ns)}
    line.pop('_final', None)
    emit(line)


if __name__ == '__main__':
    main()
