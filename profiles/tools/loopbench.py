"""Quick A/B: device loop vs host loop on the bench workload.  usage: python profiles/tools/loopbench.py [W] [steps] [iters]"""
import sys, time
sys.path.insert(0, '.')
import torch
from diffsdfsim_b200 import scenes, _lib
from diffsdfsim_b200.world import World3D
F64 = torch.float64
W = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 30
iters = int(sys.argv[3]) if len(sys.argv) > 3 else 3
modes = sys.argv[4].split(',') if len(sys.argv) > 4 else ['dev', 'host']
g = torch.Generator().manual_seed(0)
host = {'mass': 0.9 + 0.2 * torch.rand(W, generator=g, dtype=F64), 'fric_coeff': 0.01 + 0.24 * torch.rand(W, generator=g, dtype=F64),
        'push': 2.0 + 3.0 * torch.rand(W, 2, generator=g, dtype=F64)}
dev = {k: v.cuda() for k, v in host.items()}
spec = scenes.box_on_plane(steps=steps)

def it():
    leaves = {k: v.detach().requires_grad_(True) for k, v in dev.items()}
    world = scenes.build_world(spec, device='cuda', params=leaves)
    loss = 0.
    tf = time.time()
    for _ in range(steps):
        world.step(fixed_dt=True)
        loss = loss + (world.bodies[-1].pos ** 2).sum()
    torch.cuda.synchronize(); tf = time.time() - tf
    tb = time.time()
    loss.backward()
    torch.cuda.synchronize(); tb = time.time() - tb
    return world, float(loss), tf, tb, {k: v.grad for k, v in leaves.items()}

res = {}
from diffsdfsim_b200 import stepper as _st
_st.DeviceStepper.TIMING = {}
import os
if os.environ.get('FORCE_CTA'):
    _st.DeviceStepper.FORCE_CTA = os.environ['FORCE_CTA'] == '1'
for mode in modes:
    World3D.device_loop = mode == 'dev'
    for _ in range(2):
        it()
    torch.cuda.synchronize()
    t0 = time.time()
    _st.DeviceStepper.TIMING.clear()
    for _ in range(iters):
        tb0 = time.time()
        world, loss, tf, tb, grads = it()
        print('   iter %.1f ms (fwd %.1f, bwd %.1f)' % ((time.time() - tb0) * 1e3, tf * 1e3, tb * 1e3), flush=True)
    torch.cuda.synchronize()
    dt = (time.time() - t0) / iters
    res[mode] = (loss, grads)
    print('%s: %.1f ms/iter  (last: fwd %.1f ms, bwd %.1f ms)  rounds %d  syncs %s  attempts/world-step %.3f  -> %.0f world-steps/s'
          % (mode, dt * 1e3, tf * 1e3, tb * 1e3, sum(world.stats['rounds']), sum(world.stats.get('syncs', [0])),
             float(world.stats['attempts'].double().mean()) / steps, W * steps / dt), flush=True)
    print('  peak mem %.2f GB' % (torch.cuda.max_memory_allocated() / 1e9))
    from diffsdfsim_b200 import stepper
    if stepper.DeviceStepper.TIMING:
        print('  host phases (s, all iterations):', {k: round(v, 3) for k, v in stepper.DeviceStepper.TIMING.items()})
        print('  pool: %d keys, %.1f GB; history %s' % (len(stepper._SLOT_POOL), stepper._slot_pool_bytes / 1e9, stepper._ROWS_HISTORY))
        stepper.DeviceStepper.TIMING.clear()
if len(res) == 2:
    a, b = res['dev'], res['host']
    print('loss equal:', a[0] == b[0], a[0], b[0])
    for k in a[1]:
        d = (a[1][k] - b[1][k]).abs().max() / b[1][k].abs().max()
        print('  grad', k, 'max rel diff %.2e' % float(d))
