import sys, time, ctypes, torch
sys.path.insert(0, '.')
from diffsdfsim_b200 import scenes, _lib
from diffsdfsim_b200.utils import Defaults3D
W = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
S = int(sys.argv[2]) if len(sys.argv) > 2 else 12
gen = torch.Generator().manual_seed(0)
mass = (0.9 + 0.2 * torch.rand(W, generator=gen, dtype=torch.float64)).cuda().requires_grad_(True)
fric = (0.01 + 0.24 * torch.rand(W, generator=gen, dtype=torch.float64)).cuda().requires_grad_(True)
push = (2.0 + 3.0 * torch.rand(W, 2, generator=gen, dtype=torch.float64)).cuda().requires_grad_(True)
spec = scenes.box_on_plane(steps=S)
import os
world = scenes.build_world(spec, device='cuda', params=dict(mass=mass, fric_coeff=fric, push=push), capK=int(os.environ.get('CAPK', 512)))
for k in range(S):
    world.step(fixed_dt=True)
torch.cuda.synchronize()
print('contacts: mean %.1f max %d' % (world.contact_set.count.double().mean().item(), int(world.contact_set.count.max())))
p = world.state.p.detach().contiguous()
L = _lib.lib()
buf = (ctypes.c_ulonglong * 16)()
def timeit(fn, n=5):
    fn(); torch.cuda.synchronize()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(n)]
    for a, b in ev:
        a.record(); fn(); b.record()
    torch.cuda.synchronize()
    return sum(a.elapsed_time(b) for a, b in ev) / n
cs = world.contact_set.clone()
act = torch.ones(W, dtype=torch.uint8, device='cuda')
det = lambda: world.detector.detect(p, world.shape, cs, act, eps=world.eps, tol=world.tol, fd_eps=Defaults3D.EPSILON, body_eps=world.body_eps)
L.dsdf_contacts_phase_cycles(buf, 1)
ms = timeit(det)
rc = L.dsdf_contacts_phase_cycles(buf, 1)
print('contacts_detect %.3f ms / launch (W=%d)' % (ms, W))
if rc == 0:
    names = ['overlap', 'gather', 'sort+init', 'fw', 'push+compact', 'geometry', 'filter', 'append']
    tot = sum(buf[:8])
    print('   per world-launch: fw iters %.1f (both dirs), candidates %.0f, prefilter contacts %.0f' % (buf[8] / 6 / W, buf[9] / 6 / W, buf[10] / 6 / W))
    names += ['iters', 'cand', 'pre', 'f.cluster', 'f.stats', 'f.akl', 'f.sort(+dedupe)', 'f.chain']
    for n, v in zip(names, buf):
        print('   %-14s %5.1f %%   %8.0f cycles/world/launch' % (n, 100.0 * v / max(tot, 1), v / 6 / W))
dbuf = (ctypes.c_ulonglong * 11)()
DYN_NAMES = ['load', 'residuals', 'factor', 'assembly', 'lu', 'solve0', 'ratio+corr', 'solve1', 'update', 'best']
def dyn_phases(label, nworlds):
    # per world-launch; the counters cover every timed launch and the warm-up one
    if L.dsdf_dynamics_phase_cycles(dbuf, 1) != 0:
        return
    tot = sum(dbuf[:10])
    launches = 6 * nworlds
    print('   %s: %.1f loop passes per world, %.0f cycles per world' % (label, dbuf[10] / launches, tot / launches))
    for n, v in zip(DYN_NAMES, dbuf):
        print('   %-14s %5.1f %%   %8.0f cycles/world/launch' % (n, 100.0 * v / max(tot, 1), v / launches))
with torch.no_grad():
    dt = torch.full((W,), world.dt, dtype=torch.float64, device='cuda')
    L.dsdf_dynamics_phase_cycles(dbuf, 1)
    ms = timeit(lambda: world.engine.solve(world, dt, act))
print('dynamics_solve %.3f ms / launch, max_nc %d' % (ms, world.max_nc))
dyn_phases('dense', W)
one = torch.zeros(W, dtype=torch.uint8, device='cuda'); one[7] = 1
ms1 = timeit(lambda: world.detector.detect(p, world.shape, cs, one, eps=world.eps, tol=world.tol, fd_eps=Defaults3D.EPSILON, body_eps=world.body_eps))
with torch.no_grad():
    L.dsdf_dynamics_phase_cycles(dbuf, 1)
    ms2 = timeit(lambda: world.engine.solve(world, dt, one))
print('single active world: contacts %.3f ms, dynamics %.3f ms' % (ms1, ms2))
dyn_phases('single world', 1)
