"""Cost of World3D(record_substeps=True) on the bench workload: the 4096-world box-on-plane rollout (30 steps, loss on the
box position after every step, backward), recording off and on, alternated in one process.

    python profiles/tools/substep_record_cost.py [W] [steps] [runs]

Both settings compute the same loss; recording adds the gather of the sub-step states from the tape, the extra
outputs of every step node and their (zero) gradients in the reverse sweep.  Prints the card and its power limit."""
import subprocess
import sys
import time

sys.path.insert(0, '.')
import torch

from diffsdfsim_b200 import scenes

F64 = torch.float64
W = int(sys.argv[1]) if len(sys.argv) > 1 else 4096
steps = int(sys.argv[2]) if len(sys.argv) > 2 else 30
runs = int(sys.argv[3]) if len(sys.argv) > 3 else 5
g = torch.Generator().manual_seed(0)
params = {'mass': 0.9 + 0.2 * torch.rand(W, generator=g, dtype=F64),
          'fric_coeff': 0.01 + 0.24 * torch.rand(W, generator=g, dtype=F64),
          'push': 2.0 + 3.0 * torch.rand(W, 2, generator=g, dtype=F64)}
params = {k: v.cuda() for k, v in params.items()}
spec = scenes.box_on_plane(steps=steps)


def rollout(record):
    leaves = {k: v.detach().requires_grad_(True) for k, v in params.items()}
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    world = scenes.build_world(spec, device='cuda', params=leaves, record_substeps=record)
    loss = 0.
    for _ in range(steps):
        world.step(fixed_dt=True)
        loss = loss + (world.bodies[-1].pos ** 2).sum()
    loss.backward()
    torch.cuda.synchronize()
    return time.perf_counter() - t0, float(loss.detach()), {k: v.grad for k, v in leaves.items()}, len(world.trajectory)


power = subprocess.run(['nvidia-smi', '--query-gpu=power.limit', '--format=csv,noheader', '-i',
                        str(torch.cuda.current_device())], capture_output=True, text=True).stdout.strip()
print('device: %s (%s)' % (torch.cuda.get_device_name(), power or 'power limit not reported'))
for record in (False, True):                                     # warm-up: module loads, tape-slot pool
    rollout(record)
times = {False: [], True: []}
for _ in range(runs):
    for record in (False, True):
        dt, loss, grads, n = rollout(record)
        times[record].append(dt)
        print('record_substeps=%-5s %.1f ms  loss %.17g  entries %d' % (record, dt * 1e3, loss, n), flush=True)
off, on = sorted(times[False]), sorted(times[True])
print('off: %.1f-%.1f ms (median %.1f)   on: %.1f-%.1f ms (median %.1f)   median overhead %+.1f%%'
      % (off[0] * 1e3, off[-1] * 1e3, off[len(off) // 2] * 1e3, on[0] * 1e3, on[-1] * 1e3, on[len(on) // 2] * 1e3,
         100 * (on[len(on) // 2] / off[len(off) // 2] - 1)))
