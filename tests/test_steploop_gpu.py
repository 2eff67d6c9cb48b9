"""Device-resident step loop (stepper.py / csrc/dsdf_steploop.cu) vs the host-driven round loop of world.py.

Both run the same kernels on the same attempts, so poses, velocities, contact sets, simulated time and attempt counts
must be IDENTICAL bit for bit; gradients come from a hand-written reverse sweep over the tape instead of the per-round
autograd graph, so they agree to summation-order round-off (rtol 1e-9).  The oracle / reference-golden parity of the
device loop itself is asserted by tests/test_world_gpu.py (it is the default path).
"""
import numpy as np
import pytest
import torch

from diffsdfsim_b200 import scenes
from diffsdfsim_b200.world import World3D

pytestmark = pytest.mark.gpu
F64 = torch.float64


def _rollout(spec, make_params, steps, device_loop, loss_fn, fixed_dt=True, **kw):
    World3D.device_loop = device_loop
    try:
        params = make_params()
        world = scenes.build_world(spec, device='cuda', params=params, **kw)
        loss = 0.
        for _ in range(steps):
            world.step(fixed_dt=fixed_dt)
            loss = loss + loss_fn(world)
        loss.backward()
        return dict(p=world.get_p().detach().clone(), v=world.v.detach().clone(), t=world.t.clone(),
                    count=world.contact_set.count.clone(), body=world.contact_set.body.clone(),
                    geo=world.contact_set.geo.clone(), attempts=world.stats['attempts'].clone(), loss=float(loss),
                    grads={k: t.grad.clone() for k, t in params.items() if t.requires_grad},
                    rounds=sum(world.stats['rounds']), syncs=sum(world.stats.get('syncs', [0])), world=world)
    finally:
        World3D.device_loop = True


def _same(a, b, grad_rtol=1e-9):
    for k in ('p', 'v', 't', 'count', 'attempts'):
        assert torch.equal(a[k], b[k]), k
    n = int(a['count'].max())
    for w in range(a['count'].shape[0]):
        c = int(a['count'][w])
        assert torch.equal(a['body'][w, :c], b['body'][w, :c]) and torch.equal(a['geo'][w, :c], b['geo'][w, :c]), w
    assert a['loss'] == b['loss']
    for k in a['grads']:
        x, y = a['grads'][k].cpu().numpy(), b['grads'][k].cpu().numpy()
        np.testing.assert_allclose(x, y, rtol=grad_rtol, atol=grad_rtol * max(1e-12, np.abs(y).max()), err_msg=k)
    return n


def test_box_on_plane_batch_identical_to_host_loop():
    W, steps = 256, 12
    gen = torch.Generator().manual_seed(0)
    mass = 0.9 + 0.2 * torch.rand(W, generator=gen, dtype=F64)
    fric = 0.01 + 0.24 * torch.rand(W, generator=gen, dtype=F64)
    push = 2.0 + 3.0 * torch.rand(W, 2, generator=gen, dtype=F64)
    spec = scenes.box_on_plane(steps=steps)
    mk = lambda: dict(mass=mass.cuda().requires_grad_(True), fric_coeff=fric.cuda().requires_grad_(True),
                      push=push.cuda().requires_grad_(True))
    lf = lambda w: (w.bodies[-1].pos ** 2).sum() + 0.1 * (w.bodies[-1].v ** 2).sum()
    dev, host = _rollout(spec, mk, steps, True, lf), _rollout(spec, mk, steps, False, lf)
    assert _same(dev, host) >= 4
    # the device loop speculates, the host loop retries one halving at a time; a round in which worlds of the device loop
    # pause for buffer growth (tape slots, contact capacity) counts as a round too
    assert dev['rounds'] <= host['rounds'] + 6, 'device loop rounds %d, host loop rounds %d' % (dev['rounds'], host['rounds'])
    assert dev['syncs'] <= 2 * steps, 'host synchronisations: one per step + one per buffer growth (%d for %d steps)' % (dev['syncs'], steps)


def test_time_of_contact_batch_identical_to_host_loop():
    """Bouncing spheres dropped from per-world heights: first touches (World.H) at different steps, tilted pushes."""
    W, steps = 64, 14
    gen = torch.Generator().manual_seed(3)
    pos = torch.zeros(W, 3, dtype=F64)
    pos[:, 1] = 0.62 + 0.5 * torch.rand(W, generator=gen, dtype=F64)
    vel = torch.tensor([0, 0, 0, 1.0, -0.5, 0.2], dtype=F64) + 0.3 * (torch.rand(W, 6, generator=gen, dtype=F64) - 0.5)
    mass = 0.8 + 0.4 * torch.rand(W, generator=gen, dtype=F64)
    spec = scenes.bouncing_sphere(floor=(6.0, 1.0, 6.0), steps=steps, floor_tri=0.2, subdivisions=3)
    mk = lambda: dict(pos=pos.cuda().requires_grad_(True), vel=vel.cuda().requires_grad_(True),
                      mass=mass.cuda().requires_grad_(True))
    lf = lambda w: (w.bodies[-1].pos ** 2).sum() + 0.1 * (w.bodies[-1].v ** 2).sum()
    dev, host = _rollout(spec, mk, steps, True, lf), _rollout(spec, mk, steps, False, lf)
    _same(dev, host)
    assert dev['world']._any_toc_flag and host['world']._any_toc_flag, 'the scene must exercise the time-of-contact path'


def test_variable_dt_and_strict_mode_identical_to_host_loop():
    W, steps = 16, 10
    gen = torch.Generator().manual_seed(5)
    pos = torch.zeros(W, 3, dtype=F64)
    pos[:, 1] = 0.6 + 0.4 * torch.rand(W, generator=gen, dtype=F64)
    spec = scenes.bouncing_sphere(floor=(4.0, 1.0, 4.0), steps=steps, floor_tri=0.2, subdivisions=3)
    mk = lambda: dict(pos=pos.cuda().requires_grad_(True))
    lf = lambda w: (w.bodies[-1].pos ** 2).sum()
    dev = _rollout(spec, mk, steps, True, lf, fixed_dt=False)
    host = _rollout(spec, mk, steps, False, lf, fixed_dt=False)
    _same(dev, host)


def test_capacity_growth_inside_the_device_loop():
    """Candidate list, contact list, dynamics shared memory and tape slots all start too small: the paused worlds are
    retried after the host enlarged the buffers, and the result is identical to a run that had room."""
    from diffsdfsim_b200.stepper import DeviceStepper
    W, steps = 8, 6
    mass = torch.linspace(0.9, 1.2, W, dtype=F64)
    spec = scenes.box_on_plane(floor=(4.0, 1.0, 4.0), steps=steps)
    mk = lambda: dict(mass=mass.cuda().requires_grad_(True))
    lf = lambda w: (w.bodies[-1].pos ** 2).sum()
    ref = _rollout(spec, mk, steps, True, lf)
    old = DeviceStepper.INITIAL_SLOTS
    DeviceStepper.INITIAL_SLOTS = 1
    try:
        small = _rollout(spec, mk, steps, True, lf, capK=32, maxc=2)
    finally:
        DeviceStepper.INITIAL_SLOTS = old
    _same(ref, small, grad_rtol=1e-10)
    assert small['world'].maxc > 2 and small['world'].detector.capK > 32


def test_undo_step_after_contact_count_change():
    """ADVICE r1: undo a step in which the contact set changed (and the capacity grew): the restored world steps on
    exactly like a fresh copy."""
    spec = scenes.box_on_plane(floor=(4.0, 1.0, 4.0), steps=6)
    a = scenes.build_world(spec, device='cuda', maxc=4)
    b = scenes.build_world(spec, device='cuda', maxc=4)
    for _ in range(2):
        a.step(fixed_dt=True)
        b.step(fixed_dt=True)
    a.step(fixed_dt=True)
    a.undo_step()
    assert torch.equal(a.get_p(), b.get_p()) and torch.equal(a.t, b.t)
    for _ in range(3):
        a.step(fixed_dt=True)
        b.step(fixed_dt=True)
        assert torch.equal(a.get_p(), b.get_p()) and torch.equal(a.v, b.v)
        assert torch.equal(a.contact_set.count, b.contact_set.count)


def test_many_contacts_identical_to_host_loop():
    """16 bodies resting on a floor with more than 64 contacts per world: the library picks the one-CTA dynamics kernel
    for both loops, so they run the same kernels on the same attempts."""
    W, steps = 3, 4
    spec = scenes.mixed16_floor(seed=0, steps=steps)
    gen = torch.Generator().manual_seed(7)
    vel = torch.tensor([b['vel'] for b in spec['bodies']], dtype=F64).repeat(W, 1, 1)
    drift = 0.1 * (torch.rand(W, vel.shape[1] - 1, 3, generator=gen, dtype=F64) - 0.5)
    vel[:, 1:, 3:] += drift * torch.tensor([1.0, 0.0, 1.0], dtype=F64)           # per-world horizontal drift
    mk = lambda: dict(vel_all=vel.cuda().requires_grad_(True))
    lf = lambda w: (w.state.p[:, 1:, 4:] ** 2).sum()
    dev = _rollout(spec, mk, steps, True, lf, maxc=128)
    host = _rollout(spec, mk, steps, False, lf, maxc=128)
    assert _same(dev, host) > 64, 'the scene must exceed 64 contacts'
