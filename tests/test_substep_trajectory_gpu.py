"""World3D(record_substeps=True): one trajectory entry per accepted sub-step, as the reference records them
(lcp_physics/physics/world.py:372-379, restated by oracle/sim.py step_dt), on both step loops, with gradients through
the entries (time of contact included), per-world ``valid`` masks in a batch, the reference's undo rule and the C1
fitting loss (experiments/trajectory_fitting/optim_sphere.py:114-160)."""
import numpy as np
import pytest
import torch

from diffsdfsim_b200 import scenes
from diffsdfsim_b200.losses import run_world_fixed_dt, trajectory_loss
from diffsdfsim_b200.world import World3D
from oracle.scenes import build as build_oracle

pytestmark = pytest.mark.gpu
F64 = torch.float64
VEL = (0.0, 0.0, 0.0, 1.0, 0.0, 0.3)


def _sphere_spec(steps):
    return scenes.bouncing_sphere(floor=(4.0, 1.0, 4.0), steps=steps, floor_tri=0.2, height=0.75, subdivisions=3,
                                  vel=VEL)


class _host_loop:
    """World3D.device_loop = False inside the block."""

    def __init__(self, on=True):
        self.on = on

    def __enter__(self):
        World3D.device_loop = not self.on

    def __exit__(self, *exc):
        World3D.device_loop = True


def _reference_trajectory_loss(traj, traj_target):
    """optim_sphere.py:114-160 transcribed for one world: lists of (t, p, ...)."""
    loss, last_j = 0., 0
    for s in traj:
        min_diff, last_diff, min_s, new_j = 1e100, 1e100, None, 0
        for j, st in enumerate(traj_target[last_j:]):
            diff = abs(s[0] - st[0])
            if diff <= min_diff:
                min_diff, min_s, new_j = diff, st, last_j + j
            if diff > last_diff:
                break
            last_diff = diff
        loss = loss + ((s[1][-3:] - min_s[1][-3:]) ** 2).sum()
        last_j = new_j
    return loss / len(traj)


def _entries_of(world, w):
    """World w's valid entries as (t, p, v) on the host; a single world's entries are all valid."""
    out = []
    for e in world.trajectory:
        if not world.batched:
            out.append((e[0], e[1].detach().cpu(), e[2].detach().cpu()))
        elif bool(e.valid[w]):
            out.append((float(e[0][w]), e[1][w].detach().cpu(), e[2][w].detach().cpu()))
    return out


def _assert_same_entries(a, b, msg=''):
    assert len(a) == len(b), msg
    for k, (x, y) in enumerate(zip(a, b)):
        assert x[0] == y[0] and torch.equal(x[1], y[1]) and torch.equal(x[2], y[2]), '%s entry %d' % (msg, k)


def _assert_matches_oracle(entries, ow, vtol=1e-6):
    assert len(entries) == len(ow.trajectory)
    for k, (e, o) in enumerate(zip(entries, ow.trajectory)):
        assert abs(e[0] - float(o[0])) < 1e-12, k
        np.testing.assert_allclose(e[1].numpy(), o[1].detach().numpy(), atol=1e-8, rtol=0, err_msg='entry %d' % k)
        np.testing.assert_allclose(e[2].numpy(), o[2].detach().numpy(), atol=vtol, rtol=0, err_msg='entry %d' % k)


@pytest.mark.parametrize('host', [False, True])
def test_single_sphere_substep_entries_match_oracle(host):
    """Two bounces with time of contact: as many entries as the oracle, at the same start times, with the same states."""
    steps = 24
    spec = _sphere_spec(steps)
    with _host_loop(host):
        world = scenes.build_world(spec, device='cuda', record_substeps=True)
        per_step = []
        for _ in range(steps):
            n0 = len(world.trajectory)
            world.step(fixed_dt=True)
            per_step.append(len(world.trajectory) - n0)
    assert max(per_step) >= 2, 'the rollout must sub-step: %s' % per_step
    assert world._any_toc_flag
    ow = build_oracle(spec, {})
    for _ in range(steps):
        ow.step()
    assert all(len(e) == 5 and e[3] is None and e[4] is None for e in world.trajectory)
    _assert_matches_oracle(_entries_of(world, 0), ow)


def _fit_rollout(steps, rad, pos, vel):
    spec = _sphere_spec(steps)
    world = scenes.build_world(spec, device='cuda', params=dict(rad=rad, pos=pos, vel=vel), record_substeps=True)
    for _ in range(steps):
        world.step(fixed_dt=True)
    return world


def test_c1_trajectory_loss_and_gradients_match_reference_loop_and_oracle():
    """trajectory_loss between two sub-step trajectories (target: other radius and velocity) == the reference loop, and
    its gradients w.r.t. radius, initial position and velocity == oracle autograd on the same loss; likewise a loss on
    the one contact sub-step entry, which reaches the leaves through the time-of-contact backward."""
    steps = 20
    rad0, pos0, vel0 = 0.5, torch.tensor([0.0, 0.75, 0.0], dtype=F64), torch.tensor(VEL, dtype=F64)
    target = _fit_rollout(steps, torch.tensor(0.45, dtype=F64, device='cuda'), pos0.cuda(),
                          (vel0 + torch.tensor([0, 0, 0, 0.2, 0.1, -0.1], dtype=F64)).cuda())
    leaves = dict(rad=torch.tensor(rad0, dtype=F64, device='cuda', requires_grad=True),
                  pos=pos0.cuda().requires_grad_(True), vel=vel0.cuda().requires_grad_(True))
    world = _fit_rollout(steps, leaves['rad'], leaves['pos'], leaves['vel'])
    loss = trajectory_loss(world, target)
    grads = torch.autograd.grad(loss, list(leaves.values()), retain_graph=True)
    ref = _reference_trajectory_loss([(e[0], e[1].detach().cpu()) for e in world.trajectory],
                                     [(e[0], e[1].detach().cpu()) for e in target.trajectory])
    np.testing.assert_allclose(float(loss.detach()), float(ref), rtol=1e-12)

    spec = _sphere_spec(steps)
    ot = build_oracle(spec, dict(rad=torch.tensor(0.45, dtype=F64), pos=pos0.clone(),
                                 vel=vel0 + torch.tensor([0, 0, 0, 0.2, 0.1, -0.1], dtype=F64)))
    oleaves = dict(rad=torch.tensor(rad0, dtype=F64, requires_grad=True), pos=pos0.clone().requires_grad_(True),
                   vel=vel0.clone().requires_grad_(True))
    ow = build_oracle(spec, dict(oleaves))
    for _ in range(steps):
        ot.step()
        ow.step()
    assert len(ow.trajectory) == len(world.trajectory) > steps
    oloss = _reference_trajectory_loss(ow.trajectory, [(o[0], o[1].detach()) for o in ot.trajectory])
    ogr = torch.autograd.grad(oloss, list(oleaves.values()), retain_graph=True)
    np.testing.assert_allclose(float(loss.detach()), float(oloss.detach()), rtol=1e-6)
    for name, g, og in zip(leaves, grads, ogr):
        og = og.numpy()
        np.testing.assert_allclose(g.cpu().numpy(), og, rtol=1e-4, atol=1e-6 * max(1e-9, np.abs(og).max()), err_msg=name)

    # the first entry after which the oracle has contacts: the time-of-contact sub-step of the first bounce
    j = next(k for k, o in enumerate(ow.trajectory) if o[3])
    assert abs(world.trajectory[j][0] - float(ow.trajectory[j][0])) < 1e-12
    e, o = world.trajectory[j], ow.trajectory[j]
    lj = (e[1][-3:] ** 2).sum() + 0.1 * (e[2] ** 2).sum()
    olj = (o[1][-3:] ** 2).sum() + 0.1 * (o[2] ** 2).sum()
    gj = torch.autograd.grad(lj, list(leaves.values()))
    ogj = torch.autograd.grad(olj, list(oleaves.values()))
    for name, g, og in zip(leaves, gj, ogj):
        og = og.numpy()
        np.testing.assert_allclose(g.cpu().numpy(), og, rtol=1e-4, atol=1e-6 * max(1e-9, np.abs(og).max()),
                                   err_msg='contact entry ' + name)


def test_ragged_batch_entries_and_gradients_match_each_world_alone():
    """64 spheres dropped from heights over 2 m (speculative halving active, worlds sub-step at different steps): each
    world's valid entries are bit-identical to the same world stepped alone, and so are its loss and gradients."""
    W, steps = 64, 22
    heights = torch.linspace(0.62, 2.62, W, dtype=F64)
    pos0 = torch.stack([torch.zeros(W, dtype=F64), heights, torch.zeros(W, dtype=F64)], 1)
    vel0 = torch.tensor(VEL, dtype=F64).expand(W, 6).clone()
    velt = vel0 + torch.tensor([0, 0, 0, 0.2, 0.0, -0.1], dtype=F64)
    spec = _sphere_spec(steps)

    def roll(pos, vel):
        world = scenes.build_world(spec, device='cuda', params=dict(pos=pos, vel=vel), record_substeps=True)
        for _ in range(steps):
            world.step(fixed_dt=True)
        return world

    target = roll(pos0.cuda(), velt.cuda())
    pos, vel = pos0.cuda().requires_grad_(True), vel0.cuda().requires_grad_(True)
    batch = roll(pos, vel)
    assert batch._stepper.spec_threshold > 0
    counts = torch.stack([e.valid for e in batch.trajectory]).sum(0).cpu()
    loss = trajectory_loss(batch, target)
    gpos, gvel = torch.autograd.grad(loss.sum(), [pos, vel])
    # four worlds with different numbers of sub-steps
    pick, seen = [], set()
    for w in range(W):
        if int(counts[w]) not in seen:
            seen.add(int(counts[w]))
            pick.append(w)
    assert len(pick) >= 4, 'sub-step counts must differ between worlds: %s' % counts.tolist()
    for w in pick[:2] + pick[-2:]:
        pw, vw = pos0[w:w + 1].cuda().requires_grad_(True), vel0[w:w + 1].cuda().requires_grad_(True)
        alone = roll(pw, vw)
        _assert_same_entries(_entries_of(batch, w), _entries_of(alone, 0), 'world %d' % w)
        lw = trajectory_loss(alone, roll(pos0[w:w + 1].cuda(), velt[w:w + 1].cuda()))
        np.testing.assert_allclose(float(loss[w]), float(lw), rtol=1e-12)
        gp, gv = torch.autograd.grad(lw, [pw, vw])
        np.testing.assert_allclose(gpos[w].cpu().numpy(), gp[0].cpu().numpy(), rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(gvel[w].cpu().numpy(), gv[0].cpu().numpy(), rtol=1e-12, atol=1e-14)


def test_device_loop_entries_equal_host_loop_entries():
    """The device loop gathers the entries from its tape, the host loop selects them from its rounds: same entries and
    valid masks bit for bit, same gradients of trajectory_loss."""
    W, steps = 8, 16
    gen = torch.Generator().manual_seed(3)
    pos0 = torch.zeros(W, 3, dtype=F64)
    pos0[:, 1] = 0.62 + 0.5 * torch.rand(W, generator=gen, dtype=F64)
    vel0 = torch.tensor(VEL, dtype=F64) + 0.3 * (torch.rand(W, 6, generator=gen, dtype=F64) - 0.5)
    spec = _sphere_spec(steps)
    out = {}
    for host in (False, True):
        with _host_loop(host):
            target = scenes.build_world(spec, device='cuda', params=dict(pos=pos0.cuda(), vel=0.9 * vel0.cuda()),
                                        record_substeps=True)
            params = dict(pos=pos0.cuda().requires_grad_(True), vel=vel0.cuda().requires_grad_(True))
            world = scenes.build_world(spec, device='cuda', params=params, record_substeps=True)
            for _ in range(steps):
                target.step(fixed_dt=True)
                world.step(fixed_dt=True)
        loss = trajectory_loss(world, target)
        out[host] = (world.trajectory, loss.detach(), torch.autograd.grad(loss.sum(), list(params.values())))
    (ta, la, ga), (tb, lb, gb) = out[False], out[True]
    assert len(ta) == len(tb) > steps
    assert not all(bool(e.valid.all()) for e in ta), 'some worlds must sub-step more than others'
    for ea, eb in zip(ta, tb):
        assert torch.equal(ea.valid, eb.valid)
        for x, y in zip(ea[:3], eb[:3]):
            assert torch.equal(x, y)
    assert torch.equal(la, lb)
    for a, b in zip(ga, gb):
        np.testing.assert_allclose(a.cpu().numpy(), b.cpu().numpy(), rtol=1e-9, atol=1e-12 * float(b.abs().max()))


def test_post_stabilised_substep_entries_match_oracle():
    """post_stab=True (host loop): the entries hold the post-stabilised poses, as the reference records them."""
    steps = 5
    spec = dict(scenes.box_on_plane(floor=(4.0, 1.0, 4.0), steps=steps), post_stab=True)
    world = scenes.build_world(spec, device='cuda', record_substeps=True)
    assert not world._use_device_loop()
    ow = build_oracle(spec, {})
    for _ in range(steps):
        world.step(fixed_dt=True)
        ow.step()
    _assert_matches_oracle(_entries_of(world, 0), ow)


def test_undo_step_keeps_the_entries_the_oracle_keeps():
    """undo_step drops the entries stamped after the restored time (the undone step's first entry stays): a single world
    against the oracle doing the same, and a batch under run_world_fixed_dt(detach_2nd_bounce=True), whose masked
    undo fires at different steps in different worlds, against each world alone."""
    spec = _sphere_spec(0)
    world = scenes.build_world(spec, device='cuda', record_substeps=True)
    ow = build_oracle(spec, {})
    undone = 0
    for k in range(24):
        had, had_o = world.step(fixed_dt=True), ow.step()
        assert had == had_o
        if had and k % 2:
            n = len(world.trajectory)
            world.undo_step()
            ow.undo_step()
            undone += len(world.trajectory) < n - 1
    assert undone, 'an undone step must have sub-stepped'
    _assert_matches_oracle(_entries_of(world, 0), ow)

    heights = [0.62, 0.75, 0.9, 1.05]
    W = len(heights)
    pos0 = torch.tensor([[0.0, h, 0.0] for h in heights], dtype=F64)
    vel0 = torch.tensor([VEL] * W, dtype=F64)
    pos, vel = pos0.cuda().requires_grad_(True), vel0.cuda().requires_grad_(True)
    batch = scenes.build_world(spec, device='cuda', params=dict(pos=pos, vel=vel), record_substeps=True)
    n_steps = run_world_fixed_dt(batch, 0.9, detach_2nd_bounce=True)
    term = lambda world: sum((e[1].reshape(world.W, -1)[:, -3:] ** 2).sum(-1) * getattr(e, 'valid', 1)
                             for e in world.trajectory)
    gpos, gvel = torch.autograd.grad(term(batch).sum(), [pos, vel])
    for w in range(W):
        pw, vw = pos0[w:w + 1].cuda().requires_grad_(True), vel0[w:w + 1].cuda().requires_grad_(True)
        alone = scenes.build_world(spec, device='cuda', params=dict(pos=pw, vel=vw), record_substeps=True)
        contact_steps = 0
        for _ in range(n_steps):
            had = alone.step(fixed_dt=True)
            contact_steps += int(had)
            if had and contact_steps > 1:
                alone.undo_step()
                alone.detach_state()
                contact_steps = 0
        _assert_same_entries(_entries_of(batch, w), _entries_of(alone, 0), 'world %d' % w)
        gp, gv = torch.autograd.grad(term(alone).sum(), [pw, vw])
        np.testing.assert_allclose(gpos[w].cpu().numpy(), gp[0].cpu().numpy(), rtol=1e-12, atol=1e-14)
        np.testing.assert_allclose(gvel[w].cpu().numpy(), gv[0].cpu().numpy(), rtol=1e-12, atol=1e-14)
