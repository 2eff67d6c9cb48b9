"""Batched losses of the fitting experiments (diffsdfsim_b200/losses.py) against direct restatements of the reference
loops (experiments/trajectory_fitting/optim_sphere.py:114-160, optim_pointcloud.py:191-199)."""
import numpy as np
import pytest
import torch

pytestmark = pytest.mark.gpu
F64 = torch.float64


def _reference_trajectory_loss(traj, traj_target):
    """optim_sphere.py:114-160 transcribed for one world: lists of (t, p, v)."""
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


def test_trajectory_loss_matches_reference_loop_per_world():
    from diffsdfsim_b200 import scenes
    from diffsdfsim_b200.losses import trajectory_loss
    W = 3
    pos = torch.tensor([[0.0, 0.7, 0.0], [0.0, 0.9, 0.0], [0.0, 1.2, 0.0]], dtype=F64)
    spec = scenes.bouncing_sphere(floor=(4.0, 1.0, 4.0), steps=10, floor_tri=0.2, subdivisions=3)
    target = scenes.build_world(spec, device='cuda', params=dict(pos=(pos + 0.05).cuda()))
    for k in range(12):
        target.step(fixed_dt=(k % 2 == 0))             # mixed stepping: target times are not aligned with the model's
    leaf = pos.cuda().requires_grad_(True)
    world = scenes.build_world(spec, device='cuda', params=dict(pos=leaf))
    for _ in range(10):
        world.step(fixed_dt=True)
    loss = trajectory_loss(world, target)
    assert loss.shape == (W,)
    loss.sum().backward()
    assert torch.isfinite(leaf.grad).all() and float(leaf.grad.abs().sum()) > 0
    for w in range(W):
        tr = [(float(s[0][w]), s[1][w].detach().cpu(), None) for s in world.trajectory]
        tt = [(float(s[0][w]), s[1][w].detach().cpu(), None) for s in target.trajectory]
        ref = _reference_trajectory_loss(tr, tt)
        np.testing.assert_allclose(float(loss[w]), float(ref), rtol=1e-12)


def test_pointcloud_sdf_loss_matches_oracle_query():
    from diffsdfsim_b200 import bodies
    from diffsdfsim_b200.losses import pointcloud_sdf_loss
    from oracle import sdf as S, transforms as T
    gen = torch.Generator().manual_seed(0)
    q = torch.nn.functional.normalize(torch.randn(4, generator=gen, dtype=F64), dim=0)
    p7 = torch.cat([q, torch.tensor([0.3, 0.8, -0.2], dtype=F64)])
    sph = bodies.SDFSphere(p7, 0.5, device='cuda')
    pts = torch.randn(500, 3, generator=gen, dtype=F64) * 0.5 + p7[4:]
    pose = p7.clone().cuda().requires_grad_(True)
    sph.p = pose
    loss, n = pointcloud_sdf_loss(sph, pts.cuda())
    loss.backward()
    # oracle: the same transform + query in torch on the CPU
    pose_c = p7.clone().requires_grad_(True)
    R = T.quaternion_to_matrix(pose_c[:4])
    loc = (R.T.unsqueeze(0) @ (pts - pose_c[4:]).unsqueeze(-1)).squeeze(-1)
    scale = torch.tensor(0.75, dtype=F64)
    sd = S.query(S.SPHERE, [torch.tensor(0.5, dtype=F64) / scale], scale, loc, want_dir=False)
    mask = (loc.abs() <= scale).all(1)
    ref = (torch.where(mask, sd, torch.zeros_like(sd)) ** 2).sum()
    ref.backward()
    assert int(n) == int(mask.sum())
    np.testing.assert_allclose(float(loss), float(ref), rtol=1e-12)
    np.testing.assert_allclose(pose.grad.cpu().numpy(), pose_c.grad.numpy(), rtol=1e-8, atol=1e-10)


@pytest.mark.parametrize('flag', [False, True])
def test_run_world_fixed_dt_matches_the_reference_function(flag):
    """losses.run_world_fixed_dt vs the reference's OWN run_world_fixed_dt (experiments/trajectory_fitting/optim_sphere.py:
    163-177, executed unmodified on the reference World3D by tests/golden/make_golden.py): number of step() calls,
    final state, and the gradients of a loss collected after every step -- with detach_2nd_bounce the second contact
    step of a bounce is undone and the history cut there."""
    import os
    from diffsdfsim_b200 import scenes
    from diffsdfsim_b200.losses import run_world_fixed_dt
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'detach_2nd_bounce.npz'))
    k = 'detach' if flag else 'plain'
    spec = scenes.bouncing_sphere(floor=(4.0, 1.0, 4.0), steps=0, floor_tri=0.2, height=0.75, subdivisions=3,
                                  vel=(0, 0, 0, 1.0, 0, 0.3))
    pos = torch.tensor([[0.0, 0.75, 0.0]], dtype=F64, device='cuda', requires_grad=True)
    vel = torch.tensor([[0.0, 0.0, 0.0, 1.0, 0.0, 0.3]], dtype=F64, device='cuda', requires_grad=True)
    world = scenes.build_world(spec, device='cuda', params=dict(pos=pos, vel=vel))
    terms, step = [], world.step

    def recording_step(fixed_dt=False):
        had = step(fixed_dt=fixed_dt)
        terms.append((world.bodies[-1].pos ** 2).sum() + 0.1 * (world.bodies[-1].v ** 2).sum())
        return had
    world.step = recording_step
    run_world_fixed_dt(world, 0.8, detach_2nd_bounce=flag)
    assert len(terms) == int(g[k + '_nsteps'])
    loss = sum(terms)
    loss.backward()
    np.testing.assert_allclose(world.get_p().detach().cpu().numpy().reshape(-1), g[k + '_p'], atol=1e-6, rtol=0)   # (after two bounces: ~1e-7 per 10-iteration solve)
    np.testing.assert_allclose(world.v.detach().cpu().numpy().reshape(-1), g[k + '_v'], atol=1e-5, rtol=0)
    np.testing.assert_allclose(float(loss), float(g[k + '_loss']), rtol=1e-6)
    for name, leaf in (('gpos', pos), ('gvel', vel)):
        ref = g[k + '_' + name]
        np.testing.assert_allclose(leaf.grad.cpu().numpy().reshape(-1), ref, rtol=1e-4, atol=1e-5 * max(1e-9, np.abs(ref).max()))


def test_batched_detach_2nd_bounce_matches_each_world_alone():
    """run_world_fixed_dt(detach_2nd_bounce=True) on a batch of spheres dropped from different heights: the masked
    undo_step / detach_state fire at different steps in different worlds, and every world ends bit for bit where it
    ends alone.  A batch steps in lock-step on the host clock, so 'alone' is that world stepped as many times, with the
    same rule applied through the unmasked undo_step() / detach_state() (the single-world path the reference golden
    above pins)."""
    from diffsdfsim_b200 import scenes
    from diffsdfsim_b200.losses import run_world_fixed_dt
    heights = [0.62, 0.75, 0.9, 1.05]
    W = len(heights)
    spec = scenes.bouncing_sphere(floor=(4.0, 1.0, 4.0), steps=0, floor_tri=0.2, subdivisions=3)
    pos0 = torch.tensor([[0.0, h, 0.0] for h in heights], dtype=F64)
    vel0 = torch.tensor([[0.0, 0.0, 0.0, 1.0, 0.0, 0.3]] * W, dtype=F64)
    term = lambda world: (world.bodies[-1].pos ** 2).sum(-1) + 0.1 * (world.bodies[-1].v ** 2).sum(-1)

    pos, vel = pos0.cuda().requires_grad_(True), vel0.cuda().requires_grad_(True)
    batch = scenes.build_world(spec, device='cuda', params=dict(pos=pos, vel=vel))
    terms, step = [], batch.step

    def recording_step(fixed_dt=False):
        had = step(fixed_dt=fixed_dt)
        terms.append(term(batch))
        return had
    batch.step = recording_step
    n_steps = run_world_fixed_dt(batch, 0.9, detach_2nd_bounce=True)
    sum(terms).sum().backward()

    fired = []
    for w in range(W):
        pw, vw = pos0[w:w + 1].cuda().requires_grad_(True), vel0[w:w + 1].cuda().requires_grad_(True)
        world = scenes.build_world(spec, device='cuda', params=dict(pos=pw, vel=vw))
        loss, contact_steps, fired_w = 0., 0, []
        for k in range(n_steps):
            had = world.step(fixed_dt=True)
            loss = loss + term(world).sum()
            contact_steps += int(had)
            if had and contact_steps > 1:
                world.undo_step()
                world.detach_state()
                contact_steps = 0
                fired_w.append(k)
        loss.backward()
        fired.append(fired_w)
        assert torch.equal(batch.get_p()[w], world.get_p()), w
        assert torch.equal(batch.v[w], world.v), w
        assert torch.equal(batch.t[w:w + 1], world.t), w
        assert torch.equal(batch.contact_set.count[w:w + 1], world.contact_set.count), w
        for leaf, lw in ((pos, pw), (vel, vw)):
            np.testing.assert_allclose(leaf.grad[w].cpu().numpy(), lw.grad[0].cpu().numpy(), rtol=1e-12,
                                       atol=1e-14, err_msg='world %d' % w)
    assert sum(1 for f in fired if f) >= 2 and len({tuple(f) for f in fired}) > 1, \
        'the undo must fire in several worlds, at different steps: %s' % fired
