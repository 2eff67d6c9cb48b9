"""Structure-exploiting fused dynamics kernel (one warp per world) vs the dense LCP path on identical worlds."""
import numpy as np
import pytest
import torch

from diffsdfsim_b200 import scenes

pytestmark = pytest.mark.gpu
F64 = torch.float64


def _rollout(engine, steps, W, seed=0):
    gen = torch.Generator().manual_seed(seed)
    mass = (0.9 + 0.2 * torch.rand(W, generator=gen, dtype=F64)).cuda().requires_grad_(True)
    fric = (0.05 + 0.2 * torch.rand(W, generator=gen, dtype=F64)).cuda().requires_grad_(True)
    push = (2.0 + 3.0 * torch.rand(W, 2, generator=gen, dtype=F64)).cuda().requires_grad_(True)
    spec = scenes.box_on_plane(floor=(4.0, 1.0, 4.0), steps=steps)
    world = scenes.build_world(spec, device='cuda', params=dict(mass=mass, fric_coeff=fric, push=push), engine=engine,
                               maxc=12)
    loss, traj = 0., []
    for _ in range(steps):
        world.step(fixed_dt=True)
        traj.append((world.get_p().detach().clone(), world.v.detach().clone(), world.contact_set.count.clone()))
        loss = loss + (world.bodies[-1].pos ** 2).sum()
    loss.backward()
    return traj, (mass.grad, fric.grad, push.grad), world


def test_fused_engine_matches_dense_engine():
    steps, W = 6, 8
    ta, ga, wa = _rollout('PdipmEngine', steps, W)
    tb, gb, wb = _rollout('DensePdipmEngine', steps, W)
    assert torch.equal(wa.stats['attempts'], wb.stats['attempts'])
    for (pa, va, ca), (pb, vb, cb) in zip(ta, tb):
        assert torch.equal(ca, cb)
        np.testing.assert_allclose(pa.cpu().numpy(), pb.cpu().numpy(), atol=1e-9, rtol=0)
        np.testing.assert_allclose(va.cpu().numpy(), vb.cpu().numpy(), atol=1e-7, rtol=0)
    for a, b in zip(ga, gb):
        ref = b.cpu().numpy()
        np.testing.assert_allclose(a.cpu().numpy(), ref, rtol=1e-4, atol=1e-5 * max(1e-9, np.abs(ref).max()))


def test_dense_engine_runs_the_dense_operator_in_every_round():
    """64 spheres dropped from heights spread over 2 m: at every step only a few worlds touch the floor and retry with
    a halved dt, so most retry rounds have a handful of active worlds.  Every round of the dense engine, forward and
    backward, still goes through the dense LCP kernels and never through the fused solver."""
    from diffsdfsim_b200 import _lib
    W, steps = 64, 14
    gen = torch.Generator().manual_seed(3)
    pos = torch.zeros(W, 3, dtype=F64)
    pos[:, 1] = 0.62 + 2.0 * torch.rand(W, generator=gen, dtype=F64)
    pos = pos.cuda().requires_grad_(True)
    spec = scenes.bouncing_sphere(floor=(6.0, 1.0, 6.0), steps=steps, floor_tri=0.2, subdivisions=3)
    world = scenes.build_world(spec, device='cuda', params=dict(pos=pos), engine='DensePdipmEngine', maxc=12)
    _lib.reset_counters()
    loss = 0.
    for _ in range(steps):
        world.step(fixed_dt=True)
        loss = loss + (world.bodies[-1].pos ** 2).sum()
    loss.backward()
    assert int(world.stats['attempts'].max()) > steps, 'the scene must reject and retry sub-steps'
    assert 'dsdf_dynamics_solve' not in _lib.LAUNCHES and 'dsdf_dynamics_solve_backward' not in _lib.LAUNCHES
    assert 'dsdf_lcp_forward' in _lib.LAUNCHES


def test_fused_plan_has_no_contact_limit_of_the_dense_kernel():
    """16+ contacts per world exceed the dense kernel's shared memory; the fused kernel takes them (one launch of the
    one-warp kernel, no workspace)."""
    from diffsdfsim_b200 import _lib
    L = _lib.lib()
    assert L.dsdf_lcp_smem_bytes(12, 6, 170) > 227 * 1024
    assert _lib.dynamics_plan(1, 2, 6, 8, 32, 32) == (1, 0)


def test_forced_one_cta_kernel_matches_one_warp_kernel():
    """The one-CTA instantiation of the solver (per-contact data in a global workspace, block-wide reductions and LU)
    solves the same Newton systems as the one-warp kernel: identical attempts / contact sets, states and gradients to
    round-off."""
    from diffsdfsim_b200.stepper import DeviceStepper
    steps, W = 8, 16
    ta, ga, wa = _rollout('PdipmEngine', steps, W)
    DeviceStepper.FORCE_CTA = True
    try:
        tb, gb, wb = _rollout('PdipmEngine', steps, W)
        assert wb._stepper.force_cta and wb._stepper.dyn_ws is not None
    finally:
        DeviceStepper.FORCE_CTA = False
    assert torch.equal(wa.stats['attempts'], wb.stats['attempts'])
    for (pa, va, ca), (pb, vb, cb) in zip(ta, tb):
        assert torch.equal(ca, cb)
        np.testing.assert_allclose(pa.cpu().numpy(), pb.cpu().numpy(), atol=1e-11, rtol=0)
        np.testing.assert_allclose(va.cpu().numpy(), vb.cpu().numpy(), atol=1e-9, rtol=0)
    for a, b in zip(ga, gb):
        ref = b.cpu().numpy()
        np.testing.assert_allclose(a.cpu().numpy(), ref, rtol=1e-7, atol=1e-9 * max(1e-9, np.abs(ref).max()))


def test_more_than_64_contacts_per_world_on_the_one_cta_kernel():
    """Config 3, gravity + floor variant (16 primitives resting on a pinned floor): ~80-100 simultaneous contacts per
    world, beyond the one-warp kernel's 64 -- runs on the one-CTA kernel, forward and backward, finite and consistent
    between a batch and a single world."""
    from diffsdfsim_b200 import _lib
    spec = scenes.mixed16_floor(seed=0, steps=5)
    outs = []
    for W in (1, 3):
        vel = torch.tensor([b['vel'] for b in spec['bodies']], dtype=F64).repeat(W, 1, 1).cuda().requires_grad_(True)
        world = scenes.build_world(spec, device='cuda', params=dict(vel_all=vel), maxc=128)
        loss = 0.
        for _ in range(5):
            world.step(fixed_dt=True)
            loss = loss + (world.state.p[:, 1:, 4:] ** 2).sum()
        loss.backward()
        # 16 bodies: every world runs on the one-CTA kernel, which needs a workspace even for one contact
        assert world._stepper.dyn_ws is not None
        assert _lib.dynamics_plan(W, world.nb, world.num_constraints, world.fric_dirs, 1, 1)[1] > 0
        assert int(world.contact_set.count.max()) > 64, 'the scene must exceed 64 contacts'
        assert torch.isfinite(vel.grad).all() and float(vel.grad.abs().sum()) > 0
        outs.append((world.state.p.detach()[0].clone(), vel.grad[0].clone(), world.contact_set.count[0].clone()))
    assert torch.equal(outs[0][0], outs[1][0]) and torch.equal(outs[0][2], outs[1][2])
    np.testing.assert_allclose(outs[0][1].cpu().numpy(), outs[1][1].cpu().numpy(), rtol=1e-9, atol=1e-12)
