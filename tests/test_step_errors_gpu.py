"""Errors ``World3D.step`` raises: the device-resident loop (stepper.py) and the host-driven loop of world.py give up on
the same step with the same message."""
import pytest
import torch

from diffsdfsim_b200 import scenes
from diffsdfsim_b200.world import World3D

pytestmark = pytest.mark.gpu
F64 = torch.float64


def _run(spec, make_params, steps, device_loop, setup=None, fixed_dt=True, **kw):
    """Step a new world until ``step`` raises.  Returns (world, capacity after construction, index of the step that
    raised or None, its message or None)."""
    World3D.device_loop = device_loop
    try:
        world = scenes.build_world(spec, device='cuda', params=make_params(), **kw)
        built = (world.detector.capK, world.maxc)
        if setup is not None:
            setup(world)
        for k in range(steps):
            try:
                world.step(fixed_dt=fixed_dt)
            except RuntimeError as e:
                return world, built, k, str(e)
        return world, built, None, None
    finally:
        World3D.device_loop = True


def test_strict_mode_gives_up_with_the_same_error_in_both_loops():
    """Bouncing spheres in strict mode (the scene of test_variable_dt_and_strict_mode_identical_to_host_loop): touching
    down takes halvings, so with one attempt per step allowed both loops raise on the same step."""
    W, steps = 16, 10
    gen = torch.Generator().manual_seed(5)
    pos = torch.zeros(W, 3, dtype=F64)
    pos[:, 1] = 0.6 + 0.4 * torch.rand(W, generator=gen, dtype=F64)
    spec = scenes.bouncing_sphere(floor=(4.0, 1.0, 4.0), steps=steps, floor_tri=0.2, subdivisions=3)
    mk = lambda: dict(pos=pos.cuda())

    def one_attempt(world):
        world.max_rounds_per_step = 1

    world, _, k, msg = _run(spec, mk, steps, True, fixed_dt=False)
    assert k is None and world.strict_no_pen and max(world.stats['rounds']) > 1, 'the scene must halve dt'
    dev = _run(spec, mk, steps, True, one_attempt, fixed_dt=False)[2:]
    host = _run(spec, mk, steps, False, one_attempt, fixed_dt=False)[2:]
    assert dev[0] is not None and dev[1].startswith('step did not complete in 1 attempts: worlds ['), dev
    assert dev == host


def test_capacity_limit_raises_the_same_error_from_step_in_both_loops():
    """The box-on-plane scene of test_capacity_growth_inside_the_device_loop grows its contact capacity while it steps.
    With the limits pinned to the capacity the constructor settled on, both loops raise the same capacity error on the
    same step."""
    W, steps = 8, 6
    mass = torch.linspace(0.9, 1.2, W, dtype=F64)
    spec = scenes.box_on_plane(floor=(4.0, 1.0, 4.0), steps=steps)
    mk = lambda: dict(mass=mass.cuda())

    def pin(world):
        world.MAX_CAPK, world.MAX_MAXC = world.detector.capK, world.maxc

    for device_loop in (True, False):
        world, built, k, _ = _run(spec, mk, steps, device_loop, capK=32, maxc=2)
        assert k is None and (world.detector.capK, world.maxc) != built, 'the capacity must grow inside step()'
    dev = _run(spec, mk, steps, True, pin, capK=32, maxc=2)[2:]
    host = _run(spec, mk, steps, False, pin, capK=32, maxc=2)[2:]
    assert dev[0] is not None, 'step() must raise at the pinned limits'
    assert ('contact candidate capacity exceeded' in dev[1] or 'contacts in one world' in dev[1]), dev
    assert dev == host
