"""Batched losses of the reference's fitting experiments, on top of the stepping path (SURVEY.md s8f rank 2).

* ``trajectory_loss``       experiments/trajectory_fitting/optim_sphere.py:114-160 -- nearest-time matching of two
                            recorded trajectories, squared position error of the LAST body, averaged over the states
* ``pointcloud_sdf_loss``   the SDF part of experiments/trajectory_fitting/optim_pointcloud.py:166-201 -- observed points
                            moved into the estimated body frame, sum of squared SDF values inside the body's cube

Both are plain torch on top of ``World3D.trajectory`` / ``SDF3D.query_sdfs`` (the CUDA SDF-query operator); every world
of a batch is matched on its own.
"""
import torch


def _stack_times(traj, W, device):
    ts = []
    for s in traj:
        t = s[0]
        t = t if isinstance(t, torch.Tensor) else torch.full((W,), float(t), dtype=torch.float64, device=device)
        ts.append(t.reshape(-1).expand(W))
    return torch.stack(ts, 0)                                   # (S, W)


def _stack_valid(traj):
    """(S, W) bool of the rows that hold a recorded state (sub-step entries of a batch carry ``valid``), or None when no
    entry carries it."""
    if not any(hasattr(s, 'valid') for s in traj):
        return None
    return torch.stack([s.valid.reshape(-1) for s in traj], 0)


def nearest_time_index(t, t_target, valid_target=None):
    """For every recorded state (S,W) the index (S,W) of the target state (S',W) closest in time; on a tie the LATER
    target state wins (the reference's ``diff <= min_diff`` scan in ascending time order).  Target rows outside
    ``valid_target`` (S',W) are never matched."""
    diff = (t[:, None, :] - t_target[None, :, :]).abs()         # (S, S', W)
    if valid_target is not None:
        diff = torch.where(valid_target[None], diff, torch.full_like(diff, float('inf')))
    Sp = t_target.shape[0]
    rev = torch.flip(diff, dims=[1])
    return Sp - 1 - rev.argmin(dim=1)                           # argmin returns the first minimum of the reversed scan


def trajectory_loss(world, world_target):
    """Mean over the recorded states of |pos_last_body - pos_last_body_target(nearest time)|^2, per world.

    Returns a 0-d tensor for single worlds, (W,) for a batch; differentiable w.r.t. ``world``'s trajectory (the target
    is used as recorded, like the reference).  Sub-step entries of a batch (``World3D(record_substeps=True)``) carry a
    ``valid`` mask: each world averages over its own valid entries and is matched only to its valid target entries."""
    W, dev = world.W, world.device
    t = _stack_times(world.trajectory, W, dev)
    tt = _stack_times(world_target.trajectory, W, dev)
    pos = torch.stack([s[1].reshape(W, -1)[:, -3:] for s in world.trajectory], 0)               # (S, W, 3)
    pos_t = torch.stack([s[1].reshape(W, -1)[:, -3:] for s in world_target.trajectory], 0)      # (S', W, 3)
    valid, valid_t = _stack_valid(world.trajectory), _stack_valid(world_target.trajectory)
    idx = nearest_time_index(t, tt, valid_t)                                                   # (S, W)
    matched = torch.gather(pos_t, 0, idx[:, :, None].expand(-1, -1, 3))
    err = ((pos - matched) ** 2).sum(-1)
    if valid is None:
        loss = err.sum(0) / len(world.trajectory)
    else:
        loss = torch.where(valid, err, torch.zeros_like(err)).sum(0) / valid.sum(0)
    return loss if world.batched else loss[0]


def run_world_fixed_dt(world, run_time, detach_2nd_bounce=False):
    """experiments/trajectory_fitting/optim_sphere.py:163-177: step with fixed dt until ``run_time``; with
    ``detach_2nd_bounce`` the second step of every bounce (the second consecutive step that had contacts) is undone and
    the state detached, so that only the first contact step of each bounce is differentiated.  Every world of a batch
    keeps its own contact-step counter; the undo / detach is applied to the worlds whose counter fires."""
    W, dev = world.W, world.device
    num_contact_steps = torch.zeros(W, dtype=torch.int64, device=dev)
    n_steps = 0
    # a single world follows the reference's `while world.t < run_time` on the simulated time itself (the sum of its
    # accepted sub-steps); a batch steps in lock-step on the host clock
    now = (lambda: float(world.t[0])) if W == 1 else (lambda: world.t_host)
    while now() < run_time:
        had = world.step(fixed_dt=True)
        had = had if isinstance(had, torch.Tensor) else torch.tensor([had], device=dev)
        n_steps += 1
        if not detach_2nd_bounce:
            continue
        num_contact_steps = num_contact_steps + had.to(torch.int64)
        fire = had & (num_contact_steps > 1)
        if bool(fire.any()):                                 # (one host read per step, like the reference's own `if`)
            if W == 1:
                world.undo_step()
                world.detach_state()
            else:
                world.undo_step(fire)
                world.detach_state(fire)
            num_contact_steps = torch.where(fire, torch.zeros_like(num_contact_steps), num_contact_steps)
    return n_steps


def pointcloud_sdf_loss(body, points_world, pos=None, rot=None, exact=False):
    """(sum of squared SDF values of the observed points inside the body's cube, number of such points).

    points_world (N,3) or (W,N,3); pos (.,3) / rot (.,3,3) default to the body's current pose.  Points outside the cube
    |p| <= scale contribute nothing (optim_pointcloud.py:195-196)."""
    from .transforms import quaternion_to_matrix
    p = body.p if body.p.dim() == 2 else body.p.unsqueeze(0)
    pos = p[:, 4:] if pos is None else pos.reshape(-1, 3)
    rot = quaternion_to_matrix(p[:, :4]) if rot is None else rot.reshape(-1, 3, 3)
    pts = points_world if points_world.dim() == 3 else points_world.unsqueeze(0)
    B = max(pts.shape[0], pos.shape[0])
    pts = pts.expand(B, -1, 3)
    loc = torch.einsum('bji,bnj->bni', rot.expand(B, 3, 3), pts - pos.expand(B, 3)[:, None, :])   # R^T (x - pos)
    if exact:          # neural-SDF bodies: the decoder itself, differentiable w.r.t. its parameters (single world)
        sdf, mask = body.query_sdfs(loc[0].contiguous(), return_grads=False, return_overlapmask=True, exact=True)
        sdf, mask = sdf[None], mask[None]
    else:
        sdf, mask = body.query_sdfs(loc.contiguous(), return_grads=False, return_overlapmask=True)
    sdf = torch.where(mask, sdf, torch.zeros_like(sdf))
    loss, n = (sdf ** 2).sum(-1), mask.sum(-1)
    single = points_world.dim() == 2 and body.p.dim() == 1
    return (loss[0], n[0]) if single else (loss, n)
