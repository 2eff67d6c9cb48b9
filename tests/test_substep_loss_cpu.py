"""losses.trajectory_loss on sub-step entries of a batch (World3D(record_substeps=True)): every world averages over its
own ``valid`` entries and is matched only to its own valid target entries."""
import os
from types import SimpleNamespace

import numpy as np
import torch

from diffsdfsim_b200.losses import trajectory_loss
from diffsdfsim_b200.world import SubstepEntry


def _reference_trajectory_loss(traj, traj_target):
    """experiments/trajectory_fitting/optim_sphere.py:114-160 transcribed for one world: lists of (t, p)."""
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


def test_trajectory_loss_honours_valid_per_world():
    """The golden trajectories of tests/golden/trajectory_loss.npz (irregular times, exact ties), truncated to a different
    length per world through ``valid``: each world's loss and gradients equal the reference loop on that world's
    truncated lists.  Rows past a world's length hold finite values that must neither count nor be matched."""
    g = np.load(os.path.join(os.path.dirname(__file__), 'golden', 'trajectory_loss.npz'))
    W, S, St = g['t'].shape[0], g['t'].shape[1], g['tt'].shape[1]
    n, nt = [S, S - 3, 7, 2], [St - 5, St, 4, St - 1]            # valid entries of each world
    T = lambda a: torch.tensor(a, dtype=torch.float64)
    ps = [T(g['p'][:, k]).reshape(W, 2, 7).requires_grad_(True) for k in range(S)]
    mask = lambda k, lens: torch.tensor([k < m for m in lens])
    a = SimpleNamespace(W=W, device=torch.device('cpu'), batched=True, trajectory=[
        SubstepEntry((T(g['t'][:, k]), ps[k], T(g['v'][:, k]).reshape(W, 2, 6), None, None), mask(k, n)) for k in range(S)])
    b = SimpleNamespace(W=W, device=torch.device('cpu'), batched=True, trajectory=[
        SubstepEntry((T(g['tt'][:, k]), T(g['pt'][:, k]).reshape(W, 2, 7), T(g['vt'][:, k]).reshape(W, 2, 6), None, None),
                     mask(k, nt)) for k in range(St)])
    assert all(len(e) == 5 for e in a.trajectory)
    loss = trajectory_loss(a, b)
    loss.sum().backward()
    for w in range(W):
        pw = [T(g['p'][w, k]).requires_grad_(True) for k in range(n[w])]
        ref = _reference_trajectory_loss([(float(g['t'][w, k]), pw[k]) for k in range(n[w])],
                                         [(float(g['tt'][w, k]), T(g['pt'][w, k])) for k in range(nt[w])])
        ref.backward()
        np.testing.assert_allclose(float(loss[w]), float(ref), rtol=1e-12, err_msg='world %d' % w)
        for k in range(S):
            got = ps[k].grad[w].reshape(-1).numpy()
            want = pw[k].grad.numpy() if k < n[w] else np.zeros(14)
            np.testing.assert_allclose(got, want, rtol=1e-12, atol=1e-15, err_msg='world %d entry %d' % (w, k))
