"""Engine plug-in: ``PdipmEngine.solve_dynamics(world, dt) -> new_v`` (lcp_physics/physics/engines.py:22-83), batched.

``World3D(engine='PdipmEngine')`` resolves this class by name exactly like the reference (utils.get_instance);
``B200Engine`` is an alias.  One call assembles the mixed LCP of every active world on the device
(dsdf_dynamics_assemble), solves it (dsdf_lcp_forward, one CTA per world) and negates the solution.
Backward = dsdf_lcp_backward + dsdf_dynamics_assemble_backward.
"""
import torch

from . import _lib, ops
from .lcp import lcp_backward_raw, lcp_solve_raw

F64 = torch.float64


def _assemble(L, p, v, mass, Ibody, fric, rest, f, dt, active, count, cbody, geo, fd):
    W, nb = p.shape[0], p.shape[1]
    maxc = geo.shape[1]
    nz, ni = 6 * nb, maxc * (2 + fd)
    dev = p.device
    Q = torch.empty(W, nz, nz, dtype=F64, device=dev)
    pv = torch.empty(W, nz, dtype=F64, device=dev)
    G = torch.empty(W, ni, nz, dtype=F64, device=dev)
    h = torch.empty(W, ni, dtype=F64, device=dev)
    Fm = torch.empty(W, ni, ni, dtype=F64, device=dev)
    nin = torch.empty(W, dtype=torch.int32, device=dev)
    rc = _lib.call('dsdf_dynamics_assemble', _lib.ptr(p), _lib.ptr(v), _lib.ptr(mass), _lib.ptr(Ibody), _lib.ptr(fric),
                                  _lib.ptr(rest), _lib.ptr(f), _lib.ptr(dt), _lib.ptr(active), _lib.ptr(count),
                                  _lib.ptr(cbody), _lib.ptr(geo), W, nb, maxc, fd, _lib.ptr(Q), _lib.ptr(pv),
                                  _lib.ptr(G), _lib.ptr(h), _lib.ptr(Fm), _lib.ptr(nin), _lib.stream())
    _lib.check(rc, 'dsdf_dynamics_assemble')
    return Q, pv, G, h, Fm, nin


class _Dynamics(torch.autograd.Function):
    @staticmethod
    def forward(ctx, p, v, mass, Ibody, fric, rest, f, dt, geo, count, cbody, A, b, active, cfg):
        L = _lib.lib()
        _lib.require_cuda(p, v)
        c = lambda t: t.contiguous()
        p, v, mass, Ibody, fric, rest, f, dt, geo = [c(t) for t in (p, v, mass, Ibody, fric, rest, f, dt, geo)]
        A = c(A) if A is not None else None
        fd, max_iter = cfg['fric_dirs'], cfg['max_iter']
        Q, pv, G, h, Fm, nin = _assemble(L, p, v, mass, Ibody, fric, rest, f, dt, active, count, cbody, geo, fd)
        x, nu, lam, s, status, iters = lcp_solve_raw(Q, pv, G, h, A, b, Fm, nin, max_iter=max_iter, check_spd=False,
                                                     nineq_smem=cfg['ni_smem'])
        W, nb = p.shape[0], p.shape[1]
        new_v = (-x).reshape(W, nb, 6)
        if active is not None:
            new_v = torch.where(active.bool().reshape(W, 1, 1), new_v, v)
        ctx.save_for_backward(p, v, mass, Ibody, fric, rest, f, dt, geo, count, cbody, A, x, nu, lam, s, nin,
                              active if active is not None else p.new_empty(0))
        ctx.cfg = cfg
        cfg['last_status'], cfg['last_iters'] = status, iters
        ctx.mark_non_differentiable(status)
        return new_v, status

    @staticmethod
    def backward(ctx, gv_new, _gstatus):
        L = _lib.lib()
        (p, v, mass, Ibody, fric, rest, f, dt, geo, count, cbody, A, x, nu, lam, s, nin, active) = ctx.saved_tensors
        active = active if active.numel() else None
        cfg = ctx.cfg
        fd = cfg['fric_dirs']
        W, nb = p.shape[0], p.shape[1]
        maxc = geo.shape[1]
        Q, pv, G, h, Fm, _ = _assemble(L, p, v, mass, Ibody, fric, rest, f, dt, active, count, cbody, geo, fd)
        gz = (-gv_new).reshape(W, 6 * nb).contiguous()
        gpass = None
        if active is not None:
            am = active.bool().reshape(W, 1)
            gpass = torch.where(am, torch.zeros_like(gz), -gz).reshape(W, nb, 6)   # inactive worlds: new_v = v
            gz = torch.where(am, gz, torch.zeros_like(gz))
        want_A = bool(ctx.needs_input_grad[11]) and A is not None and A.numel() > 0
        dQ, dp, dG, dh, dA, _, dF = lcp_backward_raw(Q, G, A, Fm, x, nu, lam, s, gz, nin,
                                                     need=(True, True, True, True, want_A, False, True),
                                                     nineq_smem=cfg['ni_smem'])
        dev = p.device
        gp = torch.empty_like(p)
        gv = torch.empty_like(v)
        gmass, gI = torch.empty_like(mass), torch.empty_like(Ibody)
        gfric, grest, gf = torch.empty_like(fric), torch.empty_like(rest), torch.empty_like(f)
        gdt, ggeo = torch.empty(W, dtype=F64, device=dev), torch.empty_like(geo)
        rc = _lib.call(
            'dsdf_dynamics_assemble_backward', _lib.ptr(p), _lib.ptr(v), _lib.ptr(mass), _lib.ptr(Ibody), _lib.ptr(fric), _lib.ptr(rest), _lib.ptr(f),
            _lib.ptr(dt), _lib.ptr(active), _lib.ptr(count), _lib.ptr(cbody), _lib.ptr(geo), W, nb, maxc, fd,
            int(cfg['stop_contact_grad']), int(cfg['stop_friction_grad']), _lib.ptr(Q), _lib.ptr(G), _lib.ptr(dQ),
            _lib.ptr(dp), _lib.ptr(dG), _lib.ptr(dh), _lib.ptr(dF), _lib.ptr(gp), _lib.ptr(gv), _lib.ptr(gmass),
            _lib.ptr(gI), _lib.ptr(gfric), _lib.ptr(grest), _lib.ptr(gf), _lib.ptr(gdt), _lib.ptr(ggeo), _lib.stream())
        _lib.check(rc, 'dsdf_dynamics_assemble_backward')
        if gpass is not None:
            gv = gv + gpass
        return gp, gv, gmass, gI, gfric, grest, gf, gdt, ggeo, None, None, (dA if want_A else None), None, None, None


class _DynamicsFused(torch.autograd.Function):
    """dsdf_dynamics_solve / dsdf_dynamics_solve_backward: structure-exploiting KKT, one class of ``nc_smem`` contacts
    (the library picks the kernels, as for the device-resident step loop).

    The kernels write new_v (= -x, inactive worlds: v) and consume dL/dnew_v directly: no torch arithmetic around them.
    """

    @staticmethod
    def forward(ctx, p, v, mass, Ibody, fric, rest, f, dt, geo, count, cbody, eq_rows, active, cfg):
        _lib.lib()
        _lib.require_cuda(p, v)
        c = lambda t: t.contiguous()
        p, v, mass, Ibody, fric, rest, f, dt, geo = [c(t) for t in (p, v, mass, Ibody, fric, rest, f, dt, geo)]
        W, nb = p.shape[0], p.shape[1]
        maxc, fd = geo.shape[1], cfg['fric_dirs']
        neq = eq_rows.shape[0]
        dev = p.device
        x = torch.empty(W, 6 * nb, dtype=F64, device=dev)
        new_v = torch.empty(W, nb, 6, dtype=F64, device=dev)
        nu = torch.empty(W, neq, dtype=F64, device=dev)
        lam = torch.empty(W, maxc * (2 + fd), dtype=F64, device=dev)
        s = torch.empty_like(lam)
        status = torch.zeros(W, dtype=torch.int32, device=dev)
        iters = torch.zeros(W, dtype=torch.int32, device=dev)
        C = cfg['nc_smem']
        n, ws = ops.dynamics_workspace(W, nb, neq, fd, C, C, False, dev)
        rc = _lib.call('dsdf_dynamics_solve', _lib.ptr(p), _lib.ptr(v), _lib.ptr(mass), _lib.ptr(Ibody),
                       _lib.ptr(fric), _lib.ptr(rest), _lib.ptr(f), _lib.ptr(dt), _lib.ptr(active), _lib.ptr(count),
                       _lib.ptr(cbody), _lib.ptr(geo), _lib.ptr(eq_rows), W, nb, neq, maxc, C, C, 0, fd,
                       1e-12, 3, cfg['max_iter'], _lib.ptr(x), _lib.ptr(new_v), _lib.ptr(nu), _lib.ptr(lam),
                       _lib.ptr(s), _lib.ptr(status), _lib.ptr(iters), None, None, _lib.ptr(ws), _lib.stream(),
                       kernels=n)
        _lib.check(rc, 'dsdf_dynamics_solve')
        ctx.save_for_backward(p, v, mass, Ibody, fric, rest, f, dt, geo, count, cbody, eq_rows, x, lam, s,
                              active if active is not None else p.new_empty(0))
        ctx.cfg = cfg
        cfg['last_iters'] = iters
        ctx.mark_non_differentiable(status)
        return new_v, status

    @staticmethod
    def backward(ctx, gv_new, _gstatus):
        (p, v, mass, Ibody, fric, rest, f, dt, geo, count, cbody, eq_rows, x, lam, s, active) = ctx.saved_tensors
        cfg, C = ctx.cfg, ctx.cfg['nc_smem']
        grads = ops.dynamics_solve_backward(p, v, mass, Ibody, fric, rest, f, dt, active if active.numel() else None,
                                            count, cbody, geo, eq_rows, C, C, False, cfg['fric_dirs'],
                                            cfg['stop_contact_grad'], cfg['stop_friction_grad'], x, lam, s, gv_new)
        return grads + (None,) * 5


class Engine:
    """engines.py:16-20."""

    def solve_dynamics(self, world, dt):
        raise NotImplementedError


class PdipmEngine(Engine):
    """Primal-dual interior-point LCP engine (engines.py:22-83) over all worlds at once."""

    dense = False    # True: assemble dense matrices and run the general LCP kernels (dsdf_lcp_*) instead

    def __init__(self, max_iter=10):
        self.max_iter = max_iter
        self.last_status = None

    def solve_dynamics(self, world, dt, active=None):
        """The reference's plug-in entry point (engines.py:31): ``dt`` is a float, a 0-d tensor (may carry grad,
        world.py:256-259) or a (W,) tensor; returns the new generalized velocity -- ``(nz,)`` for a single world like the
        reference, ``(W, nz)`` for a batch.  ``World3D`` itself calls ``solve`` (same thing, (W,nb,6) layout, with the
        active mask)."""
        if active is None and not (isinstance(dt, torch.Tensor) and dt.dim() == 1 and dt.shape[0] == world.W):
            dt = world._dt_tensor(dt)
        with world._on_device():
            new_v = self.solve(world, dt, active).reshape(world.W, -1)
        return new_v if world.batched else new_v[0]

    def solve(self, world, dt, active=None):
        """dt: (W,) tensor (may carry grad).  Returns new_v (W,nb,6)."""
        st = world.state
        f = world.step_forces()
        cfg = dict(fric_dirs=world.fric_dirs, max_iter=self.max_iter, stop_contact_grad=world.stop_contact_grad,
                   stop_friction_grad=world.stop_friction_grad,
                   ni_smem=max(world.max_nc, 1) * (2 + world.fric_dirs), nc_smem=max(world.max_nc, 1))
        cs = world.contact_set
        if self.dense or world._general_joints:
            new_v, status = _Dynamics.apply(st.p, st.v, st.mass, st.Ibody, st.fric, st.rest, f, dt, world.contact_geo,
                                            cs.count, cs.body, world.A, world.b, active, cfg)
        else:
            new_v, status = _DynamicsFused.apply(st.p, st.v, st.mass, st.Ibody, st.fric, st.rest, f, dt,
                                                 world.contact_geo, cs.count, cs.body, world.eq_rows, active, cfg)
        self.last_status = status
        return new_v

    def post_stabilization(self, world):
        """engines.py:85-121 for all worlds at once: dp = -argmin 1/2 z'Mz  s.t.  Jc z <= Jc v (1 - e),  Je z = Je v, with the
        contacts, velocities and mass matrix the world has after its accepted sub-step.  The reference builds a fresh
        ``LCPFunction()`` for it (20 iterations, not the engine's ``max_iter``); so does this.  Runs on the general dense LCP
        operator (``dsdf_lcp_forward / backward`` with per-world inequality counts) and is differentiable like the
        reference's.  Returns (W, nb, 6) -- ``(nz,)`` for a single world through ``World3D``'s own call."""
        from .transforms import quaternion_to_matrix
        st, cs = world.state, world.contact_set
        W, nb, maxc, dev = world.W, world.nb, world.maxc, world.device
        nz = 6 * nb
        v = st.v.reshape(W, nz)
        R = quaternion_to_matrix(st.p[..., :4])                                        # (W,nb,3,3)
        Iw = R @ st.Ibody.reshape(W, nb, 3, 3) @ R.transpose(-1, -2)
        M = torch.zeros(W, nb, 6, nb, 6, dtype=F64, device=dev)
        eye3 = torch.eye(3, dtype=F64, device=dev)
        for b in range(nb):
            M[:, b, :3, b, :3] = Iw[:, b]
            M[:, b, 3:, b, 3:] = st.mass[:, b, None, None] * eye3
        M = M.reshape(W, nz, nz)
        neq = world.A.shape[1] if world.A is not None else 0
        geo = world.contact_geo.detach() if world.stop_contact_grad else world.contact_geo
        n, p1, p2 = geo[..., 0:3], geo[..., 3:6], geo[..., 6:9]
        valid = (torch.arange(maxc, device=dev)[None, :] < cs.count[:, None])
        i1, i2 = cs.body[..., 0].long().clamp(0, nb - 1), cs.body[..., 1].long().clamp(0, nb - 1)
        r1 = torch.cat([torch.linalg.cross(p1, n), n], -1) * valid[..., None]           # world.py:56-71 (physics3d)
        r2 = -torch.cat([torch.linalg.cross(p2, n), n], -1) * valid[..., None]
        Jc = torch.zeros(W, maxc, nb, 6, dtype=F64, device=dev)
        Jc = Jc.scatter_add(2, i1[:, :, None, None].expand(-1, -1, 1, 6), r1[:, :, None, :])
        Jc = Jc.scatter_add(2, i2[:, :, None, None].expand(-1, -1, 1, 6), r2[:, :, None, :]).reshape(W, maxc, nz)
        e = 0.5 * (torch.gather(st.rest, 1, i1) + torch.gather(st.rest, 1, i2))
        jv = (Jc @ v[..., None])[..., 0]
        gc = jv + jv * -e
        # a world without contacts gets one inert row (0 z <= 1): the solution is then the equality-constrained one the
        # reference computes by a direct solve (engines.py:99-110)
        none = (cs.count == 0)
        gc = torch.where(none[:, None] & (torch.arange(maxc, device=dev)[None, :] == 0), torch.ones_like(gc), gc)
        nin = torch.clamp(cs.count, min=1).to(torch.int32).contiguous()
        A = world.A if neq else None
        ge = (world.A @ v[..., None])[..., 0] if neq else None
        x = _LcpRagged.apply(M, torch.zeros(W, nz, dtype=F64, device=dev), Jc, gc, A, ge,
                             torch.zeros(W, maxc, maxc, dtype=F64, device=dev), nin)
        return (-x).reshape(W, nb, 6)


class _LcpRagged(torch.autograd.Function):
    """LCPFunction (lcp.py:48-213) with a per-world number of inequality rows (the first nin[w] rows of G, h, F count)."""

    @staticmethod
    def forward(ctx, Q, p, G, h, A, b, F, nin):
        c = lambda t: t.contiguous()
        Q, p, G, h, F = c(Q), c(p), c(G), c(h), c(F)
        A, b = (c(A), c(b)) if A is not None else (None, None)
        x, nu, lam, s, status, _ = lcp_solve_raw(Q, p, G, h, A, b, F, nin, max_iter=20, check_spd=False)
        ctx.save_for_backward(x, nu, lam, s, Q, G, A if A is not None else Q.new_empty(0), F, nin)
        ctx.has_eq = A is not None
        return x

    @staticmethod
    def backward(ctx, gz):
        x, nu, lam, s, Q, G, A, F, nin = ctx.saved_tensors
        A = A if ctx.has_eq else None
        need = list(ctx.needs_input_grad[:7])
        dQ, dp, dG, dh, dA, db, dF = lcp_backward_raw(Q, G, A, F, x, nu, lam, s, gz, nin, need)
        rows = (torch.arange(G.shape[1], device=G.device)[None, :] < nin[:, None])
        if dG is not None:
            dG = dG * rows[..., None]
        if dh is not None:
            dh = dh * rows
        if dF is not None:
            dF = dF * rows[..., None] * rows[:, None, :]
        return dQ, dp, dG, dh, dA, db, dF, None


class DensePdipmEngine(PdipmEngine):
    """Same engine through the dense LCP kernels (the LCPFunction path); limited to ~15 contacts per world."""
    dense = True


B200Engine = PdipmEngine
