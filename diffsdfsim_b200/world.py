"""``World3D`` -- drop-in for sdf_physics.physics3d.world.World3D, stepping W independent worlds at once.

Constructor and ``step`` signatures follow the reference (sdf_physics/physics3d/world.py:33-46,
lcp_physics/physics/world.py:43-139, 241-379).  Each world runs the reference's per-world state machine
(solve -> move -> find_contacts -> accept | halve dt and retry | give up below dt/2^10 when not strict;
after a short accepted sub-step the remaining time is taken next; time-of-contact differential on first
touch), expressed with per-world masks: one "round" = one attempt of every still-active world.
All arithmetic of the round runs in the CUDA kernels (engines.py, contacts.py, ops.py); this file only
routes tensors and merges accepted/rejected worlds with ``torch.where``.
"""
import weakref

import torch

from . import contacts as contacts_module
from . import engines as engines_module
from . import _lib, ops
from .contacts import ContactDetector, GeometryTable, differentiable_geometry
from .stepper import DeviceStepper, _StepFn
from .transforms import quaternion_to_matrix, so3_exponential_map
from .utils import Defaults3D, default_device, get_instance

F64 = torch.float64


class WorldState:
    """SoA over worlds: p (W,nb,7), v (W,nb,6), mass (W,nb), Ibody (W,nb,3,3), fric (W,nb), rest (W,nb)."""
    __slots__ = ('p', 'v', 'mass', 'Ibody', 'fric', 'rest')


class TimeOfContact(torch.autograd.Function):
    """World.H (lcp_physics/physics/world.py:141-237), all worlds at once.

    Forward: identity on dt.  Backward: dL/dtheta = -(dD/dh)^+ dD/dtheta dL/dh per world over its new contacts,
    with D the gap function of world.py:151-171.  Every contact's D depends only on its own rows, so the
    Jacobians the reference takes with autograd.functional.jacobian are the per-row gradients of sum(D).
    """

    @staticmethod
    def gap(h, c1, c2, v1, v2, x1, x2, R1, R2, n2, a1, a2):
        hh = h[..., None]
        Rih = so3_exponential_map(hh * v1[..., :3]) @ R1
        Rjh = so3_exponential_map(hh * v2[..., :3]) @ R2
        xi = x1 + hh * v1[..., 3:] + 0.5 * a1[..., 3:] * hh * hh
        xj = x2 + hh * v2[..., 3:] + 0.5 * a2[..., 3:] * hh * hh
        ci_w = (Rih @ c1[..., None])[..., 0] + xi
        ci_j = (Rjh.transpose(-1, -2) @ (ci_w - xj)[..., None])[..., 0]
        return (n2 * (c2 - ci_j)).sum(-1)

    @staticmethod
    def forward(ctx, h, mask, *args):
        ctx.save_for_backward(h, mask, *args)
        return h.clone()

    @staticmethod
    def backward(ctx, gh):
        h, mask, *args = ctx.saved_tensors
        C = mask.shape[1]
        with torch.enable_grad():
            hk = h.detach()[:, None].expand(-1, C).clone().requires_grad_(True)
            ins = [a.detach().clone().requires_grad_(True) for a in args]
            D = TimeOfContact.gap(hk, *ins)
            grads = torch.autograd.grad((D * mask).sum(), [hk] + ins)
        dD_dh = grads[0] * mask
        dD_dh = torch.where(dD_dh < ops.BASE_TOL / h.detach()[:, None], torch.zeros_like(dD_dh), dD_dh)
        den = (dD_dh ** 2).sum(1, keepdim=True)
        inv = torch.where(den > 1e-5, dD_dh / torch.where(den > 1e-5, den, torch.ones_like(den)), torch.zeros_like(dD_dh))
        outs = [gh, None]
        for g in grads[1:]:
            wgt = (-inv * gh[:, None]).reshape(inv.shape + (1,) * (g.dim() - 2))
            outs.append(wgt * g)
        return tuple(outs)


class TimeOfContactNative(torch.autograd.Function):
    """World.H + its gather (world.py:141-237, 275-327) for ALL worlds through dsdf_toc_backward: identity forward,
    one kernel backward; worlds without a new contact pass dL/ddt through unchanged."""

    @staticmethod
    def forward(ctx, dt_, p_try, new_v, geo, f, mass, toc_mask, cbody):
        ctx.save_for_backward(dt_, p_try, new_v, geo, f, mass, toc_mask, cbody)
        return dt_.clone()

    @staticmethod
    def backward(ctx, gh):
        dt_, p_try, new_v, geo, f, mass, toc_mask, cbody = ctx.saved_tensors
        return ops.toc_backward(dt_, toc_mask, cbody, p_try, new_v, geo, f, mass, gh) + (None, None)


class World3D:
    max_rounds_per_step = 256
    toc_native = True      # False: the torch-autograd restatement of World.H (TimeOfContact) on the affected worlds
    device_loop = True     # the per-world step state machine runs on the device (stepper.py / csrc/dsdf_steploop.cu);
                           # False: the host-driven round loop below (one synchronisation per round)

    def __init__(self, bodies, constraints=[], dt=Defaults3D.DT, engine=Defaults3D.ENGINE,
                 contact_callback=Defaults3D.CONTACT, eps=Defaults3D.EPSILON, tol=Defaults3D.TOL,
                 fric_dirs=Defaults3D.FRIC_DIRS, post_stab=Defaults3D.POST_STABILIZATION,
                 strict_no_penetration=True, time_of_contact_diff=True, stop_contact_grad=False,
                 stop_friction_grad=False, detach_contact_b2=False, device=None, capK=384, maxc=32,
                 record_prefilter=False):
        self.post_stab = bool(post_stab)          # world.py:358-370; runs on the host-driven loop + the dense LCP operator
        self.engine = get_instance(engines_module, engine)
        self.contact_callback = get_instance(contacts_module, contact_callback)
        self.bodies = list(bodies)
        if device is None:
            # the device the bodies live on (first CUDA tensor found), else the default device
            devs = [b.p.device for b in self.bodies if b.p.is_cuda] + [b.mass.device for b in self.bodies if b.mass.is_cuda]
            device = devs[0] if devs else default_device()
        self.device = torch.device(device)
        if self.device.type == 'cuda' and self.device.index is None:
            self.device = torch.device('cuda', torch.cuda.current_device())
        self.nb = len(self.bodies)
        self.W = max(b.batch() for b in self.bodies)
        self.batched = self.W > 1
        self.vec_len = 6
        self.dt, self.eps, self.tol, self.fric_dirs = dt, eps, tol, fric_dirs
        self.strict_no_pen = strict_no_penetration
        self.time_of_contact_diff = time_of_contact_diff
        self.stop_contact_grad, self.stop_friction_grad = stop_contact_grad, stop_friction_grad
        self.detach_contact_b2 = detach_contact_b2
        self.maxc = maxc
        W, nb, dev = self.W, self.nb, self.device
        for i, b in enumerate(self.bodies):
            b._world, b._index = weakref.ref(self), i      # weak: a finished world is freed by refcount, not by the GC

        def ex(t, *shape):
            return t.to(dev).expand(W, *shape)

        st = self.state = WorldState()
        st.p = torch.stack([ex(b.p, 7) for b in self.bodies], 1).contiguous()
        st.v = torch.stack([ex(b.v, 6) for b in self.bodies], 1).contiguous()
        st.mass = torch.stack([ex(b.mass) for b in self.bodies], 1).contiguous()
        st.Ibody = torch.stack([ex(b.ang_inertia, 3, 3) for b in self.bodies], 1).contiguous()
        st.fric = torch.stack([ex(b.fric_coeff) for b in self.bodies], 1).contiguous()
        st.rest = torch.stack([ex(b.restitution) for b in self.bodies], 1).contiguous()
        # [a, b, c, scale] rows of every body: the kernels read the values; shape_t keeps the autograd link to radius /
        # dimension leaves (radius and size fitting differentiate the contact geometry through them, contacts.py:262-264)
        shape_t = torch.stack([ex(b.shape_rows(), 4) for b in self.bodies], 1)
        self.shape = shape_t.detach().contiguous()
        self.shape_t = shape_t if shape_t.requires_grad else None
        self.body_eps = float(self.bodies[0].eps)

        # equality rows: constant 0/1 selections (constraints.py)
        self.joints = []
        rows, plan = [], []          # plan: Je row blocks in constraint order -- ('sel', first row, n) / ('gen', first row, joint)
        for j in constraints:
            i1 = self.bodies.index(j.body1)
            i2 = self.bodies.index(j.body2) if getattr(j, 'body2', None) is not None else None
            self.joints.append((j, i1, i2))
            if getattr(j, 'general', False):
                plan.append(('gen', len(rows), (j, i1, i2)))
                rows += [(-1, -1)] * j.num_constraints
            else:
                sel = [(i1, a) for a in j.rows()]
                plan.append(('sel', len(rows), len(sel)))
                rows += sel
        self.num_constraints = len(rows)
        self._general_joints = [blk for kind, _, blk in plan if kind == 'gen']
        self._je_plan = plan
        nz = 6 * nb
        A = torch.zeros(len(rows), nz, dtype=F64)
        for r, (i, a) in enumerate(rows):
            if i >= 0:
                A[r, 6 * i + a] = 1
        self._A_static = A.to(dev).unsqueeze(0).expand(W, -1, -1).contiguous() if rows else None
        self.b = torch.zeros(W, len(rows), dtype=F64, device=dev) if rows else None
        if self._general_joints:
            rows = []                # the fused kernels only know selection rows: such a world uses the dense operator
        self.eq_rows = torch.tensor(rows, dtype=torch.int32, device=dev).reshape(-1, 2).contiguous()

        # contact detection set-up (replaces the py3ode HashSpace of world.py:69-72)
        self.table = GeometryTable(self.bodies, W, dev)
        self.vert_leaves = [self.bodies[i].verts.to(dev) for i in self.table.vert_leaf_ids]   # differentiable meshes
        self.pairs = [(i, j) for i in range(nb) for j in range(i + 1, nb)
                      if self.bodies[j] not in self.bodies[i].no_contact]
        self.detector = ContactDetector(self.table, self.pairs, W, nb, dev, capK=capK, maxc=maxc,
                                        record_prefilter=record_prefilter)

        self.t = torch.zeros(W, dtype=F64, device=dev)
        self.t_host = 0.0
        self.last_dt = torch.zeros(W, dtype=F64, device=dev)
        self.toc_flag = torch.zeros(W, dtype=torch.uint8, device=dev)
        self.trajectory, self.observations = [], []
        self.stats = {'rounds': [], 'attempts': torch.zeros(W, dtype=torch.int64, device=dev)}
        self.static_inverse = False
        self._f_cache, self._any_toc_flag = None, False
        self._f_vectorized = any(getattr(f, 'vectorized', False) for b in self.bodies for f in b.forces)
        self.contact_set = self.detector.new_set()
        self.contact_geo = None
        self._stepper, self._last_tape = None, None
        with self._on_device():
            while True:
                self.find_contacts()
                bits = self._capacity_bits(self.contact_set)
                if not bits:
                    break
                self._grow_capacity(bits)
        if self.strict_no_pen:
            assert not bool(((self.contact_set.status & 8) != 0).any()), \
                'Interpenetration at start:\n{}'.format(self.contacts_of(0))

    # ------------------------------------------------------------------ reference-style accessors
    @property
    def v(self):
        v = self.state.v.reshape(self.W, -1)
        return v if self.batched else v[0]

    @v.setter
    def v(self, new_v):
        """The reference's drivers write ``world.v = world.v.detach().clone()`` before ``set_v`` (optim_sphere.py:172-175)."""
        self.set_v(new_v)

    def get_v(self):
        return self.v

    def set_v(self, new_v):
        self.state.v = new_v.reshape(self.W, self.nb, 6).to(self.device)
        self._sync_bodies()

    def get_p(self):
        p = self.state.p.reshape(self.W, -1)
        return p if self.batched else p[0]

    def set_p(self, new_p):
        self.state.p = new_p.reshape(self.W, self.nb, 7).to(self.device)
        self._sync_bodies()

    def _body_pose_changed(self, i):
        B = self.bodies[i]
        p = self.state.p.clone()
        p[:, i] = B.p.to(self.device).expand(self.W, 7)
        self.state.p = p

    def _sync_bodies(self):
        for i, b in enumerate(self.bodies):
            b.p, b.v = self.state.p[:, i], self.state.v[:, i]

    def apply_forces(self, t):
        """(W,nb,6) generalized forces; t is the step start time (host float) -- see forces.py."""
        fs = []
        for b in self.bodies:
            if not b.forces:
                fs.append(torch.zeros(self.W, 6, dtype=F64, device=self.device))
                continue
            tot = 0
            for f in b.forces:
                tt = self.t if getattr(f, 'vectorized', False) else self.t_host
                tot = tot + f.force(tt).to(self.device)
            fs.append(tot.expand(self.W, 6))
        return torch.stack(fs, 1).contiguous()

    def M(self):
        """Block-diagonal world-frame mass matrix (physics3d/world.py:48-50) from the assembly kernel: (W,nz,nz)."""
        Q = self.lcp_matrices()[0]
        return Q if self.batched else Q[0]

    @property
    def A(self):
        """Je for all worlds (W,neq,nz), rows in constraint order (world.py:411-428).  Constant for the selection
        constraints; joints coupling two bodies (GripperJoint) contribute pose-dependent, differentiable blocks."""
        if not self._general_joints:
            return self._A_static
        st = self.state
        A = self._A_static.clone()
        for kind, r0, blk in self._je_plan:
            if kind != 'gen':
                continue
            j, i1, i2 = blk
            J1, J2 = j.J(st.p[:, i1], st.p[:, i2])
            n = j.num_constraints
            A[:, r0:r0 + n, 6 * i1:6 * i1 + 6] = J1
            A[:, r0:r0 + n, 6 * i2:6 * i2 + 6] = J2
        return A

    def Je(self):
        if self.A is None:
            return torch.zeros(0, 6 * self.nb, dtype=F64, device=self.device)
        return self.A if self.batched else self.A[0]

    def lcp_matrices(self, dt=None):
        """(Q, p, G, h, A, b, F, nineq_w) exactly as handed to the LCP kernel (engines.py:56-79 layout)."""
        st = self.state
        dtt = self._dt_tensor(self.dt if dt is None else dt)
        f = self.apply_forces(self.t)
        Q, pv, G, h, Fm, nin = engines_module._assemble(
            _lib.lib(), st.p.detach().contiguous(), st.v.detach().contiguous(), st.mass.detach().contiguous(),
            st.Ibody.detach().contiguous(), st.fric.detach().contiguous(), st.rest.detach().contiguous(),
            f.detach().contiguous(), dtt, None, self.contact_set.count, self.contact_set.body,
            self.contact_geo.detach().contiguous(), self.fric_dirs)
        return Q, pv, G, h, self.A, self.b, Fm, nin

    def contacts_of(self, w=0):
        """Reference-format contact list of world w: [((normal, p1, p2, pen), i1, i2), ...] (contacts.py:266-270)."""
        n = int(self.contact_set.count[w])
        g, bd = self.contact_geo[w], self.contact_set.body[w]
        return [((g[k, 0:3], g[k, 3:6], g[k, 6:9], g[k, 9]), int(bd[k, 0]), int(bd[k, 1])) for k in range(n)]

    @property
    def contacts(self):
        return self.contacts_of(0) if not self.batched else [self.contacts_of(w) for w in range(self.W)]

    def _dt_tensor(self, dt):
        if isinstance(dt, torch.Tensor):
            return dt.to(self.device).expand(self.W).contiguous() if dt.dim() <= 1 else dt
        return torch.full((self.W,), float(dt), dtype=F64, device=self.device)

    def _capacity_bits(self, cs):
        """bit 0: candidate-list overflow (capK) in some world; bit 1: contact overflow (maxc) on a non-penetrating state."""
        st = cs.status
        return int((st & 1).max().item()) | (int(((st & 2) != 0).logical_and((st & 8) == 0).any().item()) << 1)

    # ------------------------------------------------------------------ contact detection
    def find_contacts(self, active=None):
        """world.py:396-399 for all (active) worlds; keeps the geometry attached to the pose graph."""
        cs = self.contact_set.clone() if active is not None else self.detector.new_set()
        self.detector.detect(self.state.p.detach().contiguous(), self.shape, cs, active, eps=self.eps, tol=self.tol,
                             fd_eps=Defaults3D.EPSILON, body_eps=self.body_eps, detach_b2=self.detach_contact_b2)
        self.contact_set = cs
        self.max_nc = int(cs.count.max())
        self.contact_geo = differentiable_geometry(self.state.p, self.shape, cs, self.table, Defaults3D.EPSILON,
                                                   self.detach_contact_b2, self.shape_t, self.vert_leaves)
        return cs

    # ------------------------------------------------------------------ stepping
    def _on_device(self):
        import contextlib
        return torch.cuda.device(self.device) if self.device.type == 'cuda' else contextlib.nullcontext()

    def step_forces(self):
        """Generalized forces of the current step.  Forces that only see the step's start time (the default, see
        forces.py) are evaluated once per step and reused by every sub-step attempt."""
        if self._f_cache is None or self._f_vectorized:
            self._f_cache = self.apply_forces(self.t)
        return self._f_cache

    def step(self, fixed_dt=False):
        """world.py:119-139.  Returns had_contacts: python bool for a single world, (W,) bool tensor otherwise."""
        with self._on_device():                      # kernels launch on the world's device, whatever is current
            return self._step(fixed_dt)

    def _use_device_loop(self):
        """The device-resident loop covers the default configuration; plug-in engines, the dense LCP path, the torch
        restatement of World.H, per-sub-step (vectorised) forces and pre-filter recording use the host-driven loop."""
        return (self.device_loop and self.device.type == 'cuda' and type(self.engine) is engines_module.PdipmEngine
                and self.toc_native and not self._f_vectorized and not self.detector.record_prefilter
                and not self.post_stab and not self._general_joints)

    def _snapshot(self):
        st = self.state
        return (st.p, st.v, self.contact_set, self.contact_geo, self.t, self.t_host, self.toc_flag.clone(),
                self.last_dt, len(self.trajectory), self._any_toc_flag, self.max_nc)

    def _step(self, fixed_dt):
        self._undo = self._snapshot()
        self._f_cache = None
        t_start = self.t if self.batched else float(self.t[0])
        if self._use_device_loop():
            had = self._step_device(fixed_dt)
        else:
            had = self._step_host(fixed_dt)
        # host copy of the simulated time handed to non-vectorised force functions: exact for fixed_dt stepping; a
        # variable-dt step may end early (world.py:134-137), then it is read back from the device (one sync, rare mode)
        self.t_host = self.t_host + self.dt if fixed_dt else float(self.t.max())
        self._sync_bodies()
        # one entry per step(), stamped like the reference's entries with the time the step STARTED (world.py:372-379
        # appends (self.t, ...) before self.t += dt; the reference appends once per accepted sub-step, we record the
        # state at the end of the whole step -- see INTEGRATION.md)
        self.trajectory.append((t_start, self.get_p(), self.v, self.contact_set, None))
        return had if self.batched else bool(had[0])

    def _step_device(self, fixed_dt):
        """world.py:119-139 with the whole sub-step state machine on the device: one autograd node, normally one host
        synchronisation (the 64-byte control block of stepper.DeviceStepper)."""
        st = self.state
        if self._stepper is None:
            self._stepper = DeviceStepper(self)
        p, v, geo, last_dt, had = _StepFn.apply(self, fixed_dt, st.p, st.v, self.contact_geo, self.last_dt, st.mass,
                                                st.Ibody, st.fric, st.rest, self.step_forces(), self.shape_t,
                                                *self.vert_leaves)
        tape = self._last_tape
        st.p, st.v, self.contact_geo, self.last_dt = p, v, geo, last_dt
        self.contact_set = tape.final
        self.max_nc = max(int(self.max_nc), int(self._stepper.max_count))
        self._any_toc_flag = self._any_toc_flag or tape.any_toc
        self.stats['rounds'].append(tape.rounds)
        self.stats.setdefault('syncs', []).append(tape.syncs)
        self._last_tape = None
        return had

    def _step_host(self, fixed_dt):
        W, dev = self.W, self.device
        end_t = (self.t + self.dt) if fixed_dt else None
        dt_try = torch.full((W,), float(self.dt), dtype=F64, device=dev)
        active = torch.ones(W, dtype=torch.uint8, device=dev)
        had = torch.zeros(W, dtype=torch.bool, device=dev)
        rounds = 0
        while True:
            rounds += 1
            if rounds > self.max_rounds_per_step:
                raise self._incomplete_step_error(active, dt_try)
            self.stats['attempts'] += active
            accept, dt_try, active, n_active = self._attempt(active, dt_try, end_t)
            had |= accept.bool() & (self.contact_set.count > 0)
            if not n_active:
                break
        self.stats['rounds'].append(rounds)
        return had

    def _incomplete_step_error(self, active, dt_try):
        """strict_no_penetration=True halves dt for ever in the reference too (world.py:344-348); both step loops stop
        after ``max_rounds_per_step`` rounds instead of accumulating an unbounded autograd graph."""
        stuck = active.nonzero().flatten().tolist()[:8]
        return RuntimeError('step did not complete in %d attempts: worlds %s keep penetrating (dt < %.3g); '
                            'use strict_no_penetration=False or a smaller dt'
                            % (self.max_rounds_per_step, stuck, float(dt_try.min())))

    def undo_step(self, mask=None):
        """world.py:106-116.  ``mask`` (optional (W,) bool tensor, batched extension): undo the last step only for those
        worlds -- the others keep their new state (used by the per-world detach-2nd-bounce logic of the fitting drivers).
        The contact capacity may have grown during the undone step: the restored set is brought to the current capacity,
        and the contact-count bound that sizes the dynamics kernel never shrinks."""
        st = self.state
        (p0, v0, cs, geo, t0, t_host0, toc0, last0, ntraj, any_toc0, max_nc) = self._undo
        if cs.maxc != self.maxc:
            cs = cs.resized(self.maxc)
            geo = torch.cat([geo, geo.new_zeros(self.W, self.maxc - geo.shape[1], 10)], 1)
        self.max_nc = max(int(self.max_nc), int(max_nc))
        if mask is None:
            st.p, st.v, self.contact_set, self.contact_geo = p0, v0, cs, geo
            self.t, self.t_host, self.toc_flag, self.last_dt, self._any_toc_flag = t0, t_host0, toc0, last0, any_toc0
            del self.trajectory[ntraj:]
        else:
            m = mask.to(self.device).bool()
            m3 = m[:, None, None]
            st.p, st.v = torch.where(m3, p0, st.p), torch.where(m3, v0, st.v)
            self.contact_geo = torch.where(m3, geo, self.contact_geo)
            self.contact_set = self.contact_set.where(m, cs)
            self.t = torch.where(m, t0, self.t)
            self.toc_flag = torch.where(m, toc0, self.toc_flag)
            self.last_dt = torch.where(m, last0, self.last_dt)
        self._sync_bodies()

    def detach_state(self, mask=None):
        """Cut the autograd history of the poses and velocities (of the masked worlds): what the reference drivers do with
        ``world.v = world.v.detach().clone(); world.set_v(world.v); world.set_p(cat(b.p.detach()))``
        (experiments/trajectory_fitting/optim_sphere.py:172-175)."""
        st = self.state
        if mask is None:
            st.p, st.v = st.p.detach().clone(), st.v.detach().clone()
        else:
            m3 = mask.to(self.device).bool()[:, None, None]
            st.p, st.v = torch.where(m3, st.p.detach(), st.p), torch.where(m3, st.v.detach(), st.v)
        self._sync_bodies()

    def _attempt(self, active, dt_try, end_t):
        """One solve -> move -> find_contacts attempt of every active world (body of world.py:249-356).

        ``active`` is a uint8 (W) mask.  Returns (accept, next dt_try, next active, any world still active).  The
        per-world accept / halve / remaining-time / time-of-contact bookkeeping and the merge of the new contact set
        with the previous one run in dsdf_attempt_commit; ONE host synchronisation per attempt reads its 4 flags
        [capacity error, any world still active, any new (time-of-contact) contact, max contact count].
        """
        st = self.state
        W, nb, dev = self.W, self.nb, self.device
        toc = self.time_of_contact_diff
        dt_ = dt_try
        if toc and self._any_toc_flag:
            # world.py:253-257: value == dt_try, carries -d last_dt
            dt_ = torch.where(self.toc_flag.bool(), -self.last_dt + (self.last_dt.detach() + dt_try), dt_try)
        new_v = self.engine.solve(self, dt_, active)
        p_try = ops.integrate(st.p, new_v, dt_, active)
        old = self.contact_set
        cs = old.clone()
        self.detector.detect(p_try.detach(), self.shape, cs, active, eps=self.eps, tol=self.tol,
                             fd_eps=Defaults3D.EPSILON, body_eps=self.body_eps, detach_b2=self.detach_contact_b2)
        geo = differentiable_geometry(p_try, self.shape, cs, self.table, Defaults3D.EPSILON, self.detach_contact_b2,
                                      self.shape_t, self.vert_leaves)
        u8 = lambda *shape: torch.empty(*shape, dtype=torch.uint8, device=dev)
        accept, active_next, toc_now, toc_mask = u8(W), u8(W), u8(W), u8(W, self.maxc)
        t_new, dt_next = torch.empty_like(self.t), torch.empty_like(dt_try)
        flags = torch.empty(4, dtype=torch.int32, device=dev)
        toc_flag = self.toc_flag.clone() if toc else self.toc_flag
        rc = _lib.call('dsdf_attempt_commit', W, nb, self.maxc, _lib.ptr(active), _lib.ptr(dt_try), _lib.ptr(self.t),
                       _lib.ptr(end_t), float(self.dt), int(self.strict_no_pen), int(toc),
                       _lib.ptr(old.count), _lib.ptr(old.status), _lib.ptr(old.body), _lib.ptr(old.face),
                       _lib.ptr(old.abc), _lib.ptr(old.geo), _lib.ptr(cs.count), _lib.ptr(cs.status),
                       _lib.ptr(cs.body), _lib.ptr(cs.face), _lib.ptr(cs.abc), _lib.ptr(cs.geo), _lib.ptr(toc_flag),
                       _lib.ptr(accept), _lib.ptr(t_new), _lib.ptr(dt_next), _lib.ptr(active_next), _lib.ptr(toc_now),
                       _lib.ptr(toc_mask), _lib.ptr(flags), _lib.stream())
        _lib.check(rc, 'dsdf_attempt_commit')
        fl = flags.tolist()                                              # the sync
        if fl[0]:
            # nothing of this attempt has been committed yet: enlarge the buffers and run the attempt again
            self._grow_capacity(fl[0])
            return self._attempt(active, dt_try, end_t)
        self.max_nc = int(fl[3])                   # sizes the dynamics kernel's shared memory for the next solve
        if toc:
            if fl[2]:
                if self.toc_native:
                    dt_h = TimeOfContactNative.apply(dt_, p_try, new_v, geo, self.step_forces(), st.mass, toc_mask,
                                                     cs.body)
                else:
                    dt_h = self._time_of_contact(dt_, p_try, new_v, geo, cs, toc_mask.bool())
                p_redo = ops.integrate(st.p, new_v, dt_h, toc_now)
                tn = toc_now.bool()
                p_try = torch.where(tn[:, None, None], p_redo, p_try)
                self.last_dt = torch.where(tn, dt_h, self.last_dt)
                self._any_toc_flag = True
            self.toc_flag = toc_flag

        # commit accepted worlds (the non-differentiable part of the merge already happened in the kernel)
        a3 = accept.bool()[:, None, None]
        st.p = torch.where(a3, p_try, st.p)
        st.v = torch.where(a3, new_v, st.v)
        self.contact_geo = torch.where(a3, geo, self.contact_geo)
        self.contact_set = cs
        self.t = t_new
        if self.post_stab:
            self._post_stabilize(accept, dt_try)
        return accept, dt_next, active_next, int(fl[1])

    def _post_stabilize(self, accept, dt):
        """world.py:358-370 for the worlds whose sub-step was just accepted: half of the engine's stabilising displacement is
        applied as a velocity over the sub-step's dt, the velocities are restored, the contacts are detected again."""
        st = self.state
        dp = self.engine.post_stabilization(self)
        p_ps = ops.integrate(st.p, dp / 2, dt, accept)
        while True:
            cs = self.contact_set.clone()
            self.detector.detect(p_ps.detach(), self.shape, cs, accept, eps=self.eps, tol=self.tol,
                                 fd_eps=Defaults3D.EPSILON, body_eps=self.body_eps, detach_b2=self.detach_contact_b2)
            am = accept.bool()
            over = int((torch.where(am, cs.status, torch.zeros_like(cs.status)) & 3).max())          # capK / maxc overflow
            if not over:
                break
            self._grow_capacity(over)
        geo = differentiable_geometry(p_ps, self.shape, cs, self.table, Defaults3D.EPSILON, self.detach_contact_b2,
                                      self.shape_t, self.vert_leaves)
        a3 = am[:, None, None]
        st.p = torch.where(a3, p_ps, st.p)
        self.contact_geo = torch.where(a3, geo, self.contact_geo)
        self.contact_set = cs
        self.max_nc = max(int(self.max_nc), int(cs.count.max()))

    MAX_CAPK, MAX_MAXC = 1024, 512     # candidate list: shared memory of the contact kernel; contacts: tape / workspace sizes

    def _next_capacity(self, bits):
        """(capK, maxc) after an overflow: bit 0 doubles the candidate capacity (capK), bit 1 the contact capacity
        (maxc).  Raises when one of them is already at its limit.  Both step loops grow through this rule."""
        capK, maxc = self.detector.capK, self.maxc
        if bits & 1:
            if capK >= self.MAX_CAPK:
                raise RuntimeError('contact candidate capacity exceeded at the kernel limit capK=%d (mesh too fine '
                                   'for the one-CTA-per-world contact kernel)' % capK)
            capK = min(self.MAX_CAPK, 2 * capK)
        if bits & 2:
            if maxc >= self.MAX_MAXC:
                raise RuntimeError('more than %d contacts in one world: beyond the dynamics kernel limit' % maxc)
            maxc = min(self.MAX_MAXC, 2 * maxc)
        return capK, maxc

    def _grow_capacity(self, bits):
        """Grow the capacity after an overflow (_next_capacity), with the world's contact set and geometry."""
        capK, maxc = self._next_capacity(bits)
        if maxc != self.maxc:
            self.contact_set = self.contact_set.resized(maxc)
            pad = self.contact_geo.new_zeros(self.W, maxc - self.maxc, 10)
            self.contact_geo = torch.cat([self.contact_geo, pad], 1)
        self._set_capacity(capK, maxc)

    def _set_capacity(self, capK, maxc):
        self.maxc = maxc
        self.detector = ContactDetector(self.table, self.pairs, self.W, self.nb, self.device, capK=capK, maxc=maxc,
                                        record_prefilter=self.detector.record_prefilter)

    def _time_of_contact(self, dt_, p_try, new_v, geo, cs, toc_mask):
        """Gather of world.py:275-327 (padded to maxc) + the H function, evaluated only for the worlds that have a new
        contact (a handful per step); every other world keeps its dt_ (H is the identity in value)."""
        st = self.state
        C = self.maxc
        idx = toc_mask.any(1).nonzero().squeeze(1)                # host sync; this branch is rare
        T = idx.numel()
        sel = lambda x: x.index_select(0, idx)
        body = sel(cs.body)
        i1 = body[..., 0].long().clamp(0, self.nb - 1)
        i2 = body[..., 1].long().clamp(0, self.nb - 1)

        def per_contact(x, ii):
            return torch.gather(x, 1, ii[..., None].expand(T, C, x.shape[-1]))

        new_v_s, p_try_s, geo_s, dt_s = sel(new_v), sel(p_try), sel(geo), sel(dt_)
        v1, v2 = per_contact(new_v_s, i1), per_contact(new_v_s, i2)
        pp1, pp2 = per_contact(p_try_s, i1), per_contact(p_try_s, i2)
        f = self.apply_forces(self.t)
        acc = sel(f) / sel(st.mass)[..., None]
        a1, a2 = per_contact(acc, i1), per_contact(acc, i2)
        h = dt_s[:, None, None]
        x1 = pp1[..., 4:] - h * v1[..., 3:]
        x2 = pp2[..., 4:] - h * v2[..., 3:]
        R1 = so3_exponential_map(-h * v1[..., :3]) @ quaternion_to_matrix(pp1[..., :4])
        R2 = so3_exponential_map(-h * v2[..., :3]) @ quaternion_to_matrix(pp2[..., :4])
        n, c1, c2 = geo_s[..., 0:3], geo_s[..., 3:6], geo_s[..., 6:9]
        c1 = (R1.transpose(-1, -2) @ c1[..., None])[..., 0]
        c2 = (R2.transpose(-1, -2) @ c2[..., None])[..., 0]
        n2 = (R2.transpose(-1, -2) @ n[..., None])[..., 0]
        dt_h = TimeOfContact.apply(dt_s, sel(toc_mask).to(F64), c1, c2, v1, v2, x1, x2, R1, R2, n2, a1, a2)
        return dt_.index_copy(0, idx, dt_h)
