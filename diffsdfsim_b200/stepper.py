"""Host side of the device-resident step loop (csrc/dsdf_steploop.cu): buffers, burst launches, tape, reverse sweep.

``World3D.step`` (lcp_physics/physics/world.py:119-139, 241-379) becomes ONE autograd node per step:

* forward  -- ``DeviceStepper.run`` launches rounds (prep -> solve -> move -> find_contacts -> commit) in bursts; the
  per-world accept / reject / halve / remaining-time / time-of-contact decisions are taken on the device; the host reads
  one 64-byte control block per burst (normally once per step).  Accepted sub-steps are recorded on a TAPE
  (``dsdf_step_slot``): slot k holds the k-th accepted sub-step of every world in this step.
* backward -- ``_StepFn.backward`` walks the tape slots in reverse and chains the hand-written VJP kernels
  (time-of-contact -> contact geometry -> integrator -> implicit LCP backward) with per-world masks; no autograd graph
  is recorded per round and rejected attempts leave no trace, exactly as in the reference (world.py:344-356 restores
  the state before retrying).
"""
import ctypes
import time

import torch

from . import _lib, ops
from .contacts import ContactSet, geometry_vjp, scatter_vertex_grads

F64 = torch.float64
U8 = torch.uint8
I32 = torch.int32

MAX_SLOTS = 64
STEP_CAPK, STEP_MAXC, STEP_DYN_SMEM, STEP_TAPE, STEP_MAX_ROUNDS = 1, 2, 4, 8, 16
CT_ABORT, CT_NACT, CT_MAXCOUNT, CT_ROUNDS, CT_MAXNSUB, CT_ANYTOC, CT_LCPSTAT, CT_MAXCLEAN = 0, 1, 3, 4, 5, 8, 9, 13
CT_CONSTAT = 14
CT_SLOTROWS, CT_WORDS = 16, 16 + MAX_SLOTS
CON_HULL3D, CON_STALLED = 4, 16
LCP_FACTOR_FAIL, LCP_INACCURATE, LCP_TOO_LARGE = 4, 8, 16

_SLOT_FIELDS = ['world', 'p_in', 'v_in', 'x', 'new_v', 'p_try', 'dt_raw', 'dt_used', 'lam', 's', 'toc_flag_in', 'toc_now',
                'toc_mask', 'count_in', 'body_in', 'geo_in', 'count', 'body', 'face', 'abc', 'geo']
_INT_FIELDS = ['W', 'nb', 'neq', 'maxc', 'fric_dirs', 'capK', 'npairs', 'depth', 'spec_threshold', 'depth2',
               'spec_threshold2', 'vcap', 'n_slots', 'slots_final',
               'max_iter', 'max_rounds', 'strict', 'toc_enabled', 'fixed_dt', 'detach_b2', 'force_cta']
_DBL_FIELDS = ['world_dt', 'eps', 'tol', 'fd_eps', 'body_eps']
_PTR_FIELDS = ['geom', 'pairs', 'eq_rows', 'mass', 'Ibody', 'fric', 'rest', 'f', 'shape',
               'p', 'v', 't', 'dt_try', 'end_t', 'last_dt', 'active', 'toc_flag', 'had', 'nsub', 'attempts',
               'count', 'status', 'body', 'face', 'abc', 'geo',
               'vmap', 'vidx', 'dt_raw_v', 'dt_used_v',
               'x_v', 'new_v_v', 'nu_v', 'lam_v', 's_v', 'p_try_v', 'lcp_status_v', 'iters_v',
               'count_v', 'status_v', 'body_v', 'face_v', 'abc_v', 'geo_v', 'dyn_ws', 'ctrl']


class StepSlot(ctypes.Structure):
    """dsdf_step_slot (include/dsdf_b200.h)."""
    _fields_ = [('cap', ctypes.c_int64)] + [(n, ctypes.c_void_p) for n in _SLOT_FIELDS]


class StepArgs(ctypes.Structure):
    """dsdf_step_args (include/dsdf_b200.h): every field 8 bytes wide, same order."""
    _fields_ = ([(n, ctypes.c_int64) for n in _INT_FIELDS] + [(n, ctypes.c_double) for n in _DBL_FIELDS]
                + [(n, ctypes.c_void_p) for n in _PTR_FIELDS] + [('slots', ctypes.c_void_p)])


def _ptr(t):
    return None if t is None else _lib.ptr(t)


class TapeSlot:
    """Device buffers of one dsdf_step_slot: ``cap`` self-contained rows (one accepted sub-step of one world each)."""
    F64_FIELDS = dict(p_in=('nb', 7), v_in=('nb', 6), p_try=('nb', 7), x=('nz',), new_v=('nb', 6), dt_raw=(), dt_used=(),
                      lam=('ni',), s=('ni',), geo_in=('maxc', 10), abc=('maxc', 3), geo=('maxc', 10))
    I32_FIELDS = dict(world=(), count_in=(), body_in=('maxc', 2), count=(), body=('maxc', 2), face=('maxc',))
    U8_FIELDS = dict(toc_flag_in=(), toc_now=(), toc_mask=('maxc',))

    def __init__(self, cap, nb, maxc, per, dev):
        self.cap, self.nb, self.maxc, self.per, self.dev = int(cap), nb, maxc, per, dev
        self.rows = 0                                   # rows in use (set from the control block after the step)
        dims = dict(nb=nb, nz=6 * nb, ni=maxc * per, maxc=maxc)
        for fields, dt in ((self.F64_FIELDS, F64), (self.I32_FIELDS, I32), (self.U8_FIELDS, U8)):
            for name, shape in fields.items():
                setattr(self, name, torch.empty((self.cap,) + tuple(dims.get(d, d) for d in shape), dtype=dt, device=dev))
        self.nbytes = sum(getattr(self, n).numel() * getattr(self, n).element_size()
                          for n in list(self.F64_FIELDS) + list(self.I32_FIELDS) + list(self.U8_FIELDS))

    def regrown(self, cap, maxc):
        """The same rows in a slot with room for ``cap`` rows of ``maxc`` contacts."""
        n = acquire_slot(cap, self.nb, maxc, self.per, self.dev)
        r, m, per = min(self.cap, cap), self.maxc, self.per
        for name in list(self.F64_FIELDS) + list(self.I32_FIELDS) + list(self.U8_FIELDS):
            src, dst = getattr(self, name), getattr(n, name)
            if name in ('lam', 's'):
                dst[:r, :m * per] = src[:r]
            elif src.dim() >= 2 and src.shape[1] == m and name not in ('p_in', 'v_in', 'p_try', 'x', 'new_v'):
                dst[:r, :m] = src[:r]
            else:
                dst[:r] = src[:r]
        if maxc != m:
            n.toc_mask[:r, m:] = 0
        n.rows = self.rows
        release_slot(self)
        return n

    def fill(self, c_slot):
        c_slot.cap = self.cap
        for k in _SLOT_FIELDS:
            setattr(c_slot, k, _ptr(getattr(self, k)))

    def view(self, n):
        """The first n rows as a namespace of tensors (what the reverse sweep of this slot reads)."""
        v = _Rows()
        for name in list(self.F64_FIELDS) + list(self.I32_FIELDS) + list(self.U8_FIELDS):
            setattr(v, name, getattr(self, name)[:n])
        v.maxc = self.maxc
        return v


class _Rows:
    pass


def _pow2(n):
    return 1 << max(0, int(n) - 1).bit_length()


# Tape slots are recycled: a rollout allocates tens of them per step and frees them all after backward; handing the
# whole group of buffers back and forth costs nothing, whereas the caching allocator fragments on their varying sizes
# (cudaMalloc in steady state).  Keyed by everything that determines the buffer shapes.
_SLOT_POOL = {}
_SLOT_POOL_MAX_BYTES = 48 << 30
_slot_pool_bytes = 0


def acquire_slot(cap, nb, maxc, per, dev):
    global _slot_pool_bytes
    key = (int(cap), nb, maxc, per, str(dev))
    free = _SLOT_POOL.get(key)
    if free:
        sl = free.pop()
        _slot_pool_bytes -= sl.nbytes
        sl.rows = 0
        return sl
    return TapeSlot(cap, nb, maxc, per, dev)


def clear_slot_pool():
    """Drop every recycled tape slot (their memory returns to the caching allocator)."""
    global _slot_pool_bytes
    _SLOT_POOL.clear()
    _slot_pool_bytes = 0


def release_slot(sl):
    global _slot_pool_bytes
    if _slot_pool_bytes + sl.nbytes > _SLOT_POOL_MAX_BYTES:
        return
    _SLOT_POOL.setdefault((sl.cap, sl.nb, sl.maxc, sl.per, str(sl.dev)), []).append(sl)
    _slot_pool_bytes += sl.nbytes


class Tape:
    """Everything one step leaves behind for its reverse sweep."""
    __slots__ = ('slots', 'maxsub', 'any_toc', 'maxc', 'C', 'rounds', 'p_out', 'v_out', 'geo_out',
                 'last_dt_out', 'had', 'final', 'f', 'syncs')

    def __del__(self):
        for sl in getattr(self, 'slots', None) or []:
            release_slot(sl)


_ROWS_HISTORY = {}       # (W, nb, fric_dirs, device) -> high-water mark of the rows used per tape slot


class DeviceStepper:
    """Owns the per-world work buffers of the step loop of one ``World3D`` and launches its rounds."""
    INITIAL_SLOTS = 2
    TIMING = None           # set to {} to accumulate host wall-clock seconds per phase of run() (diagnostics)
    FORCE_CTA = False       # tests: run every world through the one-CTA dynamics kernel
    # speculative halving (W >= 64): the retries dt, dt/2, ... of the few still-active worlds run in ONE round as virtual
    # worlds, the first accepted attempt in the reference's order wins (step_prep_kernel / step_commit_kernel).
    # False: one halving per round, the same results in more rounds.
    SPECULATE = True
    SPEC_DEPTH = 3          # halvings tried at once when <= W/8 worlds are still active
    SPEC_DEPTH2 = 6         # ... when <= W/32 worlds are still active

    @classmethod
    def _tick(cls, name, t0):
        if cls.TIMING is not None:
            cls.TIMING[name] = cls.TIMING.get(name, 0.0) + time.perf_counter() - t0
        return time.perf_counter()

    def __init__(self, world):
        _lib.lib()
        self.W, self.nb, self.dev = world.W, world.nb, world.device
        W, dev = self.W, self.dev
        self.depth = self.SPEC_DEPTH if self.SPECULATE else 1
        self.spec_threshold = W // 8 if (self.SPECULATE and W >= 64) else 0
        # second level: when hardly any world is left, try six halvings at once (a world that ends up giving up at
        # dt / 2^10 then needs two rounds instead of four)
        self.depth2 = self.SPEC_DEPTH2 if (self.SPECULATE and self.SPEC_DEPTH2 > self.depth) else 0
        self.spec_threshold2 = W // 32 if (self.depth2 and W >= 64) else 0
        self.vcap = max(W, self.depth * self.spec_threshold, self.depth2 * self.spec_threshold2)
        self.ctrl = torch.zeros(CT_WORDS, dtype=I32, device=dev)
        self.ctrl_host = torch.zeros(CT_WORDS, dtype=I32).pin_memory()
        self.slot_table = torch.zeros(MAX_SLOTS * ctypes.sizeof(StepSlot), dtype=U8, device=dev)
        self.dt_try = torch.zeros(W, dtype=F64, device=dev)
        self.end_t = torch.zeros(W, dtype=F64, device=dev)
        self.active = torch.zeros(W, dtype=U8, device=dev)
        self.nsub = torch.zeros(W, dtype=I32, device=dev)
        self.vidx = torch.zeros(W, dtype=I32, device=dev)
        self.maxc = None
        self.last_rounds = 1
        self.max_count = 0          # largest accepted contact count so far (any state)
        self.max_clean = 0          # ... of non-penetrating states: what the bulk of the worlds look like
        self.launches = 0
        self._alloc_virtual(world)

    def _alloc_virtual(self, world):
        V, nb, dev = self.vcap, self.nb, self.dev
        per = 2 + world.fric_dirs
        self.maxc = world.maxc
        e = lambda *s: torch.empty(*s, dtype=F64, device=dev)
        self.vmap = torch.zeros(V, dtype=I32, device=dev)
        self.dt_raw_v, self.dt_used_v = e(V), e(V)
        self.x_v, self.new_v_v, self.p_try_v = e(V, 6 * nb), e(V, 6 * nb), e(V, nb * 7)
        self.nu_v = e(V, max(world.num_constraints, 1))
        self.lam_v, self.s_v = e(V, self.maxc * per), e(V, self.maxc * per)
        self.lcp_status_v = torch.zeros(V, dtype=I32, device=dev)
        self.iters_v = torch.zeros(V, dtype=I32, device=dev)
        self.cs_v = ContactSet(V, self.maxc, dev)
        # workspace of the one-CTA dynamics kernel, if some world may run on it (csrc/dsdf_dynsolve.cu)
        self.force_cta = bool(self.FORCE_CTA)
        _, self.dyn_ws = ops.dynamics_workspace(V, nb, world.num_constraints, world.fric_dirs, self.maxc, self.maxc,
                                                self.force_cta, dev)

    # ------------------------------------------------------------------------------------------------------------
    def _args(self, world, fixed_dt, st, tape, f):
        a = StepArgs()
        a.W, a.nb, a.neq, a.maxc, a.fric_dirs = self.W, self.nb, world.num_constraints, world.maxc, world.fric_dirs
        a.capK, a.npairs = world.detector.capK, world.detector.npairs
        a.depth, a.spec_threshold, a.vcap, a.n_slots = self.depth, self.spec_threshold, self.vcap, len(tape.slots)
        a.depth2, a.spec_threshold2 = self.depth2, self.spec_threshold2
        a.slots_final = int(len(tape.slots) >= MAX_SLOTS)
        a.max_iter, a.max_rounds = world.engine.max_iter, world.max_rounds_per_step
        a.strict, a.toc_enabled = int(world.strict_no_pen), int(world.time_of_contact_diff)
        a.fixed_dt, a.detach_b2 = int(fixed_dt), int(world.detach_contact_b2)
        a.world_dt, a.eps, a.tol, a.fd_eps, a.body_eps = float(world.dt), world.eps, world.tol, 1e-3, world.body_eps
        a.geom, a.pairs, a.eq_rows = world.table.ptr(), _ptr(world.detector.pairs), _ptr(world.eq_rows)
        a.mass, a.Ibody, a.fric, a.rest = _ptr(st['mass']), _ptr(st['Ibody']), _ptr(st['fric']), _ptr(st['rest'])
        a.f, a.shape = _ptr(f), _ptr(world.shape)
        a.p, a.v, a.t, a.dt_try, a.end_t = _ptr(st['p']), _ptr(st['v']), _ptr(st['t']), _ptr(self.dt_try), _ptr(self.end_t)
        a.last_dt, a.active, a.toc_flag, a.had = _ptr(st['last_dt']), _ptr(self.active), _ptr(st['toc_flag']), _ptr(st['had'])
        a.nsub, a.attempts = _ptr(self.nsub), _ptr(world.stats['attempts'])
        cur = st['cur']
        a.count, a.status, a.body, a.face, a.abc, a.geo = (_ptr(cur.count), _ptr(cur.status), _ptr(cur.body),
                                                           _ptr(cur.face), _ptr(cur.abc), _ptr(cur.geo))
        a.vmap, a.vidx, a.dt_raw_v, a.dt_used_v = _ptr(self.vmap), _ptr(self.vidx), _ptr(self.dt_raw_v), _ptr(self.dt_used_v)
        a.x_v, a.new_v_v, a.nu_v, a.lam_v, a.s_v = (_ptr(self.x_v), _ptr(self.new_v_v), _ptr(self.nu_v), _ptr(self.lam_v),
                                                    _ptr(self.s_v))
        a.p_try_v, a.lcp_status_v, a.iters_v = _ptr(self.p_try_v), _ptr(self.lcp_status_v), _ptr(self.iters_v)
        v = self.cs_v
        a.count_v, a.status_v, a.body_v, a.face_v, a.abc_v, a.geo_v = (_ptr(v.count), _ptr(v.status), _ptr(v.body),
                                                                       _ptr(v.face), _ptr(v.abc), _ptr(v.geo))
        a.force_cta, a.dyn_ws = int(self.force_cta), _ptr(self.dyn_ws)
        a.ctrl = _ptr(self.ctrl)
        # the slot table lives in device memory (no limit from the kernel-parameter space); uploaded when it changes
        table = (StepSlot * len(tape.slots))()
        for k, s in enumerate(tape.slots):
            s.fill(table[k])
        raw = torch.frombuffer(bytearray(bytes(table)), dtype=U8)
        self.slot_table[:raw.numel()].copy_(raw)
        a.slots = _ptr(self.slot_table)
        return a

    def _smem_contacts(self, world):
        """Contacts the dynamics kernel sizes its shared memory for, as two classes (small, large): the bulk of the
        worlds (largest non-penetrating count so far + slack) and, if there are any, the few worlds that carry many more
        (a world that gave up halving keeps a penetrating state with dozens of contacts)."""
        r4 = lambda c: max(4, min((c + 2 + 3) // 4 * 4, world.maxc))
        small, large = r4(self.max_clean), r4(self.max_count)
        return small, (large if large > small else small)

    def _hist_key(self, world):
        return (self.W, self.nb, world.fric_dirs, str(self.dev))

    def _slot_cap(self, k, hist=()):
        """Rows to allocate for tape slot k: every world reaches slot 0; later slots hold the high-water mark of earlier
        steps of worlds of this size (rollouts are repeated every optimisation iteration), rounded up to a power of two
        so that recycled slots fit."""
        if k == 0:
            return self.W
        seen = hist[k] if k < len(hist) else 0
        return min(self.W, _pow2(max(64, seen + seen // 4)))

    def _read_ctrl(self):
        self.ctrl_host.copy_(self.ctrl, non_blocking=True)
        torch.cuda.current_stream().synchronize()
        return self.ctrl_host.tolist()

    def run(self, world, fixed_dt, p, v, last_dt, mass, Ibody, fric, rest, f):
        """One World3D.step for all worlds.  Returns the Tape (which carries the new state)."""
        W, nb, dev = self.W, self.nb, self.dev
        per = 2 + world.fric_dirs
        if self.maxc != world.maxc:
            self._alloc_virtual(world)
        if self.max_count == 0:                             # the contacts World3D.__init__ found (a legal, clean state)
            self.max_clean = int(world.max_nc)
        self.max_count = max(self.max_count, self.max_clean, int(world.max_nc))
        t0 = time.perf_counter()
        tape = Tape()
        hist = _ROWS_HISTORY.get(self._hist_key(world), [])
        tape.slots = [acquire_slot(self._slot_cap(k, hist), nb, world.maxc, per, dev)
                      for k in range(max(self.INITIAL_SLOTS, len(hist)))]
        tape.f = f
        t0 = self._tick('slots', t0)
        st = dict(p=p.detach().clone(), v=v.detach().clone(), t=world.t.clone(), last_dt=last_dt.detach().clone(),
                  toc_flag=world.toc_flag.clone(), had=torch.zeros(W, dtype=U8, device=dev),
                  cur=world.contact_set.clone(), mass=mass, Ibody=Ibody, fric=fric, rest=rest)
        st['cur'].pre_ids = st['cur'].pre_cnt = None
        stream = _lib.stream()
        t0 = self._tick('state', t0)
        args = self._args(world, fixed_dt, st, tape, f)
        t0 = self._tick('args', t0)
        _lib.check(_lib.call('dsdf_step_begin', ctypes.byref(args), stream), 'dsdf_step_begin')
        burst = min(max(2, self.last_rounds + 1), 24)
        syncs = 0
        while True:
            small, large = self._smem_contacts(world)
            n_dyn, _ = _lib.dynamics_plan(self.vcap, nb, world.num_constraints, world.fric_dirs, small, large,
                                          self.force_cta)
            nk = burst * (4 + n_dyn)                         # kernels of this burst
            rc = _lib.call('dsdf_step_rounds', ctypes.byref(args), burst, small, large, stream, kernels=nk)
            _lib.check(rc, 'dsdf_step_rounds')
            self.launches += nk
            t0 = self._tick('launch', t0)
            c = self._read_ctrl()
            t0 = self._tick('sync', t0)
            syncs += 1
            self.max_count = max(self.max_count, c[CT_MAXCOUNT])
            self.max_clean = max(self.max_clean, c[CT_MAXCLEAN])
            ab = c[CT_ABORT]
            if ab & STEP_MAX_ROUNDS and not world.strict_no_pen:
                # the reference would go on sub-stepping at dt / 2^10; leave these worlds where they are (reported)
                world.stats['stalled'] = world.stats.get('stalled', 0) + int(c[CT_NACT])
                self.active.zero_()
                break
            if ab & STEP_MAX_ROUNDS:
                raise world._incomplete_step_error(self.active, self.dt_try)
            if ab:
                self._grow(world, ab, tape, st, per, c)
                args = self._args(world, fixed_dt, st, tape, f)
                _lib.check(_lib.call('dsdf_step_resume', ctypes.byref(args), stream), 'dsdf_step_resume')
                t0 = self._tick('grow', t0)
                continue
            if c[CT_NACT] == 0:
                break
            burst = min(2 * burst, 32)
        self.last_rounds = c[CT_ROUNDS]
        ls = c[CT_LCPSTAT]
        if ls & LCP_TOO_LARGE:
            raise _lib.DsdfLibraryError('dynamics kernel: a world had more contacts than its shared memory holds')
        world.engine.last_status_bits = ls
        if c[CT_CONSTAT] & CON_STALLED:
            world.stats['stalled'] = world.stats.get('stalled', 0) + 1
        if c[CT_CONSTAT] & CON_HULL3D:
            # contacts.py:126-152 runs a 3-D Qhull on such clusters; so does the device filter (hull3d_vertices) unless the
            # cluster is larger than its work buffers (8 m <= 4 capK), in which case every point of the cluster is kept
            world.stats['hull3d_steps'] = world.stats.get('hull3d_steps', 0) + 1
            if world.stats['hull3d_steps'] == 1:
                import warnings
                warnings.warn('a non-planar contact cluster was too large for the device 3-D hull and was kept unfiltered '
                              '(DSDF_CON_HULL3D); raise capK to at least twice the cluster size')
        if ls & LCP_INACCURATE and getattr(world.engine, 'verbose', -1) >= 0:
            print('qpth warning: Returning an inaccurate and potentially incorrect solution.')       # batch.py:165,229
        tape.maxsub, tape.any_toc = c[CT_MAXNSUB], bool(c[CT_ANYTOC])
        tape.maxc, tape.C, tape.rounds, tape.syncs = world.maxc, self._smem_contacts(world) + (self.force_cta,), c[CT_ROUNDS], syncs
        tape.p_out, tape.v_out, tape.last_dt_out, tape.had = st['p'], st['v'], st['last_dt'], st['had'].bool()
        tape.final = st['cur']
        tape.geo_out = st['cur'].geo.clone()
        world.t, world.toc_flag = st['t'], st['toc_flag']
        for sl in tape.slots[max(tape.maxsub, 0):]:
            release_slot(sl)
        del tape.slots[max(tape.maxsub, 0):]
        for k, sl in enumerate(tape.slots):
            sl.rows = min(c[CT_SLOTROWS + k], sl.cap)
        hist = _ROWS_HISTORY.setdefault(self._hist_key(world), [])
        for k, sl in enumerate(tape.slots):
            if k >= len(hist):
                hist.append(sl.rows)
            hist[k] = max(hist[k], sl.rows)
        self._tick('finish', t0)
        return tape

    def _grow(self, world, bits, tape, st, per, c):
        """Enlarge what the paused worlds ran out of (the worlds themselves are untouched and still active)."""
        if bits & (STEP_CAPK | STEP_MAXC):
            capK, maxc = world._next_capacity(bits)          # STEP_CAPK / STEP_MAXC are its bits 0 / 1
            world._set_capacity(capK, maxc)
            if bits & STEP_MAXC:
                st['cur'] = st['cur'].resized(maxc)
                tape.slots = [sl.regrown(sl.cap, maxc) for sl in tape.slots]
                self._alloc_virtual(world)
        if bits & STEP_TAPE:
            # a paused world found its slot missing or full: double the full slots (their row counters overshot by the
            # number of paused worlds: clamp them), and add slots up to the deepest sub-step index seen + 1
            rows = list(c[CT_SLOTROWS:CT_SLOTROWS + MAX_SLOTS])
            for k, sl in enumerate(tape.slots):
                if k > 0 and rows[k] > sl.cap:
                    if sl.cap >= self.W:
                        raise RuntimeError('tape slot %d holds every world and is still full' % k)
                    # rows[k] worlds asked for a row so far: make room for them and as many again
                    tape.slots[k] = sl.regrown(min(self.W, _pow2(2 * rows[k])), world.maxc)
                    rows[k] = sl.cap
            self.ctrl[CT_SLOTROWS:CT_SLOTROWS + MAX_SLOTS].copy_(torch.tensor(rows, dtype=I32), non_blocking=False)
            if c[CT_MAXNSUB] >= len(tape.slots) and len(tape.slots) < MAX_SLOTS:
                n = min(MAX_SLOTS, max(len(tape.slots) + 2, len(tape.slots) * 3 // 2))
                tape.slots += [acquire_slot(self._slot_cap(k), self.nb, world.maxc, per, self.dev)
                               for k in range(len(tape.slots), n)]
        # STEP_DYN_SMEM needs no buffer: max_count was refreshed from the control block, so the next burst sizes the
        # dynamics launches for it (_smem_contacts)


class _StepFn(torch.autograd.Function):
    """One ``World3D.step`` of all worlds: (p, v, contact geometry, last_dt, parameters, forces) -> the same after the step.

    Per accepted sub-step (world.py:249-341), with cs_in the contacts found at the end of the previous sub-step:
        dt_    = toc_flag ? -last_dt + (last_dt.detach() + dt) : dt
        new_v  = solve(p, v, parameters, f, dt_, geo_in)                    engines.py:31-83
        p_try  = move(p, new_v, dt_)                                        bodies.py:488-496
        geo    = contact geometry(p_try)                                    contacts.py:262-264
        new contact:  dt_h = H(dt_, p_try, new_v, geo, f, mass);  p' = move(p, new_v, dt_h);  last_dt' = dt_h
        otherwise:    p' = p_try
    """

    @staticmethod
    def forward(ctx, world, fixed_dt, p, v, geo, last_dt, mass, Ibody, fric, rest, f, shape_t, *verts):
        p, v, mass, Ibody, fric, rest, f = [t.contiguous() for t in (p, v, mass, Ibody, fric, rest, f)]
        tape = world._stepper.run(world, fixed_dt, p, v, last_dt, mass, Ibody, fric, rest, f)
        ctx.tape = tape
        ctx.params = (mass, Ibody, fric, rest, f)
        ctx.geo_in_maxc = geo.shape[1]
        ctx.cfg = dict(eq_rows=world.eq_rows, fric_dirs=world.fric_dirs,
                       stop_contact_grad=world.stop_contact_grad, stop_friction_grad=world.stop_friction_grad,
                       table=world.table, shape=world.shape, detach_b2=world.detach_contact_b2,
                       want_shape=shape_t is not None,
                       leaves=[(i, vt) for i, vt in zip(world.table.vert_leaf_ids, verts)])
        world._last_tape = tape
        outs = (tape.p_out, tape.v_out, tape.geo_out, tape.last_dt_out, tape.had)
        # the tape must not keep the outputs: output -> grad_fn (this ctx) -> tape -> output would be a reference cycle
        # that only the cyclic GC frees, holding every rollout's tape alive
        tape.p_out = tape.v_out = tape.geo_out = tape.last_dt_out = tape.had = None
        ctx.mark_non_differentiable(outs[4])
        return outs

    @staticmethod
    def backward(ctx, gp, gv, ggeo, glast, _ghad):
        """Reverse sweep over the tape: slot k holds one row per world that accepted a (k+1)-th sub-step in this step, so
        slot 0 is processed in place and the later (short) slots on gathered rows of the adjoints."""
        tape, cfg = ctx.tape, ctx.cfg
        mass, Ibody, fric, rest, f = ctx.params
        W = mass.shape[0]
        maxc = tape.maxc
        small, large, force_cta = tape.C                   # the contact-count classes of the forward
        gp, gv, glast = gp.clone(), gv.clone(), glast.clone()
        if ggeo.shape[1] != maxc:
            ggeo = torch.cat([ggeo, ggeo.new_zeros(W, maxc - ggeo.shape[1], 10)], 1)
        else:
            ggeo = ggeo.clone()
        gm, gI = torch.zeros_like(mass), torch.zeros_like(Ibody)
        gfr, gre, gf = torch.zeros_like(fric), torch.zeros_like(rest), torch.zeros_like(f)
        want_shape, leaves = cfg['want_shape'] or bool(cfg['leaves']), cfg['leaves']
        gshape = torch.zeros(W, mass.shape[1], 4, dtype=F64, device=mass.device) if want_shape else None
        gverts = [torch.zeros_like(vt) for _, vt in leaves]
        for k in range(tape.maxsub - 1, -1, -1):
            n = tape.slots[k].rows
            if n == 0:
                continue
            S = tape.slots[k].view(n)
            if k == 0:
                idx = wmap = None
                a_gp, a_gv, a_ggeo, a_glast = gp, gv, ggeo, glast
                pm, pI, pfr, pre, pf = mass, Ibody, fric, rest, f
            else:
                idx = S.world.long()
                wmap = S.world
                sel = lambda t: t.index_select(0, idx)
                a_gp, a_gv, a_ggeo, a_glast = sel(gp), sel(gv), sel(ggeo), sel(glast)
                pm, pI, pfr, pre, pf = sel(mass), sel(Ibody), sel(fric), sel(rest), sel(f)
            zero_n = torch.zeros(n, dtype=F64, device=mass.device)
            gp_in_acc = gnv_acc = dgf = dgm = None
            gdt_acc, glast_pass, ggeo_tot, gptry = zero_n, a_glast, a_ggeo, a_gp
            if tape.any_toc:
                # new contacts: p' = move(p, new_v, H(dt_)); H = dsdf_toc_backward (world.py:141-237, 275-341)
                tn = S.toc_now.bool()
                gpA, gvA, gdtA = ops.integrate_backward(S.p_in, S.new_v, S.dt_used, S.toc_now, a_gp)
                gh = torch.where(tn, gdtA + a_glast, zero_n)
                g_dt_B, gp_B, gv_B, ggeo_B, gf_B, gm_B = ops.toc_backward(S.dt_used, S.toc_mask, S.body, S.p_try,
                                                                          S.new_v, S.geo, pf, pm, gh)
                tn3 = tn[:, None, None]
                gp_in_acc = torch.where(tn3, gpA, torch.zeros_like(gpA))
                gnv_acc = torch.where(tn3, gvA + gv_B, torch.zeros_like(gvA))
                gptry = torch.where(tn3, gp_B, a_gp)
                ggeo_tot = a_ggeo + torch.where(tn3, ggeo_B, torch.zeros_like(ggeo_B))
                gdt_acc = torch.where(tn, g_dt_B, zero_n)
                glast_pass = torch.where(tn, zero_n, a_glast)
                dgf = torch.where(tn3, gf_B, torch.zeros_like(gf_B))
                dgm = torch.where(tn[:, None], gm_B, torch.zeros_like(gm_B))
            gp_geo, gshape_k, gctri_k = geometry_vjp(cfg['table'], S.p_try, cfg['shape'], S.count, S.body, S.face, S.abc,
                                                     ggeo_tot, 1e-3, cfg['detach_b2'], wmap, want_shape)
            gptry = gptry + gp_geo
            if want_shape:
                if k == 0:
                    gshape += gshape_k
                else:
                    gshape.index_add_(0, idx, gshape_k)
                if leaves:
                    scatter_vertex_grads(gverts, leaves, cfg['table'], gctri_k, S.count, S.body, S.face, S.abc,
                                         None if k == 0 else idx)
            gp2, gv2, gdt2 = ops.integrate_backward(S.p_in, S.new_v, S.dt_used, None, gptry)
            gnv = a_gv + gv2 if gnv_acc is None else a_gv + gv2 + gnv_acc
            gp3, gv3, gm3, gI3, gfr3, gre3, gf3, gdt3, ggeo3 = ops.dynamics_solve_backward(
                S.p_in, S.v_in, pm, pI, pfr, pre, pf, S.dt_used, None, S.count_in, S.body_in, S.geo_in, cfg['eq_rows'],
                small, large, force_cta, cfg['fric_dirs'], cfg['stop_contact_grad'], cfg['stop_friction_grad'], S.x,
                S.lam, S.s, gnv)
            gp_new = gp2 + gp3 if gp_in_acc is None else gp2 + gp3 + gp_in_acc
            gdt_tot = gdt_acc + gdt2 + gdt3
            glast_new = glast_pass + torch.where(S.toc_flag_in.bool(), -gdt_tot, zero_n)
            if dgf is not None:
                gf3, gm3 = gf3 + dgf, gm3 + dgm
            if k == 0:
                gp, gv, ggeo, glast = gp_new, gv3, ggeo3, glast_new
                gm, gI, gfr, gre, gf = gm + gm3, gI + gI3, gfr + gfr3, gre + gre3, gf + gf3
            else:                                   # rows of one slot belong to distinct worlds: plain scatters
                gp.index_copy_(0, idx, gp_new)
                gv.index_copy_(0, idx, gv3)
                ggeo.index_copy_(0, idx, ggeo3)
                glast.index_copy_(0, idx, glast_new)
                gm.index_add_(0, idx, gm3)
                gI.index_add_(0, idx, gI3)
                gfr.index_add_(0, idx, gfr3)
                gre.index_add_(0, idx, gre3)
                gf.index_add_(0, idx, gf3)
        if ggeo.shape[1] != ctx.geo_in_maxc:
            ggeo = ggeo[:, :ctx.geo_in_maxc]
        return (None, None, gp, gv, ggeo, glast, gm, gI, gfr, gre, gf, gshape if cfg['want_shape'] else None) + tuple(gverts)
