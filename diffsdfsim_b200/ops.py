"""Thin wrappers over the C-ABI kernels (pointer marshalling only, no arithmetic): torch.autograd functions, and the
plain backward calls they share with the reverse sweep of the device step loop (stepper.py)."""
import torch

from . import _lib

F64 = torch.float64
BASE_TOL = 1e-6      # lcp_physics/physics/utils.py:43 -- the TOL read by World.H.backward (world.py:204)
KIND = {'box': 0, 'sphere': 1, 'cylinder': 2, 'grid': 3, 'box_rounded': 4, 'brick': 5, 'bowl': 6}


def _c(t):
    return t.contiguous() if t is not None else None


class _SdfQuery(torch.autograd.Function):
    """SDF3D.query_sdfs (bodies.py:721-760): pts (W,N,3) -> sdf (W,N), dir (W,N,3)."""

    @staticmethod
    def forward(ctx, pts, shape, grid, kind, want_dir, extra=(0.0, 0.0)):
        L = _lib.lib()
        _lib.require_cuda(pts, shape)
        pts, shape = _c(pts), _c(shape)
        W, N = pts.shape[0], pts.shape[1]
        res, stride = 0, 0
        if kind == 3:
            grid = _c(grid)
            res = grid.shape[-1]
            assert grid.dim() == 3 or grid.shape[0] == W, 'grid must be (R,R,R) shared or (W,R,R,R) per world'
            stride = res ** 3 if grid.dim() == 4 else 0
        sdf = torch.empty(W, N, dtype=F64, device=pts.device)
        d = torch.empty(W, N, 3, dtype=F64, device=pts.device) if want_dir else None
        rc = _lib.call('dsdf_sdf_query', kind, _lib.ptr(shape), float(extra[0]), float(extra[1]),
                       _lib.ptr(grid) if kind == 3 else None, res, stride, _lib.ptr(pts), W, N, int(want_dir), _lib.ptr(sdf),
                       _lib.ptr(d), _lib.stream())
        _lib.check(rc, 'dsdf_sdf_query')
        ctx.save_for_backward(pts, shape, grid if kind == 3 else pts.new_empty(0))
        ctx.meta = (kind, res, stride, want_dir, extra)
        if want_dir:
            return sdf, d
        ctx.mark_non_differentiable()
        return sdf, pts.new_empty(0)

    @staticmethod
    def backward(ctx, gsdf, gdir):
        L = _lib.lib()
        pts, shape, grid = ctx.saved_tensors
        kind, res, stride, want_dir, extra = ctx.meta
        W, N = pts.shape[0], pts.shape[1]
        gpts = torch.empty_like(pts)
        gdir = _c(gdir) if (want_dir and gdir is not None and gdir.numel()) else None
        gsdf = _c(gsdf)                  # contiguous copies stay bound to locals until the launch has been enqueued
        rc = _lib.call('dsdf_sdf_query_backward', kind, _lib.ptr(shape), float(extra[0]), float(extra[1]),
                       _lib.ptr(grid) if kind == 3 else None, res, stride, _lib.ptr(pts), W, N, _lib.ptr(gsdf), _lib.ptr(gdir),
                       _lib.ptr(gpts), _lib.stream())
        _lib.check(rc, 'dsdf_sdf_query_backward')
        return gpts, None, None, None, None, None


def sdf_query(kind, shape, pts, grid=None, want_dir=True, extra=(0.0, 0.0)):
    """kind: 'box'|'sphere'|'cylinder'|'grid'|'box_rounded'|'brick'|'bowl' (or int); shape (W,4); pts (W,N,3);
    grid (W,R,R,R) or (R,R,R); extra: the kind's further parameters (rounded box / brick: r / scale)."""
    k = KIND[kind] if isinstance(kind, str) else int(kind)
    sdf, d = _SdfQuery.apply(pts, shape, grid, k, want_dir, tuple(extra))
    return (sdf, d) if want_dir else sdf


class _Integrate(torch.autograd.Function):
    """Body3D.move (bodies.py:488-496) for all worlds/bodies: p (W,nb,7), v (W,nb,6), dt (W)."""

    @staticmethod
    def forward(ctx, p, v, dt, active):
        L = _lib.lib()
        _lib.require_cuda(p, v, dt)
        p, v, dt = _c(p), _c(v), _c(dt)
        W, nb = p.shape[0], p.shape[1]
        out = torch.empty_like(p)
        rc = _lib.call('dsdf_integrate', _lib.ptr(p), _lib.ptr(v), _lib.ptr(dt), _lib.ptr(active), W, nb, _lib.ptr(out),
                              _lib.stream())
        _lib.check(rc, 'dsdf_integrate')
        ctx.save_for_backward(p, v, dt, active if active is not None else p.new_empty(0))
        return out

    @staticmethod
    def backward(ctx, g):
        p, v, dt, active = ctx.saved_tensors
        return integrate_backward(p, v, dt, active if active.numel() else None, g) + (None,)


def integrate(p, v, dt, active=None):
    """active: optional uint8 (W) mask; inactive worlds pass their pose through."""
    return _Integrate.apply(p, v, dt, active)


def integrate_backward(p, v, dt, active, g):
    """dsdf_integrate_backward: (gp, gv, gdt) for dL/d(integrate) = g; gdt (W) is summed over the bodies."""
    W, nb = p.shape[0], p.shape[1]
    gp, gv = torch.empty_like(p), torch.empty_like(v)
    gdt = torch.empty(W, nb, dtype=F64, device=p.device)
    g = _c(g)
    rc = _lib.call('dsdf_integrate_backward', _lib.ptr(p), _lib.ptr(v), _lib.ptr(dt), _lib.ptr(active), W, nb,
                   _lib.ptr(g), _lib.ptr(gp), _lib.ptr(gv), _lib.ptr(gdt), _lib.stream())
    _lib.check(rc, 'dsdf_integrate_backward')
    return gp, gv, gdt.sum(1)


def toc_backward(dt, toc_mask, body, p, v, geo, f, mass, gh):
    """dsdf_toc_backward: the backward of World.H and its gather (world.py:141-237, 275-327) for all worlds, given
    dL/dh = gh.  Returns (g_dt, gp, gv, ggeo, gf, gmass); worlds without a new contact pass gh through to g_dt."""
    W, nb, maxc = p.shape[0], p.shape[1], geo.shape[1]
    # contiguous copies stay bound to locals until the launch has been enqueued
    dt, toc_mask, body, p, v, geo, f, mass, gh = [_c(t) for t in (dt, toc_mask, body, p, v, geo, f, mass, gh)]
    g_dt, gp, gv = torch.empty_like(dt), torch.empty_like(p), torch.empty_like(v)
    ggeo, gf, gm = torch.empty_like(geo), torch.empty_like(f), torch.empty_like(mass)
    rc = _lib.call('dsdf_toc_backward', W, nb, maxc, _lib.ptr(dt), _lib.ptr(toc_mask), _lib.ptr(body), _lib.ptr(p),
                   _lib.ptr(v), _lib.ptr(geo), _lib.ptr(f), _lib.ptr(mass), _lib.ptr(gh), BASE_TOL, _lib.ptr(g_dt),
                   _lib.ptr(gp), _lib.ptr(gv), _lib.ptr(ggeo), _lib.ptr(gf), _lib.ptr(gm), _lib.stream())
    _lib.check(rc, 'dsdf_toc_backward')
    return g_dt, gp, gv, ggeo, gf, gm


def dynamics_workspace(W, nb, neq, fric_dirs, small, large, force_cta, device):
    """(kernel launches, one-CTA workspace or None) of one dsdf_dynamics_solve / dsdf_dynamics_solve_backward call
    with contact-count classes ``small`` and ``large``."""
    n, nbytes = _lib.dynamics_plan(W, nb, neq, fric_dirs, small, large, force_cta)
    return n, (torch.empty(nbytes // 8 + 1, dtype=F64, device=device) if nbytes else None)


def dynamics_solve_backward(p, v, mass, Ibody, fric, rest, f, dt, active, count, body, geo, eq_rows, small, large,
                            force_cta, fric_dirs, stop_contact_grad, stop_friction_grad, x, lam, s, gnv):
    """dsdf_dynamics_solve_backward with the classes (``small``, ``large``, ``force_cta``) of the forward solve.
    Returns (gp, gv, gmass, gIbody, gfric, grest, gf, gdt, ggeo)."""
    W, nb = p.shape[0], p.shape[1]
    neq, maxc = eq_rows.shape[0], geo.shape[1]
    gnv = _c(gnv)
    gp, gv = torch.empty_like(p), torch.empty_like(v)
    gmass, gI = torch.empty_like(mass), torch.empty_like(Ibody)
    gfric, grest, gf = torch.empty_like(fric), torch.empty_like(rest), torch.empty_like(f)
    gdt, ggeo = torch.empty(W, dtype=F64, device=p.device), torch.empty_like(geo)
    n, ws = dynamics_workspace(W, nb, neq, fric_dirs, small, large, force_cta, p.device)
    rc = _lib.call('dsdf_dynamics_solve_backward', _lib.ptr(p), _lib.ptr(v), _lib.ptr(mass), _lib.ptr(Ibody),
                   _lib.ptr(fric), _lib.ptr(rest), _lib.ptr(f), _lib.ptr(dt), _lib.ptr(active), _lib.ptr(count),
                   _lib.ptr(body), _lib.ptr(geo), _lib.ptr(eq_rows), W, nb, neq, maxc, small, large, int(force_cta),
                   fric_dirs, int(stop_contact_grad), int(stop_friction_grad), _lib.ptr(x), _lib.ptr(lam), _lib.ptr(s),
                   _lib.ptr(gnv), _lib.ptr(gp), _lib.ptr(gv), _lib.ptr(gmass), _lib.ptr(gI), _lib.ptr(gfric),
                   _lib.ptr(grest), _lib.ptr(gf), _lib.ptr(gdt), _lib.ptr(ggeo), _lib.ptr(ws), _lib.stream(), kernels=n)
    _lib.check(rc, 'dsdf_dynamics_solve_backward')
    return gp, gv, gmass, gI, gfric, grest, gf, gdt, ggeo


def filter_contacts(normals, p1, eps=1e-3, count=None):
    """``_filter_contacts`` (sdf_physics/physics3d/contacts.py:97-158) on the device, batched: normals, p1 (W,K,3) (or (K,3)),
    ``count`` (W) valid rows per list (default: all K).  Returns the boolean keep mask (W,K) (the reference returns the
    kept indices cluster by cluster; the SET is the same) and the per-list status bits."""
    _lib.require_cuda(normals, p1)
    single = normals.dim() == 2
    if single:
        normals, p1 = normals[None], p1[None]
    W, K = normals.shape[0], normals.shape[1]
    # work-buffer capacity: the device 3-D hull needs capK >= 2 x the largest cluster (dsdf_contacts.cu hull3d_vertices)
    capK = min(1024, max(32, (2 * K + 3) // 4 * 4))
    if K > capK:
        raise ValueError('filter_contacts: at most 1024 contacts per list')
    pad = lambda t: torch.cat([t, t.new_zeros(W, capK - K, 3)], 1).contiguous() if capK != K else t.contiguous()
    nrm, pts = pad(normals.detach().double()), pad(p1.detach().double())
    n = (torch.full((W,), K, dtype=torch.int32, device=nrm.device) if count is None else count.to(torch.int32).contiguous())
    keep = torch.zeros(W, capK, dtype=torch.int32, device=nrm.device)
    status = torch.zeros(W, dtype=torch.int32, device=nrm.device)
    rc = _lib.call('dsdf_filter_contacts', _lib.ptr(nrm), _lib.ptr(pts), _lib.ptr(n), W, capK, float(eps), _lib.ptr(keep),
                   _lib.ptr(status), _lib.stream())
    _lib.check(rc, 'dsdf_filter_contacts')
    mask = keep[:, :K].bool()
    return (mask[0], status[0]) if single else (mask, status)
