"""SDF collision query host side: geometry table, detection launch, differentiable contact geometry.

Mirrors the reference's contact-handler plug-in (sdf_physics/physics3d/contacts.py:217-272): the class
``FWContactHandler`` (alias ``B200ContactHandler``) is what ``World3D(contact_callback=...)`` resolves by name;
in this batched implementation it detects the contacts of ALL worlds with one launch sequence instead of
being called back per body pair by py3ode.
"""
import numpy as np
import torch

from . import _lib

F64 = torch.float64
_GEOM_DTYPE = np.dtype([('kind', 'i4'), ('nverts', 'i4'), ('nfaces', 'i4'), ('res', 'i4'), ('verts', 'u8'),
                        ('faces', 'u8'), ('grid', 'u8'), ('vstride', 'i8'), ('gstride', 'i8'),
                        ('cell_lo', 'f8', (3,)), ('cell_inv', 'f8'), ('cell_dims', 'i4', (3,)), ('has_cells', 'i4'),
                        ('fcell_start', 'u8'), ('fcell_items', 'u8'), ('vcell_start', 'u8'), ('vcell_items', 'u8'),
                        ('max_face_rad', 'f8'), ('fstride', 'i8'), ('nfaces_w', 'u8'), ('nverts_w', 'u8'),
                        ('extra', 'f8', (2,))],
                       align=True)
assert _GEOM_DTYPE.itemsize == 184


_CELL_CACHE = {}


def cached_cell_index(verts_np, faces_np, device):
    """Cell index of a (shared) mesh on `device`, memoised on the mesh content (worlds are rebuilt every
    optimisation iteration with the same meshes)."""
    key = (verts_np.shape, faces_np.shape, hash(verts_np.tobytes()), hash(faces_np.tobytes()), str(device))
    hit = _CELL_CACHE.get(key)
    if hit is None:
        lo, inv, dims, fs, fi, vs, vi = build_cell_index(verts_np, faces_np)
        tri = np.asarray(verts_np, dtype=np.float64)[np.asarray(faces_np, dtype=np.int64)]
        cen = tri.mean(1, keepdims=True)
        max_rad = float(np.linalg.norm(tri - cen, axis=2).max()) * (1.0 + 1e-9)
        hit = (lo, inv, dims, [torch.from_numpy(a).to(device) for a in (fs, fi, vs, vi)], max_rad)
        if len(_CELL_CACHE) > 64:
            _CELL_CACHE.clear()
        _CELL_CACHE[key] = hit
    return hit


def build_cell_index(verts, faces, target=32, max_cells=1 << 18):
    """Uniform grid over a body-frame mesh: faces binned by centroid, vertices by position (CSR, int32).

    Cell size ~ sqrt(target * mean face area) so a cell of a surface patch holds about `target` faces.
    Returns (lo (3,), inv_h, dims (3,), fstart, fitems, vstart, vitems) as numpy arrays.
    """
    v = np.asarray(verts, dtype=np.float64)
    f = np.asarray(faces, dtype=np.int64)
    tri = v[f]
    cen = (tri[:, 0] + tri[:, 1] + tri[:, 2]) / 3.0
    area = 0.5 * np.linalg.norm(np.cross(tri[:, 1] - tri[:, 0], tri[:, 2] - tri[:, 0]), axis=1)
    h = float(np.sqrt(max(target * area.mean(), 1e-12)))
    lo = np.minimum(v.min(0), cen.min(0))
    hi = np.maximum(v.max(0), cen.max(0))
    ext = np.maximum(hi - lo, 1e-9)
    while True:
        dims = np.maximum(np.ceil(ext / h).astype(np.int64), 1)
        if dims.prod() <= max_cells:
            break
        h *= 1.5
    lo = lo - 1e-9 * (1.0 + np.abs(lo))
    inv = 1.0 / h

    def csr(pts):
        ijk = np.clip(np.floor((pts - lo) * inv).astype(np.int64), 0, dims - 1)
        cell = (ijk[:, 0] * dims[1] + ijk[:, 1]) * dims[2] + ijk[:, 2]
        order = np.argsort(cell, kind='stable')
        start = np.zeros(dims.prod() + 1, dtype=np.int64)
        np.add.at(start, cell + 1, 1)
        return np.cumsum(start).astype(np.int32), order.astype(np.int32)

    fs, fi = csr(cen)
    vs, vi = csr(v)
    return lo, inv, dims.astype(np.int32), fs, fi, vs, vi


class GeometryTable:
    """Device array of ``dsdf_body_geom`` (include/dsdf_b200.h) + the tensors it points into."""

    def __init__(self, bodies, W, device):
        self.keep = []
        rows = np.zeros(len(bodies), dtype=_GEOM_DTYPE)
        self.nfaces = []
        self.faces = []                      # per body: (F,3) or (W,F,3) int32 on the device
        self.vert_leaf_ids = [i for i, b in enumerate(bodies) if b.verts.requires_grad]
        for i, b in enumerate(bodies):
            verts = b.verts.to(device=device, dtype=F64).contiguous()
            faces = b.faces.to(device=device, dtype=torch.int32).contiguous()
            per_world = verts.dim() == 3
            if per_world:
                assert verts.shape[0] == W
            nverts = verts.shape[-2]
            # per-world topology: faces (W,F,3) padded to a common F, with the true counts per world
            fstride, nf_ptr, nv_ptr = 0, 0, 0
            if faces.dim() == 3:
                assert per_world and faces.shape[0] == W, 'per-world faces need per-world vertices'
                nf = getattr(b, 'nfaces_w', None)
                nv = getattr(b, 'nverts_w', None)
                nf = (torch.full((W,), faces.shape[1]) if nf is None else torch.as_tensor(nf)).to(device=device, dtype=torch.int32)
                nv = (torch.full((W,), nverts) if nv is None else torch.as_tensor(nv)).to(device=device, dtype=torch.int32)
                self.keep += [nf, nv]
                fstride, nf_ptr, nv_ptr = faces.shape[1] * 3, nf.data_ptr(), nv.data_ptr()
            grid = getattr(b, 'sdf_grid', None)
            res, gptr, gstride = 0, 0, 0
            if grid is not None:
                grid = grid.to(device=device, dtype=F64).contiguous()
                res = grid.shape[-1]
                gstride = res ** 3 if grid.dim() == 4 else 0
                gptr = grid.data_ptr()
                self.keep.append(grid)
            self.keep += [verts, faces]
            self.faces.append(faces)
            cell = (np.zeros(3), 0.0, np.zeros(3, dtype=np.int32), 0, 0, 0, 0, 0)
            max_rad = 0.0
            if not per_world:
                lo, inv, dims, dev_arrays, max_rad = cached_cell_index(verts.detach().cpu().numpy(), faces.cpu().numpy(),
                                                                       device)
                self.keep += dev_arrays
                cell = (lo, inv, dims, 1) + tuple(a.data_ptr() for a in dev_arrays)
            rows[i] = (b.kind, nverts, faces.shape[-2], res, verts.data_ptr(), faces.data_ptr(), gptr,
                       nverts * 3 if per_world else 0, gstride) + cell + (max_rad, fstride, nf_ptr, nv_ptr,
                                                                         tuple(getattr(b, 'sdf_extra', (0.0, 0.0))))
            self.nfaces.append(int(faces.shape[-2]))
        self.rows = rows
        self.dev = torch.from_numpy(rows.view(np.uint8).copy()).to(device)

    def ptr(self):
        return self.dev.data_ptr()


class ContactSet:
    """Contacts of all worlds after one detection pass (padded to ``maxc`` per world).

    All six arrays live in ONE flat allocation (segments 8-byte aligned) so that a copy of the whole set is a single
    device-to-device copy: count (W) i32 | status (W) i32 | body (W,maxc,2) i32 | face (W,maxc) i32 |
    abc (W,maxc,3) f64 | geo (W,maxc,10) f64.
    """
    __slots__ = ('flat', 'W', 'maxc', 'count', 'status', 'body', 'face', 'abc', 'geo', 'pre_ids', 'pre_cnt')

    def __init__(self, W, maxc, device, flat=None):
        self.W, self.maxc = W, maxc
        Wp = (W + 1) // 2 * 2                       # keep every segment 8-byte aligned
        sizes = [4 * Wp, 4 * Wp, 8 * W * maxc, 4 * Wp * maxc, 24 * W * maxc, 80 * W * maxc]
        offs = [0]
        for n in sizes:
            offs.append(offs[-1] + n)
        self.flat = torch.zeros(offs[-1], dtype=torch.uint8, device=device) if flat is None else flat
        seg = lambda i, dt: self.flat[offs[i]:offs[i + 1]].view(dt)
        self.count = seg(0, torch.int32)[:W]
        self.status = seg(1, torch.int32)[:W]
        self.body = seg(2, torch.int32).view(W, maxc, 2)
        self.face = seg(3, torch.int32)[:W * maxc].view(W, maxc)
        self.abc = seg(4, F64).view(W, maxc, 3)
        self.geo = seg(5, F64).view(W, maxc, 10)
        self.pre_ids = self.pre_cnt = None

    def resized(self, maxc):
        """The same contacts in a set of larger per-world capacity."""
        c = ContactSet(self.W, maxc, self.flat.device)
        m = self.maxc
        c.count.copy_(self.count)
        c.status.copy_(self.status)
        c.body[:, :m], c.face[:, :m], c.abc[:, :m], c.geo[:, :m] = self.body, self.face, self.abc, self.geo
        c.pre_ids, c.pre_cnt = self.pre_ids, self.pre_cnt
        return c

    def where(self, mask, other):
        """New set with the contacts of ``other`` in the worlds where ``mask`` ((W,) bool), else those of ``self``."""
        c = self.clone()
        for k in ('count', 'status', 'body', 'face', 'abc', 'geo'):
            a = getattr(c, k)
            a.copy_(torch.where(mask.reshape((-1,) + (1,) * (a.dim() - 1)), getattr(other, k), a))
        return c

    def clone(self):
        c = ContactSet(self.W, self.maxc, self.flat.device, self.flat.clone())
        if self.pre_ids is not None:
            c.pre_ids, c.pre_cnt = self.pre_ids.clone(), self.pre_cnt.clone()
        return c


class ContactDetector:
    """Owns the work buffers of ``dsdf_contacts_detect`` for one batched world."""

    def __init__(self, table, pairs, W, nb, device, capK=384, maxc=32, record_prefilter=False):
        _lib.lib()
        self.table, self.W, self.nb, self.capK, self.maxc = table, W, nb, capK, maxc
        self.npairs = len(pairs)
        self.pairs = torch.tensor(pairs, dtype=torch.int32, device=device).reshape(-1, 2).contiguous()
        self.device = device
        self.record_prefilter = record_prefilter

    def new_set(self):
        c, W, d = ContactSet(self.W, self.maxc, self.device), self.W, self.device
        if self.record_prefilter:
            c.pre_ids = torch.zeros(W, max(2 * self.npairs, 1), self.capK, dtype=torch.int32, device=d)
            c.pre_cnt = torch.zeros(W, max(2 * self.npairs, 1), dtype=torch.int32, device=d)
        return c

    def detect(self, p, shape, out, active=None, eps=1e-3, tol=1e-8, fd_eps=1e-3, body_eps=1e-3, detach_b2=False):
        """Fill ``out`` (a ContactSet) for the active worlds; values only (no autograd graph)."""
        L = _lib.lib()
        _lib.require_cuda(p, shape)
        rc = _lib.call('dsdf_contacts_detect', self.table.ptr(), _lib.ptr(self.pairs), self.npairs, _lib.ptr(p),
                       _lib.ptr(shape), _lib.ptr(active), out.W, self.nb, eps, tol, fd_eps, body_eps, int(detach_b2),
                       self.capK, self.maxc, _lib.ptr(out.count), _lib.ptr(out.body), _lib.ptr(out.face),
                       _lib.ptr(out.abc), _lib.ptr(out.geo), _lib.ptr(out.status), _lib.ptr(out.pre_ids),
                       _lib.ptr(out.pre_cnt), None, None, _lib.stream())
        _lib.check(rc, 'dsdf_contacts_detect')
        return out


def geometry_vjp(table, p, shape, count, body, face, abc, ggeo, fd_eps, detach_b2, wmap=None, want_shape=False):
    """VJP of the contact tuples [n, p1, p2, pen] (contacts.py:262-264) for a batch of rows: gp (R,nb,7) and, with
    ``want_shape``, gshape (R,nb,4) = d/d[a,b,c,scale] and gctri (R,maxc,3) = gradient w.r.t. the body-frame point
    sum(abc * face vertices) on the mesh body of each contact.  ``wmap`` (R,) int32: world of each row (None: row = world)."""
    R, nb, maxc = p.shape[0], p.shape[1], body.shape[1]
    gp = torch.empty_like(p)
    gshape = torch.empty(R, nb, 4, dtype=F64, device=p.device) if want_shape else None
    gctri = torch.empty(R, maxc, 3, dtype=F64, device=p.device) if want_shape else None
    ggeo = ggeo.contiguous()
    rc = _lib.call('dsdf_contact_geometry_backward', table.ptr(), _lib.ptr(p), _lib.ptr(shape), R, nb, fd_eps,
                   int(detach_b2), maxc, _lib.ptr(count), _lib.ptr(body), _lib.ptr(face), _lib.ptr(abc), _lib.ptr(ggeo),
                   _lib.ptr(gp), _lib.ptr(wmap), _lib.ptr(gshape), _lib.ptr(gctri), _lib.stream())
    _lib.check(rc, 'dsdf_contact_geometry_backward')
    return gp, gshape, gctri


def scatter_vertex_grads(grads, leaves, table, gctri, count, body, face, abc, worlds=None):
    """Accumulate d loss / d vertices from gctri: c_tri = sum_i abc_i * verts[faces[face, i]] on the mesh body (body[...,0])
    of every contact.  ``leaves`` = [(body index, verts tensor)], ``grads`` the matching accumulators ((V,3) shared or
    (W,V,3) per world); ``worlds`` (R,) long: world of each row (None: row = world)."""
    R, maxc = face.shape
    live = torch.arange(maxc, device=face.device)[None, :] < count[:, None].clamp(max=maxc)
    for (b, verts), g in zip(leaves, grads):
        m = live & (body[..., 0] == b)
        faces_b = table.faces[b]                                        # (F,3) shared or (W,F,3)
        fidx = face.long().clamp(min=0)
        if faces_b.dim() == 3:
            wsel = (worlds if worlds is not None else torch.arange(R, device=face.device))[:, None].expand(R, maxc)
            vids = faces_b[wsel, fidx.clamp(max=faces_b.shape[1] - 1)].long()     # (R,maxc,3)
        else:
            vids = faces_b[fidx.clamp(max=faces_b.shape[0] - 1)].long()
        contrib = abc[..., :, None] * gctri[..., None, :] * m[..., None, None].to(gctri.dtype)   # (R,maxc,3 verts,3)
        if verts.dim() == 3:                                            # per-world vertices
            V = verts.shape[1]
            wsel = (worlds if worlds is not None else torch.arange(R, device=face.device))[:, None, None]
            g.view(-1, 3).index_add_(0, (wsel * V + vids).reshape(-1), contrib.reshape(-1, 3))
        else:
            g.index_add_(0, vids.reshape(-1), contrib.reshape(-1, 3))


class _ContactGeometry(torch.autograd.Function):
    """Attach the detected contact geometry to the autograd graph of the poses (and, when they carry gradients, of the
    shape parameters and mesh vertices).

    Forward returns the values the detection pass already computed (identical arithmetic to the reference's
    second, grad-enabled ``_compute_contacts``, contacts.py:262-264); backward is its VJP.
    """

    @staticmethod
    def forward(ctx, p, shape, geo, count, body, face, abc, table, fd_eps, detach_b2, shape_t, *verts):
        ctx.save_for_backward(p, shape, count, body, face, abc)
        ctx.table, ctx.fd_eps, ctx.detach_b2 = table, fd_eps, detach_b2
        ctx.want_shape = shape_t is not None
        ctx.leaves = [(i, v) for i, v in zip(table.vert_leaf_ids, verts)]
        return geo.clone()

    @staticmethod
    def backward(ctx, ggeo):
        p, shape, count, body, face, abc = ctx.saved_tensors
        gp, gshape, gctri = geometry_vjp(ctx.table, p, shape, count, body, face, abc, ggeo, ctx.fd_eps, ctx.detach_b2,
                                         None, ctx.want_shape or bool(ctx.leaves))
        if not ctx.want_shape:
            gshape = None
        gverts = []
        if ctx.leaves:
            gverts = [torch.zeros_like(v) for _, v in ctx.leaves]
            scatter_vertex_grads(gverts, ctx.leaves, ctx.table, gctri, count, body, face, abc)
        return (gp,) + (None,) * 9 + (gshape,) + tuple(gverts)


def geo_cap(body):
    return body.shape[1]


def differentiable_geometry(p, shape, cs, table, fd_eps=1e-3, detach_b2=False, shape_t=None, verts=()):
    """(W,maxc,10) contact geometry [n,p1,p2,pen] connected to ``p`` (and to ``shape_t`` (W,nb,4) / the vertex tensors
    ``verts`` of the bodies listed in table.vert_leaf_ids, when given) for autograd."""
    return _ContactGeometry.apply(p, shape, cs.geo, cs.count, cs.body, cs.face, cs.abc, table, fd_eps, detach_b2,
                                  shape_t, *verts)


class FWContactHandler:
    """Name-compatible with sdf_physics.physics3d.contacts.FWContactHandler (contacts.py:217-272).

    ``World3D`` detects the contacts of all worlds and all body pairs with one launch (``ContactDetector``); this
    callable keeps the reference's per-pair plug-in signature ``handler(args=[world], geom1, geom2)`` (the py3ode
    callback of world.py:399) for code that drives a handler directly: it searches that one pair -- both directions,
    same kernels -- and appends the reference tuples ``((normal, p1, p2, pen), i1, i2)`` to ``world.contacts_debug``
    (and returns them).  ``geom1`` / ``geom2`` are the bodies (or their indices); ``no_contact`` is honoured
    (contacts.py:224).
    """

    def __call__(self, args, geom1, geom2):
        world = args[0]
        idx = lambda g: g if isinstance(g, int) else world.bodies.index(g)
        i1, i2 = idx(geom1), idx(geom2)
        b1, b2 = world.bodies[i1], world.bodies[i2]
        if b2 in b1.no_contact or b1 in b2.no_contact:
            return []
        with world._on_device():
            det = ContactDetector(world.table, [(min(i1, i2), max(i1, i2))], world.W, world.nb, world.device,
                                  capK=world.detector.capK, maxc=world.maxc)
            cs = det.new_set()
            det.detect(world.state.p.detach().contiguous(), world.shape, cs, None, eps=world.eps, tol=world.tol,
                       fd_eps=1e-3, body_eps=world.body_eps, detach_b2=world.detach_contact_b2)
            geo = differentiable_geometry(world.state.p, world.shape, cs, world.table, 1e-3, world.detach_contact_b2)
        out = []
        for w in range(world.W):
            lst = [((geo[w, k, 0:3], geo[w, k, 3:6], geo[w, k, 6:9], geo[w, k, 9]), int(cs.body[w, k, 0]),
                    int(cs.body[w, k, 1])) for k in range(int(cs.count[w]))]
            out.append(lst)
        res = out if world.batched else out[0]
        if not hasattr(world, 'contacts_debug'):
            world.contacts_debug = []
        world.contacts_debug += res if not world.batched else [res]
        return res


B200ContactHandler = FWContactHandler
