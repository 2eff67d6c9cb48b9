"""Scene specifications (pure data) for the BASELINE.json configurations.

A spec is a plain dict so the same scene can be instantiated by the product
(``build_world``), by the CPU oracle (oracle/scenes.py) and -- in the build
container only -- by the unmodified reference (tests/golden/make_golden.py).

Scene shapes follow the reference experiments:
* box_on_plane      experiments/system_identification/optim_sysid.py:105-131  (config 2 / 5)
* bouncing_sphere   experiments/trajectory_fitting/optim_sphere.py:78-111      (config 1)
* grid_on_pole      demos/demo_meshsdf.py:121-142                              (config 4)
"""
import math

import numpy as np

EPS = 1e-3


def body(kind, pos, *, dims=None, rad=None, height=None, grid=None, scale=None, vel=(0, 0, 0, 0, 0, 0),
         mass=1.0, restitution=0.5, fric_coeff=0.9, pinned=False, gravity=False, ext_force=None,
         ext_until=None, max_tri_length=0.1, mesh=None):
    return dict(kind=kind, pos=list(pos), dims=dims, rad=rad, height=height, grid=grid, scale=scale,
                vel=list(vel), mass=mass, restitution=restitution, fric_coeff=fric_coeff, pinned=pinned,
                gravity=gravity, ext_force=ext_force, ext_until=ext_until, max_tri_length=max_tri_length,
                mesh=mesh)


def scene(bodies, *, no_contact=(), axis_locks=(), dt=1.0 / 30, eps=EPS, tol=1e-8, fric_dirs=8,
          strict_no_penetration=True, time_of_contact_diff=True, steps=10, post_stab=False, grippers=()):
    return dict(post_stab=post_stab, grippers=[tuple(g) for g in grippers], bodies=bodies, no_contact=list(no_contact), axis_locks=list(axis_locks), dt=dt, eps=eps,
                tol=tol, fric_dirs=fric_dirs, strict_no_penetration=strict_no_penetration,
                time_of_contact_diff=time_of_contact_diff, steps=steps)


def make_bodies(spec, device=None, params=None, W=1):
    """Instantiate the product's bodies for a spec.  ``params`` may override, for the LAST body, 'mass' (W,),
    'pos' (W,3|7), 'vel' (W,6), 'push' (W,2) and, for all bodies, 'fric_coeff' (W,) -- mirroring how the
    reference experiments parametrise their scenes (optim_sysid.py:105-131).  Returns (bodies, constraints)."""
    import torch
    from . import bodies as B, constraints as C, forces as Fo, meshes
    params = params or {}
    out, cons = [], []
    n = len(spec['bodies'])
    for i, b in enumerate(spec['bodies']):
        last = i == n - 1
        vel = params['vel'] if (last and 'vel' in params) else b['vel']
        mass = params['mass'] if (last and 'mass' in params) else b['mass']
        if 'vel_all' in params:                    # (W,nb,6) / (W,nb): per-world initial velocities / masses of EVERY body
            vel = params['vel_all'][:, i]
        if 'mass_all' in params:
            mass = params['mass_all'][:, i]
        kw = dict(vel=vel, mass=mass,
                  restitution=b['restitution'],
                  fric_coeff=params['fric_coeff'] if 'fric_coeff' in params else b['fric_coeff'], device=device)
        pos = params['pos'] if (last and 'pos' in params) else b['pos']
        k = b['kind']
        if k == 'box':
            dims = params['dims'] if (last and 'dims' in params) else b['dims']
            ob = B.SDFBox(pos, dims, max_tri_length=b['max_tri_length'], **kw)
        elif k == 'sphere':
            rad = params['rad'] if (last and 'rad' in params) else b['rad']      # (W,) / scalar tensor: radius fitting
            ob = B.SDFSphere(pos, rad, subdivisions=(b['mesh'] or {}).get('subdivisions', 4), **kw)
        elif k == 'cylinder':
            ob = B.SDFCylinder(pos, b['rad'], b['height'], max_tri_length=b['max_tri_length'], **kw)
        elif k in ('box_rounded', 'brick'):
            ob = (B.SDFBoxRounded if k == 'box_rounded' else B.SDFBrick)(pos, b['dims'], b['rad'], mesh=extra_kind_mesh(b), **kw)
        elif k == 'bowl':
            ob = B.SDFBowl(pos, b['rad'], b['height'], mesh=extra_kind_mesh(b), **kw)
        elif k == 'grid':
            grid, mesh = grid_array(b), grid_mesh(b)
            if last and 'grid' in params:          # per-world grids (W,R,R,R) and, optionally, per-world vertices
                grid = params['grid']
                if 'verts' in params:
                    mesh = (params['verts'], params.get('faces', mesh[1]))
                    if 'nverts' in params:             # per-world topologies, padded to common sizes
                        mesh = mesh + (params['nverts'], params['nfaces'])
            inertia = params['inertia'] if (last and 'inertia' in params) else grid_unit_inertia(b)
            ob = B.SDFGrid3D(pos, b['scale'], grid, mesh, inertia=inertia, **kw)
        else:
            raise ValueError(k)
        if b['gravity']:
            ob.add_force(Fo.Gravity3D())
        if b['ext_force'] is not None:
            f = torch.tensor(b['ext_force'], dtype=torch.float64, device=ob.p.device)
            if last and 'push' in params:
                push = params['push']
                z = push.new_zeros(push.shape[0])
                f = torch.stack([z, z, z, push[:, 0], z + float(b['ext_force'][4]), push[:, 1]], 1)
            ob.add_force(Fo.ExternalForce3D(Fo.constant_force(f, b['ext_until']), multiplier=1.0))
        out.append(ob)
        if b['pinned']:
            cons.append(C.TotalConstraint3D(ob))
    for i, j in spec['no_contact']:
        out[i].add_no_contact(out[j])
    axis_cls = {3: C.XConstraint, 4: C.YConstraint, 5: C.ZConstraint}
    for i, a in spec['axis_locks']:
        cons.append(axis_cls[a](out[i]))
    for i1, i2, axis in spec.get('grippers', ()):
        cons.append(C.GripperJoint(out[i1], out[i2], axis))
    return out, cons


def build_world(spec, device=None, params=None, **world_kw):
    """World3D for a spec (batched when any parameter carries a leading world dimension)."""
    from .world import World3D
    bodies, cons = make_bodies(spec, device, params)
    kw = dict(dt=spec['dt'], eps=spec['eps'], tol=spec['tol'], fric_dirs=spec['fric_dirs'],
              strict_no_penetration=spec['strict_no_penetration'],
              time_of_contact_diff=spec['time_of_contact_diff'], post_stab=spec.get('post_stab', False))
    kw.update(world_kw)
    kw.setdefault('device', device)
    return World3D(bodies, cons, **kw)


def box_on_plane(floor=(20.0, 1.0, 20.0), box=(1.0, 1.0, 1.0), mass=1.0, fric=0.2, push=(3.0, 2.0),
                 restitution=0.5, tilt=0.0, gap=2 * EPS, steps=30, toc=True, floor_tri=0.1):
    """Box resting ``gap`` above a pinned floor slab, pushed along x,z (system-identification shape)."""
    h = box[1] / 2 + gap
    pos = [0.0, h, 0.0]
    if tilt:
        # rotate about z by ``tilt``: q = (cos t/2, 0, 0, sin t/2); lift so the lowest corner keeps the gap
        c, s = math.cos(tilt / 2), math.sin(tilt / 2)
        lift = (abs(math.sin(tilt)) * box[0] + abs(math.cos(tilt)) * box[1]) / 2 + gap
        pos = [c, 0.0, 0.0, s, 0.0, lift, 0.0]
    return scene([
        body('box', [0, -floor[1] / 2, 0], dims=list(floor), pinned=True, fric_coeff=fric,
             restitution=restitution, max_tri_length=floor_tri),
        body('box', pos, dims=list(box), mass=mass, fric_coeff=fric, restitution=restitution, gravity=True,
             ext_force=[0, 0, 0, push[0], 0, push[1]]),
    ], strict_no_penetration=False, time_of_contact_diff=toc, steps=steps)


def gripper_pair(steps=8):
    """Two boxes coupled by a GripperJoint (sdf_physics/physics3d/constraints.py:148-195): the large one rests on a pinned
    floor, the small one hangs beside it, may only slide along the large one's x axis and is pushed along x (free) and z
    (transmitted through the joint).  11 equality rows (6 pin + 5 joint), contacts between floor and large box."""
    return scene([
        body('box', [0, -0.5, 0], dims=[4.0, 1.0, 4.0], pinned=True, fric_coeff=0.2, restitution=0.2, max_tri_length=0.25),
        body('box', [0, 0.5 + 2 * EPS, 0], dims=[1.0, 1.0, 1.0], mass=1.0, fric_coeff=0.2, restitution=0.2, gravity=True),
        body('box', [1.4, 0.9, 0], dims=[0.5, 0.5, 0.5], mass=0.4, fric_coeff=0.2, restitution=0.2, gravity=True,
             ext_force=[0, 0, 0, 1.5, 0, 0.8]),
    ], no_contact=[(1, 2)], grippers=[(1, 2, (1.0, 0.0, 0.0))], strict_no_penetration=False, steps=steps)


def bouncing_sphere(rad=0.5, height=1.0, vel=(0, 0, 0, 2.0, 0, 0), floor=(20.0, 1.0, 20.0), steps=20,
                    toc=True, floor_tri=0.1, gravity=True, subdivisions=4):
    return scene([
        body('box', [0, -floor[1] / 2, 0], dims=list(floor), pinned=True, fric_coeff=0.25, restitution=0.5,
             max_tri_length=floor_tri),
        body('sphere', [0, height, 0], rad=rad, vel=list(vel), fric_coeff=0.25, restitution=0.5,
             gravity=gravity, mesh=dict(subdivisions=subdivisions)),
    ], time_of_contact_diff=toc, steps=steps)


def mixed_primitives(floor=(6.0, 1.0, 6.0), floor_tri=0.3, steps=8, toc=True, subdivisions=3):
    """Sphere, box and cylinder falling onto a pinned floor and onto each other (trajectory-fitting shape, config 3:
    several mixed primitives per world, every body pair searched).  The LAST body (cylinder) takes the per-world
    parameters ('mass', 'vel')."""
    q = [math.cos(math.pi / 4), math.sin(math.pi / 4), 0.0, 0.0]       # cylinder axis (local z) -> world -y
    return scene([
        body('box', [0, -floor[1] / 2, 0], dims=list(floor), pinned=True, fric_coeff=0.4, restitution=0.3,
             max_tri_length=floor_tri),
        body('sphere', [-0.55, 0.45, 0.0], rad=0.4, vel=[0, 0, 0, 0.3, 0, 0], fric_coeff=0.4, restitution=0.3,
             gravity=True, mesh=dict(subdivisions=subdivisions)),
        body('box', [0.5, 0.35, 0.05], dims=[0.6, 0.6, 0.6], fric_coeff=0.4, restitution=0.3, gravity=True,
             max_tri_length=0.15),
        body('cylinder', q + [0.05, 1.15, 0.0], rad=0.25, height=0.6, vel=[0, 0, 0, 0, -1.0, 0], fric_coeff=0.4,
             restitution=0.3, gravity=True, max_tri_length=0.15),
    ], time_of_contact_diff=toc, steps=steps)


def inertia_fitting(dims=(1.0, 0.5, 0.25), torque=(1.0, 0.5, 0.25), until=0.3, mass=1.0, steps=20):
    """One box whose translation is locked by X/Y/Z constraints, spun up by a torque for t < until (inertia-fitting
    shape of the scaling sweep, config 5: experiments/inertia_fitting/optim_primitives.py:97-117).  No contacts:
    nz = 6, neq = 3."""
    return scene([body('box', [0.0, 0.0, 0.0], dims=list(dims), mass=mass, ext_force=list(torque) + [0.0, 0.0, 0.0],
                       ext_until=until)],
                 axis_locks=[(0, 3), (0, 4), (0, 5)], steps=steps, time_of_contact_diff=False)


_GRID_CACHE = {}


def extra_kind_mesh(b, res=64):
    """(verts, faces) of a rounded box / brick / bowl body spec: iso-surface of its sampled SDF (memoised); the sampling
    resolution comes from the spec's mesh=dict(res=...)."""
    from . import bodies as B
    res = (b.get('mesh') or {}).get('res', res)
    key = ('xmesh', b['kind'], tuple(b['dims'] or ()), b['rad'], b['height'], res)
    if key not in _GRID_CACHE:
        if b['kind'] == 'bowl':
            r, d = float(b['rad']), float(b['height'])
            sc = (r + d) * 1.3333
            shape, extra = [r / sc, d / sc, 0.0], (0.0, 0.0)
        else:
            dims, r = np.asarray(b['dims'], dtype=np.float64), float(b['rad'])
            sc = dims.max() * 1.5 / 2
            shape = ((dims - 2 * r) / sc if b['kind'] == 'box_rounded' else dims / sc).tolist()
            extra = (r / sc, 0.0)
        _GRID_CACHE[key] = B._sampled_mesh(b['kind'], shape, extra, sc, res)
    return _GRID_CACHE[key]


def grid_array(b):
    """(R,R,R) float64 samples of a grid body's SDF: an explicit array, or a recipe dict(res, kind, seed)."""
    g = b['grid']
    if not isinstance(g, dict):
        return np.asarray(g, dtype=np.float64)
    key = (g['res'], g['kind'], g.get('seed', 0))
    if key not in _GRID_CACHE:
        _GRID_CACHE[key] = baked_grid(*key)
    return _GRID_CACHE[key]


def grid_mesh(b):
    """(verts, faces) of a grid body in its body frame: the iso-surface of its own grid (mesh=dict(kind='isosurface'),
    what the reference extracts with marching cubes, bodies.py:652-712) or an icosphere of the given radius."""
    m = b['mesh']
    if m.get('kind') == 'isosurface':
        from . import meshes
        g = b['grid']
        key = ('mesh', id(g) if not isinstance(g, dict) else (g['res'], g['kind'], g.get('seed', 0)), float(b['scale']))
        hit = _GRID_CACHE.get(key)
        if hit is None or (not isinstance(g, dict) and hit[2] is not g):
            v, f = meshes.surface_nets(grid_array(b))
            hit = (v * float(b['scale']), f, g)
            _GRID_CACHE[key] = hit
        return hit[0], hit[1]
    from . import meshes
    return meshes.icosphere(m['radius'], m.get('subdivisions', 3))


def grid_unit_inertia(b):
    """Unit-mass body-frame inertia of a grid body: volume integrals of its mesh (bodies.py:380-395) for iso-surface
    meshes, the solid-sphere closed form for the icosphere stand-ins."""
    m = b['mesh']
    if m.get('kind') == 'isosurface':
        from . import meshes
        return meshes.mesh_inertia(*grid_mesh(b))
    return 2 / 5 * m['radius'] ** 2 * np.eye(3)


def baked_grid(res=32, kind='ellipsoid', seed=0):
    """A res^3 float64 SDF grid on [-1,1]^3 standing in for a decoded IGR latent (no checkpoints offline).
    kind 'igr': a seeded random-init IGR-style decoder sampled on the lattice (igr.py)."""
    if kind == 'igr':
        from . import igr
        return igr.random_shape_grid(seed, res)
    t = np.linspace(-1.0, 1.0, res)
    X, Y, Z = np.meshgrid(t, t, t, indexing='ij')
    if kind == 'sphere':
        return np.sqrt(X * X + Y * Y + Z * Z) - 0.6
    rng = np.random.RandomState(seed)
    a = 0.45 + 0.25 * rng.rand(3)
    # first-order ellipsoid distance: smooth, sign-correct, |grad| ~ 1 near the surface
    k0 = np.sqrt((X / a[0]) ** 2 + (Y / a[1]) ** 2 + (Z / a[2]) ** 2)
    k1 = np.sqrt((X / a[0] ** 2) ** 2 + (Y / a[1] ** 2) ** 2 + (Z / a[2] ** 2) ** 2)
    return np.where(k1 > 1e-9, k0 * (k0 - 1.0) / np.maximum(k1, 1e-9), -a.min())


def grid_on_pole(res=32, floor=(10.0, 1.0, 10.0), drop=2.62, steps=12, floor_tri=0.25, with_floor=True):
    """Grid-SDF body falling on a pinned cylinder pole ('cow on pole' shape, demos/demo_meshsdf.py:121-142)."""
    bodies = []
    if with_floor:
        bodies.append(body('box', [0, -floor[1] / 2, 0], dims=list(floor), pinned=True, fric_coeff=0.15,
                           restitution=0.0, max_tri_length=floor_tri))
    q = [math.cos(math.pi / 4), math.sin(math.pi / 4), 0.0, 0.0]   # euler (pi/2,0,0): local z -> world -y.. up/down
    bodies.append(body('cylinder', q + [0.35, 1.0, 0.0], rad=0.2, height=2.0, pinned=True, fric_coeff=0.15,
                       restitution=0.0))
    bodies.append(body('grid', [0.0, drop, 0.0], grid=dict(res=res, kind='sphere'), scale=1.0, fric_coeff=0.15,
                       restitution=0.0, gravity=True, mesh=dict(subdivisions=3, radius=0.6)))
    nc = [(0, 1)] if with_floor else []
    return scene(bodies, no_contact=nc, steps=steps)


def cow_on_pole(grid=None, res=64, seed=0, floor=(50.0, 1.0, 50.0), floor_tri=0.1, scale=2.0, drop=6.0, steps=33):
    """BASELINE config 4 as the reference demo builds it (demos/demo_meshsdf.py:121-142, TIME = 1.1 s = 33 steps):
    pinned 50x1x50 floor, pinned pole SDFCylinder((pi/2,0,0, 0.35,1,0), r 0.2, h 2) with add_no_contact(pole, floor),
    and a grid-SDF body of scale 2 dropped from [0,6,0] (friction 0.15, restitution 0) whose res^3 grid is baked from a
    seeded random-init IGR-style decoder (igr.py) -- or handed in as ``grid`` -- and whose mesh is that grid's iso-surface.
    The demo's loss is |pos - [0, 0.64, 0]|^2 after the rollout (:88)."""
    q = [math.cos(math.pi / 4), math.sin(math.pi / 4), 0.0, 0.0]
    g = grid if grid is not None else dict(res=res, kind='igr', seed=seed)
    return scene([
        body('box', [0, -floor[1] / 2, 0], dims=list(floor), pinned=True, fric_coeff=0.15, restitution=0.0,
             max_tri_length=floor_tri),
        body('cylinder', q + [0.35, 1.0, 0.0], rad=0.2, height=2.0, pinned=True, fric_coeff=0.15, restitution=0.5),
        body('grid', [0.0, drop, 0.0], grid=g, scale=scale, fric_coeff=0.15, restitution=0.0, gravity=True,
             mesh=dict(kind='isosurface')),
    ], no_contact=[(0, 1)], steps=steps)


def mixed16(seed=0, steps=12, spacing=1.3, speed=1.0, gravity=False, subdivisions=3, tri=0.15):
    """BASELINE config 3 shape: 16 mixed primitives per world -- spheres r in [0.2,0.5], boxes dims in [0.3,0.8],
    cylinders r in [0.2,0.4], h in [0.4,0.8] (SURVEY.md s8d C3) -- on a jittered 4 x 2 x 2 lattice inside a ~4 m cube
    with random velocities ~ N(0, speed), free-floating (no gravity), colliding with each other.  The 16 shapes are drawn
    once per seed (meshes shared by all worlds); per-world parameters are the masses / initial velocities handed to
    make_bodies.  Every one of the 120 body pairs is a candidate (broad phase + both search directions)."""
    rng = np.random.RandomState(seed)
    bodies = []
    for i in range(16):
        ix, iy, iz = i % 4, (i // 4) % 2, i // 8
        pos = (np.array([ix - 1.5, iy - 0.5, iz - 0.5]) * spacing + 0.08 * (rng.rand(3) - 0.5)).tolist()
        vel = [0.0, 0.0, 0.0] + (speed * rng.randn(3)).tolist()
        kw = dict(vel=vel, fric_coeff=0.3, restitution=0.5, gravity=gravity, mass=float(0.5 + rng.rand()))
        kind = i % 3
        if kind == 0:
            bodies.append(body('sphere', pos, rad=float(0.2 + 0.3 * rng.rand()), mesh=dict(subdivisions=subdivisions), **kw))
        elif kind == 1:
            bodies.append(body('box', pos, dims=(0.3 + 0.5 * rng.rand(3)).tolist(), max_tri_length=tri, **kw))
        else:
            a = rng.rand() * math.pi
            q = [math.cos(a / 2), math.sin(a / 2), 0.0, 0.0]
            bodies.append(body('cylinder', q + pos, rad=float(0.2 + 0.2 * rng.rand()), height=float(0.4 + 0.4 * rng.rand()),
                               max_tri_length=tri, **kw))
    return scene(bodies, steps=steps)


def per_world_grid_bodies(W, res=64, seed0=0, scale=2.0, device=None, latent_scale=0.15):
    """Per-world geometry of ``W`` config-4 bodies: W seeded random-init IGR-style decoders baked to (W,res,res,res) grids,
    the iso-surface mesh of each grid (vertex / face arrays padded to the largest, true counts alongside) and the
    unit-mass inertia of each mesh.  Returns the ``params`` entries make_bodies understands for the LAST body:
    grid, verts, faces, nverts, nfaces, inertia (torch tensors on ``device``)."""
    import torch
    from . import igr, meshes
    grids, vs, fs, Is = [], [], [], []
    for w in range(W):
        seed = seed0 + w
        while True:                      # a fresh decoder occasionally has no zero level set, or one that leaves the grid
            g = igr.random_shape_grid(seed, res, latent_scale=latent_scale, device=device or 'cpu')
            ga = np.asarray(g)
            # closed surface strictly inside the grid: the field is positive on all six boundary faces (a level set clipped
            # by the grid gives an open mesh around a body whose SDF says "inside" at the cube wall -- not a valid body)
            wall = min(ga[0].min(), ga[-1].min(), ga[:, 0].min(), ga[:, -1].min(), ga[:, :, 0].min(), ga[:, :, -1].min())
            try:
                v, f = meshes.surface_nets(g) if wall > 0.02 else (None, [])
            except AssertionError:
                f = []
            if len(f) >= 200:
                break
            seed += 100003
        v = v * scale
        grids.append(g)
        vs.append(v)
        fs.append(f)
        Is.append(meshes.mesh_inertia(v, f))
    V, F = max(v.shape[0] for v in vs), max(f.shape[0] for f in fs)
    verts = np.zeros((W, V, 3))
    faces = np.zeros((W, F, 3), dtype=np.int32)
    for w in range(W):
        verts[w, :vs[w].shape[0]] = vs[w]
        faces[w, :fs[w].shape[0]] = fs[w]
    t = lambda a, dt=torch.float64: torch.as_tensor(np.asarray(a), dtype=dt, device=device)
    return dict(grid=t(np.stack(grids)), verts=t(verts), faces=t(faces, torch.int32),
                nverts=t([v.shape[0] for v in vs], torch.int32), nfaces=t([f.shape[0] for f in fs], torch.int32),
                inertia=t(np.stack(Is)))


def mixed16_floor(seed=0, steps=6, spacing=1.5, floor=(8.0, 1.0, 8.0), floor_tri=0.25, subdivisions=3, tri=0.15, gap=0.01):
    """The gravity + floor variant of config 3 (SURVEY.md s8d C3): the 16 mixed primitives of ``mixed16`` set down on a
    pinned floor slab (4 x 4 layout, ``gap`` above it), gravity on, small random drift.  Boxes rest on 4 + 4 corner
    contacts, lying cylinders on line contacts, spheres on point contacts: ~80-100 simultaneous contacts per world
    (nz = 102, 6 equality rows) -- beyond the 64-contact cap of the one-warp dynamics kernel, so this scene runs on
    the one-CTA kernel of dsdf_dynsolve.cu.  Body 0 is the floor; per-world masses / velocities via 'mass_all' / 'vel_all' (17 rows)."""
    rng = np.random.RandomState(seed)
    bodies = [body('box', [0, -floor[1] / 2, 0], dims=list(floor), pinned=True, fric_coeff=0.3, restitution=0.2,
                   max_tri_length=floor_tri)]
    for i in range(16):
        ix, iz = i % 4, i // 4
        x, z = (ix - 1.5) * spacing + 0.05 * (rng.rand() - 0.5), (iz - 1.5) * spacing + 0.05 * (rng.rand() - 0.5)
        vel = [0.0, 0.0, 0.0] + (0.3 * rng.randn(3) * np.array([1.0, 0.0, 1.0])).tolist()
        kw = dict(vel=vel, fric_coeff=0.3, restitution=0.2, gravity=True, mass=float(0.5 + rng.rand()))
        kind = i % 3
        if kind == 0:
            r = float(0.2 + 0.3 * rng.rand())
            bodies.append(body('sphere', [x, r + gap, z], rad=r, mesh=dict(subdivisions=subdivisions), **kw))
        elif kind == 1:
            d = (0.3 + 0.5 * rng.rand(3)).tolist()
            bodies.append(body('box', [x, d[1] / 2 + gap, z], dims=d, max_tri_length=tri, **kw))
        else:
            r, h = float(0.2 + 0.2 * rng.rand()), float(0.4 + 0.4 * rng.rand())
            bodies.append(body('cylinder', [x, r + gap, z], rad=r, height=h, max_tri_length=tri, **kw))   # axis = z: lying
    return scene(bodies, steps=steps)


def rounded_box_on_plane(kind='box_rounded', dims=(0.8, 0.5, 0.6), r=0.1, floor=(4.0, 1.0, 4.0), push=(3.0, 2.0), fric=0.2,
                         gap=2 * EPS, steps=6, floor_tri=0.2, mesh_res=28):
    """A rounded box (or brick) -- sdf_physics/physics3d/bodies.py:856-886 -- resting ``gap`` above a pinned floor, pushed
    along x, z; its mesh is the iso-surface of its own sampled SDF."""
    return scene([
        body('box', [0, -floor[1] / 2, 0], dims=list(floor), pinned=True, fric_coeff=fric, restitution=0.5,
             max_tri_length=floor_tri),
        body(kind, [0.0, dims[1] / 2 + gap, 0.0], dims=list(dims), rad=r, fric_coeff=fric, restitution=0.5, gravity=True,
             ext_force=[0, 0, 0, push[0], 0, push[1]], mesh=dict(res=mesh_res)),
    ], strict_no_penetration=False, steps=steps)
