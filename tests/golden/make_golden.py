"""Generate golden vectors by executing the UNMODIFIED reference (build container only).

    python tests/golden/make_golden.py            # writes tests/golden/*.npz

The reference has no tests and no golden vectors of its own (SURVEY.md s4), so
the oracle is pinned against outputs of the reference itself.  The reference is
imported from /root/reference with the third-party stand-ins in
tests/golden/ref_shims on sys.path (recipe: SURVEY.md s8c); meshes / grids are
injected through the reference's own ``custom_mesh`` hook so that reference,
oracle and CUDA path all see identical geometry buffers.

/root/reference does not exist on the GPU box: this script is never run there;
its outputs are committed.
"""
import os
import sys
import warnings

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [os.path.join(HERE, 'ref_shims'), '/root/reference', ROOT]
os.environ.setdefault('IGR_PATH', HERE)
warnings.filterwarnings('ignore')

import lcp_physics.physics  # noqa: E402  (must precede lcp_physics.lcp.lcp: circular import)
import sdf_physics.physics3d.utils as u3  # noqa: E402

u3.Defaults3D.DEVICE = torch.device('cpu')
from sdf_physics.physics3d import bodies as rb, contacts as rc, forces as rf, constraints as rcon  # noqa: E402
from sdf_physics.physics3d.world import World3D  # noqa: E402
from lcp_physics.lcp.lcp import LCPFunction  # noqa: E402

from diffsdfsim_b200 import scenes  # noqa: E402
from oracle.scenes import mesh_for  # noqa: E402

F64 = torch.float64


def _inject(cls, verts, faces, inertia=None):
    v = verts if isinstance(verts, torch.Tensor) else torch.as_tensor(verts, dtype=F64)
    f = torch.as_tensor(np.asarray(faces)).long()

    class Injected(cls):
        def _custom_create_mesh(self, *a, **k):
            return v, f

        def _create_mesh(self, *a, **k):
            return v, f

    if inertia is not None:
        Injected._get_ang_inertia = lambda self, mass: inertia(mass)
    return Injected


def build_reference(spec, params=None):
    params = params or {}
    bodies, joints = [], []
    n = len(spec['bodies'])
    for i, b in enumerate(spec['bodies']):
        last = i == n - 1
        if last and 'rad' in params:
            b = dict(b, rad=params['rad'])
        mass = params['mass'] if (last and 'mass' in params) else float(b['mass'])
        if 'mass_all' in params:
            mass = params['mass_all'][i]
        fric = params['fric_coeff'] if 'fric_coeff' in params else float(b['fric_coeff'])
        verts, faces = mesh_for(b)
        pos = params['pos'] if (last and 'pos' in params) else torch.tensor(b['pos'], dtype=F64)
        vel = params['vel'] if (last and 'vel' in params) else torch.tensor(b['vel'], dtype=F64)
        if 'vel_all' in params:
            vel = params['vel_all'][i]
        kw = dict(vel=vel, mass=mass, restitution=b['restitution'], fric_coeff=fric)
        k = b['kind']
        if k == 'box':
            ob = _inject(rb.SDFBox, verts, faces)(pos, b['dims'], custom_mesh=True, custom_inertia=True, **kw)
        elif k == 'sphere':
            # (a tensor radius keeps the mesh differentiable: mesh_for returns unit icosphere * rad, as the reference's own
            # custom mesh does, bodies.py:1001-1009)
            ob = _inject(rb.SDFSphere, verts, faces)(pos, b['rad'], custom_mesh=True, custom_inertia=True, **kw)
        elif k == 'cylinder':
            ob = _inject(rb.SDFCylinder, verts, faces)(pos, b['rad'], b['height'], custom_mesh=True,
                                                       custom_inertia=True, **kw)
        elif k == 'grid':
            grid = torch.tensor(scenes.grid_array(b), dtype=F64)
            if b['mesh'].get('kind') == 'isosurface':
                # the reference integrates the inertia of the injected mesh itself (bodies.py:380-395)
                cls = _inject(rb.SDFGrid3D, verts, faces)
            else:
                r = b['mesh']['radius']
                cls = _inject(rb.SDFGrid3D, verts, faces,
                              inertia=lambda m, r=r: 2 / 5 * m * r ** 2 * torch.eye(3, dtype=F64))
            ob = cls(pos, b['scale'], grid, **kw)
        else:
            raise ValueError(k)
        if b['gravity']:
            ob.add_force(rf.Gravity3D())
        if b['ext_force'] is not None:
            f = torch.tensor(b['ext_force'], dtype=F64)
            if last and 'push' in params:
                f = torch.cat([f[:3], params['push'][0:1], f[4:5], params['push'][1:2]])
            until = b['ext_until']
            ob.add_force(rf.ExternalForce3D(lambda t, f=f, until=until: f if (until is None or t < until) else f * 0,
                                            multiplier=1.))
        bodies.append(ob)
        if b['pinned']:
            joints.append(rcon.TotalConstraint3D(ob))
    for i, j in spec['no_contact']:
        bodies[i].add_no_contact(bodies[j])
    axis_cls = {3: rcon.XConstraint, 4: rcon.YConstraint, 5: rcon.ZConstraint}
    for i, a in spec['axis_locks']:
        joints.append(axis_cls[a](bodies[i]))
    for i1, i2, axis in spec.get('grippers', ()):
        joints.append(rcon.GripperJoint(bodies[i1], bodies[i2], axis=list(axis)))
    world = World3D(bodies, joints, dt=spec['dt'], eps=spec['eps'], tol=spec['tol'], fric_dirs=spec['fric_dirs'],
                    strict_no_penetration=spec['strict_no_penetration'],
                    time_of_contact_diff=spec['time_of_contact_diff'], post_stab=spec.get('post_stab', False))
    return world


def rollout_reference(spec, params=None, target=None, record_lcp=True):
    """Step the reference, recording states, contact sets, solver attempts, one LCP instance, and the loss."""
    world = build_reference(spec, params)
    tries = [0]
    solve = world.engine.solve_dynamics

    def counted(w, dt):
        tries[0] += 1
        return solve(w, dt)

    world.engine.solve_dynamics = counted

    fw_log = []
    fw = rc._frank_wolfe

    def fw_logged(b1, b2, eps=None, tol=None):
        abc, ids = fw(b1, b2, eps, tol)
        fw_log.append((world.bodies.index(b1), world.bodies.index(b2), ids.clone()))
        return abc, ids

    rc._frank_wolfe = fw_logged

    lcps = []

    def lcp_factory(**kw):
        fn = LCPFunction(**kw)

        def call(*a):
            z = fn(*a)
            if record_lcp:
                lcps.append([t.detach().clone() for t in a] + [z.detach().clone()])
            return z
        return call

    world.engine.lcp_solver = lcp_factory

    out = dict(p=[], v=[], tries=[], nc=[], con=[], fw=[], fw_off=[0], con_off=[0])
    obj = world.bodies[-1]
    loss = 0.
    try:
        for k in range(spec['steps']):
            tries[0] = 0
            del fw_log[:]
            world.step(fixed_dt=True)
            out['p'].append(torch.cat([b.p for b in world.bodies]).detach().numpy().copy())
            out['v'].append(world.v.detach().numpy().copy())
            out['tries'].append(tries[0])
            rows = [torch.cat([c[0][0], c[0][1], c[0][2], c[0][3].reshape(1),
                               c[0][0].new_tensor([c[1], c[2]])]).detach().numpy() for c in world.contacts]
            out['con'] += rows
            out['con_off'].append(out['con_off'][-1] + len(rows))
            # pre-filter FW index sets of the LAST find_contacts of this step (the accepted one)
            n_pairs_calls = [(a, b, ids) for a, b, ids in fw_log]
            # keep only calls after the last solve: the log is cleared per step, accepted attempt = trailing calls
            out['fw'].append(n_pairs_calls)
            tgt = target if target is not None else obj.pos.new_zeros(3)
            loss = loss + ((tgt - obj.pos) ** 2).sum()
    finally:
        rc._frank_wolfe = fw
    return world, out, loss, lcps


def pack(out):
    d = dict(p=np.stack(out['p']), v=np.stack(out['v']), tries=np.asarray(out['tries']),
             con=np.stack(out['con']) if out['con'] else np.zeros((0, 12)), con_off=np.asarray(out['con_off']))
    # FW pre-filter sets: flatten (step, call#, b1, b2, face id)
    rows = []
    for s, calls in enumerate(out['fw']):
        for c, (a, b, ids) in enumerate(calls):
            for i in ids.tolist():
                rows.append((s, c, a, b, i))
    d['fw'] = np.asarray(rows, dtype=np.int64).reshape(-1, 5)
    d['fw_calls'] = np.asarray([len(c) for c in out['fw']])
    return d


def golden_scene(name, spec, leaves):
    params = {k: torch.tensor(v, dtype=F64, requires_grad=True) for k, v in leaves.items()}
    world, out, loss, lcps = rollout_reference(spec, params, record_lcp=len(spec['bodies']) <= 6)
    d = pack(out)
    d['loss'] = float(loss)
    loss.backward()
    for k, t in params.items():
        d['grad_' + k] = t.grad.numpy().copy()
        d['leaf_' + k] = t.detach().numpy().copy()
    for b, rb_ in zip(spec['bodies'], world.bodies):
        if b['kind'] == 'grid' and b['mesh'].get('kind') == 'isosurface':
            # the grid is a fixture (float32 is exact: igr.random_shape_grid rounds through it); the reference's own
            # volume-integral inertia of the injected mesh pins meshes.mesh_inertia
            d['grid_f32'] = scenes.grid_array(b).astype(np.float32)
            assert np.array_equal(d['grid_f32'].astype(np.float64), scenes.grid_array(b))
            d['ref_inertia'] = rb_.ang_inertia.detach().numpy().copy()
            d['ref_mass'] = float(rb_.mass)
    # the largest recorded LCP instance, for the operator-level golden
    if lcps:
        big = max(lcps, key=lambda a: a[2].shape[1])
        for nm, t in zip(['Q', 'p', 'G', 'h', 'A', 'b', 'F', 'z'], big):
            d['lcp_' + nm] = t.numpy()
    np.savez_compressed(os.path.join(HERE, name + '.npz'), **d)
    print(name, 'steps', len(d['tries']), 'tries', d['tries'].tolist(), 'contacts/step',
          np.diff(d['con_off']).tolist(), 'loss', d['loss'],
          {k: d['grad_' + k].tolist() for k in leaves})


from specs import SCENES, default_leaves  # noqa: E402


def golden_sdf():
    """Operator-level vectors for SDF3D.query_sdfs on each body kind (bodies.py:721-760)."""
    g = torch.Generator().manual_seed(0)
    d = {}
    spec = scenes.grid_on_pole(with_floor=True)
    world = build_reference(spec)
    box = build_reference(scenes.box_on_plane(floor=(4.0, 1.0, 4.0))).bodies[1]
    sph = build_reference(scenes.bouncing_sphere(floor=(4.0, 1.0, 4.0), floor_tri=0.5)).bodies[1]
    for nm, b in (('box', box), ('sphere', sph), ('cylinder', world.bodies[1]), ('grid', world.bodies[2])):
        s = float(b.scale)
        pts = (torch.rand(4096, 3, generator=g, dtype=F64) * 2 - 1) * s * 1.1
        # exact-zero coordinates and surface points exercise the sign(0)/tie conventions
        pts[:64] = torch.round(pts[:64] / s * 4) / 4 * s
        sd, gr = b.query_sdfs(pts)
        d[nm + '_pts'], d[nm + '_sdf'], d[nm + '_dir'] = pts.numpy(), sd.numpy(), gr.numpy()
    # rounded box / brick / bowl (bodies.py:128-200, 856-886, 1012-1026): the reference classes with an injected mesh
    from diffsdfsim_b200 import bodies as pb
    shapes = {'box_rounded': (rb.SDFBoxRounded, pb.SDFBoxRounded, ([0.8, 0.5, 0.6], 0.1)),
              'brick': (rb.SDFBrick, pb.SDFBrick, ([1.0, 0.6, 0.5], 0.1)),
              'bowl': (rb.SDFBowl, pb.SDFBowl, (0.6, 0.15))}
    for nm, (ref_cls, our_cls, args) in shapes.items():
        ours = our_cls([0.0, 0.0, 0.0], *args)                       # (mesh generator only)
        b = _inject(ref_cls, ours.verts.numpy(), ours.faces.numpy())(torch.zeros(3, dtype=F64), *args)
        s = float(b.scale)
        pts = (torch.rand(4096, 3, generator=g, dtype=F64) * 2 - 1) * s * 1.1
        pts[:64] = torch.round(pts[:64] / s * 4) / 4 * s
        sd, gr = b.query_sdfs(pts.clone())
        d[nm + '_pts'], d[nm + '_sdf'], d[nm + '_dir'] = pts.numpy(), sd.numpy(), gr.numpy()
    # the first 3072 points of each kind (the 64 tie / surface points included) keep the file under 1 MB
    np.savez_compressed(os.path.join(HERE, 'sdf_query.npz'), **{k: v[:3072] for k, v in d.items()})
    print('sdf_query', {k: v.shape for k, v in d.items()})


def reference_function(path, name, namespace):
    """Compile ONE function of a reference script without importing the script (the experiment drivers import sacred,
    tensorboard, pyrender ... at module level): the function's own source, unmodified, executed in `namespace`."""
    import ast
    src = open(os.path.join('/root/reference', path)).read()
    for node in ast.parse(src).body:
        if isinstance(node, ast.FunctionDef) and node.name == name:
            node.decorator_list = []
            mod = ast.Module(body=[node], type_ignores=[])
            exec(compile(mod, path, 'exec'), namespace)
            return namespace[name]
    raise KeyError(name)


def golden_detach_2nd_bounce():
    """The reference's own run_world_fixed_dt(detach_2nd_bounce=True) (experiments/trajectory_fitting/optim_sphere.py:
    163-177) on a bouncing sphere: final state, number of steps, gradients of |final pos|^2 + |final v|^2 w.r.t. the
    initial position and velocity (only the first contact step of every bounce is differentiated)."""
    import io, contextlib
    run = reference_function('experiments/trajectory_fitting/optim_sphere.py', 'run_world_fixed_dt', {'torch': torch})
    spec = scenes.bouncing_sphere(floor=(4.0, 1.0, 4.0), steps=0, floor_tri=0.2, height=0.75, subdivisions=3,
                                  vel=(0, 0, 0, 1.0, 0, 0.3))
    d = {}
    for flag in (False, True):
        pos = torch.tensor([0.0, 0.75, 0.0], dtype=F64, requires_grad=True)
        vel = torch.tensor([0.0, 0.0, 0.0, 1.0, 0.0, 0.3], dtype=F64, requires_grad=True)
        world = build_reference(spec, dict(pos=pos, vel=vel))
        obj = world.bodies[-1]
        terms, step = [], world.step

        def recording_step(fixed_dt=False):      # the loss is collected after every step() the reference's loop issues
            had = step(fixed_dt=fixed_dt)
            terms.append((obj.pos ** 2).sum() + 0.1 * (world.v[-6:] ** 2).sum())
            return had
        world.step = recording_step
        with contextlib.redirect_stdout(io.StringIO()):
            run(world, 0.8, detach_2nd_bounce=flag)
        loss = sum(terms)
        loss.backward()
        d[k_ := ('detach' if flag else 'plain') + '_nsteps'] = len(terms)
        k = 'detach' if flag else 'plain'
        d[k + '_p'] = torch.cat([b.p for b in world.bodies]).detach().numpy()
        d[k + '_v'] = world.v.detach().numpy()
        d[k + '_t'] = float(world.t)
        d[k + '_loss'] = float(loss)
        d[k + '_gpos'], d[k + '_gvel'] = pos.grad.numpy().copy(), vel.grad.numpy().copy()
        print('detach_2nd_bounce', flag, 't', float(world.t), 'loss', float(loss), pos.grad.tolist(), vel.grad.tolist())
    np.savez_compressed(os.path.join(HERE, 'detach_2nd_bounce.npz'), **d)


def golden_mesh_sdf():
    """The reference's own MeshSDF (SDF3D._diff_marching_cubes, bodies.py:652-704) and get_ang_inertia (:260-395), with the
    declared marching-cubes stand-in: vertices, faces, inertia, and the gradients of
    sum(w * verts) + sum(u * inertia(2 * verts, faces, 1.3)) w.r.t. the SDF parameters."""
    from specs import mesh_sdf_cases
    rng = np.random.RandomState(5)
    d = {}
    for name, fn, params, res in mesh_sdf_cases():
        ps = [q.clone().requires_grad_(True) for q in params]
        verts, faces = rb.SDF3D._diff_marching_cubes(fn, res=res)(*ps)
        w = torch.tensor(rng.randn(*verts.shape))
        u = torch.tensor(rng.randn(3, 3))
        J = rb.get_ang_inertia(verts * 2.0, faces, torch.tensor(1.3, dtype=F64))
        loss = (w * verts).sum() + (u * J).sum()
        loss.backward()
        d[name + '_verts'], d[name + '_faces'] = verts.detach().numpy(), faces.numpy()
        d[name + '_w'], d[name + '_u'], d[name + '_J'] = w.numpy(), u.numpy(), J.detach().numpy()
        d[name + '_loss'] = float(loss)
        for k, q in enumerate(ps):
            d['%s_grad%d' % (name, k)] = q.grad.numpy()
        print('mesh_sdf', name, tuple(verts.shape), tuple(faces.shape), float(loss), [q.grad.tolist() for q in ps])
    np.savez_compressed(os.path.join(HERE, 'mesh_sdf.npz'), **d)


def golden_neural_query():
    """The reference's SDF3D.query_sdfs (bodies.py:721-760) on a neural-SDF body (sdf_func = an IGR-style decoder, params =
    [latent], no closed-form gradient): values, directions, overlap mask at points in and outside the cube, and the
    gradient of the point-cloud loss sum(sdf^2) (optim_pointcloud.py:193-199) w.r.t. the latent code."""
    from diffsdfsim_b200 import igr
    dec = igr.init_decoder(seed=3, radius_init=0.6)
    fn = lambda pts, z: igr.decode(dec, z, pts)
    latent = torch.tensor([0.12, -0.07], dtype=F64, requires_grad=True)
    tet_v = torch.tensor([[0., 0, 0], [1, 0, 0], [0, 1, 0], [0, 0, 1]], dtype=F64) * 0.3
    tet_f = torch.tensor([[0, 2, 1], [0, 1, 3], [0, 3, 2], [1, 2, 3]])
    body = _inject(rb.SDF3D, tet_v, tet_f)(torch.tensor([0.1, 0.2, -0.1], dtype=F64), 1.5, fn, [latent])
    rng = np.random.RandomState(11)
    pts = torch.tensor(rng.uniform(-1.8, 1.8, (400, 3)))
    sd, gr, mask = body.query_sdfs(pts.clone(), return_grads=True, return_overlapmask=True)
    sd2, mask2 = body.query_sdfs(pts.clone(), return_grads=False, return_overlapmask=True)
    sdz = sd2.clone()
    sdz[mask2 == False] = 0
    loss = torch.sum(sdz ** 2)
    loss.backward()
    print('neural_query', int(mask.sum()), float(loss), latent.grad.tolist())
    np.savez_compressed(os.path.join(HERE, 'neural_query.npz'), pts=pts.numpy(), sdf=sd.detach().numpy(), dir=gr.detach().numpy(),
                        mask=mask.numpy(), loss=float(loss), glatent=latent.grad.numpy())


def golden_trajectory_loss():
    """The reference's own trajectory_loss (experiments/trajectory_fitting/optim_sphere.py:114-160) on synthetic recorded
    trajectories: 4 worlds, 14 model states vs 19 target states each, irregular and partly coinciding time stamps (the
    tie rule of the nearest-time scan matters), random poses / velocities of two bodies."""
    from types import SimpleNamespace
    fn = reference_function('experiments/trajectory_fitting/optim_sphere.py', 'trajectory_loss', {})
    rng = np.random.RandomState(3)
    W, S, St = 4, 14, 19
    t = np.sort(rng.uniform(0, 1, (W, S)), 1)
    tt = np.sort(rng.uniform(0, 1, (W, St)), 1)
    tt[1, 5] = 0.5 * (t[1, 3] + t[1, 4]); tt[1] = np.sort(tt[1])     # a target state exactly between two model states
    t[2] = np.arange(S) / 30.0; tt[2] = np.arange(St) / 60.0 + 1.0 / 120.0   # ties at equal distance
    p, pt = rng.normal(size=(W, S, 14)), rng.normal(size=(W, St, 14))
    v, vt = rng.normal(size=(W, S, 12)), rng.normal(size=(W, St, 12))
    loss, grad = np.zeros(W), np.zeros((W, S, 14))
    for w in range(W):
        ps = [torch.tensor(p[w, k], dtype=F64, requires_grad=True) for k in range(S)]
        a = SimpleNamespace(trajectory=[(float(t[w, k]), ps[k], torch.tensor(v[w, k]), [], None) for k in range(S)])
        b = SimpleNamespace(trajectory=[(float(tt[w, k]), torch.tensor(pt[w, k]), torch.tensor(vt[w, k]), [], None)
                                        for k in range(St)])
        l = fn(a, b)
        l.backward()
        loss[w] = float(l)
        grad[w] = np.stack([x.grad.numpy() for x in ps])
        print('trajectory_loss world', w, float(l))
    np.savez_compressed(os.path.join(HERE, 'trajectory_loss.npz'), t=t, tt=tt, p=p, pt=pt, v=v, vt=vt, loss=loss, grad=grad)


def golden_filter_contacts():
    """The reference's own _filter_contacts (sdf_physics/physics3d/contacts.py:97-158, scipy's Qhull) on synthetic contact
    lists (specs.filter_cases): kept indices per list."""
    from specs import filter_cases
    cases = filter_cases()
    K = max(len(p) for _, p, _ in cases)
    P, N = np.zeros((len(cases), K, 3)), np.zeros((len(cases), K, 3))
    kept, off = [], [0]
    for w, (name, p, n) in enumerate(cases):
        P[w, :len(p)], N[w, :len(p)] = p, n
        idx = rc._filter_contacts(torch.as_tensor(n, dtype=F64), torch.as_tensor(p, dtype=F64), eps=1e-3)
        kept += idx.tolist()
        off.append(len(kept))
        print('filter_contacts', name, len(p), '->', len(idx))
    np.savez_compressed(os.path.join(HERE, 'filter_contacts.npz'), names=np.array([c[0] for c in cases]), p1=P, normals=N,
                        count=np.array([len(p) for _, p, _ in cases]), kept=np.array(kept, dtype=np.int64),
                        off=np.array(off, dtype=np.int64))


if __name__ == '__main__':
    torch.manual_seed(0)
    names = sys.argv[1:] or (list(SCENES) + ['sdf_query'])
    for n in names:
        if n == 'sdf_query':
            golden_sdf()
        elif n == 'detach_2nd_bounce':
            golden_detach_2nd_bounce()
        elif n == 'filter_contacts':
            golden_filter_contacts()
        elif n == 'trajectory_loss':
            golden_trajectory_loss()
        elif n == 'mesh_sdf':
            golden_mesh_sdf()
        elif n == 'neural_query':
            golden_neural_query()
        else:
            mk, leaves = SCENES[n]
            spec = mk()
            golden_scene(n, spec, default_leaves(spec, leaves))
