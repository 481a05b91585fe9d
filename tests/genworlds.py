"""Seeded generator of reference worlds for the generated-world tests.

The worlds are built through the package's own API (``core.World``, ``Body``, ``SubFrame``, the stock
joints, ``shapes``, ``constraints``, ``controllers``) and flattened with ``flatten``, so that model shapes
no fixed fixture has reach the specialisations ``build_host_model`` (arb_model_host.h) chooses: more
than 32 constraints, the general Gauss-Seidel visits, contact-aligned runs, many generator bodies,
wide and deep trees.

Rules the generator keeps, and why:

* No massless leaf, and no contact or ball-and-socket on a massless body.  A massless leaf makes Z
  singular (the oracle raises LinAlgError as the reference does).  Contacts on a massless body give
  4x4 contact admittance blocks of condition 1e24 and more: the reference's own Gauss-Seidel then
  diverges within a few steps (forces of 1e37 and sliding roots of -1e9, i.e. the root at infinity of
  a degenerate sextic), and no implementation can be compared with it there.  The sliding-root
  routine itself agrees with numpy's eigvals in such states (same "no root" verdicts, the same roots
  to 1e-15); the disagreement is the reference diverging.
* Every contact overlaps by a few mm and every ball-and-socket is closed at the initial pose
  (build()).
* A state is accepted only when the oracle steps it without raising, the first step has the stated
  minimum of active contacts (and a sliding one where the family asks for it) and no signed
  distance within 1e-9 of zero, every active constraint's admittance block is reasonably conditioned
  (COND_MAX) and no velocity exceeds GVEL_MAX.
"""
import numpy as np

from arboris_b200 import constraints as Cn
from arboris_b200 import controllers as Ct
from arboris_b200 import core
from arboris_b200 import homogeneousmatrix as Hg
from arboris_b200 import joints as J
from arboris_b200 import massmatrix as mm
from arboris_b200 import shapes
from arboris_b200.flatten import flatten

DT = 1e-3
COND_MAX = 1e10     # largest condition number of an active constraint's own admittance block
GVEL_MAX = 100.     # largest |gvel| (m/s, rad/s) after a step: beyond, the world is exploding
HINGES = (J.RzJoint, J.RyJoint, J.RxJoint)
KINDS = HINGES + (J.RzRyRxJoint, J.RzRyJoint, J.RzRxJoint, J.RyRxJoint, J.TxTyTzJoint)
CONS_LIMITS, CONS_BS, CONS_CONTACT = 0, 1, 2


def _tree(rng, nbodies, branching, massless=(), fan=None):
    """parent index (into the body list, 0 = root) of each non-root body: a chain when branching is
    0, random parents when 1; `fan` = (body, k) gives body k children in a row."""
    parents = []
    for i in range(1, nbodies):
        if fan is not None and fan[0] < i <= fan[0] + fan[1]:
            parents.append(fan[0])
        elif branching == 0 or rng.random() > branching:
            parents.append(i - 1)
        else:
            parents.append(int(rng.integers(i)))
    # a massless body must not be a leaf: give each one the next body as child
    for b in massless:
        if b not in parents and b + 1 < nbodies:
            parents[b] = b
    return parents


class Spec(object):
    """Knobs of one family of worlds (see CATALOGUE)."""

    def __init__(self, nbodies=6, branching=0.5, massless=(), visc=(), free_below=None, fan=None,
                 contact_bodies=(), spheres_per_body=4, points=(), subframe_both=True,
                 moving_plane=None, second_plane=None, sphere_sphere=(), box_sphere=None,
                 bs_ground=(), bs_bodies=(), nlimits=0, limits_at=None, pd=False, weight=True,
                 root_height=0.5, gvel_scale=0.3, min_active=2, sliding=True):
        self.__dict__.update(locals())
        del self.__dict__["self"]


def build_world(spec, seed):
    """The reference World of `spec` for `seed` (contact shapes at random places: see build())."""
    rng = np.random.default_rng(seed)
    w = core.World()
    ground_plane = shapes.Plane(w.ground, list(w.up) + [0.], "ground plane")
    w.register(ground_plane)
    bodies = [core.Body(name="root", mass=mm.box((.3, .2, .4), 5.))]
    rootj = J.FreeJoint(name="rootj")
    w.add_link(w.ground, rootj, bodies[0])
    rootj.gpos[:] = Hg.transl(0., spec.root_height, 0.)
    parents = _tree(rng, spec.nbodies, spec.branching, spec.massless, fan=spec.fan)
    joints, hinges = [rootj], []
    for i in range(1, spec.nbodies):
        if i == spec.free_below:
            cls = J.FreeJoint
        else:
            cls = KINDS[int(rng.integers(len(KINDS)))]
        mass = None if i in spec.massless else mm.box((.05, .1, .05), .3 + rng.random())
        visc = np.diag(rng.uniform(.01, .1, 6)) if i in spec.visc else None
        b = core.Body(name="b%d" % i, mass=mass, viscosity=visc)
        par = bodies[parents[i - 1]]
        f0 = core.SubFrame(par, np.dot(Hg.transl(*rng.uniform(-.1, .1, 3)), Hg.rotzyx(*rng.uniform(-.3, .3, 3))),
                           "f%d" % i)
        j = cls(name="j%d" % i)
        if spec.subframe_both and i % 2 == 0:
            f1 = core.SubFrame(b, np.dot(Hg.transl(*rng.uniform(-.05, .05, 3)), Hg.rotzyx(*rng.uniform(-.2, .2, 3))),
                               "g%d" % i)
            w.add_link(f0, j, f1)
        else:
            w.add_link(f0, j, b)
        if cls is J.FreeJoint:
            j.gpos[:] = np.dot(Hg.transl(*rng.uniform(-.05, .05, 3)), Hg.rotzyx(*rng.uniform(-.2, .2, 3)))
        bodies.append(b)
        joints.append(j)
        if cls in HINGES:
            hinges.append(j)
    if spec.weight:
        w.register(Ct.WeightController())
    cons = []

    # ground contacts: spheres then points, body by body (registration order = constraint order)
    ground = []
    for bi in spec.contact_bodies:
        for s in range(spec.spheres_per_body):
            r = .02 + .02*rng.random()
            ground.append(("sphere", bi, r))
    for bi in spec.points:
        ground.append(("point", bi, 0.))
    lim_left = list(hinges[:spec.nlimits])
    every = spec.limits_at
    for n, (kind, bi, r) in enumerate(ground):
        fr = core.SubFrame(bodies[bi], Hg.transl(*rng.uniform(-.08, .08, 3)), "c%d" % n)
        sh = shapes.Sphere(fr, r, "s%d" % n) if kind == "sphere" else shapes.Point(fr, "p%d" % n)
        w.register(sh)
        cons.append(Cn.SoftFingerContact((ground_plane, sh), .6, name="gc%d" % n))
        if every and lim_left and (n + 1) % every == 0:
            cons.append(Cn.JointLimits(lim_left.pop(0), -.25, .25))
    if spec.second_plane is not None:
        # a body on two ground planes with different normals: no longer contact-aligned
        bi = spec.second_plane
        pl = shapes.Plane(w.ground, [0., .8, .6, -.5], "tilted plane")
        w.register(pl)
        sh = shapes.Sphere(core.SubFrame(bodies[bi], Hg.transl(0., -.05, 0.), "tp"), .03, "tps")
        w.register(sh)
        cons.append(Cn.SoftFingerContact((pl, sh), .6, name="tilt"))
    if spec.moving_plane is not None:
        a, b = spec.moving_plane     # a plane carried by body a, touched by a sphere of body b
        pl = shapes.Plane(core.SubFrame(bodies[a], Hg.transl(0., 0., 0.), "mp"), [0., 1., 0., 0.], "moving plane")
        w.register(pl)
        sh = shapes.Sphere(core.SubFrame(bodies[b], Hg.transl(0., 0., 0.), "ms"), .03, "mps")
        w.register(sh)
        cons.append(Cn.SoftFingerContact((pl, sh), .5, name="mpc"))
    for a, b in spec.sphere_sphere:
        s0 = shapes.Sphere(core.SubFrame(bodies[a], Hg.transl(.02, 0., 0.), "ss0_%d" % a), .05)
        s1 = shapes.Sphere(core.SubFrame(bodies[b], Hg.transl(-.02, 0., 0.), "ss1_%d" % b), .05)
        w.register(s0); w.register(s1)
        cons.append(Cn.SoftFingerContact((s0, s1), .5, name="ss%d_%d" % (a, b)))
    if spec.box_sphere is not None:
        a, b = spec.box_sphere
        bx = shapes.Box(core.SubFrame(bodies[a], Hg.transl(0., 0., 0.), "bx"), (.1, .08, .1))
        sp = shapes.Sphere(core.SubFrame(bodies[b], Hg.transl(0., 0., 0.), "bxs"), .04)
        w.register(bx); w.register(sp)
        cons.append(Cn.SoftFingerContact((bx, sp), .5, name="bxc"))
    for bi in spec.bs_ground:
        cons.append(Cn.BallAndSocketConstraint((core.SubFrame(w.ground, Hg.transl(0., spec.root_height, 0.), "bsg%d" % bi),
                                                core.SubFrame(bodies[bi], Hg.transl(0., 0., 0.), "bsb%d" % bi))))
    for a, b in spec.bs_bodies:
        cons.append(Cn.BallAndSocketConstraint((core.SubFrame(bodies[a], Hg.transl(0., .02, 0.), "bsa%d" % a),
                                                core.SubFrame(bodies[b], Hg.transl(0., -.02, 0.), "bsc%d" % b))))
    for j in lim_left:              # limits left over: after every other constraint ("trailing limits")
        cons.append(Cn.JointLimits(j, -.25, .25))
    for c in cons:
        w.register(c)
    if spec.pd:
        lin = [j for j in joints[1:] if j.__class__ in HINGES + (J.RzRyRxJoint, J.TxTyTzJoint)][:3]
        n = sum(j.ndof for j in lin)
        w.register(Ct.ProportionalDerivativeController(lin, kp=np.diag(rng.uniform(1., 5., n)),
                                                       kd=np.diag(rng.uniform(.1, .5, n)),
                                                       gpos_des=rng.uniform(-.1, .1, n), name="pd"))
    w.init()
    return w


def _frame_world(o, b, H):
    """ground pose of the frame H (4x4) fixed on body b at the oracle's current pose"""
    return np.dot(o.pose[b], H) if b else H


def _move_to(o, d, side, b, p):
    """move the origin of shape frame `side` (0: d[0:16], 1: d[16:32]) of body b to the ground point p"""
    sl = slice(16*side, 16*side + 16)
    H = d[sl].reshape(4, 4).copy()
    P = o.pose[b] if b else np.eye(4)
    H[0:3, 3] = np.dot(P[0:3, 0:3].T, p - P[0:3, 3])
    d[sl] = H.reshape(-1)


def build(spec, seed, depth=(.002, .006)):
    """FlatModel of `spec` for `seed`, with every constraint placed on purpose at the initial pose
    (moving shape frames and anchors in their bodies' frames):

    * a sphere or point on a plane (carried by the ground or by a body) sits a depth drawn in `depth`
      (metres) into the plane, near the projection of its body's origin;
    * a sphere on a sphere or on a box face overlaps it by such a depth;
    * a ball-and-socket is closed: the anchor of side 0 is put where the anchor of side 1 is.

    Random placement leaves almost every contact separated, and an open ball-and-socket is closed by
    its force in one step (velocities of metres per millisecond), after which the reference's own
    Gauss-Seidel diverges and there is nothing to compare with."""
    from oracle.arboris_oracle import OracleWorld
    model = flatten(build_world(spec, seed))
    o = OracleWorld(model.to_dict())
    o.update_dynamic()
    rng = np.random.default_rng(10_000 + seed)
    for c, (t, ci) in enumerate(zip(model.cons_type, model.cons_int)):
        d = model.cons_dbl[c]
        b0, b1, pair = int(ci[0]), int(ci[1]), int(ci[2])
        if int(t) == CONS_BS:
            _move_to(o, d, 0, b0, _frame_world(o, b1, d[16:32].reshape(4, 4))[0:3, 3])
            continue
        if int(t) != CONS_CONTACT:
            continue
        H0 = _frame_world(o, b0, d[0:16].reshape(4, 4))
        r1, dep = d[42], rng.uniform(*depth)
        if pair == 0:
            n = np.dot(H0[0:3, 0:3], d[32:35])
            q = o.pose[b1][0:3, 3] + rng.uniform(-.08, .08, 3)
            q = q - (np.dot(n, q - H0[0:3, 3]) - d[35])*n          # onto the plane
            p = q + (r1 - dep)*n
        elif pair == 1:
            n = rng.normal(size=3)
            n /= np.linalg.norm(n)
            p = H0[0:3, 3] + (d[41] + r1 - dep)*n
        else:
            k, sign = int(rng.integers(3)), rng.choice((-1., 1.))
            f = rng.uniform(-.5, .5, 3)*d[32:35]
            f[k] = sign*(d[32 + k] + r1 - dep)
            p = np.dot(H0[0:3, 0:3], f) + H0[0:3, 3]
        _move_to(o, d, 1, b1, p)
    return model


def group_record_bytes(model):
    """shared memory the group prepare stage needs per CTA (arb_fused.cu group_smem_bytes: 2 worlds of
    gl.total doubles); above GROUP_SMEM_MAX the step falls back to the lane stages"""
    import harness
    return 8*2*harness.HostBatch(model, 1).group_doubles()


GROUP_SMEM_MAX = 227*1024


def ngrows(model):
    """rows of the generator-space Gauss-Seidel: 6 per generator body, 1 per joint limit"""
    ct, ci = np.asarray(model.cons_type), np.asarray(model.cons_int)
    gen = {int(b) for t, c in zip(ct, ci) if t != CONS_LIMITS for b in c[0:2] if b}
    return 6*len(gen) + int((ct == CONS_LIMITS).sum())


def free_spec(seed):
    """a random mix of every knob (the free seeds next to the catalogue)"""
    rng = np.random.default_rng(30_000 + seed)
    nb = int(rng.integers(5, 11))
    massless = (int(rng.integers(2, nb - 1)),) if rng.random() < .5 else ()
    ok = [b for b in range(nb) if b not in massless]
    pick = lambda k: tuple(int(x) for x in rng.choice(ok, size=k, replace=False))    # noqa: E731
    return Spec(nbodies=nb, branching=float(rng.uniform(0., 1.)), massless=massless, visc=pick(2),
                free_below=int(rng.integers(2, nb)) if rng.random() < .5 else None,
                contact_bodies=pick(int(rng.integers(1, 4))), spheres_per_body=int(rng.integers(2, 6)),
                points=pick(1), bs_bodies=(pick(2),) if rng.random() < .5 else (),
                sphere_sphere=(pick(2),) if rng.random() < .5 else (),
                nlimits=int(rng.integers(0, 4)), limits_at=int(rng.integers(2, 5)), pd=bool(rng.random() < .5),
                min_active=1, sliding=False)


FREE_SEEDS = (2, 3, 4)


# One world family per specialisation of the fused step that the fixed fixtures never reach.
CATALOGUE = {
    # 5 contact bodies x 7 spheres + limits every 6 contacts: nc > 32 and a run of one body across index 32
    "nc_over_32": Spec(nbodies=7, branching=.3, contact_bodies=(0, 1, 2, 3, 4), spheres_per_body=7, nlimits=4,
                       limits_at=6, min_active=8),
    # ball-and-socket to the ground and between bodies, sphere/sphere and box/sphere contacts: the general
    # visits of the staged Gauss-Seidel (gs_plain off)
    "general_visits": Spec(nbodies=7, branching=.5, contact_bodies=(0,), spheres_per_body=4, bs_ground=(3,),
                           bs_bodies=((2, 5),), sphere_sphere=((1, 4),), box_sphere=(1, 2),
                           nlimits=2, min_active=3),
    # a plane carried by a moving body (the root) touched by a sphere of another body, next to ground contacts
    "moving_plane": Spec(nbodies=6, branching=.5, contact_bodies=(0, 3), spheres_per_body=3, moving_plane=(0, 4),
                         nlimits=2, min_active=3, sliding=False),
    # contact-aligned bodies interleaved with limits, a body on two planes of different normals, a body
    # with contacts and a ball-and-socket, trailing limits
    "aligned_mixed": Spec(nbodies=6, branching=.5, contact_bodies=(0, 2, 3), spheres_per_body=4, points=(0,),
                          second_plane=2, bs_bodies=((3, 5),), nlimits=4, limits_at=3, min_active=4),
    # wide tree: a fan of 5 below body 1, a FreeJoint below the root, a massless intermediate body,
    # viscous bodies, diagonal PD, 7 generator bodies (NG > 32 for the group stage), limits off the paths
    "wide_tree": Spec(nbodies=12, branching=.6, fan=(1, 5), free_below=7, massless=(1,), visc=(2, 5, 9),
                      contact_bodies=(0, 2, 3, 4, 5, 6, 8), spheres_per_body=2, nlimits=3, pd=True, min_active=4),
    # 110 bodies: the group prepare stage's record no longer fits in shared memory (group_supported false)
    "group_fallback": Spec(nbodies=110, branching=.3, contact_bodies=(0, 5), spheres_per_body=3, nlimits=4,
                           min_active=2, sliding=False),
}


def expect(name, model):
    """Asserts that the model of catalogue entry `name` has the shape that reaches its branch."""
    ct = np.asarray(model.cons_type)
    ci = np.asarray(model.cons_int)
    contact = ct == CONS_CONTACT
    if name == "nc_over_32":
        assert len(ct) > 32
        run = [c for c in range(29, min(35, len(ct))) if contact[c]]
        assert any(c < 32 for c in run) and any(c >= 32 for c in run)
        assert len({int(ci[c][1]) for c in run}) == 1, "a run of one body crosses index 32"
    elif name == "general_visits":
        two_body = contact & (ci[:, 0] != 0) & (ci[:, 1] != 0)
        assert two_body.sum() >= 2 and (ci[contact, 2] == 1).any() and (ci[contact, 2] == 2).any()
        assert (ct == CONS_BS).sum() >= 2
    elif name == "aligned_mixed":
        lim = np.nonzero(ct == CONS_LIMITS)[0]
        assert any(0 < c < len(ct) - 1 and contact[c - 1] and contact[c + 1] for c in lim), "limits inside runs"
        assert len({tuple(d[32:35]) for d, t, i in zip(model.cons_dbl, ct, ci) if t == CONS_CONTACT and i[0] == 0}) == 2
    elif name == "wide_tree":
        jt = np.asarray(model.joint_type)
        assert (jt[1:] == 0).any(), "a FreeJoint below the root"
        assert ngrows(model) > 32, "NG > 32: world_fused_finish_k's branch without the K matrix"
        assert group_record_bytes(model) <= GROUP_SMEM_MAX, "the group stage runs"
    elif name == "moving_plane":
        moving = contact & (ci[:, 0] != 0) & (ci[:, 2] == 0)
        assert moving.sum() == 1
    elif name == "group_fallback":
        assert group_record_bytes(model) > GROUP_SMEM_MAX
    else:
        raise KeyError("no branch assertion for catalogue entry %r" % name)


def states(model, spec, seed, W, steps=1):
    """(gpos, gvel) of W worlds: the initial pose with random velocities.  A world is replaced (next draw)
    when the oracle raises within `steps` steps, or its first step breaks the contact rules (see the
    module docstring).  Returns also the number of draws rejected."""
    rng = np.random.default_rng(20_000 + seed)
    gp, gv, rejected = [], [], 0
    for _ in range(50*W):
        if len(gp) == W:
            break
        v = rng.normal(scale=spec.gvel_scale, size=model.ndof)
        if accept(model, spec, model.gpos0, v, steps):
            gp.append(np.array(model.gpos0, dtype=float)); gv.append(v)
        else:
            rejected += 1
    assert len(gp) == W, "too few states meet the contact rules"
    return np.stack(gp, 1), np.stack(gv, 1), rejected


def accept(model, spec, gpos, gvel, steps):
    from oracle.arboris_oracle import OracleWorld, CONS_SOFT_FINGER
    o = OracleWorld(model.to_dict())
    o.gpos[:], o.gvel[:] = gpos, gvel
    try:
        with np.errstate(over="raise", invalid="raise", divide="raise"):
            for s in range(steps):
                o.step(DT)
                act = [c for c in range(o.nc) if o.active[c]]
                for c, sl in o.cons_dol.items():
                    if np.linalg.cond(o.cons_adm[sl, sl]) > COND_MAX:
                        return False
                if s == 0:
                    contacts = [c for c in act if o.ct[c] == CONS_SOFT_FINGER]
                    if len(contacts) < spec.min_active:
                        return False
                    if spec.sliding and not any(o.branch[c] == 3 for c in contacts):
                        return False
                    if any(abs(o.sdist[c]) < 1e-9 for c in range(o.nc) if o.ct[c] == CONS_SOFT_FINGER):
                        return False
                if not np.abs(o.gvel).max() <= GVEL_MAX:
                    return False
    except (np.linalg.LinAlgError, FloatingPointError):
        return False
    return bool(np.isfinite(o.gvel).all())
