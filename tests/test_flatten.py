"""Host logic: the model-building mirror of the reference API and the flattener."""
import numpy as np
import pytest

from conftest import load_golden
from arboris_b200 import World, Body, SubFrame, flatten, FlatModel
from arboris_b200 import scenarios
from arboris_b200.joints import RzJoint, FreeJoint, RzRyRxJoint, RyJoint, RxJoint
from arboris_b200.constraints import JointLimits, SoftFingerContact, get_all_contacts
from arboris_b200.shapes import Sphere, Plane, Point
from arboris_b200.core import Joint, Constraint, NamedObjectsList

ALL = ["simplearm", "human36_free", "human36_contact", "snake_loop", "ball_socket",
       "simplearm_limits", "balls", "zoo"]


@pytest.mark.parametrize("name", ALL)
def test_mirror_models_equal_reference_models(name):
    """The committed model fixtures were flattened from the REAL reference objects
    (oracle/make_goldens.py); this package's robots must flatten to the same arrays."""
    ref, _ = load_golden(name)
    mine = flatten(scenarios.BUILDERS[name]())
    a, b = ref.to_dict(), mine.to_dict()
    for k in a:
        if k in ("gpos0", "gvel0"):
            continue
        assert a[k].shape == b[k].shape, k
        assert (a[k] == b[k]).all(), k


def test_reference_robots_drop_in_unchanged():
    """The reference's own robot factories, run against the reference classes, flatten through
    the same duck-typed walk: the committed model fixtures are that flattening
    (oracle/make_goldens.py), and every array of it, initial state included, equals this
    package's."""
    for name in ALL:
        ref, _ = load_golden(name)
        mine = flatten(scenarios.BUILDERS[name]())
        assert sorted(ref.to_dict()) == sorted(mine.to_dict()), name
        for k, v in ref.to_dict().items():
            assert (v == mine.to_dict()[k]).all(), (name, k)


def test_dof_numbering_human36():
    """SURVEY.md section 8(a) a2: dof map of human36 in depth-first joint order."""
    m = flatten(scenarios.human36_free_world())
    assert m.ndof == 42 and m.ngpos == 52 and m.nj == 17
    assert list(m.joint_dof) == [0, 6, 9, 10, 12, 15, 16, 18, 21, 23, 26, 28, 30, 32, 35, 37, 39]
    assert list(m.joint_parent) == [0, 1, 2, 3, 1, 5, 6, 1, 8, 9, 10, 11, 8, 13, 14, 15, 8]
    k = [len(p) for p in m.ancestors_dofs()[1:]]
    assert k == [6, 9, 10, 12, 9, 10, 12, 9, 11, 14, 16, 18, 11, 14, 16, 18, 12]


def test_contact_order_and_rows():
    m = flatten(scenarios.human36_contact_world())
    assert list(m.cons_type) == [2]*8 + [0, 0]
    assert list(m.cons_row) == [0, 4, 8, 12, 16, 20, 24, 28, 32, 33] and m.nrows == 34
    assert [int(c[1]) for c in m.cons_int[:8]] == [4]*4 + [7]*4    # FootR x4 then FootL x4
    assert [int(c[1]) for c in m.cons_int[8:]] == [9, 15]           # knee dofs


def test_world_building_errors():
    w = World()
    b = Body("b")
    w.add_link(w.ground, RzJoint(name="j"), b)
    with pytest.raises(ValueError):           # kinematic loop (core.py:459-463)
        w.add_link(w.ground, RzJoint(), b)
    with pytest.raises(ValueError):           # joints are not registered (core.py:538-539)
        w.register(RzJoint())
    with pytest.raises(ValueError):
        w.register(3.)
    with pytest.raises(ValueError):           # core.py:1012-1013
        SubFrame(None, np.eye(4))
    with pytest.raises(AssertionError):       # core.py:1010
        SubFrame(b, np.ones((4, 4)))
    with pytest.raises(ValueError):           # constraints.py:37-38
        JointLimits(FreeJoint(), 0, 1)
    with pytest.raises(ValueError):
        RzJoint().dof
    w.init()
    assert w.ndof == 1 and w.getjoints()["j"].dof == slice(0, 1)
    with pytest.raises(KeyError):
        w.getbodies()["nope"]


def test_unknown_plugins_are_refused():
    class MyJoint(Joint):
        ndof = 1
        gpos = np.zeros(1)
        gvel = np.zeros(1)

    class MyConstraint(Constraint):
        pass
    w = World()
    w.add_link(w.ground, MyJoint(), Body())
    with pytest.raises(NotImplementedError):
        flatten(w)
    w = World()
    w.add_link(w.ground, RzJoint(), Body())
    w.register(MyConstraint())
    w.init()
    with pytest.raises(NotImplementedError):
        flatten(w)
    w = World()
    ball = Body(mass=np.eye(6))
    w.add_link(w.ground, FreeJoint(), ball)
    w.register(Sphere(ball, 1.))
    w.register(Plane(w.ground))
    from arboris_b200.shapes import Box, Cylinder
    w.register(Box(w.ground, (1., 1., 1.)))
    w.register(Cylinder(w.ground, 1., 1.))
    w.register(Point(ball))
    # pairs without a collision solver are skipped like the reference's NotImplementedError pairs
    # (collisions.py:35-64): here everything with the cylinder, and box/point, which the reference
    # names but never defines; sphere/plane is ordered (plane, sphere) as choose_solver does
    cs = get_all_contacts(w, friction_coeff=.5)
    assert [(type(c._shapes[0]).__name__, type(c._shapes[1]).__name__) for c in cs] == \
        [("Plane", "Sphere"), ("Box", "Sphere"), ("Plane", "Point")]
    for c in cs:
        w.register(c)
    w.init()
    m = flatten(w)
    assert m.cons_int[:, 2].tolist() == [0, 2, 0] and m.cons_dbl[:, 42].tolist() == [1., 1., 0.]


def test_replace_joint_and_gvel_views():
    w = scenarios.simplearm_world()
    joints = w.getjoints()
    w.replace_joint(joints["Elbow"], RzJoint(name="Elbow2"))
    assert [j.name for j in w.iterjoints()] == ["Shoulder", "Elbow2", "Wrist"]
    w._gvel[1] = 3.
    assert w.getjoints()["Elbow2"].gvel[0] == 3.     # joint.gvel is a view (core.py:626-629)


def test_flatmodel_roundtrip(tmp_path):
    m = flatten(scenarios.human36_contact_world())
    p = str(tmp_path / "m.npz")
    m.save(p)
    m2 = FlatModel.load(p)
    for k, v in m.to_dict().items():
        assert (v == m2.to_dict()[k]).all()


def test_rzyx_equals_rz_ry_rx_chain_model():
    """reference tests/test_joints.py:13-31 builds this two-branch world"""
    w = World()
    ba, bb = Body(), Body()
    w.add_link(w.ground, RzRyRxJoint(), ba)
    bzy, byx = Body(name="zy"), Body(name="yx")
    w.add_link(w.ground, RzJoint(), bzy)
    w.add_link(bzy, RyJoint(), byx)
    w.add_link(byx, RxJoint(), bb)
    w.init()
    m = flatten(w)
    assert list(m.joint_parent) == [0, 0, 2, 3] and m.ndof == 6
