"""Model compiler (mbd_b200/model) against the known-answer facts of SURVEY App. B/section 4."""
import os

import numpy as np
import pytest

from mbd_b200.model import blob, kinematics, mjcf, system_io

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "humanoid_xml_models.npz")
A = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "mbd_b200", "assets")


@pytest.fixture(scope="module")
def hr():
    return system_io.load(os.path.join(A, "humanoidrun.json"))


def test_humanoid_masses_kat(hr):
    # the well-known Gym humanoid body masses (density 1000, feet fused into the shins)
    exp = [8.907, 2.262, 6.616, 4.752, 2.756 + 1.767, 4.752, 2.756 + 1.767, 1.661, 1.230, 1.661, 1.230]
    assert np.allclose(hr.mass, exp, atol=2e-3)


def test_humanoid_structure(hr):
    assert hr.link_parents == [-1, 0, 1, 2, 3, 2, 5, 0, 7, 0, 9]
    assert hr.link_types == "f2131312121"
    assert (hr.q_size(), hr.qd_size(), hr.act_size()) == (24, 23, 17)
    assert hr.act_qd_id.tolist() == [7, 6, 8, 9, 10, 11, 12, 13, 14, 15, 16, 17, 18, 19, 20, 21, 22]
    assert hr.act_gear.tolist() == [350.0] * 11 + [100.0] * 6
    assert np.allclose(hr.act_ctrl_range, [[-0.4, 0.4]] * 17)
    assert hr.dt == 0.006 and np.allclose(hr.init_q[:7], [0, 0, 1.4, 1, 0, 0, 0])
    assert [c["link"] for c in hr.contacts] == [4, 6]  # exactly two foot-sphere / floor contacts
    assert np.allclose(hr.contacts[0]["pos"], [0, 0, -0.35]) and hr.contacts[0]["radius"] == 0.075
    assert hr.joint_parity.tolist() == [1, 1, 1, -1, 1, -1, 1, 1, 1, 1, 1]  # hips are left-handed x,z,y triples
    assert hr.custom["spring_inertia_scale"] == 1.0 and hr.custom["joint_scale_pos"] == 0.5
    assert np.allclose(hr.dof_limit[6], np.deg2rad([-45, 45]))  # abdomen_z, degrees -> radians


def test_compiled_assets_match_reference_xml():
    """the committed assets equal what mjcf.load made of the original project's mbd/assets/<name>.xml, stored field by field
    in tests/golden/humanoid_xml_models.npz (keys "<name>.<field>")"""
    g = np.load(GOLDEN)
    for name in ("humanoidrun", "humanoidtrack", "humanoidstandup"):
        a = system_io.load(os.path.join(A, name + ".json"))
        assert a.link_names == g[name + ".link_names"].tolist() and a.link_types == str(g[name + ".link_types"])
        for f in ("mass", "com", "joint_rot", "joint_pos", "link_pos", "link_rot", "dof_limit", "dof_stiffness", "dof_damping"):
            assert np.array_equal(getattr(a, f), g[f"{name}.{f}"]), (name, f)


def test_fk_ik_roundtrip(hr):
    """kinematics.forward (axis-angle in the link frame) and kinematics.inverse (joint-frame Euler
    angles, the decomposition the physics uses) agree: validates joint frames and parity."""
    rng = np.random.default_rng(1)
    q = hr.init_q.copy()
    q[7:] = rng.uniform(-0.6, 0.6, size=17)
    qd = np.zeros(23)
    xp, xr, xa, xv = kinematics.forward(hr, q, qd)
    q2, _ = kinematics.inverse(hr, xp, xr, xa, xv)
    assert np.abs(q2[7:] - q[7:]).max() < 1e-6
    # single-dof rates are exact projections
    qd = np.zeros(23); qd[12] = 0.7  # right knee
    xp, xr, xa, xv = kinematics.forward(hr, q, qd)
    _, qd2 = kinematics.inverse(hr, xp, xr, xa, xv)
    assert abs(qd2[12] - 0.7) < 1e-6


def test_blob_pack(hr):
    b = blob.pack(hr, 7, blob.REWARD_HUMANOIDRUN)
    assert b.dtype == np.uint32 and b.size == blob.BLOB_WORDS
    i32, f32 = b.view(np.int32), b.view(np.float32)
    assert b[0] == blob.MAGIC and i32[blob.H_NLINK] == 11 and i32[blob.H_NU] == 17 and i32[blob.H_NFRAMES] == 7
    lf = lambda f, l: blob.HDR_WORDS + f * blob.MAXL + l
    assert [i32[lf(blob.F_PARENT, l)] for l in range(11)] == hr.link_parents
    assert [i32[lf(blob.F_CHILD0 + c, 0)] for c in range(4)] == [1, 7, 9, -1]
    assert i32[lf(blob.F_NCON, 4)] == 1 and i32[lf(blob.F_NCON, 3)] == 0
    assert np.isclose(f32[blob.H_ANG_DAMP], np.exp(-0.05 * 0.006))
    # actuator map: abdomen_y (actuator 0) drives dof 1 of link 1
    base = blob.F_DOF0 + 1 * blob.DOF_STRIDE
    assert i32[lf(base + blob.D_ACT, 1)] == 0 and f32[lf(base + blob.D_GEAR, 1)] == 350.0
    with pytest.raises(NotImplementedError):
        bad = system_io.loads(system_io.dumps(hr)); bad.custom["spring_inertia_scale"] = 0.0
        blob.pack(bad, 7, 0)


def test_humanoidtrack_subset():
    s = system_io.load(os.path.join(A, "humanoidtrack.json"))
    assert s.link_types == "f213131212111111" and s.link_parents[11:] == [-1] * 5
    links = list(range(11))
    b = blob.pack(s, 5, blob.REWARD_HUMANOIDTRACK, links=links, track_links=(0, 5, 3, 6, 4))
    i32 = b.view(np.int32)
    assert i32[blob.H_NTRACK] == 5 and i32[blob.H_TRACK0:blob.H_TRACK0 + 5].tolist() == [0, 5, 3, 6, 4]
    # the 5 cosmetic *_ref bodies hang on slide joints off the world: packable since round 2 (slide dofs on
    # world-parented links), although the env keeps simulating the 11 live links only (SURVEY App. B)
    full = blob.pack(s, 5, blob.REWARD_HUMANOIDTRACK).view(np.int32)
    assert [full[blob.HDR_WORDS + blob.F_SLIDE * blob.MAXL + l] for l in range(16)] == [0] * 11 + [1] * 5


def test_generic_quadruped_fixture():
    """a model outside the reference tree goes through the same compiler (GenericPositionalEnv's path)"""
    s = mjcf.load(os.path.join(os.path.dirname(__file__), "fixtures", "quadruped.xml"))
    assert s.link_types == "f11111111" and s.link_parents == [-1, 0, 1, 0, 3, 0, 5, 0, 7]
    assert len(s.contacts) == 9 and s.act_size() == 8 and np.allclose(s.act_gear, 60.0)
    b = blob.pack(s, 5, blob.REWARD_HUMANOIDRUN)
    i32 = b.view(np.int32)
    lf = lambda f, l: blob.HDR_WORDS + f * blob.MAXL + l
    assert [i32[lf(blob.F_CHILD0 + c, 0)] for c in range(4)] == [1, 3, 5, 7]
    assert i32[lf(blob.F_NCON, 0)] == 1 and i32[lf(blob.F_NCON, 2)] == 2
    assert np.allclose(s.dof_limit[7], np.deg2rad([30, 70]))
