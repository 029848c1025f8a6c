"""Model compiler / loader shim: golden numbers of SURVEY.md section 7.1 and Appendix B, regeneration of the
checked-in blob from the reference URDF (skipped unless TREX_GYM_REFERENCE names a trex-gym checkout: the reference's
URDF, meshes and parser are not part of this repository)."""
import json
import os
import sys

import numpy as np
import pytest

REF = os.environ.get("TREX_GYM_REFERENCE", "")
URDF = os.path.join(REF, "assets", "trex.urdf")
needs_ref = pytest.mark.skipif(not (REF and os.path.isfile(URDF)), reason="reference checkout not present (set TREX_GYM_REFERENCE)")


def test_golden_numbers(model):
    g = model.meta["golden"]
    assert abs(g["total_mass"] - 5180.275860952213) < 1e-9
    assert abs(g["links_mass_excluding_base"] - 4834.87) < 0.01  # "_total_mass" of trex_robot.py:318-320
    assert np.allclose(g["reset_head_position"], [0.000, 3.100, 3.208], atol=1e-3)
    assert np.allclose(g["reset_com"], [0.002, 1.278, 2.425], atol=1e-3)
    assert abs(g["reset_lowest_vertex_z"] - 0.250) < 1e-3
    assert model.meta["n_links"] == 132 and model.meta["n_bodies"] == 26 and model.meta["n_dof"] == 25
    assert model.meta["root_link"] == "link_vertebrae_sacral"


def test_merged_body_table(model):
    # SURVEY.md Appendix B: merged-body table (root link, parent, #links, mass)
    mass = model["mb_mass"]
    assert abs(mass[0] - 2183.997) < 1e-3 and model.meta["body_n_links"][0] == 40
    assert abs(mass[13] - 947.701) < 1e-3 and model.meta["body_root_links"][13] == "link_cranium"
    assert abs(mass[25] - 1.808) < 1e-3 and model.meta["body_root_links"][25] == "link_toe_04_d_left"
    assert sum(model.meta["body_n_links"]) == 133
    assert model["mb_parent"].tolist() == [-1, 0, 1, 2, 3, 4, 3, 6, 3, 8, 0, 10, 11, 12, 0, 14, 15, 0, 17, 18, 19, 20, 19, 22, 19, 24]


def test_sorted_joint_order_and_pybullet_indices(model):
    # SURVEY.md section 8a: name-sorted order with pybullet joint indices
    names = [n[len("joint_"):] for n in model.meta["obs_joint_names"]]
    assert names[:8] == ["atlas_axis", "cranium", "femur_left", "femur_right", "tarsometatarsus_left",
                         "tarsometatarsus_right", "tibia_left", "tibia_right"]
    assert model.meta["obs_pybullet_link_index"] == [41, 42, 113, 0, 115, 2, 114, 1, 119, 6, 120, 7, 122, 9, 124, 11,
                                                      126, 13, 129, 16, 70, 78, 92, 38, 32]
    assert model.meta["head_pybullet_link_index"] == 41


def test_subtree_inertia_about_joint_axis(model):
    """Appendix B: diagonal of the (fixed-base) joint-space mass matrix = inertia of the joint's subtree
    about its axis at the reset pose -- checks composite inertias, frames and the crouch."""
    S = model.sections
    nb = 26
    parent = S["mb_parent"]
    E0 = S["mb_E0"].reshape(nb, 3, 3)
    r0 = S["mb_r0"].reshape(nb, 3)
    q = S["mb_start_q"]
    R, x = [np.eye(3)], [np.zeros(3)]
    for b in range(1, nb):
        c, s = np.cos(q[b]), np.sin(q[b])
        Rz = np.array([[c, -s, 0], [s, c, 0], [0, 0, 1.0]])
        R.append(R[parent[b]] @ E0[b] @ Rz)
        x.append(x[parent[b]] + R[parent[b]] @ r0[b])

    def sym(v):
        return np.array([[v[0], v[1], v[2]], [v[1], v[3], v[4]], [v[2], v[4], v[5]]])

    def subtree(b):
        out = [b]
        for c in range(1, nb):
            if parent[c] == b:
                out += subtree(c)
        return out

    expect = {"atlas_axis": (959.8004, 778.042530), "femur_right": (723.8576, 1367.687173),
              "tibia_left": (334.0766, 339.905413), "toe_04_d_left": (1.8084, 0.040968),
              "vertebra_caudal_02": (404.1827, 958.947119), "vertebra_cervical_09": (1146.0215, 1550.624604)}
    names = model.meta["body_joint_names"]
    for key, (m_exp, I_exp) in expect.items():
        b = names.index("joint_" + key)
        axis, o = R[b][:, 2], x[b]
        m_tot, I_tot = 0.0, 0.0
        for k in subtree(b):
            m = S["mb_mass"][k]
            Ik = sym(S["mb_I"].reshape(nb, 6)[k])  # about body origin, body axes
            mc = S["mb_mc"].reshape(nb, 3)[k]
            # inertia about the joint axis through o: shift from body origin x[k] to o
            Iw = R[k] @ Ik @ R[k].T
            d = x[k] - o
            cw = R[k] @ mc
            # parallel axis for an inertia given about a point that is not the COM
            Io = Iw + m * ((d @ d) * np.eye(3) - np.outer(d, d)) + (2 * (d @ cw) * np.eye(3) - np.outer(d, cw) - np.outer(cw, d))
            I_tot += axis @ Io @ axis
            m_tot += m
        assert abs(m_tot - m_exp) < 1e-3, key
        assert abs(I_tot - I_exp) < 1e-4 * I_exp, (key, I_tot, I_exp)


def test_legacy_name_mapping():
    from trex_gym_b200.model_compiler import map_legacy_joint_name, map_legacy_link_name

    assert map_legacy_joint_name("femur_L_joint") == "joint_femur_left"
    assert map_legacy_joint_name("tibia_R_joint") == "joint_tibia_right"
    assert map_legacy_joint_name("tarsometatarsus_L_joint") == "joint_tarsometatarsus_left"
    assert map_legacy_link_name("atlas_axis_link") == "link_atlas_axis"


def test_blob_roundtrip(model):
    from trex_gym_b200 import model_blob

    again = model_blob.unpack(model.blob())
    assert list(again.keys()) == list(model.sections.keys())
    for k in again:
        assert np.array_equal(again[k], model.sections[k])
    with pytest.raises(ValueError):
        model_blob.unpack(b"NOTABLOB" + b"\0" * 64)


def test_noncontact_order_is_a_permutation(model):
    order = model["noncontact_order"].tolist()
    assert sorted(order) == list(range(50))
    assert order[:6] == [33, 32, 31, 36, 35, 34]  # Bullet quickSort on 50 equal keys


def test_contact_candidates(model):
    bodies = model["mb_cand_body"]
    assert 0 < len(bodies) <= 64
    # every toe segment and the cranium carry candidates; femurs do not
    names = model.meta["body_root_links"]
    with_pts = {names[b] for b in bodies}
    assert "link_toe_03_c_left" in with_pts and "link_cranium" in with_pts and "link_femur_left" not in with_pts


@needs_ref
def test_loader_shim_and_parser_defects():
    """The reference parser imports only through the shim (geometry.py:53) and parses every mass as 0
    (urdf_parsing.py:82) -- the two defects the compiler works around."""
    from trex_gym_b200.reference_loader import find_tools_dir, load_urdf_parsing

    up = load_urdf_parsing(find_tools_dir(URDF))
    with open(URDF) as f:
        urdf = up.Urdf.from_string(f.read())
    assert len(urdf.joints) == 132 and len(urdf.links) == 133
    j = urdf.joints["joint_femur_right"]
    assert j.type == "revolute" and np.allclose(j.axis, [0, 0, 1])
    assert np.allclose(j.limits.position, [-1.57079633, 1.57079633])
    assert np.allclose(j.origin.translation, [0.01719666, -0.22076976, 0.24924649], atol=1e-8)
    link = urdf.links["link_femur_right"]
    assert link.inertia.mass == 0.0  # the :82 bug
    assert np.allclose(np.diag(link.inertia.inertia), [68.57667542, 65.79754639, 19.34805107])


@needs_ref
def test_reference_parser_tests_pass_through_shim():
    """tools/urdf_parsing_test.py and tools/geometry_test.py, run against the shim-loaded modules."""
    import importlib.util
    import types
    import unittest

    from trex_gym_b200.reference_loader import _PKG, find_tools_dir, load_urdf_parsing

    tools = find_tools_dir(URDF)
    load_urdf_parsing(tools)
    ran = 0
    for name in ("geometry_test", "urdf_parsing_test"):
        path = os.path.join(tools, name + ".py")
        src = open(path).read()
        mod = types.ModuleType(_PKG + "." + name)
        mod.__package__ = _PKG
        mod.__file__ = path
        # the tests import their subject as a sibling module or as `tools.x`; point both at the shim
        sys.modules.setdefault("tools", sys.modules[_PKG])
        sys.modules.setdefault("tools.geometry", sys.modules[_PKG + ".geometry"])
        sys.modules.setdefault("tools.urdf_parsing", sys.modules[_PKG + ".urdf_parsing"])
        sys.modules.setdefault("geometry", sys.modules[_PKG + ".geometry"])
        sys.modules.setdefault("urdf_parsing", sys.modules[_PKG + ".urdf_parsing"])
        exec(compile(src, path, "exec"), mod.__dict__)
        suite = unittest.defaultTestLoader.loadTestsFromModule(mod)
        res = unittest.TextTestRunner(verbosity=0).run(suite)
        assert res.wasSuccessful(), name
        ran += res.testsRun
    assert ran >= 5


def test_topology_header_matches_checked_in_model(model):
    """The kernels' compile-time topology (csrc/trex_topology.h) is the one of the checked-in blob."""
    from trex_gym_b200.model_compiler import TOPOLOGY_HEADER, emit_topology_header

    assert open(TOPOLOGY_HEADER).read() == emit_topology_header(model)


@needs_ref
def test_checked_in_blob_regenerates(model):
    from trex_gym_b200.model_compiler import compile_model, emit_topology_header, TOPOLOGY_HEADER

    fresh = compile_model(URDF)
    assert list(fresh.sections.keys()) == list(model.sections.keys())
    for k in fresh.sections:
        a, b = fresh.sections[k], model.sections[k]
        assert a.shape == b.shape, k
        assert np.allclose(a, b, rtol=0, atol=1e-12), k
    assert json.loads(json.dumps(fresh.meta))["golden"] == model.meta["golden"]
    assert open(TOPOLOGY_HEADER).read() == emit_topology_header(fresh)


@needs_ref
def test_bullet_default_inertia_option():
    from trex_gym_b200.model_compiler import compile_model

    m = compile_model(URDF, inertia_source="bullet_default", with_contacts=False)
    mass = m["full_mass"]
    I = m["full_inertia"].reshape(-1, 3)
    assert np.allclose(I[:, 0], mass / 12.0 * 2 * 0.002 ** 2)


@needs_ref
def test_derived_urdf_with_collision_elements(model, tmp_path):
    """SURVEY.md N2: the 48 contact candidates written as <collision> meshes through the reference's own Urdf.to_string
    (tools/urdf_parsing.py:217), for a pybullet run on the same contact geometry.  Re-parsed by the reference parser the
    file has the collision shapes on the expected links at the expected places, and it compiles back to the same model
    (masses, damping and limits survive the reference serialiser's defects)."""
    from scipy.spatial.transform import Rotation

    from trex_gym_b200.model_compiler import CONTACT_POINT_MESH, compile_model, emit_derived_urdf
    from trex_gym_b200.reference_loader import find_tools_dir, load_urdf_parsing

    out = emit_derived_urdf(URDF, str(tmp_path / "trex_contacts.urdf"), model=model)
    assert os.path.isfile(str(tmp_path / CONTACT_POINT_MESH))
    up = load_urdf_parsing(find_tools_dir(URDF))
    with open(out) as f:
        text = f.read()
    parsed = up.Urdf.from_string(text)  # the reference's parser reads its own serialiser's output
    assert len(parsed.joints) == 132 and len(parsed.links) == 133
    shapes = {n: l.collision_shapes for n, l in parsed.links.items() if l.collision_shapes}
    assert sum(len(v) for v in shapes.values()) == len(model["full_cand_link"]) == 48
    names = model.meta["link_names"]
    want_links = {names[int(li) + 1] for li in model["full_cand_link"]}
    assert set(shapes) == want_links and "link_toe_04_d_left" in want_links and "link_cranium" in want_links
    assert all(s.filename == CONTACT_POINT_MESH for v in shapes.values() for s in v)
    # placement: link-frame origin -> inertial frame reproduces the candidate table
    from xml.etree import ElementTree

    et = ElementTree.fromstring(text)
    local = model["full_cand_local"].reshape(-1, 3)
    seen = {n: 0 for n in shapes}
    for li, p in zip(model["full_cand_link"], local):
        n = names[int(li) + 1]
        org = et.find("link[@name='%s']/inertial/origin" % n)
        cin = np.array([float(v) for v in org.get("xyz").split()])
        rin = Rotation.from_euler("xyz", [float(v) for v in org.get("rpy").split()]).as_matrix()
        got = rin.T @ (shapes[n][seen[n]].origin.translation - cin)
        seen[n] += 1
        assert np.abs(got - p).max() < 1e-9
    # the reference serialiser's defects are patched: mass, damping, effort/velocity survive
    assert et.find("link[@name='link_femur_right']/inertial/mass").get("value") == "390.7456359863281"
    assert et.find("joint[@name='joint_femur_right']/dynamics").get("damping") == "1.0"
    assert et.find("joint[@name='joint_femur_right']/limit").get("effort") == "100.0"
    m2 = compile_model(out)
    for k, a in model.sections.items():
        b = m2.sections[k]
        assert a.shape == b.shape and np.abs(a.astype(float) - b.astype(float)).max() < 1e-9, k


# ---------------------------------------------------------------------------------------------------------------
# Contact primitives from meshes (SURVEY.md section 8f row 3; reference pattern: tools/mesh_primitives.py:323-402)
# ---------------------------------------------------------------------------------------------------------------
def _capsule_cloud(rng, radius, length, n=4000):
    """Points on the surface of a capsule along z (length = distance of the end-sphere centres)."""
    d = rng.normal(size=(n, 3))
    d /= np.linalg.norm(d, axis=1, keepdims=True)
    z = rng.uniform(-0.5 * length - radius, 0.5 * length + radius, n)
    pts = np.zeros((n, 3))
    cyl = np.abs(z) <= 0.5 * length
    ang = rng.uniform(0, 2 * np.pi, n)
    pts[cyl] = np.stack([radius * np.cos(ang[cyl]), radius * np.sin(ang[cyl]), z[cyl]], 1)
    cap = ~cyl
    pts[cap] = radius * d[cap]
    pts[cap, 2] = np.abs(pts[cap, 2]) * np.sign(z[cap]) + np.sign(z[cap]) * 0.5 * length
    return pts


def test_fit_contact_primitives_recovers_a_capsule_and_a_sphere():
    from scipy.spatial.transform import Rotation

    from trex_gym_b200.model_compiler import fit_contact_primitives

    rng = np.random.default_rng(0)
    R = Rotation.from_euler("xyz", [0.4, -0.9, 1.3]).as_matrix()
    t = np.array([0.3, -1.2, 0.7])
    pts = _capsule_cloud(rng, 0.11, 0.8) @ R.T + t
    (prim,) = fit_contact_primitives(pts, max_radius=1.0, max_divisions=0)
    assert prim.kind == "capsule"
    assert abs(prim.radius - 0.11) < 2e-3 and abs(prim.length - 0.8) < 5e-3
    assert np.abs(prim.center - t).max() < 5e-3 and abs(abs(prim.axis @ R[:, 2]) - 1.0) < 1e-4
    ends = sorted((c @ R[:, 2] for c, _ in prim.spheres()))
    assert abs((ends[1] - ends[0]) - 0.8) < 5e-3
    ball = rng.normal(size=(3000, 3))
    ball = 0.25 * ball / np.linalg.norm(ball, axis=1, keepdims=True) + t
    (sph,) = fit_contact_primitives(ball, max_radius=1.0, max_divisions=0)
    assert sph.kind == "sphere" and abs(sph.radius - 0.25) < 5e-3 and np.abs(sph.center - t).max() < 5e-3
    assert len(sph.spheres()) == 1


def test_fit_contact_primitives_subdivides_by_octants():
    """A fat box-shaped cloud: one primitive when the radius bound allows it, the 8 octants of the PCA frame when it does
    not, 64 after two splits; octants with too few points are dropped; every piece respects the bound when it can."""
    from trex_gym_b200.model_compiler import fit_contact_primitives

    rng = np.random.default_rng(1)
    pts = rng.uniform(-1, 1, size=(40000, 3)) * np.array([0.5, 0.7, 1.0])
    assert len(fit_contact_primitives(pts, max_radius=10.0, max_divisions=4)) == 1
    one = fit_contact_primitives(pts, max_radius=0.5, max_divisions=1)
    assert len(one) == 8 and all(p.radius < 0.5 for p in one)
    two = fit_contact_primitives(pts, max_radius=0.2, max_divisions=2)
    assert len(two) == 64
    assert len(fit_contact_primitives(pts, max_radius=0.5, max_divisions=0)) == 1  # no divisions allowed
    # min_points: 7 of the 8 octants hold too few points and are dropped
    lopsided = np.concatenate([np.abs(pts[:5000]), -np.abs(pts[:40])])
    kept = fit_contact_primitives(lopsided, max_radius=0.2, max_divisions=1, min_points=100)
    assert 1 <= len(kept) < 8
    # the union of the pieces covers the cloud: every point is inside some primitive (inflated by 2 %)
    def inside(p, prim):
        d = p - prim.center
        a = np.clip(d @ prim.axis, -0.5 * prim.length, 0.5 * prim.length)
        return np.linalg.norm(d - np.outer(a, prim.axis), axis=1) <= 1.02 * prim.radius
    cov = np.zeros(len(pts), bool)
    for prim in one:
        cov |= inside(pts, prim)
    assert cov.mean() > 0.7  # (a capsule of radius = half the larger minor extent leaves the corners of a box outside)


def test_primitives_model_candidates():
    from trex_gym_b200.model_compiler import load_builtin

    pts, prim = load_builtin(), load_builtin("primitives")
    assert prim.meta["contact_model"] == "primitives"
    r = prim["mb_cand_r"]
    assert 32 <= len(r) <= 64 and (r > 0.04).all() and (r < 0.7).all() and len(prim["full_cand_r"]) == len(r)
    assert (pts["mb_cand_r"] == 0).all()
    # the same bodies carry candidates in both contact models, and nothing else differs between the two blobs
    assert set(prim["mb_cand_body"].tolist()) == set(pts["mb_cand_body"].tolist())
    for k in pts.sections:
        if "cand" not in k:
            assert np.array_equal(pts.sections[k], prim.sections[k]), k
    # toes are capsules: two end spheres of equal radius per toe body
    toe = prim.meta["body_root_links"].index("link_toe_03_a_left")
    assert (prim["mb_cand_body"] == toe).sum() == 2 and len(set(r[prim["mb_cand_body"] == toe])) == 1


@needs_ref
def test_checked_in_primitives_blob_regenerates():
    from trex_gym_b200.model_compiler import compile_model, load_builtin

    fresh, stored = compile_model(URDF, contact_model="primitives"), load_builtin("primitives")
    assert list(fresh.sections.keys()) == list(stored.sections.keys())
    for k in fresh.sections:
        assert fresh.sections[k].shape == stored.sections[k].shape and np.allclose(fresh.sections[k], stored.sections[k], rtol=0, atol=1e-12), k
