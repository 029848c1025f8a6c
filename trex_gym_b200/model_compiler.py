"""Load-time model compiler: ``assets/trex.urdf`` -> flat model blob.

The URDF is read through the reference's own parser (``tools/urdf_parsing.py``,
``Urdf.from_string`` :237-239, ``UrdfJoint.from_element`` :49-59,
``UrdfInertial.from_element`` :77-86) via :mod:`reference_loader`.  Two parser
defects are worked around here and nowhere else (SURVEY.md section 0.5):

* ``tools/urdf_parsing.py:82`` reads the mass from a non-existent attribute so
  every link parses with mass 0.0 -> ``<mass value>`` is read directly;
* ``<dynamics damping>`` is dropped by the parser -> read directly.

Two granularities are produced:

``full``   base + 132 links in pybullet's link order (DFS pre-order, children
           in joint file order), link frames = URDF *inertial* frames, fixed
           joints kept as 0-DoF links.  This is what ``oracle/trex_oracle.c``
           simulates (a restatement of Bullet's btMultiBody pipeline).
``merged`` fixed joints folded: 26 rigid bodies / 31 DoF.  Body frame of a
           revolute body = its URDF joint frame re-oriented so the joint axis is
           the local +z axis; body 0 keeps the base link's inertial frame so the
           base state is exactly pybullet's base state.  This is what the CUDA
           kernels simulate.

Contact geometry is *reference-undefined* (the URDF has no ``<collision>``;
SURVEY.md section 8a-N2): a fixed set of candidate contact points per body is
derived here from the visual meshes and used identically by kernels and oracle.
"""
from __future__ import annotations

import dataclasses
import json
import os
from collections import OrderedDict, defaultdict
from xml.etree import ElementTree

import numpy as np
from scipy.spatial.transform import Rotation

from . import model_blob
from .reference_loader import find_tools_dir, load_urdf_parsing

# ---------------------------------------------------------------------------
# Name mapping N1 (SURVEY.md section 8a): the env addresses joints/links by the
# names of an older URDF (trex_env.py:81-87, trex_robot.py:316).
# ---------------------------------------------------------------------------


def map_legacy_joint_name(name: str) -> str:
    """``femur_L_joint`` -> ``joint_femur_left`` (trex_env.py:81-87 vs trex.urdf:1020)."""
    if name.startswith("joint_"):
        return name
    if name.endswith("_joint"):
        core = name[: -len("_joint")]
        if core.endswith("_L"):
            core = core[:-2] + "_left"
        elif core.endswith("_R"):
            core = core[:-2] + "_right"
        return "joint_" + core
    return name


def map_legacy_link_name(name: str) -> str:
    """``atlas_axis_link`` -> ``link_atlas_axis`` (trex_robot.py:316 vs trex.urdf:2413)."""
    if name.startswith("link_"):
        return name
    if name.endswith("_link"):
        core = name[: -len("_link")]
        if core.endswith("_L"):
            core = core[:-2] + "_left"
        elif core.endswith("_R"):
            core = core[:-2] + "_right"
        return "link_" + core
    return name


HEAD_LINK_NAME = "link_atlas_axis"  # trex_robot.py:316 after N1

# Solver / engine constants.  Everything tagged [RECALL] restates pybullet /
# Bullet defaults from knowledge of the Bullet3 sources (SURVEY.md Appendix A);
# pybullet is not vendored in the reference nor installable here, so these are
# parameters of the model blob rather than hard-coded literals.
DEFAULT_PARAMS = OrderedDict(
    [
        ("time_step", 0.01),  # trex_env.py:54 (divided by substeps at :71)
        ("solver_iterations", 300.0),  # trex_env.py:57 (divided at :72)
        ("num_substeps", 5.0),  # trex_env.py:18
        ("gravity", 9.81),  # trex_env.py:20,117
        ("motor_kp", 5.0e-3),  # trex_robot.py:421
        ("motor_kd", 0.1),  # trex_robot.py:398  sqrt(2*1.0*kp)
        ("motor_max_torque", 3.0e5),  # trex_robot.py:260
        ("linear_damping", 0.04),  # [RECALL] btMultiBody default
        ("angular_damping", 0.04),  # [RECALL] btMultiBody default
        ("max_coordinate_velocity", 100.0),  # [RECALL] btMultiBody default
        ("erp", 0.2),  # [RECALL] btContactSolverInfo::m_erp (non-contact rows)
        ("contact_erp", 0.08),  # [RECALL] pybullet sets m_erp2 = 0.08
        ("split_impulse_threshold", -0.04),  # [RECALL] m_splitImpulsePenetrationThreshold
        ("linear_slop", 1.0e-5),  # [RECALL] pybullet sets m_linearSlop = 1e-5
        ("residual_threshold", 1.0e-7),  # [RECALL] m_leastSquaresResidualThreshold
        ("warmstart_factor", 0.1),  # [RECALL] pybullet sets m_warmstartingFactor = 0.1
        ("friction", 0.25),  # [RECALL] 0.5 (link) * 0.5 (floor), product combine
        ("contact_breaking_threshold", 0.02),  # [RECALL] gContactBreakingThreshold
        ("floor_height", 0.0005),  # assets/floor.urdf:21 box 0.001 thick centred at 0
        ("limit_max_impulse", 100.0),  # [RECALL] btMultiBodyConstraint::m_maxAppliedImpulse default
        ("reset_height", 3.0),  # trex_env.py:105
        ("reward_target_height", 2.5),  # trex_env.py:189
        ("max_contacts", 16.0),  # contact definition N2: capacity per environment (deepest first), = kernel TREX_KMAX
    ]
)

# Starting crouch, trex_env.py:81-87 with N1 applied.
STARTING_CONFIGURATION = OrderedDict(
    [
        ("joint_femur_left", -0.6),
        ("joint_tibia_left", 0.4),
        ("joint_tarsometatarsus_left", -1.2),
        ("joint_femur_right", -0.6),
        ("joint_tibia_right", 0.4),
        ("joint_tarsometatarsus_right", -1.2),
    ]
)

# Candidate contact points per merged body (keyed by the body's root link with
# the ``link_`` prefix and side suffix removed).  The link set is the one the
# orphaned hulls in assets/collisions/ cover (SURVEY.md section 2 #6).
# value = (count, "lower" | "all"): directions considered at the reset pose.
CONTACT_POINT_PLAN = {
    "vertebrae_sacral": (6, "all"),
    "tibia": (1, "lower"),
    "tarsometatarsus": (2, "lower"),
    "toe_02_a": (2, "lower"),
    "toe_02_b": (2, "lower"),
    "toe_03_a": (2, "lower"),
    "toe_03_c": (2, "lower"),
    "toe_04_a": (2, "lower"),
    "toe_04_d": (2, "lower"),
    "vertebra_cervical_09": (1, "lower"),
    "vertebra_cervical_03": (1, "lower"),
    "cranium": (4, "all"),
    "vertebra_caudal_02": (2, "lower"),
    "vertebra_caudal_10": (2, "lower"),
    "vertebra_caudal_24": (2, "lower"),
}
MAX_CONTACT_CANDIDATES = 64


def _rot_z_to(axis: np.ndarray) -> np.ndarray:
    """Rotation matrix A with A @ z = axis (axis is a unit vector)."""
    axis = axis / np.linalg.norm(axis)
    z = np.array([0.0, 0.0, 1.0])
    c = float(z @ axis)
    if c > 1.0 - 1e-12:
        return np.eye(3)
    if c < -1.0 + 1e-12:
        return np.diag([1.0, -1.0, -1.0])
    v = np.cross(z, axis)
    s = np.linalg.norm(v)
    vx = np.array([[0, -v[2], v[1]], [v[2], 0, -v[0]], [-v[1], v[0], 0]])
    return np.eye(3) + vx + vx @ vx * ((1 - c) / (s * s))


def _bullet_quicksort_equal_keys(n: int) -> list:
    """Permutation Bullet's ``btAlignedObjectArray::quickSort`` applies to ``n``
    elements whose sort keys are all equal.

    [RECALL] ``btMultiBodyDynamicsWorld::solveConstraints`` quick-sorts the
    constraint array by island id each step; all constraints of the one
    multibody share an island, the predicate is a strict ``<`` and the Hoare
    partition swaps on ties, so the (unstable) sort permutes the array
    deterministically.  The non-contact rows are solved in this order.
    """
    a = list(range(n))

    def qs(lo, hi):
        i, j = lo, hi
        while True:
            # all keys equal: neither inner while loop advances
            if i <= j:
                a[i], a[j] = a[j], a[i]
                i += 1
                j -= 1
            if not (i <= j):
                break
        if lo < j:
            qs(lo, j)
        if i < hi:
            qs(i, hi)

    if n > 1:
        qs(0, n - 1)
    return a


@dataclasses.dataclass
class CompiledModel:
    sections: "OrderedDict[str, np.ndarray]"
    meta: dict

    def blob(self) -> bytes:
        return model_blob.pack(self.sections)

    def __getitem__(self, k):
        return self.sections[k]


def _load_obj_vertices(path: str) -> np.ndarray:
    vs = []
    with open(path, "r") as f:
        for line in f:
            if line.startswith("v "):
                p = line.split()
                vs.append((float(p[1]), float(p[2]), float(p[3])))
    return np.asarray(vs, dtype=np.float64).reshape(-1, 3)


_DIRS26 = np.array(
    [
        (x, y, z)
        for x in (-1, 0, 1)
        for y in (-1, 0, 1)
        for z in (-1, 0, 1)
        if (x, y, z) != (0, 0, 0)
    ],
    dtype=np.float64,
)
_DIRS26 /= np.linalg.norm(_DIRS26, axis=1, keepdims=True)


def _select_contact_points(world_pts: np.ndarray, count: int, mode: str) -> list:
    """Pick ``count`` vertex indices: the lowest point at the reset pose first,
    then farthest-point sampling among support points of 26 fixed directions
    (lower hemisphere only for ``mode == 'lower'``)."""
    dirs = _DIRS26 if mode == "all" else _DIRS26[_DIRS26[:, 2] <= 1e-9]
    pool = []
    for d in dirs:
        idx = int(np.argmax(world_pts @ d))
        if idx not in pool:
            pool.append(idx)
    first = int(np.argmin(world_pts[:, 2]))
    chosen = [first]
    while len(chosen) < count:
        best, best_d = None, -1.0
        for idx in pool:
            if idx in chosen:
                continue
            dmin = min(np.linalg.norm(world_pts[idx] - world_pts[c]) for c in chosen)
            if dmin > best_d + 1e-12:
                best, best_d = idx, dmin
        if best is None or best_d < 1e-6:
            break
        chosen.append(best)
    return chosen


# ---------------------------------------------------------------------------
# Contact primitives from meshes (SURVEY.md section 8f row 3).  The reference's tooling direction
# (tools/mesh_primitives.py:323-402: PCA-aligned bounding box -> sphere or capsule, recursive octant subdivision while
# the radius is too large) restated here for the model compiler: a body's visual-mesh vertex cloud becomes a few
# spheres / capsules, and every sphere -- a capsule contributes its two end spheres -- is one floor-contact candidate.
# ---------------------------------------------------------------------------
@dataclasses.dataclass
class ContactPrimitive:
    kind: str            # "sphere" | "capsule"
    center: np.ndarray   # in the frame of the input points
    axis: np.ndarray     # unit vector of the capsule axis (the dominant PCA axis); unused for spheres
    radius: float
    length: float        # distance between the end-sphere centres (0 for spheres)

    def spheres(self):
        """(centre, radius) of the sphere(s) that can touch a plane: the sphere itself or the capsule's two end spheres."""
        if self.kind == "sphere":
            return [(self.center, self.radius)]
        h = 0.5 * self.length * self.axis
        return [(self.center - h, self.radius), (self.center + h, self.radius)]


def _pca_box(points: np.ndarray):
    """Oriented bounding box of a point cloud: axes = principal axes of the second moment about the centroid (columns
    x, y, z with z the dominant one, right handed), centre and full extents in that frame
    (cf. tools/mesh_primitives.py:323-344)."""
    pts = np.asarray(points, float)
    centroid = pts.mean(axis=0)
    d = pts - centroid
    u, _, _ = np.linalg.svd(d.T @ d)
    z, y = u[:, 0], u[:, 1]
    x = np.cross(y, z)
    axes = np.stack([x, y, z], axis=1)
    local = d @ axes
    lo, hi = local.min(axis=0), local.max(axis=0)
    return axes, centroid + axes @ (0.5 * (lo + hi)), hi - lo


def _sphere_or_capsule(axes, center, size) -> ContactPrimitive:
    """cf. tools/mesh_primitives.py:347-362: radius = half the larger minor extent; a capsule along the dominant axis when
    the box is longer than one diameter, else a sphere."""
    radius = 0.5 * float(max(size[0], size[1]))
    length = float(size[2]) - 2.0 * radius
    if length > 0.0:
        return ContactPrimitive("capsule", center, axes[:, 2].copy(), radius, length)
    return ContactPrimitive("sphere", center, axes[:, 2].copy(), radius, 0.0)


def fit_contact_primitives(points: np.ndarray, max_radius: float, max_divisions: int = 4, min_points: int = 100, _depth: int = 0) -> list:
    """Spheres / capsules covering ``points`` (N x 3): fit one primitive to the PCA box; while its radius exceeds
    ``max_radius`` (and fewer than ``max_divisions`` splits were made) split the cloud into the octants of the box frame
    -- octants with at most ``min_points`` points are dropped -- and recurse (cf. tools/mesh_primitives.py:296-402)."""
    pts = np.asarray(points, float)
    axes, center, size = _pca_box(pts)
    prim = _sphere_or_capsule(axes, center, size)
    if prim.radius > max_radius and _depth < max_divisions:
        local = (pts - center) @ axes
        out = []
        sx, sy, sz = local[:, 0] >= 0, local[:, 1] >= 0, local[:, 2] >= 0
        for mx in (sx, ~sx):
            for my in (sy, ~sy):
                for mz in (sz, ~sz):
                    m = mx & my & mz
                    if m.sum() > min_points:
                        out.extend(fit_contact_primitives(pts[m], max_radius, max_divisions, min_points, _depth + 1))
        if out:
            return out
    return [prim]


# primitives per merged body for contact_model="primitives": (max_radius in metres, max_divisions); bodies as in CONTACT_POINT_PLAN
CONTACT_PRIMITIVE_PLAN = {
    "vertebrae_sacral": (0.45, 1),
    "tibia": (1.0, 0), "tarsometatarsus": (1.0, 0),
    "toe_02_a": (1.0, 0), "toe_02_b": (1.0, 0), "toe_03_a": (1.0, 0), "toe_03_c": (1.0, 0), "toe_04_a": (1.0, 0), "toe_04_d": (1.0, 0),
    "vertebra_cervical_09": (1.0, 0), "vertebra_cervical_03": (1.0, 0),
    "cranium": (0.35, 1),
    "vertebra_caudal_02": (1.0, 0), "vertebra_caudal_10": (1.0, 0), "vertebra_caudal_24": (1.0, 0),
}


def compile_model(
    urdf_path: str,
    *,
    inertia_source: str = "urdf",
    with_contacts: bool = True,
    params: dict | None = None,
    contact_model: str = "points",
) -> CompiledModel:
    """Compile ``urdf_path`` (normally ``<reference>/assets/trex.urdf``).

    ``inertia_source``: ``"urdf"`` uses the ``<inertia>`` tensors of the file
    (pybullet ``URDF_USE_INERTIA_FROM_FILE``); ``"bullet_default"`` restates
    what pybullet does with default ``loadURDF`` flags on a link without a
    collision shape [RECALL, SURVEY.md H6 / Appendix A.1]: the diagonal becomes
    that of a box with half extents = the 0.001 m collision margin.

    ``contact_model``: ``"points"`` (default) takes support points of each body's visual-mesh vertex cloud as floor
    contact candidates (CONTACT_POINT_PLAN); ``"primitives"`` fits spheres / capsules to the clouds
    (``fit_contact_primitives``, CONTACT_PRIMITIVE_PLAN) and every sphere / capsule end sphere is a candidate with a
    radius (it touches the floor at centre - r * normal).
    """
    if contact_model not in ("points", "primitives"):
        raise ValueError("contact_model must be 'points' or 'primitives'")
    tools_dir = find_tools_dir(urdf_path)
    up = load_urdf_parsing(tools_dir)
    with open(urdf_path, "r") as f:
        text = f.read()
    urdf = up.Urdf.from_string(text)  # tools/urdf_parsing.py:237
    et = ElementTree.fromstring(text)

    # --- parser defect work-arounds (SURVEY.md section 0.5) --------------------
    link_mass = {}
    for ln in et.findall("link"):
        m = ln.find("inertial/mass")
        link_mass[ln.get("name")] = float(m.get("value")) if m is not None else 0.0
    joint_damping = {}
    for jn in et.findall("joint"):
        d = jn.find("dynamics")
        joint_damping[jn.get("name")] = float(d.get("damping", 0.0)) if d is not None else 0.0

    roots = urdf.root_link_names  # tools/urdf_parsing.py:133
    if len(roots) != 1:
        raise ValueError("expected a single root link, got %r" % (roots,))
    root = roots[0]

    # --- pybullet link order: DFS pre-order, children in joint file order -----
    children = defaultdict(list)
    for j in urdf.joints.values():
        children[j.parent_name].append(j)
    order = []

    def dfs(link_name):
        for j in children.get(link_name, []):
            order.append(j)
            dfs(j.child_name)

    dfs(root)
    n_links = len(order)
    link_names = [root] + [j.child_name for j in order]  # index 0 = base, i+1 = link i
    link_index = {n: i - 1 for i, n in enumerate(link_names)}  # base = -1
    joint_names = [j.name for j in order]

    def rin(name):
        return urdf.links[name].inertia.origin.rotation.as_matrix()

    def cin(name):
        return np.asarray(urdf.links[name].inertia.origin.translation, dtype=np.float64)

    def principal(name):
        I = np.asarray(urdf.links[name].inertia.inertia, dtype=np.float64)
        off = abs(I[0, 1]) + abs(I[0, 2]) + abs(I[1, 2])
        if off > 0:
            raise ValueError("link %s: non-diagonal <inertia> not supported" % name)
        return np.array([I[0, 0], I[1, 1], I[2, 2]])

    full_parent = np.zeros(n_links, np.int32)
    full_jtype = np.zeros(n_links, np.int32)
    full_dof = -np.ones(n_links, np.int32)
    full_mass = np.zeros(n_links + 1)
    full_inertia = np.zeros((n_links + 1, 3))
    full_rot0 = np.zeros((n_links, 9))
    full_axis = np.zeros((n_links, 3))
    full_d = np.zeros((n_links, 3))
    full_e = np.zeros((n_links, 3))
    full_lower = np.zeros(n_links)
    full_upper = np.zeros(n_links)
    full_damping = np.zeros(n_links)

    def inertia_of(name):
        m = link_mass[name]
        if inertia_source == "urdf":
            return principal(name)
        if inertia_source == "bullet_default":
            h = 0.001  # gUrdfDefaultCollisionMargin, empty btCompoundShape AABB [RECALL]
            l2 = (2 * h) ** 2
            v = m / 12.0 * (l2 + l2)
            return np.array([v, v, v])
        raise ValueError("inertia_source must be 'urdf' or 'bullet_default'")

    full_mass[0] = link_mass[root]
    full_inertia[0] = inertia_of(root)
    n_dof = 0
    for i, j in enumerate(order):
        p, c = j.parent_name, j.child_name
        full_parent[i] = link_index[p]
        rj = j.origin.rotation.as_matrix()
        xj = np.asarray(j.origin.translation, dtype=np.float64)
        full_rot0[i] = (rin(c).T @ rj.T @ rin(p)).reshape(-1)
        full_d[i] = rin(c).T @ cin(c)
        full_e[i] = rin(p).T @ (xj - cin(p))
        full_mass[i + 1] = link_mass[c]
        full_inertia[i + 1] = inertia_of(c)
        full_damping[i] = joint_damping.get(j.name, 0.0)
        if j.type == "revolute":
            full_jtype[i] = 1
            full_dof[i] = n_dof
            n_dof += 1
            a = np.asarray(j.axis, dtype=np.float64)
            a = a / np.linalg.norm(a)
            full_axis[i] = rin(c).T @ a
            full_lower[i] = j.limits.position[0]
            full_upper[i] = j.limits.position[1]
        elif j.type != "fixed":
            raise ValueError("joint %s: unsupported type %s" % (j.name, j.type))

    # --- zero-pose link frames (base URDF link frame at identity) -------------
    W_R = {root: np.eye(3)}
    W_x = {root: np.zeros(3)}
    for j in order:
        rp, xp = W_R[j.parent_name], W_x[j.parent_name]
        W_R[j.child_name] = rp @ j.origin.rotation.as_matrix()
        W_x[j.child_name] = xp + rp @ np.asarray(j.origin.translation, dtype=np.float64)

    # --- merged bodies ----------------------------------------------------------
    body_of_link = {root: 0}
    body_root = [root]
    body_parent = [-1]
    body_joint = [None]
    for j in order:
        if j.type == "revolute":
            body_of_link[j.child_name] = len(body_root)
            body_root.append(j.child_name)
            body_parent.append(body_of_link[j.parent_name])
            body_joint.append(j)
        else:
            body_of_link[j.child_name] = body_of_link[j.parent_name]
    nb = len(body_root)

    # body frames in the zero-pose "world" (base URDF link frame)
    B_R = [W_R[root] @ rin(root)]
    B_x = [W_x[root] + W_R[root] @ cin(root)]
    for b in range(1, nb):
        j = body_joint[b]
        a = np.asarray(j.axis, dtype=np.float64)
        B_R.append(W_R[j.child_name] @ _rot_z_to(a))
        B_x.append(W_x[j.child_name].copy())

    mb_parent = np.asarray(body_parent, np.int32)
    mb_E0 = np.zeros((nb, 9))
    mb_r0 = np.zeros((nb, 3))
    mb_E0[0] = np.eye(3).reshape(-1)
    for b in range(1, nb):
        p = body_parent[b]
        mb_E0[b] = (B_R[p].T @ B_R[b]).reshape(-1)  # child axes in parent coordinates
        mb_r0[b] = B_R[p].T @ (B_x[b] - B_x[p])  # child origin in parent coordinates

    mb_mass = np.zeros(nb)
    mb_mc = np.zeros((nb, 3))
    mb_I = np.zeros((nb, 3, 3))
    mb_damp_rot = np.zeros((nb, 3, 3))
    mb_nlinks = np.zeros(nb, np.int32)
    task_body, task_r, task_m = [], [], []
    for idx, name in enumerate(link_names):
        b = body_of_link[name]
        m = full_mass[idx]
        Rk = B_R[b].T @ (W_R[name] @ rin(name))
        pk = B_R[b].T @ (W_x[name] + W_R[name] @ cin(name) - B_x[b])
        Ik = Rk @ np.diag(full_inertia[idx]) @ Rk.T
        mb_mass[b] += m
        mb_mc[b] += m * pk
        mb_I[b] += Ik + m * ((pk @ pk) * np.eye(3) - np.outer(pk, pk))
        mb_damp_rot[b] += Ik
        mb_nlinks[b] += 1
        task_body.append(b)
        task_r.append(pk)
        task_m.append(m)

    def sym6(M):
        return np.array([M[0, 0], M[0, 1], M[0, 2], M[1, 1], M[1, 2], M[2, 2]])

    mb_lower = np.zeros(nb)
    mb_upper = np.zeros(nb)
    mb_damping = np.zeros(nb)
    mb_link = -np.ones(nb, np.int32)  # pybullet link index of the body's joint
    for b in range(1, nb):
        j = body_joint[b]
        mb_lower[b] = j.limits.position[0]
        mb_upper[b] = j.limits.position[1]
        mb_damping[b] = joint_damping.get(j.name, 0.0)
        mb_link[b] = link_index[j.child_name]

    # name-sorted revolute joints = action / observation order (trex_robot.py:311-314;
    # pybullet returns names as bytes: a bytes-wise sort == str sort for ASCII)
    rev = [(body_joint[b].name, b) for b in range(1, nb)]
    rev_sorted = sorted(rev, key=lambda t: t[0].encode())
    obs_body = np.asarray([b for _, b in rev_sorted], np.int32)  # obs slot k -> body index
    obs_dof = obs_body - 1  # merged joint dof index (0..24) == full revolute dof index

    start_q = np.zeros(nb)  # per body
    for jn, val in STARTING_CONFIGURATION.items():
        for b in range(1, nb):
            if body_joint[b].name == jn:
                start_q[b] = val

    # head point: COM of link_atlas_axis (trex_robot.py:330-335: getLinkState()[0])
    hb = body_of_link[HEAD_LINK_NAME]
    head_p = B_R[hb].T @ (W_x[HEAD_LINK_NAME] + W_R[HEAD_LINK_NAME] @ cin(HEAD_LINK_NAME) - B_x[hb])
    head_link = link_index[HEAD_LINK_NAME]

    # --- reset-pose FK (for contact-point selection and golden numbers) ---------
    def body_world_poses(q_body, base_R=np.eye(3), base_x=np.array([0.0, 0.0, 3.0])):
        R = [base_R]
        x = [base_x]
        for b in range(1, nb):
            p = body_parent[b]
            c, s = np.cos(q_body[b]), np.sin(q_body[b])
            Rz = np.array([[c, -s, 0], [s, c, 0], [0, 0, 1.0]])
            R.append(R[p] @ mb_E0[b].reshape(3, 3) @ Rz)
            x.append(x[p] + R[p] @ mb_r0[b])
        return R, x

    RW, XW = body_world_poses(start_q)

    # --- contact candidates -------------------------------------------------------
    cand_body, cand_p, cand_link, cand_local, cand_r = [], [], [], [], []
    mesh_stats = {}
    asset_dir = os.path.dirname(os.path.abspath(urdf_path))
    lowest_vertex_z = None
    if with_contacts:
        body_pts = defaultdict(list)
        for ln in et.findall("link"):
            name = ln.get("name")
            b = body_of_link[name]
            for vis in ln.findall("visual"):
                mesh = vis.find("geometry/mesh")
                if mesh is None:
                    continue
                path = os.path.join(asset_dir, mesh.get("filename"))
                if not os.path.isfile(path):
                    continue
                org = vis.find("origin")
                xyz = np.array([float(v) for v in org.get("xyz").split()]) if org is not None else np.zeros(3)
                rpy = [float(v) for v in org.get("rpy").split()] if org is not None else [0, 0, 0]
                Rv = Rotation.from_euler("xyz", rpy).as_matrix()  # tools/urdf_parsing.py:267-269
                v = _load_obj_vertices(path)
                if v.size == 0:
                    continue
                vl = v @ Rv.T + xyz  # link frame
                vw0 = vl @ W_R[name].T + W_x[name]  # zero-pose world
                vb = (vw0 - B_x[b]) @ B_R[b]  # body frame
                body_pts[b].append(vb)
        for b in range(nb):
            if b in body_pts:
                pts = np.concatenate(body_pts[b], axis=0)
                zw = (pts @ RW[b].T + XW[b])[:, 2]
                lo = float(zw.min())
                lowest_vertex_z = lo if lowest_vertex_z is None else min(lowest_vertex_z, lo)
        for b in range(nb):
            key = body_root[b][len("link_"):]
            for suf in ("_left", "_right"):
                if key.endswith(suf):
                    key = key[: -len(suf)]
            if key not in CONTACT_POINT_PLAN or b not in body_pts:
                continue
            count, mode = CONTACT_POINT_PLAN[key]
            pts = np.concatenate(body_pts[b], axis=0)
            if contact_model == "primitives":
                max_radius, max_div = CONTACT_PRIMITIVE_PLAN[key]
                spheres = [sp for prim in fit_contact_primitives(pts, max_radius, max_div) for sp in prim.spheres()]
                # lowest-reaching spheres first (reset pose), as many as the point plan grants this body at most twice over
                spheres.sort(key=lambda cr: float((RW[b] @ cr[0] + XW[b])[2] - cr[1]))
                for centre, radius in spheres[: max(2, 2 * count)]:
                    cand_body.append(b)
                    cand_p.append(centre)
                    cand_r.append(float(radius))
                continue
            wpts = pts @ RW[b].T + XW[b]
            for idx in _select_contact_points(wpts, count, mode):
                cand_body.append(b)
                cand_p.append(pts[idx])
                cand_r.append(0.0)
        if len(cand_body) > MAX_CONTACT_CANDIDATES:
            raise ValueError("too many contact candidates")
        # oracle view: attach each point to the body's root link, in that link's inertial frame
        for b, p in zip(cand_body, cand_p):
            name = body_root[b]
            pw0 = B_x[b] + B_R[b] @ p
            Rl = W_R[name] @ rin(name)
            xl = W_x[name] + W_R[name] @ cin(name)
            cand_link.append(link_index[name])
            cand_local.append(Rl.T @ (pw0 - xl))

    # --- non-contact constraint order [RECALL] ------------------------------------
    # creation order: one joint-limit constraint per revolute link (added while the
    # URDF is converted, link order), then one motor per revolute link.
    # id k in [0,25): limit of dof k ; id 25+k: motor of dof k.
    n_rev = nb - 1
    perm = _bullet_quicksort_equal_keys(2 * n_rev)
    noncontact_order = np.asarray(perm, np.int32)

    p = OrderedDict(DEFAULT_PARAMS)
    if params:
        for k, v in params.items():
            if k not in p:
                raise KeyError("unknown model parameter %r" % k)
            p[k] = float(v)

    S = OrderedDict()
    S["param_values"] = np.asarray(list(p.values()), dtype=np.float64)
    S["full_n_links"] = np.asarray([n_links], np.int32)
    S["full_parent"] = full_parent
    S["full_jtype"] = full_jtype
    S["full_dof"] = full_dof
    S["full_mass"] = full_mass
    S["full_inertia"] = full_inertia.reshape(-1)
    S["full_rot0"] = full_rot0.reshape(-1)
    S["full_axis"] = full_axis.reshape(-1)
    S["full_d"] = full_d.reshape(-1)
    S["full_e"] = full_e.reshape(-1)
    S["full_lower"] = full_lower
    S["full_upper"] = full_upper
    S["full_damping"] = full_damping
    S["full_head_link"] = np.asarray([head_link], np.int32)
    S["full_start_q"] = np.asarray(
        [start_q[body_of_link[j.child_name]] if j.type == "revolute" else 0.0 for j in order]
    )
    S["full_cand_link"] = np.asarray(cand_link, np.int32).reshape(-1)
    S["full_cand_local"] = np.asarray(cand_local, np.float64).reshape(-1)
    S["full_cand_r"] = np.asarray(cand_r, np.float64).reshape(-1)
    S["noncontact_order"] = noncontact_order
    S["obs_dof"] = obs_dof.astype(np.int32)
    S["mb_n_bodies"] = np.asarray([nb], np.int32)
    S["mb_parent"] = mb_parent
    S["mb_link"] = mb_link
    S["mb_E0"] = mb_E0.reshape(-1)
    S["mb_r0"] = mb_r0.reshape(-1)
    S["mb_mass"] = mb_mass
    S["mb_mc"] = mb_mc.reshape(-1)
    S["mb_I"] = np.stack([sym6(M) for M in mb_I]).reshape(-1)
    S["mb_damp_rot"] = np.stack([sym6(M) for M in mb_damp_rot]).reshape(-1)
    S["mb_lower"] = mb_lower
    S["mb_upper"] = mb_upper
    S["mb_damping"] = mb_damping
    S["mb_start_q"] = start_q
    S["mb_head_body"] = np.asarray([hb], np.int32)
    S["mb_head_p"] = head_p
    S["mb_task_body"] = np.asarray(task_body, np.int32)
    S["mb_task_r"] = np.asarray(task_r).reshape(-1)
    S["mb_task_m"] = np.asarray(task_m)
    S["mb_cand_body"] = np.asarray(cand_body, np.int32).reshape(-1)
    S["mb_cand_p"] = np.asarray(cand_p, np.float64).reshape(-1)
    S["mb_cand_r"] = np.asarray(cand_r, np.float64).reshape(-1)

    # golden numbers (SURVEY.md section 7.1 / Appendix B)
    total_mass = float(full_mass.sum())
    com = sum(
        mb_mass[b] * XW[b] + RW[b] @ mb_mc[b] for b in range(nb)
    ) / total_mass
    head_w = XW[hb] + RW[hb] @ head_p
    meta = {
        "urdf": os.path.basename(urdf_path),
        "inertia_source": inertia_source,
        "contact_model": contact_model,
        "root_link": root,
        "n_links": n_links,
        "n_bodies": nb,
        "n_dof": n_dof,
        "link_names": link_names,
        "joint_names": joint_names,
        "body_root_links": body_root,
        "body_joint_names": [None] + [body_joint[b].name for b in range(1, nb)],
        "body_n_links": mb_nlinks.tolist(),
        "obs_joint_names": [n for n, _ in rev_sorted],
        "obs_pybullet_link_index": [int(mb_link[b]) for _, b in rev_sorted],
        "head_link": HEAD_LINK_NAME,
        "head_pybullet_link_index": int(head_link),
        "param_names": list(p.keys()),
        "params": dict(p),
        "starting_configuration": dict(STARTING_CONFIGURATION),
        "contact_candidate_bodies": [int(b) for b in cand_body],
        "golden": {
            "total_mass": total_mass,
            "links_mass_excluding_base": float(full_mass[1:].sum()),
            "reset_head_position": head_w.tolist(),
            "reset_com": com.tolist(),
            "reset_lowest_vertex_z": lowest_vertex_z,
        },
    }
    return CompiledModel(S, meta)


# ---------------------------------------------------------------------------
# Derived URDF with <collision> elements (SURVEY.md section 8a-N2): the contact geometry this repository
# defines, in a form pybullet can load, so that a pybullet run uses the same contact points.
# ---------------------------------------------------------------------------
CONTACT_POINT_MESH = "contact_point.obj"


def _write_contact_point_mesh(path: str, radius: float) -> None:
    """A tiny octahedron centred on the origin: the only collision geometry the reference serialiser can express is a
    mesh (tools/urdf_parsing.py:359-369), so every contact point becomes one instance of this mesh."""
    r = float(radius)
    v = [(r, 0, 0), (-r, 0, 0), (0, r, 0), (0, -r, 0), (0, 0, r), (0, 0, -r)]
    f = [(1, 3, 5), (3, 2, 5), (2, 4, 5), (4, 1, 5), (3, 1, 6), (2, 3, 6), (4, 2, 6), (1, 4, 6)]
    with open(path, "w") as fh:
        fh.write("# contact point marker: octahedron of radius %g m\n" % r)
        for x, y, z in v:
            fh.write("v %.9g %.9g %.9g\n" % (x, y, z))
        for a, b, c in f:
            fh.write("f %d %d %d\n" % (a, b, c))


def emit_derived_urdf(urdf_path: str, out_path: str, model: CompiledModel | None = None, point_radius: float = 1.0e-3,
                      absolute_visual_paths: bool = True) -> str:
    """Write ``out_path``: the reference URDF plus one ``<collision>`` mesh per contact candidate of ``model``.

    The file is produced by the reference's own ``Urdf.to_string`` (tools/urdf_parsing.py:217) from the parsed
    ``Urdf`` with ``GeometryMesh`` collision shapes added (tools/urdf_parsing.py:108-112, 359-369).  That serialiser
    loses what its parser never read -- ``<mass value>`` (``:82`` parses 0.0), ``<dynamics damping>`` and the
    ``effort`` / ``velocity`` limits -- so those attributes are patched back from the source file afterwards.
    Each point is a ``point_radius`` octahedron (``contact_point.obj`` next to ``out_path``): against the floor it
    touches ``point_radius`` lower than the candidate point itself (1 mm against a 20 mm breaking distance).
    """
    tools_dir = find_tools_dir(urdf_path)
    up = load_urdf_parsing(tools_dir)
    geo = up.geometry
    with open(urdf_path, "r") as f:
        text = f.read()
    urdf = up.Urdf.from_string(text)
    src = ElementTree.fromstring(text)
    if model is None:
        model = compile_model(urdf_path)
    link_names = list(model.meta["link_names"])  # pybullet link order, entry 0 = base
    cand_link = model.sections["full_cand_link"]
    cand_local = model.sections["full_cand_local"].reshape(-1, 3)
    inertial = {}
    for ln in src.findall("link"):
        org = ln.find("inertial/origin")
        xyz = np.array([float(v) for v in org.get("xyz").split()]) if org is not None else np.zeros(3)
        rpy = [float(v) for v in org.get("rpy").split()] if org is not None else [0.0, 0.0, 0.0]
        inertial[ln.get("name")] = (xyz, Rotation.from_euler("xyz", rpy).as_matrix())
    per_link = defaultdict(int)
    for li, p in zip(cand_link, cand_local):
        name = link_names[int(li) + 1]
        cin, rin = inertial[name]
        p_link = cin + rin @ p  # candidate points are stored in the link's inertial frame (Bullet's link frame)
        urdf.links[name].collision_shapes.append(
            geo.GeometryMesh(filename=CONTACT_POINT_MESH, origin=geo.Transform(translation=p_link)))
        per_link[name] += 1
    if absolute_visual_paths:  # keep the visuals loadable wherever the derived file is written
        asset_dir = os.path.dirname(os.path.abspath(urdf_path))
        for link in urdf.links.values():
            for shape in link.visual_shapes:
                if isinstance(shape, geo.GeometryMesh) and not os.path.isabs(shape.filename):
                    shape.filename = os.path.join(asset_dir, shape.filename)
    out = ElementTree.fromstring(urdf.to_string())  # the reference's serialiser
    # patch back what the reference's parser drops (SURVEY.md section 0.5)
    src_links = {ln.get("name"): ln for ln in src.findall("link")}
    for ln in out.findall("link"):
        m_src = src_links[ln.get("name")].find("inertial/mass")
        m_out = ln.find("inertial/mass")
        if m_src is not None and m_out is not None:
            m_out.set("value", m_src.get("value"))
    src_joints = {jn.get("name"): jn for jn in src.findall("joint")}
    for jn in out.findall("joint"):
        sj = src_joints[jn.get("name")]
        dyn = sj.find("dynamics")
        if dyn is not None and jn.find("dynamics") is None:
            jn.append(ElementTree.Element("dynamics", dict(dyn.attrib)))
        lim_s, lim_o = sj.find("limit"), jn.find("limit")
        if lim_s is not None and lim_o is not None:
            for k in ("effort", "velocity"):
                if lim_s.get(k) is not None:
                    lim_o.set(k, lim_s.get(k))
    os.makedirs(os.path.dirname(os.path.abspath(out_path)) or ".", exist_ok=True)
    _write_contact_point_mesh(os.path.join(os.path.dirname(os.path.abspath(out_path)), CONTACT_POINT_MESH), point_radius)
    from xml.dom import minidom

    pretty = minidom.parseString(ElementTree.tostring(out, encoding="utf-8")).toprettyxml(indent="  ")
    pretty = "\n".join(line for line in pretty.splitlines() if line.strip())
    with open(out_path, "w") as f:
        f.write(pretty + "\n")
    return out_path


# ---------------------------------------------------------------------------
# Checked-in compiled model (the GPU box has no /root/reference)
# ---------------------------------------------------------------------------
DATA_DIR = os.path.join(os.path.dirname(os.path.abspath(__file__)), "data")
BLOB_PATH = os.path.join(DATA_DIR, "trex_model.blob")
META_PATH = os.path.join(DATA_DIR, "trex_model.json")
TOPOLOGY_HEADER = os.path.join(os.path.dirname(os.path.abspath(__file__)), "csrc", "trex_topology.h")


PRIMITIVES_BLOB_PATH = os.path.join(DATA_DIR, "trex_model_primitives.blob")
PRIMITIVES_META_PATH = os.path.join(DATA_DIR, "trex_model_primitives.json")
LITERAL_BLOB_PATH = os.path.join(DATA_DIR, "trex_model_literal.blob")
LITERAL_META_PATH = os.path.join(DATA_DIR, "trex_model_literal.json")


def load_builtin(contact_model: str = "points") -> CompiledModel:
    """The checked-in compiled model: ``"points"`` (default: URDF inertia tensors, derived floor-contact points),
    ``"primitives"`` (the same with spheres / capsules fitted to the meshes as contact geometry) or ``"literal"`` -- what
    the reference's own pybullet call does with the checked-in URDF [RECALL, SURVEY.md H6 and section 0.4]:
    ``loadURDF`` without flags recomputes every link's inertia from its (absent) collision shape, and without any
    ``<collision>`` element nothing ever touches the floor."""
    bp, mp = {"points": (BLOB_PATH, META_PATH), "primitives": (PRIMITIVES_BLOB_PATH, PRIMITIVES_META_PATH),
              "literal": (LITERAL_BLOB_PATH, LITERAL_META_PATH)}[contact_model]
    with open(bp, "rb") as f:
        sections = model_blob.unpack(f.read())
    with open(mp, "r") as f:
        meta = json.load(f)
    return CompiledModel(sections, meta)


def with_params(model: CompiledModel, **overrides) -> CompiledModel:
    """Copy of ``model`` with some ``param_values`` replaced."""
    names = model.meta["param_names"]
    vals = model.sections["param_values"].copy()
    params = dict(model.meta["params"])
    for k, v in overrides.items():
        vals[names.index(k)] = float(v)
        params[k] = float(v)
    sections = OrderedDict(model.sections)
    sections["param_values"] = vals
    meta = dict(model.meta)
    meta["params"] = params
    return CompiledModel(sections, meta)


def with_body_mass_scale(model: CompiledModel, scales) -> CompiledModel:
    """Copy of ``model`` with the mass of every merged body scaled: uniform density scaling, what pybullet's
    ``changeDynamics(mass=s * m, localInertiaDiagonal=s * I)`` does to each URDF link of the body.  The COM stays; the
    mass, first moment, rotational inertia, angular-damping tensor and link-damping task masses of the body, and the
    mass and principal inertia of each of its links, are multiplied by the body's scale.

    ``scales``: 26 factors in the order of a per-environment parameter row (``TrexBatchSim.set_env_params``):
    ``scales[L]`` for the body of joint ``L`` (body ``L + 1``), ``scales[25]`` for the base."""
    s = np.asarray(scales, np.float64).reshape(-1)
    nb = int(model.sections["mb_n_bodies"][0])
    if s.shape != (nb,) or not np.all(np.isfinite(s)) or np.any(s <= 0):
        raise ValueError("scales must be %d finite factors > 0" % nb)
    by_body = np.concatenate([s[nb - 1:], s[:nb - 1]])  # body index order: base first
    S = OrderedDict(model.sections)
    S["mb_mass"] = model.sections["mb_mass"] * by_body
    for name, width in (("mb_mc", 3), ("mb_I", 6), ("mb_damp_rot", 6)):
        S[name] = (model.sections[name].reshape(nb, width) * by_body[:, None]).reshape(-1)
    task_body = model.sections["mb_task_body"]
    link_scale = by_body[task_body]  # one task per URDF link, in link order
    S["mb_task_m"] = model.sections["mb_task_m"] * link_scale
    S["full_mass"] = model.sections["full_mass"] * link_scale
    S["full_inertia"] = (model.sections["full_inertia"].reshape(-1, 3) * link_scale[:, None]).reshape(-1)
    return CompiledModel(S, dict(model.meta))


def link_wrenches(model: CompiledModel, body_wrench) -> np.ndarray:
    """The links' share of per-body external wrenches, for the reference simulator (``oracle``), which keeps every URDF link.

    ``body_wrench``: [26, 6] in the order of an external-wrench record (``TrexBatchSim.set_external_forces``: ``[k]`` for
    the body of joint ``k`` (body ``k + 1``), ``[25]`` for the base), world force at the body's COM then world torque.
    Returns [n_links + 1, 6], base first: each link carries the body's force times its share of the body's mass (the
    mass-weighted link COMs average to the body COM, so the split adds no moment), and the body's torque sits on its first
    link."""
    w = np.asarray(body_wrench, np.float64)
    nb = int(model.sections["mb_n_bodies"][0])
    if w.shape != (nb, 6):
        raise ValueError("body_wrench must have shape (%d, 6)" % nb)
    by_body = np.concatenate([w[nb - 1:], w[:nb - 1]])  # body index order: base first
    task_body = np.asarray(model.sections["mb_task_body"])  # body of every link, in link order (base first)
    mass = np.asarray(model.sections["full_mass"], np.float64)
    body_mass = np.bincount(task_body, weights=mass, minlength=nb)
    out = np.zeros((task_body.shape[0], 6))
    out[:, :3] = by_body[task_body, :3] * (mass / body_mass[task_body])[:, None]
    for b in range(nb):
        out[int(np.flatnonzero(task_body == b)[0]), 3:] = by_body[b, 3:]
    return out


def emit_topology_header(model: CompiledModel) -> str:
    """C header with the merged tree as compile-time constants.

    The kernels unroll over the 26-body tree with static register allocation, so
    the topology is baked in; ``trex_create`` verifies that the blob it is given
    matches these constants and fails loudly otherwise.
    """
    S = model.sections
    nb = int(S["mb_n_bodies"][0])
    parent = S["mb_parent"].tolist()
    depth = [0] * nb
    for b in range(1, nb):
        depth[b] = depth[parent[b]] + 1
    order = S["noncontact_order"].tolist()
    tb = S["mb_task_body"].tolist()

    def fn(name, vals):
        return (
            "TREX_TOPO_FN int %s(int i) { constexpr int T[%d] = {%s}; return T[i]; }"
            % (name, len(vals), ", ".join(str(v) for v in vals))
        )

    lines = [
        "// GENERATED by trex_gym_b200/model_compiler.py (emit_topology_header) -- do not edit.",
        "// Merged T-rex tree (fixed joints folded) as compile-time constants.",
        "#pragma once",
        "#ifdef __CUDACC__",
        "#define TREX_TOPO_FN __host__ __device__ constexpr",
        "#else",
        "#define TREX_TOPO_FN constexpr",
        "#endif",
        "namespace trex_topo {",
        "static constexpr int NB = %d;      // rigid bodies (body 0 = floating base)" % nb,
        "static constexpr int NJ = %d;      // revolute joints, joint j drives body j+1" % (nb - 1),
        "static constexpr int NDOF = %d;    // 6 + NJ" % (nb + 5),
        "static constexpr int MAX_DEPTH = %d;" % max(depth),
        "static constexpr int N_TASKS = %d;   // original URDF links (per-link damping)" % len(tb),
        "static constexpr int N_CAND = %d;    // contact candidate points" % len(S["mb_cand_body"]),
        fn("parent_of", parent),
        fn("depth_of", depth),
        fn("noncontact_order", order),
        fn("obs_dof", S["obs_dof"].tolist()),
        "}  // namespace trex_topo",
        "",
    ]
    return "\n".join(lines)


def write_builtin(model: CompiledModel) -> None:
    os.makedirs(DATA_DIR, exist_ok=True)
    primitives = model.meta.get("contact_model") == "primitives"
    literal = model.meta.get("inertia_source") == "bullet_default"
    bp, mp = (LITERAL_BLOB_PATH, LITERAL_META_PATH) if literal else ((PRIMITIVES_BLOB_PATH, PRIMITIVES_META_PATH) if primitives else (BLOB_PATH, META_PATH))
    with open(bp, "wb") as f:
        f.write(model.blob())
    with open(mp, "w") as f:
        json.dump(model.meta, f, indent=1, sort_keys=True)
    if not primitives and not literal:  # (the topology does not depend on the contact model or the inertia source)
        with open(TOPOLOGY_HEADER, "w") as f:
            f.write(emit_topology_header(model))


if __name__ == "__main__":  # python -m trex_gym_b200.model_compiler [urdf]
    import sys

    path = sys.argv[1] if len(sys.argv) > 1 else "/root/reference/assets/trex.urdf"
    mdl = compile_model(path)
    write_builtin(mdl)
    print(json.dumps(mdl.meta["golden"], indent=1))
    print("bodies", mdl.meta["n_bodies"], "links", mdl.meta["n_links"], "candidates", len(mdl["mb_cand_body"]))
    prim = compile_model(path, contact_model="primitives")
    write_builtin(prim)
    print("contact primitives:", len(prim["mb_cand_body"]), "sphere candidates, radii %.3f..%.3f m" % (prim["mb_cand_r"].min(), prim["mb_cand_r"].max()))
    lit = compile_model(path, inertia_source="bullet_default", with_contacts=False)
    write_builtin(lit)
    print("literal reference model: bullet-default inertia, %d contact candidates" % len(lit["mb_cand_body"]))
