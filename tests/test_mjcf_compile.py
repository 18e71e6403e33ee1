"""The MJCF -> structure-of-arrays compiler (mjcf/parser.py + mjcf/compile.py) run FROM THE XML: every other test loads the
committed models/*.npz, so a regression in the parser or the compiler would go unnoticed (VERDICT r1, weak #9).

The first three tests compile a small scene stored with the tests (tests/golden/mjcf/: an included defaults file, a
non-convex STL mesh) and compare with first-principles values and with the model this compiler produced from it when it
was stored.  The last three compile the reference project's own Sawyer / kitchen scenes, whose MJCF / STL files are not
part of this repository: they run where EARL_REFERENCE names a checkout of the reference and skip elsewhere."""
import os
import sys

import numpy as np
import pytest

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
SCENE = os.path.join(REPO, "tests", "golden", "mjcf", "scene.xml")
REF = os.environ.get("EARL_REFERENCE", "")
needs_reference = pytest.mark.skipif(not REF or not os.path.isdir(os.path.join(REF, "earl_benchmark", "envs", "metaworld_assets")),
                                     reason="set EARL_REFERENCE to a checkout of the reference project (its MJCF / STL assets)")


def compile_scene(spec):
    from earl_benchmark_b200.mjcf import compile as C
    return C.compile_model(spec, keep_geoms=("handle",), frame_sites=("hand",), keep_sites=("ee",))


def test_compile_of_the_stored_scene_reproduces_the_stored_model():
    from earl_benchmark_b200.mjcf import parser
    from earl_benchmark_b200.mjcf.compile import Model
    fresh = compile_scene(parser.load(SCENE))
    fresh._ext_defaults()
    stored = Model.load(os.path.join(REPO, "tests", "golden", "mjcf", "scene_compiled.npz"))
    stored._ext_defaults()
    for k, _ in Model.FIELDS + Model.EXT_FIELDS:
        a, b = np.asarray(getattr(fresh, k)), np.asarray(getattr(stored, k))
        assert a.shape == b.shape, k
        assert np.array_equal(a, b), (k, np.abs(a.astype(float) - b.astype(float)).max())
    assert fresh.names == stored.names
    assert fresh.to_blob() == stored.to_blob()


def test_parser_semantics_on_the_stored_scene():
    """<include> expansion, last-one-wins <compiler>, nested default classes through `childclass` and `class`, explicit
    <inertial> against inertiafromgeom="auto" with inertiagrouprange 4-5, massless bodies, mocap, weld, position actuator."""
    from earl_benchmark_b200.mjcf import compile as C, parser
    spec = parser.load(SCENE)
    assert spec.compiler["angle"] == "radian" and spec.compiler["inertiagrouprange"] == "4 5"
    assert spec.option["timestep"] == "0.0025" and spec.option["cone"] == "elliptic" and spec.option["iterations"] == "50"
    by = {b["name"]: b for b in spec.bodies}
    geoms = {g["name"]: g for b in spec.bodies for g in b["geoms"]}
    assert geoms["arm_col"]["group"] == "4" and geoms["arm_col"]["condim"] == "4" and geoms["arm_col"]["contype"] == "1"
    assert geoms["arm_col"]["friction"] == "1 0.1 0.002"                              # class base_col
    assert geoms["arm_vis"]["group"] == "1" and geoms["arm_vis"]["contype"] == "0"      # childclass xyz_base
    assert geoms["pad"]["group"] == "4" and geoms["table"]["group"] == "4" and geoms["table"]["condim"] == "3"
    j = {x["name"]: x for b in spec.bodies for x in b["joints"]}
    assert j["slide_x"]["damping"] == "10" and j["slide_x"]["armature"] == "0.001" and j["slide_x"]["limited"] == "true"
    assert j["grip"]["armature"] == "100" and j["grip"]["damping"] == "1000" and j["hinge"]["damping"] == "2"
    assert j["hinge"]["armature"] == "0" and j["ball_free"]["type"] == "free"
    assert by["mocap"]["mocap"] and len(spec.actuators) == 1 and spec.actuators[0]["kp"] == "400"
    assert [e["tag"] for e in spec.equalities] == ["weld"] and spec.equalities[0]["body2"] == "hand"
    assert np.allclose(by["finger"]["quat"], [np.sqrt(0.5), 0, 0, np.sqrt(0.5)])        # euler in radians
    raw = C.RawModel(spec)
    mass = dict(zip(raw.names, raw.mass))
    assert abs(mass["arm"] - 1000 * 8 * 0.02 * 0.03 * 0.04) < 1e-15                    # arm_vis (mass 1) is in group 1
    assert np.allclose(raw.inertia[raw.names.index("arm")], np.diag([0.03 ** 2 + 0.04 ** 2, 0.02 ** 2 + 0.04 ** 2,
                                                                     0.02 ** 2 + 0.03 ** 2]) * mass["arm"] / 3, rtol=0, atol=1e-18)
    assert abs(mass["finger"] - 1000 * (np.pi * 0.01 ** 2 * 0.04 + 4 / 3 * np.pi * 0.01 ** 3)) < 1e-15   # fromto capsule
    assert mass["door"] == 0.5 and np.array_equal(raw.ipos[raw.names.index("door")], [0.01, 0, 0])   # explicit <inertial>
    assert mass["hand"] == 0.0 and np.allclose(raw.ipos[raw.names.index("hand")], [0, 0, 0.12])      # massless: ipos <- pos
    assert raw.nq == 10 and raw.nv == 9
    m = compile_scene(spec)
    assert m.names["body"] == ["world", "arm", "finger", "door", "ball"]     # hand is fused into arm, mocap is not a body
    assert int(m.nweld) == 1 and int(m.nu) == 1 and m.names["site"] == ["ee", "body:hand"]


def test_legacy_mesh_centre_of_the_stored_mesh():
    """A U-shaped prism of five unit cubes: MuJoCo 2.1's legacy centre is not the centroid of a non-convex mesh, and the
    mesh geom's frame sits at that centre (scaled)."""
    from earl_benchmark_b200.mjcf import mesh, parser
    tris = mesh.load_stl(os.path.join(REPO, "tests", "golden", "mjcf", "meshes", "ushape.stl"), np.ones(3))
    assert len(tris) == 44
    signed = np.einsum("ij,ij->i", tris[:, 0], np.cross(tris[:, 1], tris[:, 2])) / 6
    assert abs(signed.sum() - 5.0) < 1e-12
    centroid = (signed[:, None] * (tris.sum(1) / 4)).sum(0) / signed.sum()
    assert np.abs(centroid - [1.5, 0.9, 0.5]).max() < 1e-12
    assert np.abs(mesh.legacy_center(tris) - [1.5, 21 / 22, 0.5]).max() < 1e-12
    scale = np.array([0.01, 0.02, 0.01])
    c = mesh.legacy_center(mesh.load_stl(os.path.join(REPO, "tests", "golden", "mjcf", "meshes", "ushape.stl"), scale))
    # a non-uniform scale re-weights the face areas, so the centre does not scale with the mesh along y
    assert np.abs(c[[0, 2]] - [0.015, 0.005]).max() < 1e-15 and 1e-6 < abs(c[1] - 0.02 * 21 / 22) < 1e-4
    m = compile_scene(parser.load(SCENE))
    assert np.abs(m.geom_pos[m.geom_id("handle")] - ([0.05, -0.05, 0] + c)).max() < 1e-15
    assert int(m.nhullvert) == 8                                             # the convex hull of the prism is a box


@pytest.fixture(scope="module")
def CM():
    sys.path.insert(0, os.path.join(REPO, "tools"))
    import compile_models
    return compile_models


@needs_reference
@pytest.mark.parametrize("name", ["sawyer_door", "sawyer_peg", "kitchen"])
def test_compile_from_xml_reproduces_the_committed_model(CM, name):
    from earl_benchmark_b200.mjcf.compile import Model
    fresh = getattr(CM, name)()
    fresh._ext_defaults()
    stored = Model.load(os.path.join(REPO, "earl_benchmark_b200", "models", name + ".npz"))
    stored._ext_defaults()
    for k, _ in Model.FIELDS + Model.EXT_FIELDS:
        a, b = np.asarray(getattr(fresh, k)), np.asarray(getattr(stored, k))
        assert a.shape == b.shape, k
        assert np.array_equal(a, b), (name, k, np.abs(a.astype(float) - b.astype(float)).max())
    assert fresh.names == stored.names
    assert fresh.to_blob() == stored.to_blob()


@needs_reference
def test_parser_semantics_on_the_sawyer_scene(CM):
    """Spot checks of what the parser must get right for the physics to be MuJoCo's (SURVEY Appendix B): nested default
    classes through `childclass`, last-one-wins <compiler>, explicit <inertial> against inertiafromgeom="auto" with
    inertiagrouprange 4-5, mocap bodies, weld equality, position actuators."""
    from earl_benchmark_b200.mjcf import compile as C, parser
    spec = parser.load(os.path.join(CM.MW, "sawyer_door_pull.xml"))
    assert spec.compiler["angle"] == "radian" and spec.compiler["inertiagrouprange"] == "4 5"
    assert spec.option["timestep"] == "0.0025" and spec.option["cone"] == "elliptic" and spec.option["iterations"] == "50"
    by = {b["name"]: b for b in spec.bodies}
    pad = {g.get("name"): g for g in by["rightpad"]["geoms"]}["rightpad_geom"]
    assert pad["group"] == "1" and pad["condim"] == "4" and pad["mass"] == "1"     # group from childclass xyz_base: NOT in 4-5
    claw = {g.get("name"): g for g in by["rightclaw"]["geoms"]}["rightclaw_it"]
    assert claw["group"] == "4" and claw["contype"] == "1"                          # class base_col
    j = {x["name"]: x for b in spec.bodies for x in b["joints"]}
    assert j["right_j3"]["damping"] == "10" and j["right_j3"]["armature"] == "0.001" and j["right_j3"]["limited"] == "true"
    assert j["r_close"]["armature"] == "100" and j["r_close"]["damping"] == "1000" and j["doorjoint"]["damping"] == "2"
    assert by["mocap"]["mocap"] and len(spec.actuators) == 2 and spec.actuators[0]["kp"] == "400"
    raw = C.RawModel(spec)
    hand = raw.names.index("hand")
    assert raw.mass[hand] == 0.0 and np.allclose(raw.ipos[hand], [0, 0, 0.12])      # massless: ipos <- pos (MuJoCo compiler)
    assert abs(raw.mass[raw.names.index("rightclaw")] - 0.0162) < 1e-12             # 1000 kg/m^3 x the claw box
    assert raw.mass[raw.names.index("rightpad")] == 0.0                             # mass="1" geom is outside the group range
    assert raw.nq == 10 and raw.nv == 10
    assert abs(raw.mass[raw.names.index("door_link")] - 0.111491) < 1e-6         # five density-50 collision geoms (group 4)
    biw, diw = raw.invweight0()
    assert abs(biw[hand, 0] - 6.1056) < 1e-3 and abs(biw[hand, 1] - 284.895) < 1e-2


@needs_reference
def test_legacy_mesh_centre_of_the_door_handle(CM):
    """SURVEY Appendix E.1: MuJoCo 2.1's LEGACY mesh centring of door_handle.stl (the observed object position)."""
    from earl_benchmark_b200.mjcf import mesh
    tris = mesh.load_stl(os.path.join(REF, "earl_benchmark/envs/metaworld_assets/objects/meshes/doorlock/door_handle.stl"), np.ones(3))
    assert len(tris) == 896
    assert np.abs(mesh.legacy_center(tris) - np.array([5.07216292e-02, 2.594e-09, 4.51399102e-02])).max() < 5e-9
