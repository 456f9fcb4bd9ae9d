"""Cross-checks of the restatement against the reference's own compiled code: the same seeded inputs as the reference build got, in the same
order, against what it returned (tests/golden/ref_crosscheck.npz, recorded by tests/golden/make_golden.py).  Visible sets (ids in ascending
order with their types) and poses are compared bit for bit through a 16-byte digest of their bytes."""
import hashlib
import os

import numpy as np
import pytest

from lumixengine_b200 import _lib, scenes
from lumixengine_b200.hierarchy import TRANSFORM_DTYPE


def digest(*arrays):
    """16-byte digest of the bytes of `arrays`, as tests/golden/make_golden.py records it."""
    h = hashlib.blake2b(digest_size=16)
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return np.frombuffer(h.digest(), np.uint8)


@pytest.fixture(scope="module")
def ref():
    return np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "ref_crosscheck.npz"))


def same_as_ref(ref, key, ids, tys):
    """ids / types of one cull of the restatement against the recorded cull of the reference -> its result page count."""
    count, pages = (int(x) for x in ref[f"{key}_info"])
    assert count == len(ids), (key, count, len(ids))
    o = np.argsort(ids)
    assert np.array_equal(digest(ids[o].astype(np.uint32), tys[o].astype(np.uint8)), ref[f"{key}_digest"]), key
    return pages


def test_struct_sizes(ref):
    sizes = {"Sphere": 16, "Frustum": 224, "ShiftedFrustum": 256, "ShiftedFrustum.origin": 224, "Transform": 56, "CullResult": 4096,
             "CullResult.entities": 16, "LocalRigidTransform": 28, "DualQuat": 32, "Matrix": 64}
    assert dict(zip(ref["sizeof_names"].tolist(), ref["sizeof_values"].tolist())) == sizes
    # the layouts the product's host side hands across its C-ABI
    assert _lib.ShiftedFrustum.origin.offset == sizes["ShiftedFrustum.origin"] and TRANSFORM_DTYPE.itemsize == sizes["Transform"]


@pytest.mark.parametrize("workers", [1, 4])
def test_cull_sets_equal_reference_job_system(oracle, ref, workers):
    """The reference's CullingSystemImpl on its own fiber job system of `workers` workers vs the restatement: identical sorted ids and types."""
    scene = scenes.cull_scene(400_000, (3000.0, 300.0, 3000.0), seed=123, big_fraction=0.005, type_probs=(0.5, 0.3, 0.2))
    oc = oracle.OracleCulling()
    oc.add(scene["entities"], scene["types"], scene["pos"], scene["radius"])
    for v, a in enumerate((scenes.c1_frustum_args(), dict(scenes.c1_frustum_args(), position=(900.0, -50.0, 400.0), direction=(-0.7, 0.1, -0.7), far=3500.0))):
        key = f"sets_w{workers}_v{v}"
        f = oracle.frustum_perspective(a["position"], a["direction"], a["up"], a["fov"], a["ratio"], a["near"], a["far"])
        assert np.array_equal(f[:248], ref[f"{key}_frustum"][:248])
        ids, tys, st = oc.cull(f)
        assert len(ids) > 1000
        assert same_as_ref(ref, key, ids, tys) == st["pages_total"] - st["pages_filtered"]  # one result page per processed cell page (:337)


def test_random_views_and_edits_equal_reference(oracle, ref):
    """Randomised cross-check: small worlds with crowded and sparse cells, random perspective / ortho views (inside, outside, tangent
    to cell borders, huge and tiny far planes, types filtered or not), with batches of moves / radius changes / removals in between.
    The restatement must return exactly the reference's visible set every time."""
    rng = np.random.default_rng(2024)
    for world in range(3):
        n = int(rng.integers(2_000, 30_000))
        half = (float(rng.choice([250.0, 900.0, 4000.0])), float(rng.choice([50.0, 400.0])), float(rng.choice([250.0, 900.0, 4000.0])))
        scene = scenes.cull_scene(n, half, seed=300 + world, big_fraction=float(rng.choice([0.0, 0.02, 0.3])), type_probs=(0.5, 0.25, 0.25))
        oc = oracle.OracleCulling()
        oc.add(scene["entities"], scene["types"], scene["pos"], scene["radius"])
        alive = np.ones(n, bool)
        pos, rad = scene["pos"].copy(), scene["radius"].copy()
        for step in range(12):
            p = rng.normal(size=3) * np.array(half) * 1.5
            d = rng.normal(size=3); d /= np.linalg.norm(d)
            up = np.cross(np.cross(d, rng.normal(size=3)), d); up /= np.linalg.norm(up)
            if step % 5 == 0:  # snapped to a cell corner, axis-aligned: planes coincide with cell faces
                p = np.round(p / 300.0) * 300.0
                d, up = np.array([0.0, 0.0, -1.0]), np.array([0.0, 1.0, 0.0])
            far = float(rng.choice([30.0, 700.0, 5000.0, 60000.0]))
            if step % 3 == 2:
                args = (p, d.astype(np.float32), up.astype(np.float32), float(rng.uniform(10, 3000)), float(rng.uniform(10, 3000)), 0.0, far)
                f = oracle.frustum_ortho(*args)
            else:
                args = (p, d.astype(np.float32), up.astype(np.float32), float(rng.uniform(0.2, 2.4)), float(rng.uniform(0.5, 2.5)), float(rng.uniform(0.01, 2.0)), far)
                f = oracle.frustum_perspective(*args)
            assert np.array_equal(f[:248], ref[f"rv{world}_{step}_frustum"][:248])
            t = int(rng.choice([-1, -1, 0, 1, 2]))
            ids, tys, _ = oc.cull(f, t)
            same_as_ref(ref, f"rv{world}_{step}", ids, tys)
            # edits between views
            live = np.nonzero(alive)[0]
            mv = rng.choice(live, min(len(live), 400), replace=False).astype(np.int32)
            a, b, c = np.array_split(mv, 3)
            pos[a] = pos[a] + rng.normal(size=(len(a), 3)) * 200.0
            oc.set_position(a, pos[a])
            rad[b] = (rng.random(len(b)) * 500.0).astype(np.float32)
            oc.set_radius(b, rad[b])
            oc.remove(c)
            alive[c] = False


def test_random_clips_equal_reference(oracle, ref):
    """Randomised pose pin: skeletons of 1..196 bones, clips of 1..90 frames with 3..19-bit channels (tracks up to 58 bits wide, which
    exercises the 64-bit unpack path), any share of constant tracks; plain, weighted and chained samples, relative and absolute, against
    the reference's own Animation::getRelativePose + Pose::computeAbsolute."""
    rng = np.random.default_rng(99)
    expected = iter(ref["clip_digests"])
    for trial in range(25):
        bones = int(rng.choice([1, 2, 3, 4, 5, 7, 16, 33, 64, 100, 196]))
        frames = int(rng.integers(1, 91))
        pb = tuple(int(x) for x in rng.integers(3, 20, 3))
        rb = tuple(int(x) for x in rng.integers(3, 20, 3))
        sk = scenes.skeleton(bones, seed=500 + trial)
        clip = scenes.clip(sk, frames=frames, fps=float(rng.choice([1.0, 24.0, 30.0, 59.94])), seed=600 + trial, pos_bits=pb, rot_bits=rb,
                           const_fraction=float(rng.choice([0.0, 0.25, 1.0])))
        other = scenes.clip(sk, frames=int(rng.integers(1, 40)), seed=700 + trial, const_fraction=0.5)
        L = clip.length_ticks
        for t in [0, 1, max(L - 1, 0), L, L + 5000] + [int(x) for x in rng.integers(0, max(L, 1), 6)]:
            for absolute in (False, True):
                assert np.array_equal(digest(*oracle.pose_evaluate(sk, clip, t, compute_absolute=absolute)), next(expected)), (trial, t, absolute)
            rel = oracle.pose_evaluate(sk, clip, t, compute_absolute=False)
            w = float(rng.choice([0.0, 0.3, 0.9998, 0.9999, 1.0]))
            t2 = int(rng.integers(0, max(other.length_ticks, 1)))
            chained = oracle.pose_evaluate(sk, other, t2, weight=w, start_from_bind=False, compute_absolute=True, pos=rel[0], rot=rel[1])
            assert np.array_equal(digest(*chained), next(expected)), (trial, t, w)
    assert next(expected, None) is None


def test_threshold_values_equal_reference(oracle, ref):
    """Exact thresholds: radius == cell size (not big: `radius > m_cell_size`, culling_system.cpp:139) and the next float above it; positions
    exactly on cell borders, +-0.0 and just inside them (cell index = int(pos * (1 / 300.f)), truncation toward zero)."""
    r_edge = np.float32(300.0)
    radii = np.array([r_edge, np.nextafter(r_edge, np.float32(1e9)), np.nextafter(r_edge, np.float32(0)), 0.0, 1e-30], np.float32)
    coords = [0.0, -0.0, 300.0, -300.0, 299.99999999, -299.99999999, 300.00000001, 600.0, -600.0, 899.9999, 1e-300, -1e-300]
    pos = np.array([[x, y, 10.0] for x in coords for y in (0.0, -300.0, 299.99999999)], np.float64)
    n = len(pos) * len(radii)
    P = np.repeat(pos, len(radii), axis=0)
    R = np.tile(radii, len(pos))
    E = np.arange(n, dtype=np.int32)
    T = (E % 3).astype(np.uint8)
    oc = oracle.OracleCulling()
    oc.add(E, T, P, R)
    a = scenes.c1_frustum_args()
    for v, args in enumerate((dict(a, position=(0.0, 0.0, 500.0)), dict(a, position=(300.0, 0.0, 300.0), direction=(-1.0, 0.0, 0.0)),
                              dict(a, position=(-1000.0, 100.0, 0.0), direction=(1.0, 0.0, 0.0), far=5000.0))):
        f = oracle.frustum_perspective(args["position"], args["direction"], args["up"], args["fov"], args["ratio"], args["near"], args["far"])
        ids, tys, st = oc.cull(f)
        assert len(ids) > 0
        assert same_as_ref(ref, f"th_v{v}", ids, tys) == st["pages_total"] - st["pages_filtered"]
    # the same edits as the reference got: shrink the big ones to exactly the threshold, grow the exact ones past it
    big = E[R > r_edge]
    oc.set_radius(big, np.full(len(big), r_edge, np.float32))
    edge = E[R == r_edge]
    oc.set_radius(edge, np.full(len(edge), np.nextafter(r_edge, np.float32(1e9)), np.float32))
    f = oracle.frustum_perspective(a["position"], a["direction"], a["up"], a["fov"], a["ratio"], a["near"], 5000.0)
    ids, tys, _ = oc.cull(f)
    same_as_ref(ref, "th_edited", ids, tys)
