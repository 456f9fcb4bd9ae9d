"""Pins the CPU oracle (restatement) against golden vectors produced by the reference's own compiled code
(tests/golden/*.npz, generator: tests/golden/make_golden.py).  Runs anywhere: needs gcc only."""
import ctypes as C
import os

import numpy as np
import pytest

from lumixengine_b200 import scenes

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
P = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731


def bits(a):
    a = np.ascontiguousarray(a)
    return a.view(np.uint32 if a.dtype.itemsize == 4 else np.uint8)


@pytest.fixture(scope="module")
def kat():
    return {**np.load(os.path.join(G, "math_kat.npz")), **np.load(os.path.join(G, "math_kat_frustum.npz"))}


def test_math_primitives_bit_exact(oracle, kat):
    L = oracle.lib()
    n = len(kat["qa"])
    c = lambda a: np.ascontiguousarray(a)  # noqa: E731
    out = np.zeros((n, 56), np.uint8)
    L.oracle_transform_compose(P(c(kat["tr_a"])), P(c(kat["tr_b"])), P(out), C.c_uint32(n))
    assert np.array_equal(out[:, :52], kat["compose"][:, :52])  # math.cpp:801-807 (bytes 52..55 are struct padding)
    qa, qb, v, v2, t = (c(kat[k]) for k in ("qa", "qb", "v", "v2", "t"))
    o4, o3 = np.zeros((n, 4), np.float32), np.zeros((n, 3), np.float32)
    L.oracle_quat_mul(P(qa), P(qb), P(o4), C.c_uint32(n)); assert np.array_equal(bits(o4), bits(kat["quat_mul"]))
    L.oracle_quat_rotate(P(qa), P(v), P(o3), C.c_uint32(n)); assert np.array_equal(bits(o3), bits(kat["quat_rotate"]))
    L.oracle_nlerp(P(qa), P(qb), P(t), P(o4), C.c_uint32(n), C.c_int(0)); assert np.array_equal(bits(o4), bits(kat["nlerp"]))
    L.oracle_nlerp(P(qa), P(qb), P(t), P(o4), C.c_uint32(n), C.c_int(1)); assert np.array_equal(bits(o4), bits(kat["simd_nlerp"]))
    L.oracle_lerp_vec3(P(v), P(v2), P(t), P(o3), C.c_uint32(n)); assert np.array_equal(bits(o3), bits(kat["lerp"]))
    la, lb_ = c(kat["lrt_a"]), c(kat["lrt_b"])
    o7, o8, o16 = np.zeros((n, 7), np.float32), np.zeros((n, 8), np.float32), np.zeros((n, 16), np.float32)
    L.oracle_lrt_mul(P(la), P(lb_), P(o7), C.c_uint32(n)); assert np.array_equal(bits(o7), bits(kat["lrt_mul"]))
    L.oracle_lrt_inverted(P(la), P(o7), C.c_uint32(n)); assert np.array_equal(bits(o7), bits(kat["lrt_inverted"]))
    L.oracle_lrt_to_matrix(P(la), P(o16), C.c_uint32(n)); assert np.array_equal(bits(o16), bits(kat["lrt_to_matrix"]))
    L.oracle_lrt_to_dual_quat(P(la), P(o8), C.c_uint32(n))
    # the reference's SSE toDualQuat negates with 0 - x (simd.h:187-189): results agree except for the sign of zero
    assert np.array_equal(o8, kat["lrt_to_dual_quat"])
    got = oracle.skin_vertices(kat["skin_palette"], v, kat["skin_w"], kat["skin_idx"])
    assert np.array_equal(bits(got), bits(kat["skin_out"]))  # model.cpp:103-109


def test_cell_indices_and_rng(oracle, kat):
    L = oracle.lib()
    cp = np.ascontiguousarray(kat["cell_pos"])
    out = np.zeros(3, np.int32)
    for p, exp in zip(cp, kat["cell_idx"]):
        L.oracle_cell_indices(P(p), C.c_float(300.0), P(out))
        assert tuple(out) == tuple(exp)
    r, _ = oracle.rng_floats(521288629, 362436069, 64)
    assert np.array_equal(bits(r), bits(kat["rng64"]))  # math.cpp:1333-1378


def test_frustum_construction_and_cell_tests(oracle, kat):
    L = oracle.lib()
    k = 0
    for args, exp in zip(kat["fr_args"], kat["fr_out"]):
        pos, dirv, up = args[0:3], args[3:6].astype(np.float32), args[6:9].astype(np.float32)
        fov, ratio, near, far, persp = args[9:14]
        f = oracle.frustum_perspective(pos, dirv, up, fov, ratio, near, far) if persp else oracle.frustum_ortho(pos, dirv, up, 50 + far * 0.1, 30 + far * 0.05, 0.0, far)
        assert np.array_equal(f[:248], exp[:248])  # geometry.cpp:390-409,470-499
        for _ in range(25):
            o = np.ascontiguousarray(kat["rel_origin"][k])
            rel = np.zeros(224, np.uint8)
            L.oracle_frustum_get_relative.argtypes = None
            # ODVec3 by value: pass through a tiny struct
            class D3(C.Structure):
                _fields_ = [("x", C.c_double), ("y", C.c_double), ("z", C.c_double)]

            class V3(C.Structure):
                _fields_ = [("x", C.c_float), ("y", C.c_float), ("z", C.c_float)]
            L.oracle_frustum_get_relative(P(f), D3(*o), P(rel))
            assert np.array_equal(rel[:128], kat["rel_out"][k])  # the 8 planes; geometry.cpp:121-149
            sz = kat["box_size"][k]
            assert L.oracle_frustum_contains_aabb(P(f), D3(*kat["box_pos"][k]), V3(*sz)) == kat["box_contains"][k]
            assert L.oracle_frustum_intersects_aabb(P(f), D3(*kat["box_pos"][k]), V3(*sz)) == kat["box_intersects"][k]
            k += 1
    assert kat["box_contains"].sum() > 5 and kat["box_intersects"].sum() > 50  # the fixture exercises both outcomes


def test_cull_visible_sets(oracle):
    """Sorted visible ids (+ types) of the reference's CullingSystemImpl on its own job system."""
    g = np.load(os.path.join(G, "cull_kat.npz"))
    scene = scenes.cull_scene(30_000, (2500.0, 300.0, 2500.0), seed=31, big_fraction=0.01, type_probs=(0.7, 0.2, 0.1))
    oc = oracle.OracleCulling()
    oc.add(scene["entities"], scene["types"], scene["pos"], scene["radius"])

    def check(prefix):
        for i, f in enumerate(g["frusta"]):
            ids, tys, _ = oc.cull(f)
            o = np.argsort(ids)
            assert np.array_equal(ids[o], g[f"{prefix}{i}_ids"]) and np.array_equal(tys[o], g[f"{prefix}{i}_types"])
            assert len(ids) > 100
            if prefix == "vis":
                for t in range(3):
                    it, _, _ = oc.cull(f, type=t)
                    assert np.array_equal(np.sort(it), g[f"vis{i}_type{t}"])
    check("vis")
    oc.set_position(g["edit_a"], g["edit_pa"]); oc.set_radius(g["edit_b"], g["edit_rb"]); oc.set(g["edit_c"], g["edit_pc"], g["edit_rc"]); oc.remove(g["edit_e"])
    check("edited")
    # special radii (NaN of either sign, infinities, -0.0, negative): the sign bit movemask sees is the reference's
    rad = g["special_radius_bits"].view(np.float32)
    n = len(rad)
    os_ = oracle.OracleCulling()
    os_.add(np.arange(n, dtype=np.int32), np.zeros(n, np.uint8), g["special_pos"], rad)
    ids, _, _ = os_.cull(g["frusta"][0])
    assert np.array_equal(np.sort(ids), g["special_visible"])
    vis = set(int(i) for i in ids)
    assert not any(i in vis for i in range(100))          # +NaN radius: culled by every plane
    assert all(i in vis for i in range(100, 200))          # -NaN radius: passes every plane, wherever the sphere is


def test_pose_sampling_and_absolute(oracle):
    """Animation::getRelativePose (weight 1 and blended) + Pose::computeAbsolute from the reference build."""
    g = np.load(os.path.join(G, "pose_kat.npz"))
    cfgs = [(24, 17, 30.0, (11, 13, 16), (12, 14, 16), 0.25), (64, 60, 30.0, (16, 16, 16), (15, 15, 15), 0.25), (7, 3, 1.0, (5, 3, 7), (9, 9, 9), 0.0)]
    for k, (bones, frames, fps, pb, rb, cf) in enumerate(cfgs):
        sk = scenes.skeleton(bones, seed=40 + k)
        clip = scenes.clip(sk, frames=frames, fps=fps, seed=50 + k, pos_bits=pb, rot_bits=rb, const_fraction=cf)
        assert clip.length_ticks == int(g[f"c{k}_length"][0])
        L = clip.length_ticks
        for j, t in enumerate(g[f"c{k}_times"]):
            rel = np.concatenate(oracle.pose_evaluate(sk, clip, t, compute_absolute=False), axis=1)
            assert np.array_equal(bits(rel), bits(g[f"c{k}_rel"][j])), (k, t)
            ab = np.concatenate(oracle.pose_evaluate(sk, clip, t, compute_absolute=True), axis=1)
            assert np.array_equal(bits(ab), bits(g[f"c{k}_abs"][j])), (k, t)
            # dual-quaternion palette of that pose: the reference's own PipelineImpl::computeSkeletonDualQuats (4-wide SIMD batches +
            # scalar tail, pipeline.cpp:2680-2745), cut out of pipeline.cpp at build time by oracle/build_ref.sh
            dq, mtx = oracle.palettes(sk, ab[:, :3], ab[:, 3:])
            assert np.array_equal(bits(dq), bits(g[f"c{k}_dq"][j])), (k, t)
            if j < len(g[f"c{k}_mtx"]):  # computeSkinMatrices (model.cpp:132-137), and evaluateSkin (model.cpp:103-109) on a 300-vertex mesh
                assert np.array_equal(bits(mtx), bits(g[f"c{k}_mtx"][j])), (k, t)
                if j < len(g[f"c{k}_skinned"]):
                    mesh = scenes.mesh(sk, 300, seed=60 + k)
                    v = oracle.skin_vertices(mtx, mesh.positions, mesh.weights, mesh.indices)
                    assert np.array_equal(bits(v), bits(g[f"c{k}_skinned"][j])), (k, t)
            bl = np.concatenate(oracle.pose_evaluate(sk, clip, (int(t) * 7 + 11) % max(L, 1), weight=0.37, start_from_bind=False, compute_absolute=False,
                                                     pos=rel[:, :3], rot=rel[:, 3:]), axis=1)
            assert np.array_equal(bits(bl), bits(g[f"c{k}_blend"][j])), (k, t)
    for t, dt, fps, fc, exp in g["time_advance"]:  # animation_module.cpp:458-469 through the reference's own Time operators
        assert oracle.time_advance(int(t), float(dt), float(fps), int(fc)) == int(exp), (t, dt, fps, fc)
    for s, exp in zip(g["time_from_seconds_in"], g["time_from_seconds_out"]):
        assert int(np.uint32(np.float32(s) * np.float32(32768))) == int(exp)  # Time::fromSeconds, animation.h:21-24


def test_relative_matrices(oracle):
    """World::getRelativeMatrix (world.cpp:370-377): the restatement against the reference's own toMatrix/setTranslation/multiply3x3."""
    k = np.load(os.path.join(G, "world_kat.npz"))
    for i, base in enumerate(k["bases"]):
        got = oracle.relative_matrices(k["tr"], base)
        assert np.array_equal(got.view(np.uint32), k[f"rel{i}"].view(np.uint32))


def test_compute_local(oracle):
    """Transform::computeLocal (math.cpp:809-816) against the reference's own function, and as the inverse of compose."""
    k = np.load(os.path.join(G, "world_kat.npz"))
    got = oracle.transform_compute_local(k["cl_parent"], k["cl_child"])
    assert np.array_equal(got[:, :52], k["cl_out"][:, :52])
    # compose(parent, computeLocal(parent, child)) comes back to child within rounding (fp64 position, fp32 rotation / scale)
    dt = np.dtype({"names": ["pos", "rot", "scale"], "formats": [(np.float64, 3), (np.float32, 4), (np.float32, 3)], "offsets": [0, 24, 40], "itemsize": 56})
    back = oracle.transform_compose(k["cl_parent"], got).view(dt).reshape(-1)
    child = k["cl_child"].view(dt).reshape(-1)
    assert np.allclose(back["pos"], child["pos"], rtol=0, atol=2e-3 * (1 + np.abs(child["pos"]).max() * 1e-6))
    assert np.allclose(back["scale"], child["scale"], rtol=1e-5)
    assert np.allclose(np.abs((back["rot"] * child["rot"]).sum(1)), 1.0, atol=1e-5)


def test_pose_compute_relative_and_blend(oracle):
    """Pose::computeRelative (pose.cpp:136-146) and Pose::blend (pose.cpp:30-41) against outputs of the reference's own pose.cpp."""
    from lumixengine_b200 import scenes
    k = np.load(os.path.join(G, "pose_kat.npz"))
    sk = scenes.skeleton(24, seed=40)
    for i in range(len(k["c0_abs"])):
        p, r = oracle.pose_compute_relative(sk, k["c0_abs"][i][:, :3], k["c0_abs"][i][:, 3:])
        assert np.array_equal(np.concatenate([p, r], 1).view(np.uint32), k["c0_abs_to_rel"][i].view(np.uint32))
    rel = k["c0_rel"]
    for j, w in enumerate(k["blend_weights"]):
        rb = -rel[-1][:, 3:] if w == 0.5 else rel[-1][:, 3:]  # the negative-dot branch of nlerp
        p, r = oracle.pose_blend(rel[0][:, :3], rel[0][:, 3:], rel[-1][:, :3], rb, float(w))
        assert np.array_equal(np.concatenate([p, r], 1).view(np.uint32), k["pose_blend"][j].view(np.uint32)), float(w)
    # weights at or below 0.001 leave the pose untouched (pose.cpp:33)
    assert np.array_equal(k["pose_blend"][0], rel[0]) and np.array_equal(k["pose_blend"][1], rel[0])


def test_viewport_frustum(oracle):
    """Viewport::getFrustum() (geometry.cpp:793-818) from the reference build: the restatement and the product's host builder
    (lb200_frustum_from_viewport needs no GPU) both reproduce its bytes (the last 8 of the 256 are padding)."""
    import lumixengine_b200 as lb
    k = np.load(os.path.join(G, "world_kat.npz"))
    for a, exp in zip(k["vp_args"], k["vp_out"]):
        is_ortho, fov, osz, w, h = bool(a[0]), float(np.float32(a[1])), float(np.float32(a[2])), int(a[3]), int(a[4])
        pos, rot, near, far = a[5:8], a[8:12].astype(np.float32), float(np.float32(a[12])), float(np.float32(a[13]))
        got = oracle.frustum_from_viewport(pos, rot, fov, w, h, near, far, is_ortho, osz)
        assert np.array_equal(got[:248], exp[:248])
        prod = lb.culling.frustum_bytes(lb.frustum_from_viewport(pos, rot, fov, w, h, near, far, is_ortho, osz))
        assert np.array_equal(prod[:248], exp[:248])


def test_sphere_refresh_radius(oracle):
    """render_module.cpp:1554 bounding_radius * maximum(scale.x, scale.y, scale.z) with the reference's variadic maximum (math.h:468-475),
    including NaN scales (a NaN in z propagates, a NaN in x or y is dropped by the comparisons)."""
    k = np.load(os.path.join(G, "world_kat.npz"))
    got = oracle.sphere_radius(k["sr_tr"], k["sr_bound"])
    exp = k["sr_out"]
    assert np.isnan(exp).sum() > 0
    assert np.array_equal(np.isnan(got), np.isnan(exp))
    assert np.array_equal(got[~np.isnan(exp)].view(np.uint32), exp[~np.isnan(exp)].view(np.uint32))


def test_ani_image_loader():
    """AnimationClip.from_ani_bytes against what the reference's own Animation::load (animation.cpp:397-493) parsed out of the same
    compiled .ani images (tests/golden/ani_kat.npz), and to_ani_bytes reproduces the images byte for byte."""
    from lumixengine_b200.animation import AnimationClip, TRACK_DTYPE
    k = np.load(os.path.join(G, "ani_kat.npz"))
    cfgs = [(24, 17, 0.25, (11, 13, 16), (12, 14, 16)), (64, 60, 0.25, (16, 16, 16), (15, 15, 15)), (7, 3, 0.0, (5, 3, 7), (9, 9, 9)), (5, 9, 1.0, (16, 16, 16), (15, 15, 15))]
    for i, (bones, frames, cf, pb, rb) in enumerate(cfgs):
        img, hashes = k[f"a{i}_image"].tobytes(), k[f"a{i}_hashes"]
        h2b = {int(h): b for b, h in enumerate(hashes)}
        clip = AnimationClip.from_ani_bytes(img, h2b)
        fc, t_bits, r_bits, n_t, n_ct, n_r, n_cr, t_off, r_off, mem = (int(v) for v in k[f"a{i}_scalars"])
        assert (clip.frame_count, clip.translations_frame_size_bits, clip.rotations_frame_size_bits) == (fc, t_bits, r_bits)
        assert np.float32(clip.fps) == k[f"a{i}_fps"][0]
        assert (len(clip.translations), len(clip.const_translations), len(clip.rotations), len(clip.const_rotations)) == (n_t, n_ct, n_r, n_cr)
        for mine, ref, hs in ((clip.translations, k[f"a{i}_t"], k[f"a{i}_t_hash"]), (clip.rotations, k[f"a{i}_r"], k[f"a{i}_r_hash"])):
            ref = ref.reshape(-1).view(TRACK_DTYPE) if len(ref) else np.zeros(0, TRACK_DTYPE)
            assert np.array_equal([h2b[int(h)] for h in hs], mine["bone_index"])  # onBeforeReady's resolution (animation.cpp:366-395)
            for f in ("offset_bits", "bitsizes", "skipped_channel", "min", "to_range"):
                assert np.ascontiguousarray(ref[f]).tobytes() == np.ascontiguousarray(mine[f]).tobytes(), f
        assert np.array_equal([h2b[int(h)] for h in k[f"a{i}_ct_hash"]], clip.const_translations["bone_index"])
        assert k[f"a{i}_ct_value"].tobytes() == np.ascontiguousarray(clip.const_translations["value"]).tobytes()
        assert np.array_equal([h2b[int(h)] for h in k[f"a{i}_cr_hash"]], clip.const_rotations["bone_index"])
        assert k[f"a{i}_cr_value"].tobytes() == np.ascontiguousarray(clip.const_rotations["value"]).tobytes()
        body = img[24:]
        n_t_bytes, n_r_bytes = (t_bits * (fc + 1) + 7) // 8, (r_bits * (fc + 1) + 7) // 8
        assert body[t_off:t_off + n_t_bytes] == bytes(clip.translation_stream[:n_t_bytes])
        assert body[r_off:r_off + n_r_bytes] == bytes(clip.rotation_stream[:n_r_bytes])
        assert mem == len(body) + 8  # the loader's 8-byte unpacker padding, animation.cpp:439
        # and the writer is the inverse of the loader
        sk = scenes.skeleton(bones, seed=bones)
        orig = scenes.clip(sk, frames=frames, seed=bones + 3, pos_bits=pb, rot_bits=rb, const_fraction=cf)
        assert orig.to_ani_bytes(hashes) == img
        assert clip.to_ani_bytes(hashes) == img


def test_skeleton_derivation_follows_parse_bones(oracle):
    """Skeleton derives the inverse bind pose and the relative bind transforms the way Model::parseBones does (model.cpp:389-421:
    invert(transform) = LocalRigidTransform::inverted's formula, relative = inverse_bind(parent) * transform).  Both primitives are pinned
    against the reference build (math_kat: lrt_inverted, lrt_mul); here the numpy derivation must equal them bit for bit."""
    L = oracle.lib()
    for bones in (1, 5, 24, 64, 196):
        sk = scenes.skeleton(bones, seed=100 + bones)
        abs7 = np.ascontiguousarray(sk.bind_abs7, np.float32)
        inv = np.zeros_like(abs7)
        L.oracle_lrt_inverted(P(abs7), P(inv), C.c_uint32(bones))
        assert np.array_equal(bits(inv), bits(sk.inverse_bind7))
        par = np.maximum(sk.parents, 0)
        rel = np.zeros_like(abs7)
        L.oracle_lrt_mul(P(np.ascontiguousarray(inv[par])), P(abs7), P(rel), C.c_uint32(bones))
        rel[sk.parents < 0] = abs7[sk.parents < 0]  # roots keep their transform (model.cpp:416-419)
        assert np.array_equal(bits(rel), bits(sk.bind_relative7))
        assert all(int(p) < i for i, p in enumerate(sk.parents))  # parent < child, model.cpp:381-384


def test_bone_attachments(oracle):
    """RenderModuleImpl::updateBoneAttachment (render_module.cpp:399-403) against the reference's own Transform::compose(LocalRigidTransform)
    and LocalRigidTransform::operator*."""
    k = np.load(os.path.join(G, "world_kat.npz"))
    got = oracle.bone_attachments(k["ba_parent"], k["ba_bone"], k["ba_rel"], k["ba_scale"])
    assert np.array_equal(got[:, :52], k["ba_out"][:, :52])
