"""Generates tests/golden/*.npz from the REFERENCE'S OWN compiled code (oracle/_ref/libref_lumix.so, built by
oracle/build_ref.sh from /root/reference).  Run in the build container only:  python tests/golden/make_golden.py

The reference has no golden vectors of its own for this path (SURVEY.md F9), so these reference-run outputs are the pin:
inputs are seeded numpy draws, outputs come from unmodified math.cpp / geometry.cpp / culling_system.cpp / pose.cpp /
animation.cpp.  tests/test_oracle_golden.py replays them against the restatement on any box.
"""
import ctypes as C
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from lumixengine_b200 import scenes  # noqa: E402  (numpy input generators)
from oracle import pyoracle as po  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
P = lambda a: a.ctypes.data_as(C.c_void_p)  # noqa: E731


def unit_quats(rng, n):
    q = rng.normal(size=(n, 4)).astype(np.float32)
    return (q / np.linalg.norm(q, axis=1, keepdims=True)).astype(np.float32)


def math_kat():
    L = po.ref()
    rng = np.random.default_rng(1234)
    n = 2000
    tr_dtype = np.dtype({"names": ["pos", "rot", "scale"], "formats": [(np.float64, 3), (np.float32, 4), (np.float32, 3)], "offsets": [0, 24, 40], "itemsize": 56})
    a = np.zeros(n, tr_dtype); b = np.zeros(n, tr_dtype)
    for t, s in ((a, 1e5), (b, 50.0)):
        t["pos"] = rng.normal(size=(n, 3)) * s
        t["rot"] = unit_quats(rng, n)
        t["scale"] = (0.5 + rng.random((n, 3))).astype(np.float32)
    out = np.zeros(n, tr_dtype)
    L.ref_transform_compose(P(a), P(b), P(out), C.c_uint32(n))
    d = dict(tr_a=a.view(np.uint8).reshape(n, 56), tr_b=b.view(np.uint8).reshape(n, 56), compose=out.view(np.uint8).reshape(n, 56))
    qa, qb = unit_quats(rng, n), unit_quats(rng, n)
    qb[: n // 4] = -qa[: n // 4] + rng.normal(size=(n // 4, 4)).astype(np.float32) * 0.01  # negative-dot branch of nlerp
    v = (rng.normal(size=(n, 3)) * 10).astype(np.float32)
    v2 = (rng.normal(size=(n, 3)) * 10).astype(np.float32)
    t = rng.random(n).astype(np.float32)
    o4 = np.zeros((n, 4), np.float32); o3 = np.zeros((n, 3), np.float32)
    L.ref_quat_mul(P(qa), P(qb), P(o4), C.c_uint32(n)); d.update(qa=qa, qb=qb, quat_mul=o4.copy())
    L.ref_quat_rotate(P(qa), P(v), P(o3), C.c_uint32(n)); d.update(v=v, quat_rotate=o3.copy())
    L.ref_nlerp(P(qa), P(qb), P(t), P(o4), C.c_uint32(n), C.c_int(0)); d.update(t=t, nlerp=o4.copy())
    L.ref_nlerp(P(qa), P(qb), P(t), P(o4), C.c_uint32(n), C.c_int(1)); d.update(simd_nlerp=o4.copy())
    L.ref_lerp_vec3(P(v), P(v2), P(t), P(o3), C.c_uint32(n)); d.update(v2=v2, lerp=o3.copy())
    la = np.concatenate([v, qa], axis=1).astype(np.float32); lb_ = np.concatenate([v2, qb], axis=1).astype(np.float32)
    o7 = np.zeros((n, 7), np.float32); o8 = np.zeros((n, 8), np.float32); o16 = np.zeros((n, 16), np.float32)
    L.ref_lrt_mul(P(la), P(lb_), P(o7), C.c_uint32(n)); d.update(lrt_a=la, lrt_b=lb_, lrt_mul=o7.copy())
    L.ref_lrt_inverted(P(la), P(o7), C.c_uint32(n)); d.update(lrt_inverted=o7.copy())
    L.ref_lrt_to_dual_quat(P(la), P(o8), C.c_uint32(n)); d.update(lrt_to_dual_quat=o8.copy())
    L.ref_lrt_to_matrix(P(la), P(o16), C.c_uint32(n)); d.update(lrt_to_matrix=o16.copy())
    # skinning of n vertices against a 32-matrix palette
    pal = np.zeros((32, 16), np.float32)
    pl = np.concatenate([(rng.normal(size=(32, 3)) * 3).astype(np.float32), unit_quats(rng, 32)], axis=1).astype(np.float32)
    L.ref_lrt_to_matrix(P(pl), P(pal), C.c_uint32(32))
    w = rng.random((n, 4)); w = (np.round(w / w.sum(1, keepdims=True) * 65535) / 65535.0).astype(np.float32)
    idx = rng.integers(0, 32, (n, 4)).astype(np.int16)
    L.ref_skin_vertex(P(pal), P(v), P(w), P(idx), P(o3), C.c_uint32(n)); d.update(skin_palette=pal, skin_w=w, skin_idx=idx, skin_out=o3.copy())
    # cell indices incl. negative coordinates and exact multiples of 300
    cp = np.concatenate([rng.normal(size=(500, 3)) * 2000, (rng.integers(-8, 9, (200, 3)) * 300.0), (rng.integers(-8, 9, (200, 3)) * 300.0) - 1e-9])
    ci = np.zeros((len(cp), 3), np.int32)
    for i in range(len(cp)):
        L.ref_cell_indices(P(cp[i]), C.c_float(300.0), P(ci[i]))
    d.update(cell_pos=cp, cell_idx=ci)
    # frustums: construction, getRelative, contains / intersects
    fr_args, fr_out, rel_origin, rel_out, box_pos, box_size, box_c, box_i = [], [], [], [], [], [], [], []
    for k in range(40):
        pos = rng.normal(size=3) * (1000.0 if k % 2 else 1e6)
        dirv = rng.normal(size=3); dirv /= np.linalg.norm(dirv)
        up = np.cross(np.cross(dirv, rng.normal(size=3)), dirv); up /= np.linalg.norm(up)
        fov, ratio, near, far = 0.3 + rng.random() * 1.5, 0.5 + rng.random() * 2, 0.05 + rng.random(), 100 + rng.random() * 5000
        f = po.ref_frustum_perspective(pos, dirv.astype(np.float32), up.astype(np.float32), fov, ratio, near, far) if k % 4 else \
            po.ref_frustum_ortho(pos, dirv.astype(np.float32), up.astype(np.float32), 50 + far * 0.1, 30 + far * 0.05, 0.0, far)
        fr_args.append(np.concatenate([pos, dirv, up, [fov, ratio, near, far, float(k % 4 != 0)]]))
        fr_out.append(f.copy())
        for j in range(25):
            o = pos + rng.normal(size=3) * far * 0.7
            o = np.floor(o / 300.0) * 300.0
            rel = np.zeros(224, np.uint8)
            L.ref_frustum_get_relative(P(f), P(o), P(rel))
            rel_origin.append(o); rel_out.append(rel)
            sz = np.float32(300.0 * (1 + j % 2))
            size = np.array([sz, sz, sz], np.float32)
            box_pos.append(o); box_size.append(size)
            box_c.append(L.ref_frustum_contains_aabb(P(f), P(o), P(size)))
            box_i.append(L.ref_frustum_intersects_aabb(P(f), P(o), P(size)))
    d.update(fr_args=np.array(fr_args), fr_out=np.array(fr_out), rel_origin=np.array(rel_origin), rel_out=np.array(rel_out)[:, :128],
             box_pos=np.array(box_pos), box_size=np.array(box_size), box_contains=np.array(box_c, np.int8), box_intersects=np.array(box_i, np.int8))
    # RNG
    r = np.zeros(64, np.float32)
    L.ref_rng_floats(C.c_uint32(521288629), C.c_uint32(362436069), C.c_uint32(64), P(r), None)
    d.update(rng64=r)
    # two files, each under 1 MB: the cell / frustum / RNG vectors go to math_kat_frustum.npz
    frustum = ("cell_pos", "cell_idx", "fr_args", "fr_out", "rel_origin", "rel_out", "box_pos", "box_size", "box_contains", "box_intersects", "rng64")
    np.savez_compressed(os.path.join(OUT, "math_kat.npz"), **{k: v for k, v in d.items() if k not in frustum})
    np.savez_compressed(os.path.join(OUT, "math_kat_frustum.npz"), **{k: d[k] for k in frustum})
    print("math_kat.npz + math_kat_frustum.npz", sum(v.nbytes for v in d.values()))


def cull_kat():
    """Visible sets of the reference's CullingSystemImpl (on its own job system, 4 workers) for seeded scenes, incl. incremental edits."""
    d = {}
    rng = np.random.default_rng(99)
    scene = scenes.cull_scene(30_000, (2500.0, 300.0, 2500.0), seed=31, big_fraction=0.01, type_probs=(0.7, 0.2, 0.1))
    rc = po.RefCulling(workers=4)
    rc.add(scene["entities"], scene["types"], scene["pos"], scene["radius"])
    frusta = [dict(scenes.c1_frustum_args()),
              dict(scenes.c1_frustum_args(), position=(700.0, 40.0, -300.0), direction=(-0.5, -0.05, -0.8), far=2500.0),
              dict(scenes.c1_frustum_args(), position=(-2000.0, 0.0, 2000.0), direction=(1.0, 0.0, -1.0), far=6000.0, fov=0.35)]
    fb = [po.ref_frustum_perspective(a["position"], a["direction"], a["up"], a["fov"], a["ratio"], a["near"], a["far"]) for a in frusta]
    d["frusta"] = np.array(fb)
    for i, f in enumerate(fb):
        ids, tys, info = rc.cull(f, cap=30_000)
        o = np.argsort(ids)
        d[f"vis{i}_ids"], d[f"vis{i}_types"] = ids[o], tys[o]
        for t in range(3):
            ids_t, _, _ = rc.cull(f, type=t, cap=30_000)
            d[f"vis{i}_type{t}"] = np.sort(ids_t)
    # incremental edits, then cull again
    mv = rng.choice(30_000, 4000, replace=False).astype(np.int32)
    a, b, c, e = np.array_split(mv, 4)
    pa = scene["pos"][a] + rng.normal(size=(len(a), 3)) * np.array([500.0, 50.0, 500.0])
    rb = (rng.random(len(b)) * 650).astype(np.float32)
    pc = scene["pos"][c] * 0.3; rcc = (rng.random(len(c)) * 400).astype(np.float32)
    rc.set_position(a, pa); rc.set_radius(b, rb); rc.set(c, pc, rcc); rc.remove(e)
    d.update(edit_a=a, edit_pa=pa, edit_b=b, edit_rb=rb, edit_c=c, edit_pc=pc, edit_rc=rcc, edit_e=e)
    for i, f in enumerate(fb):
        ids, tys, _ = rc.cull(f, cap=30_000)
        o = np.argsort(ids)
        d[f"edited{i}_ids"], d[f"edited{i}_types"] = ids[o], tys[o]
    # special radii: +NaN / -NaN / +-inf / -0.0 / negative.  movemask reads sign bits, and t - (-radius) hands a NaN radius through with its
    # sign flipped: a +NaN radius is culled by every plane, a -NaN radius passes every plane (even outside the frustum)
    rs = np.random.default_rng(3)
    ns = 2000
    spos = np.stack([rs.uniform(-250, 250, ns), rs.uniform(-100, 100, ns), rs.uniform(-900, -100, ns)], 1)
    srad = np.full(ns, 2.0, np.float32)
    srad[:100] = np.nan
    srad[100:200] = np.array([0xFFC00000], np.uint32).view(np.float32)[0]
    srad[200:300] = np.inf; srad[300:400] = -np.inf; srad[400:500] = -0.0; srad[500:600] = -3.5
    rs2 = po.RefCulling(workers=4)
    rs2.add(np.arange(ns, dtype=np.int32), np.zeros(ns, np.uint8), spos, srad)
    sids, _, _ = rs2.cull(fb[0], cap=ns)
    d.update(special_pos=spos, special_radius_bits=srad.view(np.uint32), special_visible=np.sort(sids))
    np.savez_compressed(os.path.join(OUT, "cull_kat.npz"), **d)
    print("cull_kat.npz", sum(v.nbytes for v in d.values()))


def pose_kat():
    """The reference's Animation::getRelativePose + Pose::computeAbsolute on synthetic clips (bit widths 5..16)."""
    d = {}
    cfgs = [(24, 17, 30.0, (11, 13, 16), (12, 14, 16), 0.25), (64, 60, 30.0, (16, 16, 16), (15, 15, 15), 0.25), (7, 3, 1.0, (5, 3, 7), (9, 9, 9), 0.0)]
    for k, (bones, frames, fps, pb, rb, cf) in enumerate(cfgs):
        sk = scenes.skeleton(bones, seed=40 + k)
        clip = scenes.clip(sk, frames=frames, fps=fps, seed=50 + k, pos_bits=pb, rot_bits=rb, const_fraction=cf)
        L = clip.length_ticks
        times = np.unique(np.concatenate([[0, 1, L // 3, L // 2, L - 1, L, L + 12345, 2 ** 31], np.random.default_rng(k).integers(0, L, 40)])).astype(np.uint32)
        rel, abs_, blend = [], [], []
        for t in times:
            rel.append(np.concatenate(po.ref_pose_evaluate(sk, clip, t, compute_absolute=False), axis=1))
            abs_.append(np.concatenate(po.ref_pose_evaluate(sk, clip, t, compute_absolute=True), axis=1))
            p0, r0 = rel[-1][:, :3], rel[-1][:, 3:]
            blend.append(np.concatenate(po.ref_pose_evaluate(sk, clip, (int(t) * 7 + 11) % max(L, 1), weight=0.37, start_from_bind=False,
                                                              compute_absolute=False, pos=p0, rot=r0), axis=1))
        d[f"c{k}_times"] = times
        d[f"c{k}_rel"], d[f"c{k}_abs"], d[f"c{k}_blend"] = np.array(rel), np.array(abs_), np.array(blend)
        # PipelineImpl::computeSkeletonDualQuats (the reference's own SIMD + scalar-tail code) on the absolute poses
        d[f"c{k}_dq"] = np.array([po.ref_skeleton_dual_quats(sk, a[:, :3], a[:, 3:]) for a in abs_])
        # the reference's own computeSkinMatrices / evaluateSkin (file statics of model.cpp, cut out at build time) on the same poses
        d[f"c{k}_mtx"] = np.array([po.ref_skin_matrices(sk, a[:, :3], a[:, 3:]) for a in abs_[:12]])
        mesh = scenes.mesh(sk, 300, seed=60 + k)
        d[f"c{k}_skinned"] = np.array([po.ref_evaluate_skin(m, mesh.positions, mesh.weights, mesh.indices) for m in d[f"c{k}_mtx"][:4]])
        d[f"c{k}_length"] = np.array([po.ref().ref_clip_length_ticks(C.c_float(clip.fps), C.c_uint32(clip.frame_count))], np.uint32)
    # Pose::computeRelative and Pose::blend on the poses above (reference's own pose.cpp)
    abs0 = d["c0_abs"]
    sk = scenes.skeleton(cfgs[0][0], seed=40)  # the skeleton of config 0
    rel_back, blends = [], []
    for i in range(len(abs0)):
        p, r = po.pose_compute_relative(sk, abs0[i][:, :3], abs0[i][:, 3:], use_ref=True)
        rel_back.append(np.concatenate([p, r], axis=1))
    d["c0_abs_to_rel"] = np.array(rel_back)
    rel0 = d["c0_rel"]
    d["blend_weights"] = np.array([0.0005, 0.001, 0.0011, 0.25, 0.5, 0.9999, 1.0, 1.7, -0.3], np.float32)
    for w in d["blend_weights"]:
        p, r = po.pose_blend(rel0[0][:, :3], rel0[0][:, 3:], rel0[-1][:, :3], -rel0[-1][:, 3:] if w == 0.5 else rel0[-1][:, 3:], float(w), use_ref=True)
        blends.append(np.concatenate([p, r], axis=1))
    d["pose_blend"] = np.array(blends)
    # time step of updateAnimable through the reference's Time operators: (ticks, time_delta, fps, frame_count) -> ticks
    rng = np.random.default_rng(77)
    rows = []
    for fps, fc in ((30.0, 60), (24.0, 37), (1.0, 3), (29.97, 1000)):
        l = po.ref().ref_clip_length_ticks(C.c_float(fps), C.c_uint32(fc))
        for dt in (1 / 60, 0.5, 3.7, -0.25, -1 / 60, -100.3, 0.0, 1e-6, -1e-6, 250.0):
            for t in rng.integers(0, l, 6):
                rows.append((float(t), dt, fps, float(fc), float(po.time_advance(t, dt, fps, fc, use_ref=True))))
    d["time_advance"] = np.array(rows, np.float64)
    d["time_from_seconds_in"] = np.array([0.0, 1 / 60, 1 / 30, 0.5, 3.7, 100.25], np.float32)
    d["time_from_seconds_out"] = np.array([po.ref().ref_time_from_seconds(C.c_float(float(x))) for x in d["time_from_seconds_in"]], np.uint32)
    np.savez_compressed(os.path.join(OUT, "pose_kat.npz"), **d)
    print("pose_kat.npz", sum(v.nbytes for v in d.values()))


def world_kat():
    """World::getRelativeMatrix (world.cpp:370-377) through the reference's Quat::toMatrix / setTranslation / multiply3x3."""
    rng = np.random.default_rng(4321)
    n = 1500
    tr_dtype = np.dtype({"names": ["pos", "rot", "scale"], "formats": [(np.float64, 3), (np.float32, 4), (np.float32, 3)], "offsets": [0, 24, 40], "itemsize": 56})
    t = np.zeros(n, tr_dtype)
    t["pos"] = rng.normal(size=(n, 3)) * np.where(rng.random((n, 1)) < 0.5, 1e3, 1e7)
    t["rot"] = unit_quats(rng, n)
    t["scale"] = (0.25 + 2 * rng.random((n, 3))).astype(np.float32)
    bases = np.array([[0.0, 0.0, 0.0], [1234.5, -20.25, 987.125], [9.99e6, 1e3, -1.0001e7]])
    d = dict(tr=t.view(np.uint8).reshape(n, 56), bases=bases)
    for k, b in enumerate(bases):
        d[f"rel{k}"] = po.ref_relative_matrices(d["tr"], b)
    # Transform::computeLocal (math.cpp:809-816): parents with non-uniform scale, children near and far from them
    par = np.zeros(n, tr_dtype); chi = np.zeros(n, tr_dtype)
    par["pos"] = rng.normal(size=(n, 3)) * np.where(rng.random((n, 1)) < 0.5, 1e3, 1e6)
    par["rot"] = unit_quats(rng, n)
    par["scale"] = (0.25 + 2 * rng.random((n, 3))).astype(np.float32)
    chi["pos"] = par["pos"] + rng.normal(size=(n, 3)) * np.where(rng.random((n, 1)) < 0.5, 5.0, 5e3)
    chi["rot"] = unit_quats(rng, n)
    chi["scale"] = (0.25 + 2 * rng.random((n, 3))).astype(np.float32)
    d["cl_parent"] = par.view(np.uint8).reshape(n, 56)
    d["cl_child"] = chi.view(np.uint8).reshape(n, 56)
    d["cl_out"] = po.transform_compute_local(d["cl_parent"], d["cl_child"], use_ref=True)
    # sphere refresh of onModelInstanceMoved (render_module.cpp:1554) incl. NaN / negative / equal scales
    sr = np.zeros(400, tr_dtype)
    sr["scale"] = (rng.normal(size=(400, 3)) * 2).astype(np.float32)
    sr["scale"][::13, 1] = np.nan; sr["scale"][::17, 0] = np.nan; sr["scale"][::19] = 1.5; sr["scale"][::23, 2] = np.inf; sr["scale"][::29, 2] = np.nan
    d["sr_tr"] = sr.view(np.uint8).reshape(400, 56)
    d["sr_bound"] = (rng.random(400) * 10).astype(np.float32)
    d["sr_out"] = po.sphere_radius(d["sr_tr"], d["sr_bound"], use_ref=True)
    # updateBoneAttachment (render_module.cpp:399-403): parents far from / near the origin, non-uniform scales
    nb = 600
    bp = np.zeros(nb, tr_dtype)
    bp["pos"] = rng.normal(size=(nb, 3)) * np.where(rng.random((nb, 1)) < 0.5, 1e3, 1e6)
    bp["rot"] = unit_quats(rng, nb)
    bp["scale"] = (0.25 + 2 * rng.random((nb, 3))).astype(np.float32)
    d["ba_parent"] = bp.view(np.uint8).reshape(nb, 56)
    d["ba_bone"] = np.concatenate([(rng.normal(size=(nb, 3)) * 2).astype(np.float32), unit_quats(rng, nb)], axis=1)
    d["ba_rel"] = np.concatenate([(rng.normal(size=(nb, 3)) * 0.5).astype(np.float32), unit_quats(rng, nb)], axis=1)
    d["ba_scale"] = (0.5 + rng.random((nb, 3))).astype(np.float32)
    d["ba_out"] = po.bone_attachments(d["ba_parent"], d["ba_bone"], d["ba_rel"], d["ba_scale"], use_ref=True)
    # Viewport::getFrustum() (geometry.cpp:793-818): args = is_ortho, fov, ortho_size, w, h, pos[3], rot[4], near, far
    vp_args, vp_out = [], []
    for k in range(120):
        q = rng.normal(size=4).astype(np.float32); q /= np.linalg.norm(q)
        pos = rng.normal(size=3) * (1e3 if k % 2 else 1e6)
        w, h = int(rng.integers(1, 4000)), (int(rng.integers(1, 3000)) if k % 17 else 0)
        fov, near, far = np.float32(0.2 + rng.random() * 2), np.float32(0.05 + rng.random()), np.float32(100 + rng.random() * 5000)
        ortho, osz = (k % 3 == 0), np.float32(10 + rng.random() * 500)
        vp_args.append(np.concatenate([[float(ortho), float(fov), float(osz), w, h], pos, q.astype(np.float64), [float(near), float(far)]]))
        vp_out.append(po.frustum_from_viewport(pos, q, float(fov), w, h, float(near), float(far), ortho, float(osz), use_ref=True))
    d["vp_args"], d["vp_out"] = np.array(vp_args), np.array(vp_out)
    np.savez_compressed(os.path.join(OUT, "world_kat.npz"), **d)
    print("world_kat.npz", sum(v.nbytes for v in d.values()))


def ani_kat():
    """Compiled .ani images written by AnimationClip.to_ani_bytes and what the reference's own Animation::load (animation.cpp:397-493)
    parsed out of them."""
    d = {}
    cfgs = [(24, 17, 0.25, (11, 13, 16), (12, 14, 16)), (64, 60, 0.25, (16, 16, 16), (15, 15, 15)), (7, 3, 0.0, (5, 3, 7), (9, 9, 9)), (5, 9, 1.0, (16, 16, 16), (15, 15, 15))]
    for k, (bones, frames, cf, pb, rb) in enumerate(cfgs):
        sk = scenes.skeleton(bones, seed=bones)
        clip = scenes.clip(sk, frames=frames, seed=bones + 3, pos_bits=pb, rot_bits=rb, const_fraction=cf)
        hashes = np.array([(0x9E3779B97F4A7C15 * (i + 1)) & 0xFFFFFFFFFFFFFFFF for i in range(bones)], np.uint64)
        img = clip.to_ani_bytes(hashes)
        L = po.ref_animation_load(img)
        assert L["ok"] == 1
        d[f"a{k}_image"] = np.frombuffer(img, np.uint8).copy()
        d[f"a{k}_hashes"] = hashes
        d[f"a{k}_scalars"] = np.array([L["frame_count"], L["t_bits"], L["r_bits"], L["n_t"], L["n_ct"], L["n_r"], L["n_cr"], L["t_stream_offset"], L["r_stream_offset"],
                                       L["mem_size"]], np.int64)
        d[f"a{k}_fps"] = np.array([L["fps"]], np.float32)
        for key in ("t_hash", "ct_hash", "r_hash", "cr_hash", "ct_value", "cr_value"):
            d[f"a{k}_{key}"] = L[key]
        d[f"a{k}_t"] = L["t"].view(np.uint8).reshape(-1, 32)
        d[f"a{k}_r"] = L["r"].view(np.uint8).reshape(-1, 32)
    np.savez_compressed(os.path.join(OUT, "ani_kat.npz"), **d)
    print("ani_kat.npz", sum(v.nbytes for v in d.values()))


def sortkeys_kat():
    """The reference's own sort-key packers, Model::getLODMeshIndices and PipelineImpl::radixSort (pipeline.cpp:53-143, 4020-4144; model.h:173-179),
    compiled from the reference file by oracle/build_ref.sh."""
    rng = np.random.default_rng(2024)
    R = po.sortkey_packers("ref")
    n = 600
    d = {}
    u32 = rng.integers(0, 2**32, n, dtype=np.uint64).astype(np.uint32)
    u32[:8] = [0, 1, 0x7fffffff, 0x80000000, 0xffffffff, 0x3f800000, 0xbf800000, 0x7f800000]
    buckets = rng.integers(0, 256, n).astype(np.uint8)
    ents = rng.integers(-3, 2**24, n).astype(np.int32)
    mesh_idx = rng.integers(0, 64, n).astype(np.uint32)
    depths = (rng.random(n) * 1e7).astype(np.float32)
    depths[:4] = [0.0, 1e-30, 3.4e38, 1.0]
    d.update(u32=u32, buckets=buckets, ents=ents, mesh_idx=mesh_idx, depths=depths)
    d["float_flip"] = np.array([R["float_flip"](int(x)) for x in u32], np.uint32)
    d["mesh_key"] = np.array([R["make_mesh_sort_key"](int(k), int(b)) for k, b in zip(u32, buckets)], np.uint64)
    d["depth_key"] = np.array([R["make_depth_sort_key"](float(x), int(b)) for x, b in zip(depths, buckets)], np.uint64)
    d["inst_key"] = np.array([R["make_autoinstanced_sort_key"](int(k & 0xffff), int(b)) for k, b in zip(u32, buckets)], np.uint64)
    d["decal_key"] = np.array([R["make_decal_sort_key"](int(k), int(b)) for k, b in zip(u32, buckets)], np.uint64)
    d["decal_value"] = np.array([R["make_decal_sort_value"](int(e)) for e in ents], np.uint64)
    d["curve_decal_value"] = np.array([R["make_curve_decal_sort_value"](int(e)) for e in ents], np.uint64)
    d["skinned_value"] = np.array([R["make_skinned_sort_value"](int(e), int(m)) for e, m in zip(ents, mesh_idx)], np.uint64)
    d["mesh_value"] = np.array([R["make_mesh_sort_value"](int(e), int(m)) for e, m in zip(ents, mesh_idx)], np.uint64)
    d["inst_value"] = np.array([R["make_autoinstanced_sort_value"](int(k & 0xffff), int(m)) for k, m in zip(u32, mesh_idx)], np.uint64)
    lodd = np.sort(rng.uniform(10.0, 1e6, (n, 4)).astype(np.float32), axis=1)
    lodd[::7, 2:] = np.finfo(np.float32).max
    sq = (rng.random(n) * 1.2e6).astype(np.float32)
    sq[:5] = [lodd[0, 0], lodd[1, 1], lodd[2, 2], lodd[3, 3], 0.0]
    d.update(lod_distances=lodd, squared=sq)
    d["lod_index"] = np.array([R["lod_mesh_indices"](lodd[i].ctypes.data_as(C.c_void_p), float(sq[i])) for i in range(n)], np.uint32)
    # radix sort: realistic key layouts (bucket byte, instanced flag, 32 low bits; runs of equal keys: the sort is stable)
    for name, size in (("tiny", 5), ("below_step", 511), ("above_step", 513), ("big", 20000)):
        keys = (rng.integers(0, 6, size).astype(np.uint64) << np.uint64(56)) | (rng.integers(0, 2, size).astype(np.uint64) << np.uint64(55)) | rng.integers(0, 3000, size).astype(np.uint64)
        vals = np.arange(size, dtype=np.uint64) | (rng.integers(0, 5, size).astype(np.uint64) << np.uint64(32))
        k, v = po.ref_radix_sort(keys, vals, workers=4)
        d[f"rs_{name}_keys"], d[f"rs_{name}_values"], d[f"rs_{name}_sorted_keys"], d[f"rs_{name}_sorted_values"] = keys, vals, k, v
    keys = rng.integers(0, 2**63, 3000, dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, 3000).astype(np.uint64)  # all 64 bits in play
    vals = np.arange(3000, dtype=np.uint64)
    k, v = po.ref_radix_sort(keys, vals, workers=4)
    d["rs_full_keys"], d["rs_full_values"], d["rs_full_sorted_keys"], d["rs_full_sorted_values"] = keys, vals, k, v
    np.savez_compressed(os.path.join(OUT, "sortkeys_kat.npz"), **d)
    print("sortkeys_kat.npz", sum(v.nbytes for v in d.values()))


def digest(*arrays):
    """16-byte digest of the bytes of `arrays` (tests/test_oracle_ref.py computes the same over the restatement's outputs)."""
    import hashlib
    h = hashlib.blake2b(digest_size=16)
    for a in arrays:
        h.update(np.ascontiguousarray(a).tobytes())
    return np.frombuffer(h.digest(), np.uint8)


def record_cull(d, key, ids, tys, info):
    """A visible set of the reference's cull: count, result pages and the digest of the ids in ascending order with their types."""
    o = np.argsort(ids)
    d[f"{key}_info"], d[f"{key}_digest"] = np.array([info["count"], info["pages"]], np.int64), digest(ids[o].astype(np.uint32), tys[o].astype(np.uint8))


def cull_sets(workers, out):
    """The scene and views of test_cull_sets_equal_reference_job_system through the reference's cull on a job system of `workers` workers.
    The job system is process-wide, so every worker count is recorded by a process of its own."""
    scene = scenes.cull_scene(400_000, (3000.0, 300.0, 3000.0), seed=123, big_fraction=0.005, type_probs=(0.5, 0.3, 0.2))
    rc = po.RefCulling(workers=workers)
    assert rc.workers == workers
    rc.add(scene["entities"], scene["types"], scene["pos"], scene["radius"])
    d = {}
    for v, a in enumerate((scenes.c1_frustum_args(), dict(scenes.c1_frustum_args(), position=(900.0, -50.0, 400.0), direction=(-0.7, 0.1, -0.7), far=3500.0))):
        fr = po.ref_frustum_perspective(a["position"], a["direction"], a["up"], a["fov"], a["ratio"], a["near"], a["far"])
        ids, tys, info = rc.cull(fr, cap=len(scene["entities"]), iters=2)
        d[f"sets_w{workers}_v{v}_frustum"] = fr
        record_cull(d, f"sets_w{workers}_v{v}", ids, tys, info)
    np.savez(out, **d)


def ref_crosscheck():
    """What the reference's own code returned in the cross-checks of tests/test_oracle_ref.py and tests/test_sortkeys_oracle.py: the same
    seeded inputs, in the same order, through the reference build instead of the restatement."""
    import subprocess
    import tempfile
    L = po.ref()
    names = ["Sphere", "Frustum", "ShiftedFrustum", "ShiftedFrustum.origin", "Transform", "CullResult", "CullResult.entities", "LocalRigidTransform", "DualQuat", "Matrix"]
    d = dict(sizeof_names=np.array(names), sizeof_values=np.array([L.ref_sizeof(k.encode()) for k in names], np.int64))
    with tempfile.TemporaryDirectory() as tmp:
        for w in (1, 4):
            subprocess.check_call([sys.executable, os.path.abspath(__file__), "--cull-sets", str(w), os.path.join(tmp, f"w{w}.npz")])
            d.update(np.load(os.path.join(tmp, f"w{w}.npz")))
    # random worlds, views and edits (test_random_views_and_edits_equal_reference)
    rng = np.random.default_rng(2024)
    for world in range(3):
        n = int(rng.integers(2_000, 30_000))
        half = (float(rng.choice([250.0, 900.0, 4000.0])), float(rng.choice([50.0, 400.0])), float(rng.choice([250.0, 900.0, 4000.0])))
        scene = scenes.cull_scene(n, half, seed=300 + world, big_fraction=float(rng.choice([0.0, 0.02, 0.3])), type_probs=(0.5, 0.25, 0.25))
        rc = po.RefCulling(workers=1)
        rc.add(scene["entities"], scene["types"], scene["pos"], scene["radius"])
        alive = np.ones(n, bool)
        pos, rad = scene["pos"].copy(), scene["radius"].copy()
        for step in range(12):
            p = rng.normal(size=3) * np.array(half) * 1.5
            dv = rng.normal(size=3); dv /= np.linalg.norm(dv)
            up = np.cross(np.cross(dv, rng.normal(size=3)), dv); up /= np.linalg.norm(up)
            if step % 5 == 0:
                p = np.round(p / 300.0) * 300.0
                dv, up = np.array([0.0, 0.0, -1.0]), np.array([0.0, 1.0, 0.0])
            far = float(rng.choice([30.0, 700.0, 5000.0, 60000.0]))
            if step % 3 == 2:
                args = (p, dv.astype(np.float32), up.astype(np.float32), float(rng.uniform(10, 3000)), float(rng.uniform(10, 3000)), 0.0, far)
                fr = po.ref_frustum_ortho(*args)
            else:
                args = (p, dv.astype(np.float32), up.astype(np.float32), float(rng.uniform(0.2, 2.4)), float(rng.uniform(0.5, 2.5)), float(rng.uniform(0.01, 2.0)), far)
                fr = po.ref_frustum_perspective(*args)
            t = int(rng.choice([-1, -1, 0, 1, 2]))
            ids, tys, info = rc.cull(fr, type=t, cap=n, iters=1)
            d[f"rv{world}_{step}_frustum"] = fr
            record_cull(d, f"rv{world}_{step}", ids, tys, info)
            live = np.nonzero(alive)[0]
            mv = rng.choice(live, min(len(live), 400), replace=False).astype(np.int32)
            a, b, c = np.array_split(mv, 3)
            pos[a] = pos[a] + rng.normal(size=(len(a), 3)) * 200.0
            rc.set_position(a, pos[a])
            rad[b] = (rng.random(len(b)) * 500.0).astype(np.float32)
            rc.set_radius(b, rad[b])
            rc.remove(c)
            alive[c] = False
    # random clips (test_random_clips_equal_reference): digests of the reference's poses (positions, then rotations) in the order the test asks for them
    rng = np.random.default_rng(99)
    digests = []
    for trial in range(25):
        bones = int(rng.choice([1, 2, 3, 4, 5, 7, 16, 33, 64, 100, 196]))
        frames = int(rng.integers(1, 91))
        pb = tuple(int(x) for x in rng.integers(3, 20, 3))
        rb = tuple(int(x) for x in rng.integers(3, 20, 3))
        sk = scenes.skeleton(bones, seed=500 + trial)
        clip = scenes.clip(sk, frames=frames, fps=float(rng.choice([1.0, 24.0, 30.0, 59.94])), seed=600 + trial, pos_bits=pb, rot_bits=rb,
                           const_fraction=float(rng.choice([0.0, 0.25, 1.0])))
        other = scenes.clip(sk, frames=int(rng.integers(1, 40)), seed=700 + trial, const_fraction=0.5)
        Lt = clip.length_ticks
        for t in [0, 1, max(Lt - 1, 0), Lt, Lt + 5000] + [int(x) for x in rng.integers(0, max(Lt, 1), 6)]:
            for absolute in (False, True):
                digests.append(digest(*po.ref_pose_evaluate(sk, clip, t, compute_absolute=absolute)))
            rel = po.ref_pose_evaluate(sk, clip, t, compute_absolute=False)
            w = float(rng.choice([0.0, 0.3, 0.9998, 0.9999, 1.0]))
            t2 = int(rng.integers(0, max(other.length_ticks, 1)))
            digests.append(digest(*po.ref_pose_evaluate(sk, other, t2, weight=w, start_from_bind=False, compute_absolute=True, pos=rel[0], rot=rel[1])))
    d["clip_digests"] = np.array(digests)
    # exact thresholds (test_threshold_values_equal_reference): the restatement's frusta, the reference's cull
    r_edge = np.float32(300.0)
    radii = np.array([r_edge, np.nextafter(r_edge, np.float32(1e9)), np.nextafter(r_edge, np.float32(0)), 0.0, 1e-30], np.float32)
    coords = [0.0, -0.0, 300.0, -300.0, 299.99999999, -299.99999999, 300.00000001, 600.0, -600.0, 899.9999, 1e-300, -1e-300]
    pos = np.array([[x, y, 10.0] for x in coords for y in (0.0, -300.0, 299.99999999)], np.float64)
    n = len(pos) * len(radii)
    P_, R = np.repeat(pos, len(radii), axis=0), np.tile(radii, len(pos))
    E = np.arange(n, dtype=np.int32)
    rc = po.RefCulling(workers=1)
    rc.add(E, (E % 3).astype(np.uint8), P_, R)
    a = scenes.c1_frustum_args()
    for v, args in enumerate((dict(a, position=(0.0, 0.0, 500.0)), dict(a, position=(300.0, 0.0, 300.0), direction=(-1.0, 0.0, 0.0)),
                              dict(a, position=(-1000.0, 100.0, 0.0), direction=(1.0, 0.0, 0.0), far=5000.0))):
        f = po.frustum_perspective(args["position"], args["direction"], args["up"], args["fov"], args["ratio"], args["near"], args["far"])
        record_cull(d, f"th_v{v}", *rc.cull(f, cap=n, iters=1))
    big, edge = E[R > r_edge], E[R == r_edge]
    rc.set_radius(big, np.full(len(big), r_edge, np.float32))
    rc.set_radius(edge, np.full(len(edge), np.nextafter(r_edge, np.float32(1e9)), np.float32))
    f = po.frustum_perspective(a["position"], a["direction"], a["up"], a["fov"], a["ratio"], a["near"], 5000.0)
    record_cull(d, "th_edited", *rc.cull(f, cap=n, iters=1))
    # PipelineImpl::radixSort on its job system (test_reference_build_agrees_live)
    rng = np.random.default_rng(5)
    for size in (0, 1, 300, 700, 4096):
        keys = (rng.integers(0, 4, size).astype(np.uint64) << np.uint64(56)) | rng.integers(0, 1 << 20, size).astype(np.uint64)
        d[f"rs{size}_digest"] = digest(*po.ref_radix_sort(keys, np.arange(size, dtype=np.uint64), workers=2))
    np.savez_compressed(os.path.join(OUT, "ref_crosscheck.npz"), **d)
    print("ref_crosscheck.npz", sum(v.nbytes for v in d.values()))


if __name__ == "__main__":
    po.build()
    if sys.argv[1:2] == ["--cull-sets"]:
        cull_sets(int(sys.argv[2]), sys.argv[3])
        sys.stdout.flush()
        os._exit(0)
    po.ref().ref_clip_length_ticks.restype = C.c_uint32
    po.ref().ref_time_from_seconds.restype = C.c_uint32
    # python tests/golden/make_golden.py [name ...]: only the named sets (default: all)
    for name in sys.argv[1:] or ["math_kat", "pose_kat", "cull_kat", "world_kat", "ani_kat", "sortkeys_kat", "ref_crosscheck"]:
        globals()[name]()
    sys.stdout.flush()
    os._exit(0)
