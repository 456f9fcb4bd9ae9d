"""CPU: the sort-key oracle (oracle/oracle_sortkeys.c) against vectors the reference's own code produced (tests/golden/sortkeys_kat.npz:
packers, Model::getLODMeshIndices and PipelineImpl::radixSort cut out of pipeline.cpp / model.h by oracle/build_ref.sh, and
tests/golden/ref_crosscheck.npz: its radix sort on its job system), and properties of the createSortKeys restatement."""
import ctypes as C
import hashlib
import os

import numpy as np

from lumixengine_b200 import scenes, sortkeys

G = np.load(os.path.join(os.path.dirname(__file__), "golden", "sortkeys_kat.npz"))


def _packers_equal(P, g):
    assert np.array_equal(np.array([P["float_flip"](int(x)) for x in g["u32"]], np.uint32), g["float_flip"])
    assert np.array_equal(np.array([P["make_mesh_sort_key"](int(k), int(b)) for k, b in zip(g["u32"], g["buckets"])], np.uint64), g["mesh_key"])
    assert np.array_equal(np.array([P["make_depth_sort_key"](float(x), int(b)) for x, b in zip(g["depths"], g["buckets"])], np.uint64), g["depth_key"])
    assert np.array_equal(np.array([P["make_autoinstanced_sort_key"](int(k & 0xffff), int(b)) for k, b in zip(g["u32"], g["buckets"])], np.uint64), g["inst_key"])
    assert np.array_equal(np.array([P["make_decal_sort_key"](int(k), int(b)) for k, b in zip(g["u32"], g["buckets"])], np.uint64), g["decal_key"])
    assert np.array_equal(np.array([P["make_decal_sort_value"](int(e)) for e in g["ents"]], np.uint64), g["decal_value"])
    assert np.array_equal(np.array([P["make_curve_decal_sort_value"](int(e)) for e in g["ents"]], np.uint64), g["curve_decal_value"])
    assert np.array_equal(np.array([P["make_skinned_sort_value"](int(e), int(m)) for e, m in zip(g["ents"], g["mesh_idx"])], np.uint64), g["skinned_value"])
    assert np.array_equal(np.array([P["make_mesh_sort_value"](int(e), int(m)) for e, m in zip(g["ents"], g["mesh_idx"])], np.uint64), g["mesh_value"])
    assert np.array_equal(np.array([P["make_autoinstanced_sort_value"](int(k & 0xffff), int(m)) for k, m in zip(g["u32"], g["mesh_idx"])], np.uint64), g["inst_value"])
    lodd = np.ascontiguousarray(g["lod_distances"])
    assert np.array_equal(np.array([P["lod_mesh_indices"](lodd[i].ctypes.data_as(C.c_void_p), float(g["squared"][i])) for i in range(len(lodd))], np.uint32), g["lod_index"])


def test_packers_and_lod_index_match_reference_vectors(oracle):
    _packers_equal(oracle.sortkey_packers("oracle"), G)


def test_radix_sort_matches_reference_vectors(oracle):
    for name in ("tiny", "below_step", "above_step", "big", "full"):
        keys, vals = G[f"rs_{name}_keys"], G[f"rs_{name}_values"]
        k, v = oracle.radix_sort(keys, vals, reference_copy_back=True)  # the reference's literal tail (see oracle_sortkeys.c)
        assert np.array_equal(k, G[f"rs_{name}_sorted_keys"]) and np.array_equal(v, G[f"rs_{name}_sorted_values"]), name
        k, v = oracle.radix_sort(keys, vals)  # what its callers mean: a stable sort by key
        order = np.argsort(keys, kind="stable")
        assert np.array_equal(k, keys[order]) and np.array_equal(v, vals[order]), name


def test_reference_build_agrees_live(oracle):
    """PipelineImpl::radixSort of the reference build on its job system against the restatement: the digest of the sorted keys and values
    (tests/golden/ref_crosscheck.npz)."""
    R = np.load(os.path.join(os.path.dirname(__file__), "golden", "ref_crosscheck.npz"))
    rng = np.random.default_rng(5)
    for size in (0, 1, 300, 700, 4096):
        keys = (rng.integers(0, 4, size).astype(np.uint64) << np.uint64(56)) | rng.integers(0, 1 << 20, size).astype(np.uint64)
        vals = np.arange(size, dtype=np.uint64)
        ok, ov = oracle.radix_sort(keys, vals, reference_copy_back=True)
        assert hashlib.blake2b(ok.tobytes() + ov.tobytes(), digest_size=16).digest() == R[f"rs{size}_digest"].tobytes(), size


def _inputs(n=20000, seed=3):
    scene = scenes.cull_scene(n, (2500.0, 300.0, 2500.0), seed=seed, type_probs=(0.8, 0.08, 0.04, 0.08))
    sk = scenes.sortkey_setup(n, scene["types"], scene["pos"], seed=seed + 1)
    view = sortkeys.make_view((10.0, 5.0, 30.0), (12.0, 5.0, 28.0), 1.0 / 60.0, 1.0, 17, False, sk["max_sort_key"], sk["layer_to_bucket"], sk["depth_sorted_buckets"])
    return scene, sk, view


def test_create_sort_keys_properties(oracle):
    scene, sk, view = _inputs()
    rng = np.random.default_rng(0)
    vis = np.sort(rng.choice(len(scene["types"]), 9000, replace=False)).astype(np.uint32)
    lod, pf = sk["lod"].copy(), sk["pose_frame"].copy()
    out = oracle.create_sort_keys(vis, scene["types"][vis], sk["transforms"], sk["model_of"], lod, sk["flags"], pf, sk["decal_sort_key"], sk["decal_layer"],
                                  sk["models"], sk["meshes"], view)
    keys, values = out["keys"], out["values"]
    assert len(keys) > 1000 and np.all(keys[1:] >= keys[:-1])
    # every auto-instanced record sits in the group of its mesh's sort key, groups are dense and ordered
    assert np.array_equal(out["group_offset"], np.concatenate([[0], np.cumsum(out["group_count"])[:-1]]).astype(np.uint32))
    assert int(out["group_count"].sum()) == len(out["group_renderables"]) > 1000
    ent = (out["group_renderables"] & np.uint64(0xffffffff)).astype(np.int64)
    mesh = (out["group_renderables"] >> np.uint64(40)).astype(np.int64)
    g_of = np.repeat(np.arange(len(out["group_count"])), out["group_count"])
    assert np.array_equal(sk["meshes"]["sort_key"][sk["models"]["mesh_base"][sk["model_of"][ent]] + mesh], g_of)
    assert np.all(scene["types"][ent] == 0) and not np.any(sk["flags"][ent] & 2)
    # one AUTOINSTANCED key per non-empty group; skinned instances are on the pose list exactly once; dirty instances emit nothing
    typ = (values >> np.uint64(32)) & np.uint64(31)
    assert int((typ == 1).sum()) == int((out["group_count"] > 0).sum())
    sk_ents = np.unique((values[typ == 2] & np.uint64(0xffffffff)).astype(np.int64))
    assert np.array_equal(np.sort(out["pose_list"]).astype(np.int64), sk_ents) and np.all(pf[sk_ents] == 17)
    dirty = vis[(scene["types"][vis] == 0) & ((sk["flags"][vis] & 2) != 0)]
    assert np.array_equal(np.sort(out["dirty_list"]), np.sort(dirty))
    # instance data: camera-relative position and lod - mesh.lod of the updated lod state
    lpos = out["instance_data"][:, 16:28].copy().view(np.float32)
    assert np.array_equal(lpos, (sk["transforms"]["pos"][ent] - np.array([10.0, 5.0, 30.0])).astype(np.float32))
    lod_d = out["instance_data"][:, 28:32].copy().view(np.float32)[:, 0]
    assert np.array_equal(lod_d, lod[ent] - sk["meshes"]["lod"][sk["models"]["mesh_base"][sk["model_of"][ent]] + mesh])
    # a second frame with the same view: lod smoothing moves on, poses are due again
    view2 = view.copy(); view2["frame_number"] = 18
    lod_before = lod.copy()
    out2 = oracle.create_sort_keys(vis, scene["types"][vis], sk["transforms"], sk["model_of"], lod, sk["flags"], pf, sk["decal_sort_key"], sk["decal_layer"],
                                   sk["models"], sk["meshes"], view2)
    assert np.any(lod != lod_before) and len(out2["pose_list"]) == len(out["pose_list"])
