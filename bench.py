#!/usr/bin/env python
"""bench.py — headline benchmark of the LumixEngine hot path on B200 (contract: task brief "Measurement").

    python bench.py --gpus N --steps K --warmup W            # our arm (CUDA, liblumix_b200.so)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's own CPU cull on the host cores

Metric (BASELINE.json): M entities culled/s.  Workload at N=1: configs[1] = "10M static entities, 1 camera frustum cull,
single B200" (scene C2 of SURVEY.md §8d).  A step = one CullingSystem::cull of the whole scene for one frustum.
N>1 (torchrun, one rank per GPU): weak scaling — every rank owns its own 10 M-entity shard (whole cell pages, no
data-path collective for the cull itself) and each step carries the one exchange the path has (SURVEY.md §8e): the visibility
bitmask + per-type counts of every rank reach every other rank, stored into peer memory over NVLink by the cull kernel itself
(lb200_culling_cull_exchange); the compacted id lists stay sharded with their entities.  LB200_EXCHANGE=ids gathers the id lists
instead (fused pack + peer push; LB200_NO_P2P=1: pack + ncclAllGather).  `value` = all ranks' entities / max-over-ranks device time.
The JSON line also carries the secondary BASELINE metric (M skinned verts/s) and the other stages of the path under "paths":
configs[2] as a chain on the device (propagate -> sphere refresh -> re-binning -> cull), configs[3] (pose + palette, skin; sharded by
instance at N>1), configs[4] (50M-entity cull + id all-gather over NVLink || pose pass of 1M instances, strong scaling).
`e2e` = host frustum + view in -> cull -> createSortKeys -> radixSort on the device -> counters back (the reference arm's e2e is the same
step on the host).  `parity`: the C2 digest against the reference build; at N>1 one exchanged step checked on every rank.
DESIGN.md section 7 describes every field.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

N_ENTITIES = 10_000_000
WORKLOAD = "C2: 10M static entities, 1 camera frustum cull (BASELINE.json configs[1]); per GPU at N>1"
REPLICAS = 8  # scene copies rotated through by successive culls: 8 x ~200 MB > 126 MB L2


_REAL_STDOUT = None


def claim_stdout():
    """The contract is ONE JSON line on stdout.  Libraries loaded into this process print banners to fd 1 (NCCL's version line at any
    NCCL_DEBUG level >= VERSION, glog, ...): point fd 1 at stderr for the whole run and keep the real stdout for emit()."""
    global _REAL_STDOUT
    if _REAL_STDOUT is None:
        sys.stdout.flush()
        _REAL_STDOUT = os.dup(1)
        os.dup2(2, 1)


def emit(line):
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            j = json.load(open(p))
            return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, copy read+write bytes)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md: 6.65 TB/s)"


def traffic_from_profile(kernel):
    """dram bytes per launch from the committed ncu capture, if any (profiles/traffic.json)."""
    p = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(p):
        try:
            return json.load(open(p)).get(kernel)
        except Exception:
            return None
    return None


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the GPU is under our load (B200_PROFILING.md 'clocks line')."""
    Q = "index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, device):
        self.device = device
        self.proc = None
        self.lines = []

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.device}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits", "-lms", "50"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def stop(self, t0, t1):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        for ts, line in self.lines:
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 9 or not (t0 <= ts <= t1 + 0.1):
                continue
            try:
                sm.append(float(parts[1])); mx.append(float(parts[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), parts[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": sorted(reasons), "samples": len(sm),
                "sampled": "50 ms nvidia-smi samples over the timed regions plus a ~1.5 s probe loop of the same cull kernel"}


def shared_config(visible, pages=None):
    """The keys both arms (--impl ours / reference) put into `config`: same workload, same scene, same frustum."""
    return {"workload": WORKLOAD, "entities_per_gpu": N_ENTITIES, "visible_per_gpu": int(visible),
            "frustum": "perspective fov 60deg 16:9 near 0.1 far 4500 at origin looking -z",
            "scene_rng": "numpy default_rng(seed 2 + rank) in lumixengine_b200/scenes.py::c2_scene, shared by both arms (SURVEY 8d names the reference's "
                         "RandomGenerator(521288629, 362436069); the distribution is the one 8d gives, the generator is not)"}


def build_info():
    """Source hash recorded by build() next to the .so against the hash of the sources as they lie here: a stale prebuilt library shows."""
    try:
        from lumixengine_b200 import _lib
        cur = _lib.source_hash()
        rec = _lib.recorded_source_hash()
        return {"source_hash": cur, "library_built_from": rec, "fresh": cur == rec}
    except Exception as e:
        return {"error": repr(e)}


def cull_cpu_baseline(steps, warmup):
    """The reference's CullingSystemImpl::cull on its own job system with W = min(cores, 64) workers AND with one worker (BASELINE.md
    section 3: its job system anti-scales on this path); the faster of the two is the baseline value."""
    runs = []
    for workers in (0, 1):
        r = run_cpu_worker(["--workload", "cull", "--n", str(N_ENTITIES), "--scene", "c2", "--steps", str(steps), "--warmup", str(warmup), "--workers", str(workers)])
        runs.append(r)
    best = max(runs, key=lambda r: r["value"])
    return best, runs


def run_cpu_worker(args, timeout=900):
    cmd = [sys.executable, "-m", "oracle.cpu_baseline"] + args
    out = subprocess.run(cmd, cwd=ROOT, capture_output=True, text=True, timeout=timeout)
    for line in out.stdout.splitlines():
        if line.startswith("CPU_BASELINE_JSON "):
            return json.loads(line[len("CPU_BASELINE_JSON "):])
    raise RuntimeError("cpu baseline worker failed: " + out.stderr[-2000:])


def attach_path_baselines(paths):
    """CPU figures for the secondary stages, timed on the host next to the GPU ones (SURVEY.md 8d): the serial restatements of
    World::transformEntity, updateAnimable + palettes and evaluateSkin (kind "port": the reference itself is serial on these paths or
    cannot be linked here), on bounded samples.  Never fatal."""
    try:
        pr = run_cpu_worker(["--workload", "propagate", "--n", "1000000", "--steps", "5"], timeout=300)
        paths["propagate_1m_depth8"]["cpu_baseline"] = {"value": pr["value"], "unit": pr["unit"], "cores": pr["cores"], "kind": pr["kind"], "sample": pr["sample"]}
        if "c3_update_and_cull" in paths:
            c3 = run_cpu_worker(["--workload", "c3chain", "--n", "1000000", "--steps", "3"], timeout=600)
            paths["c3_update_and_cull"]["cpu_baseline"] = {"value": c3["value"], "unit": c3["unit"], "cores": c3["cores"], "kind": c3["kind"], "sample": c3["sample"], "ms_per_step": c3["median_s"] * 1e3,
                                                          "parts_ms": c3["parts_ms"]}
        an = run_cpu_worker(["--workload", "anim", "--n", "10000"], timeout=300)
        for key, part in (("pose_palette_100k_x64", "pose"), ("skin_100k_x5k", "skin")):
            paths[key]["cpu_baseline"] = {"value": an[part]["value"], "unit": an[part]["unit"], "cores": an["cores"], "kind": an["kind"], "sample": an[part]["sample"]}
    except Exception as e:  # the GPU numbers stand on their own
        paths["cpu_baseline_error"] = repr(e)


def reference_arm(a, rank):
    """The reference's own CPU implementation (oracle/_ref) on the host cores; rank 0 only."""
    if rank != 0:
        return
    r, runs = cull_cpu_baseline(a.steps, a.warmup)
    ms = r["median_s"] * 1e3
    cfg = shared_config(r["visible"])
    cfg["note"] = "one 10M shard culled on the host whatever --gpus is (bounded sample of the N-shard job)"
    line = {
        "impl": "reference", "metric": "M entities culled/s", "value": r["value"], "unit": "M entities/s", "n_gpus": a.gpus, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": cfg,
        "cpu_baseline": {"value": r["value"], "unit": "M entities/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"], "impl": r["impl"],
                         "by_workers": [{"workers": x["cores"], "value": x["value"], "median_ms": x["median_s"] * 1e3} for x in runs],
                         "note": "value = the faster of W = min(cores, 64) and W = 1"},
        "e2e": {"value": r["value"], "unit": "M entities/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "ms_per_step": ms,
                "stages": "CullingSystemImpl::cull only (the sort-key stage could not be timed: see e2e.error)"},
        "gpu_launches": 0,
    }
    # the same end-to-end step as the GPU arm's e2e: cull -> createSortKeys -> radixSort (pipeline.cpp:3789-4144), on the host
    try:
        sk = run_cpu_worker(["--workload", "sortkeys", "--n", str(N_ENTITIES), "--steps", "3"], timeout=600)
        total_ms = ms + sk["median_s"] * 1e3
        line["e2e"] = {"value": N_ENTITIES / total_ms / 1e3, "unit": "M entities/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0, "ms_per_step": total_ms,
                       "stages": "CullingSystemImpl::cull (reference build, the faster worker count) + PipelineImpl::createSortKeys over its visible list (C restatement, one worker: "
                                 "pipeline.cpp does not compile here) + PipelineImpl::radixSort (" + sk["radix_sort"] + ")",
                       "parts_ms": {"cull": ms, "create_sort_keys": sk["create_keys_median_s"] * 1e3, "radix_sort": sk["sort_median_s"] * 1e3},
                       "sort_keys": {"n_keys": sk["n_keys"], "n_instances": sk["n_instances"], "sample": sk["sample"]}}
    except Exception as e:
        line["e2e"]["error"] = repr(e)
    emit(line)


DUMP_BYTES = 64 << 20


def dump_outputs(out_dir, cs, ctx):
    """Writes the result of the last cull as its caller receives it: the visible ids grouped by renderable type (sorted inside a type,
    where their order is unspecified) and the per-type counts, as float64 .npy files.  A list over the size limit is written as a
    fixed, seeded sample of its entries."""
    ptr, res = cs.last_result()
    counts = np.array(res.type_count[:res.n_types], np.int64)
    ids = [np.sort(ctx.copy_to_host(ptr + 4 * int(res.type_offset[t]), int(c), np.uint32)) for t, c in enumerate(counts) if c]
    ids = np.concatenate(ids).astype(np.float64) if ids else np.zeros(0)
    if ids.nbytes + counts.nbytes > DUMP_BYTES:
        ids = ids[np.sort(np.random.default_rng(0).choice(len(ids), (DUMP_BYTES - counts.nbytes) // 8, replace=False))]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "visible_ids.npy"), ids)
    np.save(os.path.join(out_dir, "visible_type_counts.npy"), counts.astype(np.float64))


def time_region(ctx, fn, steps):
    e0, e1 = ctx.event(), ctx.event()
    ctx.synchronize()
    ctx.record(e0)
    for _ in range(steps):
        fn()
    ctx.record(e1)
    ms = ctx.elapsed_ms(e0, e1)
    return ms


def secondary_paths(ctx, lb, scenes, peak, steps, warmup):
    """Other stages of the hot path: 1M-node propagate (config 3), 100k x 64-bone pose+palette and 100k x 5k-vert skin (config 4)."""
    out = {}
    # --- propagate ---
    parents, locals_, roots = scenes.hierarchy_forest(1_000_000, 8, 7, seed=3)
    hs = []
    for _ in range(5):  # 5 x 112 MB of locals + globals > 4 x the 126 MB L2: successive steps never find their hierarchy in L2
        h = lb.Hierarchy(ctx, parents)
        h.setLocalTransforms(locals_)
        h.setRootTransforms(roots)
        hs.append(h)
    turn = [0]

    def prop():
        hs[turn[0] % len(hs)].propagate()
        turn[0] += 1
    for _ in range(max(warmup, 3) + len(hs)):
        prop()
    ms = time_region(ctx, prop, steps) / steps
    b = hs[0].algorithmic_bytes()
    out["propagate_1m_depth8"] = {"value": len(parents) / ms / 1e3, "unit": "M nodes/s", "ms_per_step": ms,
                                  "roofline": {"bound": "hbm", "achieved": b / ms / 1e6, "peak": peak, "unit": "GB/s", "frac": b / ms / 1e6 / peak, "algorithmic_bytes": b},
                                  "note": "narrow levels fused into one block + one launch per wide level; 5 hierarchies (560 MB) rotated, so every step reads its locals from HBM"}
    for h in hs:
        h.close()
    # --- config 3 as a chain: 1M-node propagate -> sphere refresh -> re-binning of the culling structure -> cull, all on the device ---
    bounding = np.full(len(parents), 1.0, np.float32)  # SURVEY 8d C3: radius = 1.0 * max(scale)
    h = lb.Hierarchy(ctx, parents)
    h.setLocalTransforms(locals_)
    h.setRootTransforms(roots)
    h.propagate()
    pos0, rad0 = h.getSpheres(bounding)
    c3 = lb.CullingSystem(ctx)
    c3.add(np.arange(len(parents), dtype=np.int32), np.zeros(len(parents), np.uint8), pos0, rad0)
    c3.flush()
    root_ids = np.nonzero(parents < 0)[0].astype(np.uint32)
    root_sets = [roots[root_ids].copy(), roots[root_ids].copy()]
    root_sets[1]["pos"] += np.array([37.0, 4.0, -29.0])  # every tree drifts back and forth: ~4 % of the nodes cross a cell border per step
    f3 = lb.frustum_perspective(**scenes.c2_frustum_args())
    state = {"k": 0, "changers": 0}

    def chain():
        state["k"] += 1
        h.setSubset(root_ids, root_sets[state["k"] & 1], globals_=True)  # World::setTransform for the roots: 3906 x 60 B over PCIe
        h.propagate()
        d_pos, d_rad = h.refreshSpheres(bounding if state["k"] == 1 else None)
        state["changers"] = c3.set_many_device(d_pos, d_rad, len(parents))
        c3.cull_device(f3, want_counts=False)
    for _ in range(max(warmup, 3)):
        chain()
    c_steps = max(3, min(steps, 20))
    ms = time_region(ctx, chain, c_steps) / c_steps
    _, r3 = c3.cull_device(f3, want_counts=True)
    out["c3_update_and_cull"] = {"value": len(parents) / ms / 1e3, "unit": "M nodes/s", "ms_per_step": ms, "nodes": len(parents), "cell_changers_per_step": int(state["changers"]),
                                 "visible": int(r3.total),
                                 "note": "BASELINE configs[2] as one chain on one stream: root transforms uploaded (3906 x 60 B), propagate, sphere refresh (render_module.cpp:1544-1554) left "
                                         "in HBM, CullingSystem::set for all 1M nodes on the device (lb200_culling_set_many_device: two 32-byte counter read-backs inside), cull. "
                                         "The 1M-entity culling structure (22 MB) is L2-resident: a latency number, not an HBM one"}
    h.close()
    c3.close()
    # --- pose + palette, skin ---
    sk = scenes.skeleton(64)
    clips = [scenes.clip(sk, frames=60, seed=s) for s in (1, 2, 3, 4)]
    mesh = scenes.mesh(sk, 5000)
    n_inst = 100_000
    anim = lb.AnimationSystem(ctx, sk, clips, mesh, max_instances=n_inst)
    ci, tt = scenes.instance_times(n_inst, clips)
    anim.setInstances(ci, tt)
    flags = lb.PALETTE_DUAL_QUAT
    for _ in range(max(warmup, 3)):
        anim.update(1.0 / 60.0, flags)
    ms = time_region(ctx, lambda: anim.update(1.0 / 60.0, flags), steps) / steps
    b = anim.algorithmic_bytes(flags)
    out["pose_palette_100k_x64"] = {"value": n_inst * 64 / ms / 1e3, "unit": "M bone-instances/s", "ms_per_step": ms,
                                    "roofline": {"bound": "hbm", "achieved": b / ms / 1e6, "peak": peak, "unit": "GB/s", "frac": b / ms / 1e6 / peak, "algorithmic_bytes": b},
                                    "note": "dual-quaternion palette (pipeline.cpp:2680-2745), 205 MB written per step (> L2)"}
    anim.update(0.0, lb.PALETTE_MATRIX)
    for _ in range(max(warmup, 3)):
        anim.skin()
    sk_steps = max(3, min(steps, 10))
    ms = time_region(ctx, anim.skin, sk_steps) / sk_steps
    b = anim.algorithmic_bytes(lb.PALETTE_MATRIX, skin=True)
    out["skin_100k_x5k"] = {"value": n_inst * 5000 / ms / 1e3, "unit": "M skinned verts/s", "ms_per_step": ms,
                            "roofline": {"bound": "hbm", "achieved": b / ms / 1e6, "peak": peak, "unit": "GB/s", "frac": b / ms / 1e6 / peak, "algorithmic_bytes": b},
                            "note": "evaluateSkin (model.cpp:103-109), 6 GB written per step"}
    anim.close()
    return out


def c4_sharded(ctx, lb, scenes, rank, world, dist, peak, steps, warmup):
    """BASELINE configs[3] at N > 1: the 100k instances x 64 bones x 5k vertices shard by instance index range (strong scaling, no exchange:
    "replicas only" in SURVEY 8e's terms) — pose + dual-quaternion palette, then matrix palette + evaluateSkin; device time, max over ranks."""
    import torch
    n_total = 100_000
    n_inst = n_total // world
    sk = scenes.skeleton(64)
    clips = [scenes.clip(sk, frames=60, seed=s) for s in (1, 2, 3, 4)]
    mesh = scenes.mesh(sk, 5000)
    anim = lb.AnimationSystem(ctx, sk, clips, mesh, max_instances=n_inst)
    ci, tt = scenes.instance_times(n_total, clips)
    anim.setInstances(ci[rank * n_inst:(rank + 1) * n_inst], tt[rank * n_inst:(rank + 1) * n_inst])
    for _ in range(max(warmup, 3)):
        anim.update(1.0 / 60.0, lb.PALETTE_DUAL_QUAT)
    dist.barrier()
    ms_pose = time_region(ctx, lambda: anim.update(1.0 / 60.0, lb.PALETTE_DUAL_QUAT), steps) / steps
    anim.update(0.0, lb.PALETTE_MATRIX)
    for _ in range(3):
        anim.skin()
    dist.barrier()
    k = max(3, min(steps, 10))
    ms_skin = time_region(ctx, anim.skin, k) / k
    t = torch.tensor([ms_pose, ms_skin], dtype=torch.float64, device="cuda")
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_pose, ms_skin = (float(x) for x in t.tolist())
    b_pose = anim.algorithmic_bytes(lb.PALETTE_DUAL_QUAT) * world
    b_skin = anim.algorithmic_bytes(lb.PALETTE_MATRIX, skin=True) * world
    anim.close()
    return {"scaling": "strong", "n_gpus": world, "instances_total": n_inst * world, "instances_per_gpu": n_inst,
            "pose_palette": {"value": n_inst * world * 64 / ms_pose / 1e3, "unit": "M bone-instances/s", "ms_per_step": ms_pose, "hbm_frac_per_gpu": b_pose / world / ms_pose / 1e6 / peak},
            "skin": {"value": n_inst * world * 5000 / ms_skin / 1e3, "unit": "M skinned verts/s", "ms_per_step": ms_skin, "hbm_frac_per_gpu": b_skin / world / ms_skin / 1e6 / peak},
            "note": "instances sharded by index range, no exchange; device time, max over ranks"}


C5_ENTITIES = 50_000_000
C5_INSTANCES = 1_000_000


def c5_mixed(ctx, lb, scenes, rank, world, dist, steps, warmup):
    """BASELINE configs[4]: 50M-entity cull + 1M skinned instances, STRONG scaling over the ranks.  Entities shard by index range (every rank
    owns whole cell pages of its 50M / N entities), instances by index range (pose + dual-quaternion palette of 1M / N instances, no
    exchange).  The one collective of the path (north_star): every step all-gathers the compacted visible id lists — fused pack + NVLink peer
    push + epoch flags (LB200_C5_EXCHANGE=nccl: pack + ncclAllGather).  One exchanged step is verified: every rank's view of the gathered
    slabs has the digest of the ranks' own id lists."""
    import numpy as np
    n_ent = C5_ENTITIES // world
    n_inst = C5_INSTANCES // world
    scene = scenes.c2_scene(n_ent, seed=500 + rank)
    cs = lb.CullingSystem(ctx)
    t0 = time.time()
    cs.add(np.arange(n_ent, dtype=np.int32), scene["types"], scene["pos"], scene["radius"])  # local ids; the global id is rank * n_ent + local
    build_s = time.time() - t0
    cs.flush()
    f = lb.frustum_perspective(**scenes.c2_frustum_args())
    sk = scenes.skeleton(64)
    clips = [scenes.clip(sk, frames=60, seed=s) for s in (1, 2, 3, 4)]
    # culling and the animation update are independent jobs of a frame (the engine runs them concurrently on its job system): here they are
    # two streams — the animation system lives on a second context of the same device — so the NVLink-bound id gather and the arithmetic-
    # bound pose pass overlap
    ctx_anim = lb.Context(ctx.device, background=True)  # lowest stream priority: the cull / gather kernels take SMs as soon as pose blocks retire
    anim = lb.AnimationSystem(ctx_anim, sk, clips, scenes.mesh(sk, 64), max_instances=n_inst)
    ci, tt = scenes.instance_times(n_inst, clips, seed=9 + rank)
    anim.setInstances(ci, tt)
    first = cs.cull(f)
    visible = int(first.total)
    own = lb.culling.digest_ids(first.ids, first.types())
    slab = visible + 1024
    mode = "single GPU: no exchange"
    if world > 1:
        import torch
        t = torch.tensor([slab], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        slab = int(t.item())
        mapped = getattr(ctx, "p2p_slab_ids", None)
        if os.environ.get("LB200_C5_EXCHANGE", "p2p") == "p2p":
            if mapped is None:
                ctx.comm_enable_p2p(slab)
                mapped = ctx.p2p_slab_ids = slab
        # lb200_culling_cull_gather pushes over NVLink when the slab fits the mapped peer buffers and goes through ncclAllGather otherwise
        if mapped is not None and slab <= mapped:
            mode = "visible id lists: fused pack + NVLink peer push + epoch flags (lb200_culling_cull_gather)"
        else:
            mode = "visible id lists: pack + ncclAllGather (lb200_culling_cull_gather; the mapped peer buffers hold %s ids, the slab needs %d)" % (mapped, slab)

    def step():
        if world > 1:
            cs.cull_gather(f, slab)
        else:
            cs.cull_device(f, want_counts=False)
        anim.update(1.0 / 60.0, lb.PALETTE_DUAL_QUAT)
    for _ in range(max(warmup, 3)):
        step()
    ctx.synchronize()
    verified = None
    if world > 1:
        import torch
        dev = cs.cull_gather(f, slab)
        ctx.synchronize()
        slabs, counts = cs.read_gathered(dev, slab, world)
        seen = []
        for r in range(world):
            off = np.concatenate([[0], np.cumsum(counts[r].astype(np.int64))])  # int64: cumsum of uint32 is uint64, which numpy promotes to float next to an int
            seen.append([[int(counts[r][t]), int(slabs[r][off[t]:off[t + 1]].astype(np.uint64).sum(dtype=np.uint64)),
                          int(np.bitwise_xor.reduce(slabs[r][off[t]:off[t + 1]].astype(np.uint64))) if counts[r][t] else 0] for t in range(4)])
        mine = torch.tensor(own, dtype=torch.int64, device="cuda")
        everyone = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(everyone, mine)
        verified = all(seen[r] == everyone[r].cpu().tolist() for r in range(world))
        flag = torch.tensor([1 if verified else 0], dtype=torch.int64, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        verified = bool(flag.item())
        dist.barrier()
    def region(fn):  # K steps between two events on the culling stream; the closing event is recorded once the animation stream has drained too
        ctx_anim.synchronize()
        e0, e1 = ctx.event(), ctx.event()
        ctx.synchronize()
        ctx.record(e0)
        fn()
        ctx_anim.synchronize()
        ctx.record(e1)
        return ctx.elapsed_ms(e0, e1)
    if world > 1:
        dist.barrier()
    ms = region(lambda: [step() for _ in range(steps)]) / steps
    ms_cull = region(lambda: [cs.cull_gather(f, slab) if world > 1 else cs.cull_device(f, want_counts=False) for _ in range(steps)]) / steps
    ea, eb = ctx_anim.event(), ctx_anim.event()
    ctx_anim.synchronize()
    ctx_anim.record(ea)
    for _ in range(steps):
        anim.update(1.0 / 60.0, lb.PALETTE_DUAL_QUAT)
    ctx_anim.record(eb)
    ms_pose = ctx_anim.elapsed_ms(ea, eb) / steps
    vis_total = visible
    if world > 1:
        import torch
        t = torch.tensor([ms, ms_cull, ms_pose], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms, ms_cull, ms_pose = (float(x) for x in t.tolist())
        v = torch.tensor([visible], dtype=torch.int64, device="cuda")
        dist.all_reduce(v)
        vis_total = int(v.item())
    anim.close()
    ctx_anim.close()
    cs.close()
    return {"value": C5_ENTITIES / ms / 1e3, "unit": "M entities/s", "ms_per_step": ms, "scaling": "strong", "n_gpus": world,
            "entities_total": C5_ENTITIES, "skinned_instances_total": C5_INSTANCES, "entities_per_gpu": n_ent, "instances_per_gpu": n_inst,
            "visible_total": vis_total, "parts_ms": {"cull_and_gather": ms_cull, "pose_palette": ms_pose}, "exchange": mode, "exchange_verified": verified,
            "gather_bytes_received_per_gpu": int(vis_total - visible) * 4, "scene_build_s": build_s,
            "note": "a step = [cull of the rank's shard + all-gather of the visible ids] on one stream and [pose / dual-quaternion palette of the rank's instances] on a second "
                    "one (independent jobs of a frame); device time of K steps until both streams have drained, max over ranks; value = 50M entities / step time at every N"}


def ours(a, rank, world):
    import lumixengine_b200 as lb
    from lumixengine_b200 import scenes

    dist = None
    if world > 1:
        # exchange steps of a lane wait for the peers' flags: more lanes in flight hide more of that (N=2: 14.5 us per step with 3 lanes, 11.1 with 6, 10.1 with 8;
        # profiles/r2_N2_time_exchange.log).  Read once by the library when the first culling system is created.
        os.environ.setdefault("LB200_CULL_LANES", "8")
        os.environ.setdefault("NCCL_DEBUG", "WARN")  # keep NCCL's version banner off stdout: the contract is ONE JSON line
        import torch
        import torch.distributed as dist
        local = int(os.environ.get("LOCAL_RANK", rank))
        torch.cuda.set_device(local)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
        device = local
    else:
        device = 0
    ctx = lb.Context(device)  # NoDeviceError without a GPU / ImportError without the .so: no fallback
    peak, peak_src = measured_peaks()

    # ---- scene: C2 shard of this rank (distinct seed per rank) ----
    scene = scenes.c2_scene(N_ENTITIES, seed=2 + rank)
    cs = lb.CullingSystem(ctx)
    cs.set_replicas(REPLICAS)
    t0 = time.time()
    cs.add(scene["entities"], scene["types"], scene["pos"], scene["radius"])
    build_s = time.time() - t0
    cs.flush()
    f = lb.frustum_perspective(**scenes.c2_frustum_args())

    if world > 1:
        import torch
        uid = torch.zeros(128, dtype=torch.uint8, device="cuda")
        if rank == 0:
            uid.copy_(torch.from_numpy(ctx.comm_unique_id()))
        dist.broadcast(uid, 0)
        ctx.comm_init(world, rank, uid.cpu().numpy())

    first = cs.cull(f)  # also the warm-up of every buffer; gives the visible count for sizing the gather slab
    visible = first.total
    slab = 0
    if world > 1:
        import torch
        t = torch.tensor([visible], dtype=torch.int64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        slab = int(t.item()) + 1024
        exchange = os.environ.get("LB200_EXCHANGE", "mask")
        if exchange == "mask":
            t = torch.tensor([cs.exchange_slab_words()], dtype=torch.int64, device="cuda")
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            # the peer buffers are mapped once per process: sized for the larger of this exchange's slabs and config 5's id lists (the same view
            # sees 18 % of the C2 distribution: 25 % of the rank's 50M / N entities + margin), so that config 5 below runs its gather over NVLink too
            p2p_ids = int(t.item()) - 256
            if not a.only_cull and not a.no_c5 and os.environ.get("LB200_C5_EXCHANGE", "p2p") == "p2p":
                p2p_ids = max(p2p_ids, C5_ENTITIES // world // 4 + 4096)
            ctx.comm_enable_p2p(p2p_ids)
            ctx.p2p_slab_ids = p2p_ids
            exchange_desc = "visibility bitmask rows + per-type counts stored into every rank's memory by the cull kernel (NVLink peer stores, epoch flags); id lists stay sharded"
        elif os.environ.get("LB200_NO_P2P") != "1":
            ctx.comm_enable_p2p(slab)  # per-frame exchange = fused pack + NVLink peer stores + epoch flags (no NCCL call per step)
            ctx.p2p_slab_ids = slab
            exchange_desc = "visible id lists: fused pack + NVLink peer push"
        else:
            exchange_desc = "visible id lists: pack + ncclAllGather"

    def steps_device(n):
        """n steps = n culls of the whole scene.  N=1: ONE lb200_culling_cull_device_n call — the engine culls its views (main,
        shadow cascades, lights) concurrently (pipeline.cpp:996-1063), so consecutive culls are independent submissions: they go
        to 3 internal streams / output lanes with programmatic dependent launch and the device overlaps them."""
        if world > 1 and exchange == "mask":
            cs.cull_exchange_n(f, n)  # independent steps on the internal lanes; every step = cull + peer stores + epoch-flag wait
        elif world > 1:
            for _ in range(n):
                step_device()
        else:
            cs.cull_device_n(f, n)

    def step_device():
        if world > 1 and exchange == "mask":
            cs.cull_exchange(f)  # one kernel: cull + peer stores of the mask rows; then the flag wait
        elif world > 1:
            cs.cull_gather(f, slab)  # cull + device-side pack + exchange of the id slabs, no host synchronisation
        else:
            cs.cull_device(f, want_counts=False)

    sampler = ClockSampler(device)
    sampler.start()
    t_load0 = time.time()
    steps_device(max(a.warmup, 3) + 50)
    ctx.synchronize()

    # ---- timed region: EXACTLY K steps, barrier + sync both sides, device time, max over ranks ----
    if world > 1:
        dist.barrier()
    launches0 = ctx.launches
    ms_total = time_region(ctx, lambda: steps_device(a.steps), 1)
    launches = ctx.launches - launches0
    if world > 1:
        import torch
        t = torch.tensor([ms_total], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
        dist.barrier()
    ms_step = ms_total / a.steps
    if a.dump_outputs and rank == 0:
        dump_outputs(a.dump_outputs, cs, ctx)

    # N>1, bitmask exchange: one exchanged step is checked — what every rank sees of rank r's slab (per-type counts, visibility rows by page
    # id) must be what rank r holds itself, and rank r's own rows must say exactly what its own cull made visible
    exchange_verified = None
    if world > 1 and exchange == "mask":
        import torch
        _, slabs_ptr, stride = cs.cull_exchange(f)
        ctx.synchronize()
        seen = cs.read_exchanged(slabs_ptr, stride, world)

        def slab_digest(sl):
            rows = sl["mask"].astype(np.uint64)
            page_w = (np.arange(rows.shape[0], dtype=np.uint64)[:, None] * np.uint64(8) + np.arange(8, dtype=np.uint64)[None, :] + np.uint64(1))
            bits = int(np.unpackbits(sl["mask"].view(np.uint8)).sum())
            return [int(sl["counts"].astype(np.int64).sum()), bits, int(sl["n_pages"]), int((rows * page_w).sum(dtype=np.uint64) & np.uint64(0x7fffffffffffffff))]
        mine = torch.tensor([slab_digest(seen[r]) for r in range(world)], dtype=torch.int64, device="cuda")  # my view of every rank
        views = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(views, mine)
        views = [v.cpu().tolist() for v in views]
        own = cs.cull(f)
        ok = all(views[q][r] == views[r][r] for q in range(world) for r in range(world))          # everybody sees rank r as rank r sees itself
        ok = ok and views[rank][rank][0] == int(own.total) and views[rank][rank][1] == int(own.total)  # counts and set bits = my visible set
        flag = torch.tensor([1 if ok else 0], dtype=torch.int64, device="cuda")
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        exchange_verified = bool(flag.item())
        dist.barrier()

    # algorithmic bytes of one cull (needs counts: one more cull, untimed)
    cs.cull_device(f, want_counts=True)
    alg_bytes = cs.last_algorithmic_bytes()
    stats = cs.cull(f).stats

    # kernel-only timing for the roofline (N>1 steps also contain the gather): K launches of the cull kernel alone
    ms_kernel = time_region(ctx, lambda: cs.cull_device_n(f, a.steps), 1) / a.steps
    # one cull on an idle device, nothing to overlap with, its launch queued behind a delay kernel (no host latency in the interval):
    # the latency of a lone view — beside what the interval costs when it holds nothing, and when it holds one empty kernel
    lone = {what: float(np.mean(cs.time_lone_cull(f, 50, mode=mode))) for mode, what in ((0, "cull"), (1, "empty_interval"), (2, "empty_kernel"))}
    ms_lone = lone["cull"]
    # parity at full size: the digest of the visible set (per type: count, sum, xor of ids) against the reference's own build below
    full = cs.cull(f)
    gpu_digest = lb.culling.digest_ids(full.ids, full.types())

    # ---- e2e: the public host API every step: frustum + view in host memory -> CullingSystem.cull_device -> SortKeys.createSortKeys
    # (the consumer of the visible list, pipeline.cpp:3789-4144) -> sorted keys / values + per-group instance data in HBM for the draw
    # stage, the counts read back to the host.  The visible ids never cross PCIe.  (The round-1 form of this number — ids delivered
    # into pinned host memory — is kept beside it as e2e.ids_to_host_ms.)
    from lumixengine_b200 import sortkeys as skm
    sk_in = scenes.sortkey_setup(N_ENTITIES, scene["types"], scene["pos"], seed=40 + rank)
    SK = lb.SortKeys(ctx, N_ENTITIES, sk_in["max_sort_key"] + 1, max_keys=1 << 22, max_instances=1 << 22)
    SK.setModels(sk_in["models"], sk_in["meshes"])
    SK.setInstances(sk_in["model_of"], sk_in["lod"], sk_in["flags"], sk_in["pose_frame"], sk_in["decal_sort_key"], sk_in["decal_layer"])
    SK.setTransforms(sk_in["transforms"])
    fa = scenes.c2_frustum_args()
    frame = [0]
    # the views of the frames to come, in host memory (the engine fills this 1.3 KB struct per view in C++; here it is numpy, kept out of the step)
    views = [skm.make_view(fa["position"], fa["position"], 1.0 / 60.0, 1.0, 101 + k, False, sk_in["max_sort_key"], sk_in["layer_to_bucket"], sk_in["depth_sorted_buckets"])
             for k in range(64)]

    def e2e_step():
        view = views[frame[0] % len(views)]
        frame[0] += 1
        cs.cull_device(f, want_counts=False)
        return SK.createSortKeys(cs, view, sort=True, want_counts=True)
    for _ in range(3):
        cs.cull(f)
        sk_res = e2e_step()
    e2e_steps = max(3, min(a.steps, 50))
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        r = cs.cull(f)
    ctx.synchronize()
    e2e_ids_s = (time.perf_counter() - t0) / e2e_steps
    if world > 1:
        dist.barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        sk_res = e2e_step()
    ctx.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    # device time of the sort-key stage alone
    view0 = skm.make_view(fa["position"], fa["position"], 1.0 / 60.0, 1.0, 7, False, sk_in["max_sort_key"], sk_in["layer_to_bucket"], sk_in["depth_sorted_buckets"])
    cs.cull_device(f, want_counts=False)
    ms_keys = time_region(ctx, lambda: SK.createSortKeys(cs, view0, sort=True, want_counts=False), 20) / 20
    if world > 1:
        import torch
        t = torch.tensor([e2e_s], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())

    # clock probe: the same kernel back to back for ~1.5 s so that nvidia-smi has samples under this load
    t_probe = time.time()
    while time.time() - t_probe < 1.5:
        for _ in range(200):
            cs.cull_device(f, want_counts=False)
        ctx.synchronize()
    clocks = sampler.stop(t_load0, time.time())

    n_pages_c2 = cs.page_count()
    c5_result = None
    if not a.only_cull and not a.no_c5:
        SK.close()
        cs.close()  # free the C2 scene's HBM and pinned host memory before the 50M scene
        cs = None
        del scene, sk_in
        try:
            c5_result = c5_mixed(ctx, lb, scenes, rank, world, dist, max(5, min(a.steps, 50)), a.warmup)
        except Exception as e:
            c5_result = {"error": repr(e)}

    c4_result = None
    if world > 1 and not a.only_cull:
        try:
            c4_result = c4_sharded(ctx, lb, scenes, rank, world, dist, peak, max(5, min(a.steps, 50)), a.warmup)
        except Exception as e:
            c4_result = {"error": repr(e)}

    if rank != 0:
        ctx.close()
        if dist:
            dist.destroy_process_group()
        return

    total_entities = N_ENTITIES * world
    line = {
        "metric": "M entities culled/s", "value": total_entities / ms_step / 1e3, "unit": "M entities/s", "n_gpus": world, "steps": a.steps, "warmup": a.warmup,
        "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {**shared_config(visible), "pages": n_pages_c2,
                   "l2": f"{REPLICAS} rotating copies of the page arrays ({REPLICAS} x ~{n_pages_c2 * 4064 // 1_000_000} MB): successive culls never re-read an L2-resident scene",
                   "parallelism": f"dp{world}: whole cell pages per rank" + (("; exchanged each step: " + exchange_desc) if world > 1 else ""),
                   "submission": "K culls = one lb200_culling_cull_device_n call: consecutive (independent) culls on 3 streams / output lanes, half-occupancy grids, programmatic dependent launch" if world == 1 else f"K exchange steps = one lb200_culling_cull_exchange_n call (steps on {os.environ.get('LB200_CULL_LANES', '3')} streams / output lanes, 3 x lanes exchange buffers per rank)",
                   "lone_cull_ms": ms_lone, "lone_empty_interval_ms": lone["empty_interval"], "lone_empty_kernel_ms": lone["empty_kernel"],
                   "scene_build_s": build_s, "page_stats": stats},
        "gpu_launches": int(launches),
        "clocks": clocks,
        "e2e": {"value": total_entities / e2e_s / 1e6, "unit": "M entities/s", "h2d_bytes_per_step": 256 + 1352 + 1024 + 8, "d2h_bytes_per_step": 32,
                "ms_per_step": e2e_s * 1e3,
                "api": "CullingSystem.cull_device(frustum) + SortKeys.createSortKeys(view): host frustum + view -> kernel params; cull, sort keys / LOD / auto-instancing "
                       "groups + instance data and the radix sort on the device; 8 counters read back (one synchronisation); ids, keys and instance data stay in HBM",
                "sort_keys": {"n_keys": int(sk_res.n_keys), "n_instances": int(sk_res.n_instances), "n_pose": int(sk_res.n_pose), "device_ms": ms_keys,
                              # DESIGN.md 4.5: 64 B record + 52 B stash written + 52 B read per visible renderable, 56 B per instance, 16 B per key written,
                              # 8 B of ids; the radix sort's 32 B per pair and pass stay in L2 (12 MB) and are not counted
                              "algorithmic_bytes": int(176 * int(visible) + 56 * int(sk_res.n_instances) + 16 * int(sk_res.n_keys)),
                              "hbm_frac": (176 * int(visible) + 56 * int(sk_res.n_instances) + 16 * int(sk_res.n_keys)) / ms_keys / 1e6 / peak,
                              "traffic": (traffic_from_profile("create_keys_kernel") or 0) + (traffic_from_profile("radix_sort_kernel") or 0),
                              "note": "counts of the last frame of the loop: the lod smoothing state evolves from frame to frame (both arms start from the same state; "
                                      "equality per frame is what tests/test_sortkeys_gpu.py checks)"},
                "ids_to_host_ms": e2e_ids_s * 1e3, "ids_to_host_d2h_bytes": int(r.total) * 4 + 264 * 4,
                "ids_to_host_api": "CullingSystem.cull(frustum): visible ids + counts written into pinned host memory by the device right behind the cull (the round-1 e2e)"},
        "roofline": {"bound": "hbm", "achieved": alg_bytes / ms_kernel / 1e6, "peak": peak, "unit": "GB/s", "frac": alg_bytes / ms_kernel / 1e6 / peak,
                     "traffic": traffic_from_profile("cull_pages_kernel"), "kernel": "cull_pages_kernel", "kernel_ms": ms_kernel, "algorithmic_bytes": int(alg_bytes),
                     "peak_source": peak_src,
                     "lone_frac": alg_bytes / ms_lone / 1e6 / peak, "lone_ms": ms_lone,
                     "lone_note": "one cull, device to itself, CUDA events (1 us ticks) around it; the interval costs lone_empty_interval_ms with nothing in it and lone_empty_kernel_ms with one empty kernel",
                     "scan_all_equivalent_gbs": (16 * N_ENTITIES + 8 * visible + N_ENTITIES / 8) / ms_kernel / 1e6},
        "build": build_info(),
        "parity": {"gpu_digest": gpu_digest, "digest": "per renderable type [count, sum of ids, xor of ids] of the visible set of one C2 cull",
                   **({"exchange_verified": exchange_verified, "exchange_check": "one exchanged step: every rank's view of every rank's slab (per-type counts, visibility rows "
                       "by page id) equals that rank's own, and a rank's rows / counts say exactly what its own cull made visible"} if exchange_verified is not None else {})},
    }
    if not a.only_cull and not a.no_c5:
        try:
            c5 = c5_result
            if rank == 0 and c5 is not None:
                line.setdefault("paths", {})["c5_mixed_50m_plus_1m_skinned"] = c5
        except Exception as e:
            line["c5_error"] = repr(e)
    if c4_result is not None:
        line.setdefault("paths", {})["c4_pose_skin_100k_sharded"] = c4_result
        if "skin" in c4_result:
            line["secondary"] = {"metric": "M skinned verts/s", "value": c4_result["skin"]["value"], "unit": c4_result["skin"]["unit"], "roofline_frac": c4_result["skin"]["hbm_frac_per_gpu"]}
    if world == 1 and not a.only_cull:
        try:
            line.setdefault("paths", {}).update(secondary_paths(ctx, lb, scenes, peak, a.steps, a.warmup))
            sk = line["paths"]["skin_100k_x5k"]
            line["secondary"] = {"metric": "M skinned verts/s", "value": sk["value"], "unit": sk["unit"], "roofline_frac": sk["roofline"]["frac"]}
            attach_path_baselines(line["paths"])
        except Exception as e:  # the headline number stands on its own
            line["paths_error"] = repr(e)
        try:
            cb, runs = cull_cpu_baseline(20, 2)
            line["cpu_baseline"] = {"value": cb["value"], "unit": "M entities/s", "cores": cb["cores"], "kind": cb["kind"], "sample": cb["sample"],
                                    "impl": cb["impl"], "median_ms": cb["median_s"] * 1e3, "visible": cb["visible"],
                                    "by_workers": [{"workers": x["cores"], "value": x["value"], "median_ms": x["median_s"] * 1e3} for x in runs],
                                    "note": "value = the faster of W = min(cores, 64) and W = 1 (the reference's job system anti-scales on this path)"}
            assert cb["visible"] == visible, "CPU reference and GPU disagree on the visible count"
            if "digest" in cb:
                line["parity"]["reference_digest"] = cb["digest"]
                line["parity"]["equal"] = cb["digest"] == gpu_digest
                assert cb["digest"] == gpu_digest, "the visible set of the 10M C2 cull differs from the reference's own CullingSystemImpl"
        except Exception as e:
            line["cpu_baseline"] = {"value": None, "unit": "M entities/s", "cores": 0, "kind": "reference", "sample": "failed: " + repr(e)}
    emit(line)
    ctx.close()
    if dist:
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=10)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--only-cull", action="store_true", help="skip the secondary paths and the CPU baseline leg (profiling runs)")
    ap.add_argument("--no-c5", action="store_true", help="skip the 50M + 1M mixed scene (BASELINE configs[4])")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the visible set of the last timed cull (rank 0's shard at N>1) to DIR/*.npy, "
                                                          "so that two builds can be compared output for output: the inputs are seeded")
    a = ap.parse_args()
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    a.warmup = max(a.warmup, 3)
    claim_stdout()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if a.impl == "reference":
        reference_arm(a, rank)
    else:
        ours(a, rank, world)


if __name__ == "__main__":
    main()
