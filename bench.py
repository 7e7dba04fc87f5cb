#!/usr/bin/env python3
"""bench.py -- headline benchmark of the hot path (BASELINE.json configs[2]).

Workload: synthetic 10 M-triangle mesh (createTriangleSphere numPhi=1581 = 9 991 920 triangles, the reference's own
benchmark generator), 64 Mi incoherent diffuse-bounce rays (33 cosine-weighted bounces per hit of a 1920x1080 pinhole
image from inside the mesh, path-tracer style: tutorials/pathtracer/pathtracer_device.cpp:1119-1120,1597-1600), traced
as batched rtcIntersect1 records.  A step = one pass of the 64 Mi-ray stream through the trace kernel.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--rays R] [--phi P]

value  : Mrays/s with the RTCRayHit[] stream resident in HBM (rtcb200Intersect1MDevice on torch's current stream),
         whole job over all ranks (weak scaling: every rank traces its own 64 Mi rays; inside the timed region the
         trace kernel itself stores a compact hit record per ray into rank 0's buffer over NVLink peer memory).
e2e    : the same stream through the host-pointer entry point rtcb200Intersect1M with pinned host buffers:
         H2D copy + trace + D2H copy inside the timed region.
--impl reference : the unmodified reference (oracle/_ref/libembree4.so.4, else the C port) on the host cores.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np
import torch

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
from embree_b200 import scenes  # noqa: E402

PRIMARY_W, PRIMARY_H, REPLICATE = 1920, 1080, 33
EYE, LOOK = (0.15, -0.1, 0.05), (0.3, 0.2, 1.0)


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p)), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    return {"hbm_gbs": 6650.0}, "fallback (B200_PROFILING.md 6.65 TB/s)"


def bounce_rays(primary_hits, ids, replicate=REPLICATE):
    """Bounce ray `i` (global index) leaves the hit of primary ray i // replicate with random numbers seeded by i.
    Primary rays that missed re-emit themselves so that indices never depend on hit/miss compaction."""
    parent = (ids // replicate).clamp_max(primary_hits.shape[0] - 1)
    src = primary_hits.index_select(0, parent)
    pri = src.view(torch.int32)
    missed = pri[:, 18] == -1
    if missed.any():
        pri[missed, 18] = 0
        src[missed, 8] = 1.0
        src[missed, 12:15] = -src[missed, 4:7]
    out = scenes.diffuse_bounce_rays(src, seed=0, replicate=1, ids=ids)
    return out


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.rows = index, False, []

    def run(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                o = subprocess.run(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                   stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows if r[0].replace(".", "").isdigit())
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [n for i, n in enumerate(names) if any(r[3 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons,
                "samples": len(self.rows)}


def usable_cores():
    """Host threads this process can really run: scheduler affinity intersected with the cgroup CPU quota (a box may
    report 128 logical CPUs while the container is limited to a fraction of them).  Returns (usable, detail)."""
    logical = os.cpu_count() or 1
    try:
        affinity = len(os.sched_getaffinity(0))
    except Exception:   # noqa: BLE001
        affinity = logical
    quota = None
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    quota = float(txt[0]) / float(txt[1])
            else:
                q = float(txt[0])
                if q > 0:
                    quota = q / float(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read().split()[0])
            break
        except Exception:   # noqa: BLE001
            continue
    usable = affinity if quota is None else max(1, min(affinity, int(quota + 0.999)))
    return usable, {"os_cpu_count": logical, "sched_affinity": affinity, "cgroup_quota_cpus": quota}


def bind_to_gpu_numa(local):
    """Multi-GPU runs: pin this rank (CPU affinity + memory policy) to the NUMA node its GPU hangs off, BEFORE any pinned
    host memory is allocated -- otherwise every rank's staging buffers land on the launching node and the ranks whose
    GPUs sit on the other socket pull their rays across the inter-socket link (round 1: e2e scaled to 50 % at 8 GPUs)."""
    info = {"node": None}
    try:
        pr = torch.cuda.get_device_properties(local)
        dom, bus, devi = getattr(pr, "pci_domain_id", 0), pr.pci_bus_id, pr.pci_device_id
        node = int(open(f"/sys/bus/pci/devices/{dom:04x}:{bus:02x}:{devi:02x}.0/numa_node").read())
        if node < 0:
            return info
        cpus = set()
        for part in open(f"/sys/devices/system/node/node{node}/cpulist").read().strip().split(","):
            a, _, b = part.partition("-")
            cpus.update(range(int(a), int(b or a) + 1))
        cpus &= os.sched_getaffinity(0)
        if not cpus:
            return info
        os.sched_setaffinity(0, cpus)
        info.update(node=node, cpus=len(cpus))
        try:   # set_mempolicy(MPOL_PREFERRED, {node}): first-touch stays local even if a thread migrates
            libc = C.CDLL(None, use_errno=True)
            mask = (C.c_ulong * 16)()
            mask[node // 64] = 1 << (node % 64)
            info["mempolicy"] = "preferred" if libc.syscall(238, 1, mask, 16 * 64) == 0 else "default (set_mempolicy failed)"
        except Exception:   # noqa: BLE001
            info["mempolicy"] = "default"
    except Exception as ex:   # noqa: BLE001
        info["error"] = str(ex)[:100]
    return info


def make_scene(phi):
    t0 = time.time()
    v, t = scenes.triangle_sphere(phi)
    log(f"scene: sphere numPhi={phi}: {len(t)} triangles, {len(v)} vertices ({time.time() - t0:.1f}s)")
    return v, t


def commit(lib, dev, v, t, quality=1):
    sc = lib.rtcNewScene(dev)
    lib.rtcSetSceneBuildQuality(sc, quality)
    _, keep = lib.add_triangle_mesh(dev, sc, v, t, mask=0xFFFFFFFF)
    t0 = time.time()
    lib.rtcCommitScene(sc)
    lib.check(dev)
    return sc, keep, time.time() - t0


# ----------------------------------------------------------------------------------------------------------------------
def run_reference(args):
    """Reference arm: the reference's own CPU implementation on the host cores, same scene / ray definition; each step
    traces a bounded strided sample of the 64 Mi-ray stream with all host threads."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from tests.parity import api_trace_mt, load_oracle, load_reference
    cores, core_detail = usable_cores()
    v, t = make_scene(args.phi)
    R = load_reference()
    kind = "reference" if R is not None else "port"
    nsample = min(args.rays, 1 << 24)
    stride = max(1, args.rays // nsample)
    ids = torch.arange(0, nsample, dtype=torch.int64) * stride
    prim = scenes.primary_rays(PRIMARY_W, PRIMARY_H, eye=EYE, look=LOOK)
    if R is not None:
        dev = R.new_device(None)
        sc, keep, bt = commit(R, dev, v, t)
        log(f"reference rtcCommitScene: {bt * 1e3:.0f} ms")
        prim_np = scenes.as_numpy_rayhits(prim)
        api_trace_mt(R, sc, prim_np, cores)
        trace = lambda recs: api_trace_mt(R, sc, recs, cores)  # noqa: E731
    else:
        o = load_oracle()
        osc = o.scene([(v, t, 0, 0xFFFFFFFF)])
        prim_np = osc.trace(scenes.as_numpy_rayhits(prim), nthreads=cores)
        trace = lambda recs: osc.trace(recs, nthreads=cores)  # noqa: E731
    prim_hits = torch.from_numpy(prim_np.view(np.float32).reshape(-1, 24).copy())
    rays = scenes.as_numpy_rayhits(bounce_rays(prim_hits, ids))
    times = []
    for it in range(args.warmup + args.steps):
        work = rays.copy()
        t0 = time.perf_counter()
        trace(work)
        dt = time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    ms = float(np.mean(times)) * 1e3
    val = nsample / (ms * 1e-3) * 1e-6
    line = {"impl": "reference", "metric": "Mrays/s incoherent diffuse-bounce, 10M-triangle scene", "value": val, "unit": "Mrays/s",
            "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, len(t)),
            "cpu_baseline": {"value": val, "unit": "Mrays/s", "cores": cores, "cores_detail": core_detail, "kind": kind,
                             "sample": f"{nsample} rays = every {stride}th ray of the {args.rays}-ray stream per step, rtcIntersect1 on {cores} host threads (FTZ|DAZ)"},
            "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    emit(line)


def workload_config(args, ntris):
    return {"workload": f"configs[2]: createTriangleSphere(numPhi={args.phi}) = {ntris} triangles, BUILD_QUALITY_MEDIUM (device binned-SAH); "
                        f"{args.rays} incoherent diffuse-bounce rays ({REPLICATE} cosine-weighted bounces per hit of a {PRIMARY_W}x{PRIMARY_H} "
                        f"pinhole image from inside the mesh), batched rtcIntersect1 over RTCRayHit[]",
            "rays_per_gpu": args.rays, "triangles": ntris, "l2": "ray stream 6.4 GB and BVH 0.6 GB per step exceed the 126 MB L2",
            "parallelism": f"ray-stream sharding x{args.gpus}, BVH replicated, compact hit records stored to rank 0 over NVLink by the trace kernel"}


def reference_counters(phi, sample, cores):
    """Traversal counters of the UNMODIFIED reference (EMBREE_STAT_COUNTERS build, kernels/common/stat.h:82-86) on a
    sample of the headline stream, next to ours: the roofline's algorithmic bytes use OUR visit counts, so a looser
    traversal would inflate `achieved`; this shows how many nodes the reference's ordered BVH8 traversal visits on the
    same rays.  Runs oracle/ref_stat.py in a subprocess (the counters print from a static destructor at exit)."""
    so = os.path.join(ROOT, "oracle", "_ref", "libembree4_stat.so.4")
    if not os.path.exists(so):
        return None
    import tempfile
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import ref_stat
    with tempfile.NamedTemporaryFile(suffix=".npy") as f:
        np.save(f.name, np.ascontiguousarray(sample).view(np.uint8))
        r = subprocess.run([sys.executable, os.path.join(ROOT, "oracle", "ref_stat.py"), str(phi), f.name, str(cores)],
                           stdout=subprocess.PIPE, stderr=subprocess.PIPE, text=True, timeout=900)
    d = ref_stat.parse(r.stdout)
    if not d.get("rays"):
        log("reference counters unavailable: " + r.stderr[-300:])
        return None
    return {"rays": int(d["rays"]), "nodes_per_ray": d["nodes"] / d["rays"], "leaves_per_ray": d["leaves"] / d["rays"],
            "triangle4_blocks_per_ray": d["blocks"] / d["rays"],
            "note": "reference BVH8<Triangle4> (256-B nodes, 4-triangle blocks), ordered traversal with pop-time distance culling"}


def dynamic_leg(lib, dev, args):
    """configs[3]b: per-frame re-commit of a dynamic scene, measured as the reference's update.* benchmarks do
    (verify.cpp:6173-6194 CreateGeometryBenchmark, update = true: rtcCommitGeometry + rtcCommitScene of an
    RTC_SCENE_FLAG_DYNAMIC scene; Mprims/s).  Ours is wall time of the same two calls: the vertex upload over PCIe, the
    device build (LBVH / binned SAH) or the refit, and the final synchronisation are all inside."""
    from tests.parity import load_reference
    out = []
    R = load_reference() if not args.no_cpu else None
    rdev = R.new_device(None) if R is not None else None
    for label, phi in (("100k", 159), ("1000k", 501)):
        v, t = scenes.triangle_sphere(phi)
        for gq_name, scene_q, geom_q in (("LOW (Morton rebuild)", 0, 0), ("MEDIUM (binned-SAH rebuild)", 1, 1), ("REFIT", 0, 3)):
            row = {"triangles": len(t), "mesh": f"createTriangleSphere(numPhi={phi})", "quality": gq_name}
            for who, L, d in (("b200", lib, dev), ("reference", R, rdev)):
                if L is None:
                    continue
                sc = L.rtcNewScene(d)
                L.rtcSetSceneFlags(sc, 1)
                L.rtcSetSceneBuildQuality(sc, scene_q)
                gid, keep = L.add_triangle_mesh(d, sc, v, t, mask=0xFFFFFFFF, quality=geom_q)
                L.rtcCommitScene(sc)
                g = L.rtcGetGeometry(sc, gid)
                ts = []
                for it in range(8):
                    keep[0][: v.size] *= 1.001                      # the vertices move every frame
                    L.rtcUpdateGeometryBuffer(g, 1, 0)
                    t0 = time.perf_counter()
                    L.rtcCommitGeometry(g)
                    L.rtcCommitScene(sc)
                    dt = time.perf_counter() - t0
                    if it >= 2:
                        ts.append(dt)
                L.check(d)
                ms = float(np.mean(ts)) * 1e3
                row[who] = {"commit_ms": ms, "Mprims_per_s": len(t) / ms * 1e-3}
                if who == "b200":
                    st = L.scene_stats(sc)
                    row[who]["device_ms"] = st.build_ms
                    row[who]["path"] = ["lbvh build", "sah build", "refit", "two-level"][st.builder]
                L.rtcReleaseScene(sc)
            out.append(row)
    if R is not None:
        R.rtcReleaseDevice(rdev)
    return out


def two_level_leg(lib, dev, args):
    """configs[3]b, the tutorial's case proper (tutorials/dynamic_scene: many meshes, a few of them move every frame): one static terrain of
    4 M triangles + 200 spheres of 5 000 triangles each in an RTC_SCENE_FLAG_DYNAMIC scene; per frame 10 spheres move and the scene is
    committed.  Wall time of rtcCommitGeometry x 10 + rtcCommitScene: the two-level path (one kept BVH per mesh, only the moved meshes are
    uploaded and rebuilt), the same library forced to rebuild one BVH over everything (RTCB200_NO_TWOLEVEL), and the reference's
    two-level builder (scene build quality LOW, as the tutorial sets it)."""
    from tests.parity import load_reference
    tv, tt = scenes.terrain(1414, seed=3)
    rng = np.random.RandomState(1)
    sv, st_ = scenes.triangle_sphere(36)
    balls = []
    for i in range(200):
        c = np.array([rng.uniform(-0.9, 0.9), rng.uniform(0.2, 0.6), rng.uniform(-0.9, 0.9)], np.float32)
        balls.append((sv * np.float32(0.03) + c).astype(np.float32))
    R = load_reference() if not args.no_cpu else None
    out = {"workload": f"terrain {len(tt)} triangles (static) + 200 spheres x {len(st_)} triangles, 10 spheres move per frame, RTC_SCENE_FLAG_DYNAMIC, scene quality LOW",
           "triangles": int(len(tt) + 200 * len(st_))}
    wv, wt = scenes.triangle_sphere(20)          # warm-up commit: one-time costs of the process (module load, occupancy queries) stay out of first_commit_ms
    wsc = lib.rtcNewScene(dev)
    wkeep = [lib.add_triangle_mesh(dev, wsc, wv, wt, geom_id=0)[1], lib.add_triangle_mesh(dev, wsc, wv + np.float32(3), wt, geom_id=1)[1]]
    lib.rtcSetSceneFlags(wsc, 1)
    lib.rtcCommitScene(wsc)
    lib.rtcReleaseScene(wsc)
    runs = [("b200_two_level", lib, dev, None), ("b200_single_bvh_rebuild", lib, dev, "1")]
    if R is not None:
        runs.append(("reference", R, R.new_device(None), None))
    for name, L, d, env in runs:
        if env:
            os.environ["RTCB200_NO_TWOLEVEL"] = env
        sc = L.rtcNewScene(d)
        L.rtcSetSceneFlags(sc, 1)
        L.rtcSetSceneBuildQuality(sc, 0)
        keep = [L.add_triangle_mesh(d, sc, tv, tt, mask=0xFFFFFFFF, geom_id=0)[1]]
        for i, bv in enumerate(balls):
            keep.append(L.add_triangle_mesh(d, sc, bv, st_, mask=0xFFFFFFFF, geom_id=1 + i)[1])
        t0 = time.perf_counter()
        L.rtcCommitScene(sc)
        first = time.perf_counter() - t0
        L.check(d)
        ts = []
        for it in range(8):
            moved = [1 + (it * 10 + k) % 200 for k in range(10)]
            for m in moved:
                keep[m][0][: sv.size] += np.float32(0.001)
                g = L.rtcGetGeometry(sc, m)
                L.rtcUpdateGeometryBuffer(g, 1, 0)
            t0 = time.perf_counter()
            for m in moved:
                L.rtcCommitGeometry(L.rtcGetGeometry(sc, m))
            L.rtcCommitScene(sc)
            dt = time.perf_counter() - t0
            if it == 0:
                frame0 = dt
            if it >= 2:
                ts.append(dt)
        L.check(d)
        row = {"first_commit_ms": first * 1e3, "second_commit_ms": frame0 * 1e3, "recommit_ms": float(np.mean(ts)) * 1e3}   # second commit: the kept per-mesh BVHs are built here (two-level path)
        if L is lib:
            row["path"] = ["lbvh build", "sah build", "refit", "two-level"][L.scene_stats(sc).builder]
            rays = scenes.as_numpy_rayhits(scenes.primary_rays(480, 270, eye=(0.0, 0.9, -0.2), look=(0.0, -1.0, 0.25)))
            hit = L.intersect(sc, rays, "1M")
            row["camera_hit_fraction"] = float((hit["geomID"] != 0xFFFFFFFF).mean())
            row["camera_hit_checksum"] = int(hit["primID"][hit["geomID"] != 0xFFFFFFFF].astype(np.uint64).sum())
        L.rtcReleaseScene(sc)
        if env:
            del os.environ["RTCB200_NO_TWOLEVEL"]
        out[name] = row
    if R is not None:
        R.rtcReleaseDevice(runs[-1][2])
    return out


def hair_leg(lib, dev, devt, stream, args, rnd=False):
    """configs[3]a (rnd: the same fur ball as RTC_GEOMETRY_TYPE_ROUND_BEZIER_CURVE, the xml loader's default hair type,
    xml_loader.cpp:1322 -- the sweep intersector): tutorials/hair_geometry with Bezier curves -- a fur ball of flat cubic Bezier curves
    (RTC_GEOMETRY_TYPE_FLAT_BEZIER_CURVE, what the tutorials' hair generators and loaders create, geometry_creation.cpp:340,
    obj_loader.cpp:641) around a triangle sphere.  Two ray sets: 1920x1080 camera rays and as many incoherent rays aimed at
    the ball; closest hit and any hit, device-resident, CUDA events; next to the unmodified reference's rtcIntersect1 on the
    usable host threads, with parity of every ray."""
    from tests.parity import api_trace_mt, compare_hits, load_reference, sweep_disagreements, unexplained_ribbon_disagreements
    strands = 120000
    cv, ci, _tg = scenes.cubic_hair(strands, "bezier", knots=10, seed=5, radius=1.0, step=0.05, width=0.0025)
    v, t = scenes.triangle_sphere(201)

    def build(L, d):
        sc = L.rtcNewScene(d)
        keep = [L.add_triangle_mesh(d, sc, v, t, mask=0xFFFFFFFF, geom_id=0)[1], L.add_flat_cubic_curves(d, sc, cv, ci, "bezier", None, None, mask=0xFFFFFFFF, geom_id=1, round=rnd)[1]]
        t0 = time.perf_counter()
        L.rtcCommitScene(sc)
        dt = time.perf_counter() - t0
        L.check(d)
        return sc, keep, dt
    sc, keep, commit_s = build(lib, dev)
    st = lib.scene_stats(sc)
    cam = scenes.primary_rays(PRIMARY_W, PRIMARY_H, eye=(0.0, 0.4, -2.6), look=(0.0, -0.15, 1.0), fov=60.0, device=devt)
    g = torch.Generator(device="cpu").manual_seed(11)
    n = cam.shape[0]
    o = torch.randn((n, 3), generator=g)
    o = o / o.norm(dim=1, keepdim=True) * (1.3 + 1.2 * torch.rand((n, 1), generator=g))
    d = -o + 0.45 * torch.randn((n, 3), generator=g)
    inc = scenes.pack_rayhits(o.to(devt), d.to(devt), 0.0, float("inf"))
    a = lib.args()
    kind = "round cubic Bezier curves (swept spheres)" if rnd else "flat cubic Bezier curves (tessellation rate 4)"
    out = {"workload": f"fur ball: {strands} strands x 3 {kind} = {len(ci)} curves + createTriangleSphere(numPhi=201) = {len(t)} triangles",
           "curves": int(len(ci)), "triangles": int(len(t)), "commit_ms": commit_s * 1e3, "build_device_ms": st.build_ms, "nodes": int(st.num_nodes)}
    cores, _detail = usable_cores()
    R = load_reference() if not args.no_cpu else None
    rsc2 = None
    if R is not None:
        rdev = R.new_device(None)
        rsc, rkeep, rcommit = build(R, rdev)
        out["reference_commit_ms"] = rcommit * 1e3
        if rnd:
            rdev2 = R.new_device("isa=avx2")
            rsc2, rkeep2, _c2 = build(R, rdev2)
    for name, rays in (("camera_1080p", cam), ("incoherent", inc)):
        work = rays.clone()
        best = 1e9
        for it in range(4):
            work.copy_(rays)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            lib.rtcb200Intersect1MDevice(sc, C.c_void_p(work.data_ptr()), n, C.byref(a), C.c_void_p(stream))
            c1.record()
            torch.cuda.synchronize()
            if it:
                best = min(best, c0.elapsed_time(c1))
        occ = rays[:, :12].contiguous()
        ow = occ.clone()
        obest = 1e9
        for it in range(3):
            ow.copy_(occ)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            lib.rtcb200Occluded1MDevice(sc, C.c_void_p(ow.data_ptr()), n, C.byref(a), C.c_void_p(stream))
            c1.record()
            torch.cuda.synchronize()
            if it:
                obest = min(obest, c0.elapsed_time(c1))
        gi = work.view(torch.int32)[:, 18]
        row = {"rays": int(n), "Mrays_per_s": n / best * 1e-3, "ms": best, "occluded_Mrays_per_s": n / obest * 1e-3,
               "curve_hit_fraction": float((gi == 1).float().mean().item()), "triangle_hit_fraction": float((gi == 0).float().mean().item())}
        if R is not None:
            got = scenes.as_numpy_rayhits(work.cpu())
            rin = scenes.as_numpy_rayhits(rays.cpu())
            rbest = 1e30
            for _ in range(2):
                w = rin.copy()
                t0 = time.perf_counter()
                api_trace_mt(R, rsc, w, cores)
                rbest = min(rbest, time.perf_counter() - t0)
            row["reference"] = {"Mrays_per_s": n / rbest * 1e-6, "cores": cores, "api": "rtcIntersect1 loop (FTZ|DAZ), best of 2"}
            rep = compare_hits(w, got)
            row["parity"] = {k: rep[k] for k in ("n", "hits", "id_mismatch", "tie", "hit_miss_disagree", "max_rel_t", "max_abs_uv")}
            if rnd:
                # The hit is the root of a Newton iteration (at most 5 steps from cylinder estimates): implementations part where it is
                # ill-conditioned -- mostly on the silhouette of the tube (|cos(Ng, dir)| < 0.1 at the nearer hit), a few at the
                # iteration limit.  The yardstick is the reference against ITSELF: its AVX2 and AVX-512 code paths (same algorithm,
                # different reciprocal / rsqrt approximations) on the same rays.
                nd, bad = sweep_disagreements(rin, w, got, {1})
                row["parity"]["differing_rays"] = nd
                row["parity"]["not_a_silhouette_graze"] = bad
                if rsc2 is not None:
                    w2 = rin.copy()
                    api_trace_mt(R, rsc2, w2, cores)
                    sd, sb = sweep_disagreements(rin, w, w2, {1})
                    row["parity"]["reference_avx512_vs_its_own_avx2_path"] = {"differing_rays": sd, "not_a_silhouette_graze": sb}
            else:
                nd, bad = unexplained_ribbon_disagreements(w, got, {1})
                row["parity"]["differing_rays"] = nd
                row["parity"]["not_on_a_ribbon_edge"] = bad     # every difference must be a ray through the very edge (|v| >= 0.999) of the nearer ribbon
            row["parity"]["checked_against"] = "reference, every ray"
        out[name] = row
        del work, occ, ow
    if R is not None:
        R.rtcReleaseScene(rsc)
        R.rtcReleaseDevice(rdev)
        if rsc2 is not None:
            R.rtcReleaseScene(rsc2)
            R.rtcReleaseDevice(rdev2)
    lib.rtcReleaseScene(sc)
    return out


def point_leg(lib, dev, devt, stream, args):
    """Point primitives (tutorials/point_geometry's geometry types at scale): 2 M sphere points / ray-facing discs / oriented discs in a
    ball, 1920x1080 camera rays; closest hit and any hit, device-resident, CUDA events; next to the unmodified reference's rtcIntersect1
    on the usable host threads with parity of every ray (differences must be rays on a decision boundary of the test)."""
    from tests.parity import api_trace_mt, compare_hits, load_reference, point_disagreements
    rng = np.random.RandomState(31)
    npts = 2000000
    c = rng.normal(size=(npts, 3)).astype(np.float32)
    c = c / np.linalg.norm(c, axis=1, keepdims=True) * (rng.uniform(0.0, 1.0, (npts, 1)) ** (1.0 / 3.0)).astype(np.float32)
    pv = np.concatenate([c, rng.uniform(0.001, 0.004, (npts, 1)).astype(np.float32)], 1).astype(np.float32)
    pn = rng.normal(size=(npts, 3)).astype(np.float32)
    cam = scenes.primary_rays(PRIMARY_W, PRIMARY_H, eye=(0.0, 0.4, -2.6), look=(0.0, -0.15, 1.0), fov=60.0, device=devt)
    n = cam.shape[0]
    a = lib.args()
    cores, _detail = usable_cores()
    R = load_reference() if not args.no_cpu else None
    out = {"workload": f"{npts} points of radius 0.001-0.004 in the unit ball, {PRIMARY_W}x{PRIMARY_H} camera rays", "points": npts}
    for kind in ("sphere", "disc", "oriented_disc"):
        def build(L, d):
            sc = L.rtcNewScene(d)
            keep = L.add_points(d, sc, pv, kind, normals=pn, mask=0xFFFFFFFF, geom_id=0)[1]
            t0 = time.perf_counter()
            L.rtcCommitScene(sc)
            dt = time.perf_counter() - t0
            L.check(d)
            return sc, keep, dt
        sc, keep, commit_s = build(lib, dev)
        work = cam.clone()
        best = 1e9
        for it in range(4):
            work.copy_(cam)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            lib.rtcb200Intersect1MDevice(sc, C.c_void_p(work.data_ptr()), n, C.byref(a), C.c_void_p(stream))
            c1.record()
            torch.cuda.synchronize()
            if it:
                best = min(best, c0.elapsed_time(c1))
        occ = cam[:, :12].contiguous()
        ow = occ.clone()
        obest = 1e9
        for it in range(3):
            ow.copy_(occ)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            lib.rtcb200Occluded1MDevice(sc, C.c_void_p(ow.data_ptr()), n, C.byref(a), C.c_void_p(stream))
            c1.record()
            torch.cuda.synchronize()
            if it:
                obest = min(obest, c0.elapsed_time(c1))
        row = {"commit_ms": commit_s * 1e3, "rays": int(n), "Mrays_per_s": n / best * 1e-3, "ms": best, "occluded_Mrays_per_s": n / obest * 1e-3,
               "hit_fraction": float((work.view(torch.int32)[:, 18] == 0).float().mean().item())}
        if R is not None:
            rdev = R.new_device(None)
            rsc, rkeep, rcommit = build(R, rdev)
            row["reference_commit_ms"] = rcommit * 1e3
            got = scenes.as_numpy_rayhits(work.cpu())
            rin = scenes.as_numpy_rayhits(cam.cpu())
            w = rin.copy()
            t0 = time.perf_counter()
            api_trace_mt(R, rsc, w, cores)
            row["reference"] = {"Mrays_per_s": n / (time.perf_counter() - t0) * 1e-6, "cores": cores, "api": "rtcIntersect1 loop (FTZ|DAZ)"}
            rep = compare_hits(w, got)
            nd, bad = point_disagreements(rin, w, got, {0: (pv, kind, pn)})
            row["parity"] = {k: rep[k] for k in ("n", "hits", "max_rel_t", "max_abs_uv")}
            row["parity"].update({"differing_rays": nd, "not_on_a_decision_boundary": bad, "checked_against": "reference, every ray"})
            R.rtcReleaseScene(rsc)
            R.rtcReleaseDevice(rdev)
        out[kind] = row
        lib.rtcReleaseScene(sc)
        del work, occ, ow
    return out


def coherent_leg(lib, dev, devt, stream, workload, phi, rays, args):
    """One coherent configuration, measured like the headline: device-resident value (CUDA events, 3 warm-up + 5 timed
    passes over a packet stream larger than L2), e2e through the host-pointer entry point rtcb200IntersectNM with pinned
    buffers, the reference's rtcIntersect16 with RTC_RAY_QUERY_FLAG_COHERENT on the usable host cores, parity of the FULL
    frame, and the algorithmic roofline of the launch.  `rays`: [n,24] RTCRayHit records on the device in packet order."""
    import embree_b200  # noqa: F401
    from embree_b200.rtc import from_packets, packet_dtype
    v1, t1 = scenes.triangle_sphere(phi)
    sc1, keep1, _ = commit(lib, dev, v1, t1)
    n = rays.shape[0]
    npk = n // 16
    pk0 = rays.view(npk, 16, 24).permute(0, 2, 1)[:, :21, :].contiguous()   # AoS -> RTCRayHit16 SoA (21 fields x 16 lanes)
    pk = pk0.clone()
    ac = lib.args(coherent=True)

    def go():
        lib.rtcb200IntersectNMDevice(None, sc1, C.c_void_p(pk.data_ptr()), 16, npk, C.byref(ac), C.c_void_p(stream))
    lib.rtcb200SetSceneStatCounters(sc1, 1)
    lib.rtcb200ResetSceneStatCounters(sc1)
    go()
    torch.cuda.synchronize()
    s2 = lib.scene_stats(sc1)
    lib.rtcb200SetSceneStatCounters(sc1, 0)
    npr, tpr = s2.trav_nodes / s2.trav_rays, s2.trav_tris / s2.trav_rays
    times = []
    for it in range(8):
        pk.copy_(pk0)
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record()
        go()
        c1.record()
        torch.cuda.synchronize()
        if it >= 3:
            times.append(c0.elapsed_time(c1))
    ms = float(np.mean(times))
    lib.check(dev)
    bytes_per_ray = 40 + 40 + npr * 96 + tpr * 48        # 10 ray fields read, tfar + 9 hit fields written, per lane
    peaks, peak_src = measured_peaks()
    out = {"workload": workload, "rays": n, "value": n / ms * 1e-3, "unit": "Mrays/s", "ms_per_step": ms, "steps": len(times), "warmup": 3,
           "hits": int((pk.view(torch.int32)[:, 18, :] != -1).sum().item()),
           "roofline": {"bound": "hbm", "achieved": bytes_per_ray * n / (ms * 1e-3) * 1e-9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                        "frac": bytes_per_ray * n / (ms * 1e-3) * 1e-9 / peaks["hbm_gbs"], "algorithmic_bytes_per_ray": bytes_per_ray,
                        "nodes_per_ray": npr, "tris_per_ray": tpr, "traffic": None, "peak_source": peak_src,
                        "kernel": "rtk::trace_kernel<K=16,OCCLUDED=false,...>", "packet_stream_bytes": n * 84}}
    if not args.no_e2e:
        H = torch.empty(pk0.shape, dtype=torch.float32).pin_memory()
        times = []
        for it in range(4):
            H.copy_(pk0)
            t0 = time.perf_counter()
            lib.rtcb200IntersectNM(None, sc1, C.c_void_p(H.data_ptr()), 16, npk, C.byref(ac))
            dt = time.perf_counter() - t0
            if it > 0:
                times.append(dt)
        lib.check(dev)
        out["e2e"] = {"value": n / float(np.mean(times)) * 1e-6, "unit": "Mrays/s", "h2d_bytes_per_step": n * 84, "d2h_bytes_per_step": n * 84,
                      "api": "rtcb200IntersectNM(NULL, scene, RTCRayHit16* host, 16, M, args), pinned host buffers"}
        out["e2e"]["host_equals_device"] = bool(torch.equal(H.view(torch.int32)[:, 8:19, :], pk.cpu().view(torch.int32)[:, 8:19, :]))   # bit-identical records
        del H
    if not args.no_cpu:
        from tests.parity import api_trace_mt, compare_hits, load_reference
        R = load_reference()
        if R is not None:
            cores, detail = usable_cores()
            rdev = R.new_device(None)
            rsc, rkeep, _ = commit(R, rdev, v1, t1)
            from embree_b200.rtc import aligned_empty
            src = pk0.cpu().numpy().reshape(-1).view(packet_dtype(16))
            best, w = 1e30, aligned_empty(npk, packet_dtype(16), align=64)    # RTCRayHit16 must be 64-byte aligned (rtcore.cpp:867)
            for _ in range(2):
                w[:] = src
                t0 = time.perf_counter()
                api_trace_mt(R, rsc, w, cores, K=16, coherent=True)
                best = min(best, time.perf_counter() - t0)
            out["cpu_baseline"] = {"value": n / best * 1e-6, "unit": "Mrays/s", "cores": cores, "cores_detail": detail, "kind": "reference",
                                   "sample": f"all {n} rays, rtcIntersect16 + RTC_RAY_QUERY_FLAG_COHERENT on {cores} host threads (FTZ|DAZ), best of 2"}
            got = from_packets(pk.cpu().numpy().reshape(-1).view(packet_dtype(16)), n)
            out["parity"] = compare_hits(from_packets(w, n), got, meshes=[(v1, t1, 0, 0xFFFFFFFF)])
            out["parity"]["checked_against"] = "reference, full frame"
            R.rtcReleaseScene(rsc)
            R.rtcReleaseDevice(rdev)
    lib.rtcReleaseScene(sc1)
    lib.check(dev)
    return out


# ----------------------------------------------------------------------------------------------------------------------
# --workload pathtracer: BASELINE configs[4] -- 10 M-triangle scene, 8 bounces, the path stream sharded over the GPUs
# ----------------------------------------------------------------------------------------------------------------------
PT_BOUNCES, PT_SPP = 8, 16
PT_LIGHT = (0.2, 0.3, -0.1, 1.0, 0.8)      # point light inside the mesh (px, py, pz, intensity), matte albedo 0.8


def pathtracer_config(args, ntris, world):
    return {"workload": f"configs[4]: createTriangleSphere(numPhi={args.phi}) = {ntris} triangles; wavefront form of tutorials/pathtracer "
                        f"(pathtracer_device.cpp:1489-1603): {args.rays} paths per GPU ({PRIMARY_W}x{PRIMARY_H} pinhole, jittered samples), "
                        f"{PT_BOUNCES} bounces, per bounce one batched rtcIntersect1 pass + one rtcOccluded1 shadow pass (matte material, one point light)",
            "paths_per_gpu": args.rays, "bounces": PT_BOUNCES, "rays_per_step_per_gpu": args.rays * PT_BOUNCES * 2, "triangles": ntris,
            "l2": "each pass streams 3.2-6.4 GB of ray records: larger than the 126 MB L2",
            "parallelism": f"path-stream sharding x{world}, BVH replicated, bounce generation local to each GPU, only the last bounce's compact "
                           "hit records are gathered to rank 0 (stored over NVLink by the trace kernel)"}


def run_pathtracer(args):
    import torch.distributed as dist
    import embree_b200
    from embree_b200 import pathstream
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    devt = torch.device("cuda", local)
    numa = bind_to_gpu_numa(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=devt)
    lib, pts = embree_b200.load(), pathstream.load()
    dev = lib.new_device(f"gpu={local},verbose={2 if rank == 0 else 0}")
    v, t = make_scene(args.phi)
    sc, keep, _ = commit(lib, dev, v, t)
    lib.rtcReleaseScene(sc)
    sc, keep, commit_s = commit(lib, dev, v, t)
    st = lib.scene_stats(sc)
    a, ao = lib.args(), lib.args()
    stream = torch.cuda.current_stream().cuda_stream
    n = args.rays
    cam = scenes.camera_basis(PRIMARY_W, PRIMARY_H, EYE, LOOK)
    cam_c = (C.c_float * 12)(*cam.tolist())
    light_c = (C.c_float * 5)(*PT_LIGHT)
    R = torch.empty((n, 24), dtype=torch.float32, device=devt)       # RTCRayHit[] path records, reused in place by every bounce
    S = torch.empty((n, 12), dtype=torch.float32, device=devt)       # RTCRay[] shadow rays
    rng = torch.empty(n, dtype=torch.int32, device=devt)
    Lw, pend, L = (torch.empty(n, dtype=torch.float32, device=devt) for _ in range(3))
    gbuf, my_out, flag = None, None, None
    if world > 1:
        handle = [None]
        if rank == 0:
            gbuf = lib.rtcb200PeerAlloc(dev, world * n * 32)
            h64 = (C.c_ubyte * 64)()
            assert lib.rtcb200PeerExport(dev, C.c_void_p(gbuf), h64) == 0
            handle = [bytes(h64)]
        dist.broadcast_object_list(handle, src=0)
        if rank != 0:
            gbuf = lib.rtcb200PeerImport(dev, (C.c_ubyte * 64).from_buffer_copy(handle[0]))
        lib.check(dev)
        my_out = gbuf + rank * n * 32
        flag = torch.zeros(1, device=devt)
    P = lambda x: C.c_void_p(x.data_ptr())   # noqa: E731
    first_path = rank * n
    ev = None

    def step(events=None, capture=None):
        L.zero_()
        assert pts.pts200_primary(P(R), P(rng), P(Lw), first_path, n, cam_c, PRIMARY_W, PRIMARY_H, PT_SPP, C.c_void_p(stream)) == 0
        for b in range(PT_BOUNCES):
            if capture is not None:
                capture["in"].append(R[capture["idx"]].clone())
            if events is not None:
                events[b][0].record()
            if world > 1 and b == PT_BOUNCES - 1:
                lib.rtcb200Intersect1MGatherDevice(sc, P(R), n, C.byref(a), C.c_void_p(stream), C.c_void_p(my_out))
            else:
                lib.rtcb200Intersect1MDevice(sc, P(R), n, C.byref(a), C.c_void_p(stream))
            if events is not None:
                events[b][1].record()
            if capture is not None:
                capture["out"].append(R[capture["idx"]].clone())
            assert pts.pts200_bounce(P(R), P(S), P(rng), P(Lw), P(pend), n, light_c, C.c_void_p(stream)) == 0
            if capture is not None:
                capture["sin"].append(S[capture["idx"]].clone())
            if events is not None:
                events[b][2].record()
            lib.rtcb200Occluded1MDevice(sc, P(S), n, C.byref(ao), C.c_void_p(stream))
            if events is not None:
                events[b][3].record()
            if capture is not None:
                capture["sout"].append(S[capture["idx"]].clone())
            assert pts.pts200_shade(P(S), P(pend), P(L), n, C.c_void_p(stream)) == 0
        if world > 1:
            dist.all_reduce(flag)

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = lib.rtcb200GetLaunchCount()
    evs = [[[torch.cuda.Event(enable_timing=True) for _ in range(4)] for _ in range(PT_BOUNCES)] for _ in range(args.steps)]
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for k in range(args.steps):
        step(events=evs[k])
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler.stop_flag = True
    launches = (lib.rtcb200GetLaunchCount() - l0) + args.steps * (1 + 2 * PT_BOUNCES)      # + primary / bounce / shade kernels
    ms = torch.tensor([e0.elapsed_time(e1) / args.steps], device=devt)
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    ms_per_step = float(ms.item())
    rays_per_step = n * PT_BOUNCES * 2
    value = rays_per_step * world / (ms_per_step * 1e-3) * 1e-6
    per_bounce = []
    for b in range(PT_BOUNCES):
        ti = float(np.mean([evs[k][b][0].elapsed_time(evs[k][b][1]) for k in range(args.steps)]))
        tb = float(np.mean([evs[k][b][1].elapsed_time(evs[k][b][2]) for k in range(args.steps)]))
        to = float(np.mean([evs[k][b][2].elapsed_time(evs[k][b][3]) for k in range(args.steps)]))
        per_bounce.append({"bounce": b, "intersect_Mrays_per_s": n / ti * 1e-3, "occluded_Mrays_per_s": n / to * 1e-3,
                           "intersect_ms": ti, "bounce_kernel_ms": tb, "occluded_ms": to})
    lib.check(dev)
    sampler.join(timeout=2)
    radiance_mean = float(L.mean().item())
    alive_last = float((R[:, 8] >= 0).float().mean().item())

    # ---- end to end: the host provides the camera, receives the radiance of every path and the final hit records
    e2e = None
    if not args.no_e2e:
        Lh = torch.empty(n, dtype=torch.float32).pin_memory()
        Hh = torch.empty((n, 24), dtype=torch.float32).pin_memory()
        times = []
        for it in range(3):
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            step()
            Lh.copy_(L, non_blocking=True)
            Hh.copy_(R, non_blocking=True)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if it > 0:
                times.append(dt)
        tt = torch.tensor([float(np.mean(times))], device=devt)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": rays_per_step * world / float(tt.item()) * 1e-6, "unit": "Mrays/s", "h2d_bytes_per_step": 48 * world,
               "d2h_bytes_per_step": n * (4 + 96) * world, "ms_per_step": float(tt.item()) * 1e3,
               "api": "pts200_primary + 8 x (rtcb200Intersect1MDevice, pts200_bounce, rtcb200Occluded1MDevice, pts200_shade); the camera goes in, "
                      "the radiance per path and the last bounce's RTCRayHit records come back to pinned host memory"}

    # ---- parity of every bounce on a strided sample + CPU baseline on the same sampled streams (rank 0, N == 1)
    parity, cpu_baseline = None, None
    if rank == 0 and world == 1 and not args.no_cpu:
        from tests.parity import api_trace_mt, compare_hits, load_reference
        ns = min(n, 1 << 19)
        cap = {"idx": torch.arange(0, n, max(1, n // ns), device=devt)[:ns], "in": [], "out": [], "sin": [], "sout": []}
        step(capture=cap)
        torch.cuda.synchronize()
        Rl = load_reference()
        if Rl is not None:
            cores, detail = usable_cores()
            rdev = Rl.new_device(None)
            rsc, rkeep, rbt = commit(Rl, rdev, v, t)
            t_int, t_occ, reps = 0.0, 0.0, []
            for b in range(PT_BOUNCES):
                w = scenes.as_numpy_rayhits(cap["in"][b].cpu())
                t0 = time.perf_counter()
                api_trace_mt(Rl, rsc, w, cores)
                t_int += time.perf_counter() - t0
                rep = compare_hits(w, scenes.as_numpy_rayhits(cap["out"][b].cpu()), meshes=[(v, t, 0, 0xFFFFFFFF)])
                from embree_b200.rtc import RAY_DTYPE, aligned_empty
                sw = aligned_empty(len(w), RAY_DTYPE)
                sw.view(np.float32).reshape(-1, 12)[:] = cap["sin"][b].cpu().numpy()
                t0 = time.perf_counter()
                api_trace_mt(Rl, rsc, sw, cores, occluded=True)
                t_occ += time.perf_counter() - t0
                got_s = cap["sout"][b].cpu().numpy()[:, 8]
                rep["shadow_disagree"] = int(((sw["tfar"] < 0) != (got_s < 0)).sum())
                rep["bounce"] = b
                reps.append(rep)
            parity = {"checked_against": "reference", "sample_paths": int(len(cap["idx"])), "per_bounce": reps,
                      "id_mismatch": sum(r["id_mismatch"] for r in reps), "tie": sum(r["tie"] for r in reps),
                      "hit_miss_disagree": sum(r["hit_miss_disagree"] for r in reps), "shadow_disagree": sum(r["shadow_disagree"] for r in reps),
                      "max_rel_t": max(r["max_rel_t"] for r in reps), "ng_bit_exact": all(r["ng_bit_exact"] for r in reps)}
            nr = len(cap["idx"]) * PT_BOUNCES * 2
            cpu_baseline = {"value": nr / (t_int + t_occ) * 1e-6, "unit": "Mrays/s", "cores": cores, "cores_detail": detail, "kind": "reference",
                            "sample": f"{len(cap['idx'])} paths (every {max(1, n // ns)}th) x {PT_BOUNCES} bounces: the GPU's own bounce / shadow streams "
                                      f"traced with rtcIntersect1 / rtcOccluded1 on {cores} host threads (FTZ|DAZ)", "commit_ms": rbt * 1e3,
                            "intersect_Mrays_per_s": nr / 2 / t_int * 1e-6, "occluded_Mrays_per_s": nr / 2 / t_occ * 1e-6}
    if rank == 0:
        peaks, peak_src = measured_peaks()
        bk = float(np.mean([pb["bounce_kernel_ms"] for pb in per_bounce]))
        bk_bytes = n * (80 + 4 + 4 + 64 + 48 + 4 + 4 + 4)   # record read (5 x 16 B) + rng/Lw r/w + next ray (4 x 16 B) + shadow ray + pending
        line = {"metric": "Mrays/s path-tracer stream (8 bounces, closest-hit + shadow rays), 10M-triangle scene", "value": value, "unit": "Mrays/s",
                "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": pathtracer_config(args, len(t), world),
                "clocks": sampler.summary(), "e2e": e2e, "gpu_launches": int(launches), "per_bounce": per_bounce,
                "radiance_mean": radiance_mean, "alive_after_last_bounce": alive_last, "numa": numa,
                "roofline": {"bound": "hbm", "kernel": "pts200 bounce_kernel (the workload's own kernel; the trace kernels' roofline is the headline bench's)",
                             "achieved": bk_bytes / (bk * 1e-3) * 1e-9, "peak": peaks["hbm_gbs"], "unit": "GB/s",
                             "frac": bk_bytes / (bk * 1e-3) * 1e-9 / peaks["hbm_gbs"], "traffic": None, "peak_source": peak_src, "kernel_ms": bk,
                             "algorithmic_bytes_per_path": bk_bytes / n},
                "cpu_baseline": cpu_baseline, "parity": parity,
                "build": {"device_ms": st.build_ms, "commit_wall_ms": commit_s * 1e3, "nodes": int(st.num_nodes)}}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


def run_pathtracer_reference(args):
    """Reference arm of the path-tracer workload: the unmodified reference traces the same kind of stream on the host
    cores -- primary rays, then per bounce rtcIntersect1 + rtcOccluded1 -- with the bounce rays generated between the timed
    calls by the torch restatement of the bounce kernel (scenes.path_bounce, untimed).  Bounded sample of paths."""
    if int(os.environ.get("RANK", "0")) != 0:
        return
    from embree_b200.rtc import RAY_DTYPE, aligned_empty
    from tests.parity import api_trace_mt, load_oracle, load_reference
    cores, detail = usable_cores()
    v, t = make_scene(args.phi)
    R = load_reference()
    kind = "reference" if R is not None else "port"
    if R is not None:
        dev = R.new_device(None)
        sc, keep, bt = commit(R, dev, v, t)
        trace = lambda recs, occ: api_trace_mt(R, sc, recs, cores, occluded=occ)   # noqa: E731
    else:
        osc = load_oracle().scene([(v, t, 0, 0xFFFFFFFF)])
        trace = lambda recs, occ: osc.trace(recs, occluded=occ, nthreads=cores)   # noqa: E731
    n = min(args.rays, 1 << 20)
    stride = max(1, args.rays // n)
    cam = scenes.camera_basis(PRIMARY_W, PRIMARY_H, EYE, LOOK)
    times = []
    for it in range(args.warmup + args.steps):
        r, rng, Lw = scenes.path_primary(0, n * stride, cam, PRIMARY_W, PRIMARY_H, PT_SPP)
        r, rng, Lw = r[::stride].contiguous(), rng[::stride].contiguous(), Lw[::stride].contiguous()
        dt = 0.0
        for b in range(PT_BOUNCES):
            w = scenes.as_numpy_rayhits(r)
            t0 = time.perf_counter()
            trace(w, False)
            dt += time.perf_counter() - t0
            r = torch.from_numpy(w.view(np.float32).reshape(-1, 24).copy())
            shadow, rng, Lw, _ = scenes.path_bounce(r, rng, Lw, PT_LIGHT)
            sw = aligned_empty(n, RAY_DTYPE)
            sw.view(np.float32).reshape(-1, 12)[:] = shadow.numpy()
            t0 = time.perf_counter()
            trace(sw, True)
            dt += time.perf_counter() - t0
        if it >= args.warmup:
            times.append(dt)
    ms = float(np.mean(times)) * 1e3
    val = n * PT_BOUNCES * 2 / (ms * 1e-3) * 1e-6
    emit({"impl": "reference", "metric": "Mrays/s path-tracer stream (8 bounces, closest-hit + shadow rays), 10M-triangle scene", "value": val,
          "unit": "Mrays/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True,
          "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": pathtracer_config(args, len(t), args.gpus),
          "cpu_baseline": {"value": val, "unit": "Mrays/s", "cores": cores, "cores_detail": detail, "kind": kind,
                           "sample": f"{n} paths (every {stride}th) x {PT_BOUNCES} bounces per step, rtcIntersect1 + rtcOccluded1 on {cores} host threads; "
                                     "bounce rays generated between the timed calls (untimed)"},
          "e2e": {"value": val, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})


# ----------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--rays", type=int, default=1 << 26)
    ap.add_argument("--phi", type=int, default=1581)
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-extras", action="store_true")
    ap.add_argument("--workload", default="diffuse", choices=["diffuse", "pathtracer"],
                    help="diffuse = configs[2] headline (default); pathtracer = configs[4] 8-bounce path stream")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write a fixed sample of the last step's hit records (and the rays they belong to) "
                         "as DIR/<field>.npy, for comparing two builds output for output (diffuse workload, one GPU)")
    args = ap.parse_args()
    if args.dump_outputs and (args.workload != "diffuse" or args.impl != "b200" or args.gpus != 1
                              or int(os.environ.get("WORLD_SIZE", "1")) != 1):
        ap.error("--dump-outputs covers the diffuse workload of --impl b200 on one GPU")
    if args.workload == "pathtracer":
        if "--rays" not in sys.argv:
            args.rays = 1 << 25          # paths per GPU; a step traces 16 rays per path
        return run_pathtracer_reference(args) if args.impl == "reference" else run_pathtracer(args)
    if args.impl == "reference":
        return run_reference(args)

    import torch.distributed as dist
    import embree_b200
    from embree_b200 import sharding
    rank, world = int(os.environ.get("RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local)
    devt = torch.device("cuda", local)
    numa = bind_to_gpu_numa(local) if world > 1 else None
    if world > 1:
        dist.init_process_group("nccl", device_id=devt)
    lib = embree_b200.load()
    for kv in filter(None, os.environ.get("RTCB200_TUNING", "").split(",")):   # A/B experiments only, e.g. gather_chunks=4
        k, val = kv.split("=")
        assert lib.rtcb200SetTuning(k.encode(), int(val)) == 0, kv
    dev = lib.new_device(f"gpu={local},verbose={2 if rank == 0 else 0}")
    v, t = make_scene(args.phi)
    sc, keep, _ = commit(lib, dev, v, t)      # first commit of the process: loads the kernels and grows the memory pool
    lib.rtcReleaseScene(sc)
    sc, keep, commit_s = commit(lib, dev, v, t)
    st = lib.scene_stats(sc)
    log(f"rank {rank}: commit {commit_s * 1e3:.0f} ms wall, device build {st.build_ms:.1f} ms, {st.num_nodes} nodes")

    a = lib.args()
    stream = torch.cuda.current_stream().cuda_stream
    n = args.rays

    def trace_dev(tensor, count):
        lib.rtcb200Intersect1MDevice(sc, C.c_void_p(tensor.data_ptr()), count, C.byref(a), C.c_void_p(stream))

    # ---- ray stream, generated in HBM
    prim = scenes.primary_rays(PRIMARY_W, PRIMARY_H, eye=EYE, look=LOOK, device=devt)
    trace_dev(prim, prim.shape[0])
    torch.cuda.synchronize()
    A = torch.empty((n, 24), dtype=torch.float32, device=devt)
    CH = 1 << 22
    for c0 in range(0, n, CH):
        ids = torch.arange(c0, min(c0 + CH, n), device=devt, dtype=torch.int64) + rank * n
        A[c0:c0 + len(ids)] = bounce_rays(prim, ids)
    del prim
    B = A.clone()
    torch.cuda.synchronize()
    lib.check(dev)

    # ---- traversal work per ray (device stat counters = EMBREE_STAT_COUNTERS analogue) on a 1 Mi-ray strided sample
    ns = min(n, 1 << 20)
    S = A[:: max(1, n // ns)][:ns].contiguous()
    lib.rtcb200SetSceneStatCounters(sc, 1)
    lib.rtcb200ResetSceneStatCounters(sc)
    trace_dev(S, S.shape[0])
    torch.cuda.synchronize()
    st2 = lib.scene_stats(sc)
    lib.rtcb200SetSceneStatCounters(sc, 0)
    nodes_per_ray, tris_per_ray = st2.trav_nodes / st2.trav_rays, st2.trav_tris / st2.trav_rays
    NODE_BYTES, TRI_BYTES = 96, 48      # sizeof(rtk::Node8), sizeof(rtk::TriRec) (embree_b200/csrc/rt_core.cuh)
    bytes_per_ray = 48 + 48 + 4 + nodes_per_ray * NODE_BYTES + tris_per_ray * TRI_BYTES
    del S

    # ---- hit gather (N > 1), fused into the trace kernel: rank 0 owns a [world, n, 8] float buffer, every rank maps it
    # through CUDA IPC and its trace kernel stores one compact 32-byte hit record per ray straight into its slice over
    # NVLink (rtcb200Intersect1MGatherDevice).  A tiny NCCL all-reduce, stream-ordered after the kernel, is the
    # per-step "all hits have arrived" signal.  No separate collective moves hit data.  Measured: 99 % / 98 % of
    # linear at 2 / 4 GPUs; at 8 GPUs the 15 GB per step that seven peers deliver into rank 0 take 86 ms (kernel alone:
    # 50 ms): rank 0 ingests only ~175 GB/s (DESIGN.md section 7).
    gbuf, my_out, flag = None, None, None
    if world > 1:
        nbytes = world * n * 32
        handle = [None]
        if rank == 0:
            gbuf = lib.rtcb200PeerAlloc(dev, nbytes)
            h64 = (C.c_ubyte * 64)()
            assert lib.rtcb200PeerExport(dev, C.c_void_p(gbuf), h64) == 0
            handle = [bytes(h64)]
        dist.broadcast_object_list(handle, src=0)
        if rank != 0:
            h64 = (C.c_ubyte * 64).from_buffer_copy(handle[0])
            gbuf = lib.rtcb200PeerImport(dev, h64)
        lib.check(dev)
        assert gbuf
        my_out = gbuf + rank * n * 32
        flag = torch.zeros(1, device=devt)
    kernel_ms = []

    def step(record_kernel_ms=False):
        B[:, 8] = float("inf")  # restore the only input field the trace overwrites (ray.tfar)
        if world > 1:
            lib.rtcb200Intersect1MGatherDevice(sc, C.c_void_p(B.data_ptr()), n, C.byref(a), C.c_void_p(stream), C.c_void_p(my_out))
            dist.all_reduce(flag)
        else:
            lib.rtcb200Intersect1MDevice(sc, C.c_void_p(B.data_ptr()), n, C.byref(a), C.c_void_p(stream))
        if record_kernel_ms:
            kernel_ms.append(lib.rtcb200GetLastTraceMs(sc))

    for _ in range(args.warmup):
        step()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler = ClockSampler(local)
    sampler.start()
    l0 = lib.rtcb200GetLaunchCount()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    torch.cuda.synchronize()
    e0.record()
    for _ in range(args.steps):
        step(record_kernel_ms=True)
    e1.record()
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
    sampler.stop_flag = True
    launches = lib.rtcb200GetLaunchCount() - l0
    ms_local = e0.elapsed_time(e1) / args.steps
    ms = torch.tensor([ms_local], device=devt)
    per_rank = None
    if world > 1:
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        # diagnostics only: every rank's own step time, trace time (direct mode: includes stalls on the peer stores) and
        # SM clock, so that a slow step can be attributed to the gather (all ranks but 0 slow) or to single GPUs
        vals = [float(ms_local), 0.0, 0.0, 0.0]
        try:   # rank-local parsing must never keep a rank out of the collective below
            vals[1] = float(np.mean(kernel_ms)) if kernel_ms else 0.0
            sampler.join(timeout=2)
            cs = sampler.summary()
            vals[2] = float(cs.get("sm_mhz") or 0.0)
            vals[3] = 1.0 if cs.get("reasons") and cs["reasons"] != ["unavailable"] else 0.0
        except Exception as ex:   # noqa: BLE001
            log(f"per-rank diagnostics incomplete: {ex}")
        mine = torch.tensor(vals, dtype=torch.float32, device=devt)
        allv = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allv, mine)
        per_rank = {"ms_per_step": [round(float(x[0]), 3) for x in allv], "trace_ms": [round(float(x[1]), 3) for x in allv],
                    "sm_mhz": [float(x[2]) for x in allv], "throttled": [bool(x[3] > 0) for x in allv]}
    ms_per_step = float(ms.item())
    value = n * world / (ms_per_step * 1e-3) * 1e-6
    lib.check(dev)
    sampler.join(timeout=2)
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, A, B)
    gather_ab = None
    if world > 1 and os.environ.get("RTCB200_GATHER_AB"):   # untimed extra: the same steps with the other delivery mode
        gather_ab = {"default_mode_ms": ms_per_step}
        for mode in (0, 1):
            assert lib.rtcb200SetTuning(b"gather_mode", mode) == 0
            for _ in range(2):
                step()
            torch.cuda.synchronize()
            dist.barrier()
            g0, g1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            g0.record()
            for _ in range(args.steps):
                step()
            g1.record()
            torch.cuda.synchronize()
            tm = torch.tensor([g0.elapsed_time(g1) / args.steps], device=devt)
            dist.all_reduce(tm, op=dist.ReduceOp.MAX)
            gather_ab[f"mode{mode}_ms"] = float(tm.item())
        lib.rtcb200SetTuning(b"gather_mode", 1)
    gather_ok = None
    if world > 1:   # untimed: the NVLink-written records on rank 0 must equal what an NCCL gather of the same hits delivers
        local = sharding.compact_hits(B)
        ri = B.view(torch.int32)
        miss = ri[:, 18] == -1
        local[miss, 1:6] = 0.0
        local.view(torch.int32)[miss, 6] = -1
        local.view(torch.int32)[miss, 7] = -1
        bufs, _ = sharding.gather_hits(local, dst=0)
        if rank == 0:
            got = torch.empty((world, n, 8), dtype=torch.float32, device=devt)
            lib.rtcb200PeerCopy(dev, C.c_void_p(got.data_ptr()), C.c_void_p(gbuf), world * n * 32)
            gather_ok = all(bool(torch.equal(got[r].view(torch.int32), bufs[r].view(torch.int32))) for r in range(world))
            log(f"fused NVLink gather == NCCL gather: {gather_ok}")

    # ---- end to end through the host-pointer entry point (pinned host memory, H2D + trace + D2H timed)
    e2e = None
    if not args.no_e2e:
        H = torch.empty((n, 24), dtype=torch.float32).pin_memory()
        H.copy_(A)
        times = []
        reps = max(1, min(args.steps, 3))
        for it in range(1 + reps):
            H[:, 8] = float("inf")
            if world > 1:
                dist.barrier()
            t0 = time.perf_counter()
            lib.rtcb200Intersect1M(sc, C.c_void_p(H.data_ptr()), n, C.byref(a))
            dt = time.perf_counter() - t0
            if it > 0:
                times.append(dt)
        tt = torch.tensor([float(np.mean(times))], device=devt)
        if world > 1:
            dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        e2e = {"value": n * world / float(tt.item()) * 1e-6, "unit": "Mrays/s", "h2d_bytes_per_step": n * 96 * world,
               "d2h_bytes_per_step": n * 96 * world, "steps": reps, "ms_per_step": float(tt.item()) * 1e3,
               "api": "rtcb200Intersect1M(scene, RTCRayHit* host, M, args), pinned host buffers, 3-stream chunked pipeline"}
        lib.check(dev)
        host_result = H
    # ---- coherent leg of the metric: RTCRayHit16 packets with RTC_RAY_QUERY_FLAG_COHERENT (rank 0, N == 1)
    coherent = None
    if rank == 0 and world == 1 and not args.no_extras:
        coherent = {}
        # (a) the reference's own coherent benchmark (tutorials/verify/verify.cpp:5757-5921): 1 M-triangle sphere, 4096^2 rays
        #     from the origin, dir = (x/W, 1, y/H), 32x32 tiles of 4x4-pixel packets
        coherent["verify_4096"] = coherent_leg(lib, dev, devt, stream, "verify CoherentRaysBenchmark: createTriangleSphere(numPhi=500) = 1 000 000 triangles, "
                                               "4096x4096 rays dir=(x/W,1,y/H) from the origin, 32x32 tiles of 4x4-pixel RTCRayHit16 packets, COHERENT flag",
                                               500, scenes.verify_coherent_rays(4096, 4096, 32, device=devt), args)
        # (b) BASELINE configs[1]: 1 M-triangle mesh, 1920x1080 pinhole primary rays as 4x4-pixel packets
        pr = scenes.primary_rays(PRIMARY_W, PRIMARY_H, eye=EYE, look=LOOK, device=devt)
        pr = pr[scenes.tile_order_16(PRIMARY_W, PRIMARY_H).to(devt)].contiguous()
        coherent["configs1_1080p"] = coherent_leg(lib, dev, devt, stream, "configs[1]: createTriangleSphere(numPhi=501) = 1 002 000 triangles, 1920x1080 pinhole "
                                                  "primary rays, 4x4-pixel RTCRayHit16 packets, COHERENT flag", 501, pr, args)
        del pr

    # ---- extras (not the headline): any-hit on the same stream, and a non-convex 10 M-triangle terrain (SURVEY 8d "S10b")
    extras = None
    if rank == 0 and world == 1 and not args.no_extras:
        ne = min(n, 1 << 24)
        Rr = A[:: max(1, n // ne)][:ne, :12].contiguous()           # RTCRay[] halves of every 4th ray
        work = Rr.clone()
        best = 1e9
        ao = lib.args()
        for it in range(3):
            work.copy_(Rr)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            lib.rtcb200Occluded1MDevice(sc, C.c_void_p(work.data_ptr()), ne, C.byref(ao), C.c_void_p(stream))
            c1.record()
            torch.cuda.synchronize()
            best = min(best, c0.elapsed_time(c1))
        extras = {"occluded_same_stream": {"Mrays_per_s": ne / best * 1e-3, "rays": ne, "occluded_fraction": float((work[:, 8] == float("-inf")).float().mean().item())}}
        tv, tt = scenes.terrain(2236, seed=7)
        sct, keept, _ = commit(lib, dev, tv, tt)
        stt = lib.scene_stats(sct)
        cam = scenes.primary_rays(PRIMARY_W, PRIMARY_H, eye=(0.0, 0.9, -0.2), look=(0.0, -1.0, 0.25), device=devt)
        trace_dev_scene = lambda scx, tensor, count: lib.rtcb200Intersect1MDevice(scx, C.c_void_p(tensor.data_ptr()), count, C.byref(a), C.c_void_p(stream))  # noqa: E731
        trace_dev_scene(sct, cam, cam.shape[0])
        torch.cuda.synchronize()
        prim_hit = float((cam.view(torch.int32)[:, 18] != -1).float().mean().item())
        T = torch.empty((ne, 24), dtype=torch.float32, device=devt)
        for c0_ in range(0, ne, CH):
            ids = torch.arange(c0_, min(c0_ + CH, ne), device=devt, dtype=torch.int64) * max(1, n // ne)
            T[c0_:c0_ + len(ids)] = bounce_rays(cam, ids)
        Tw = T.clone()
        best = 1e9
        for it in range(3):
            Tw.copy_(T)
            c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            c0.record()
            trace_dev_scene(sct, Tw, ne)
            c1.record()
            torch.cuda.synchronize()
            best = min(best, c0.elapsed_time(c1))
        extras["terrain_10M_diffuse"] = {"triangles": int(stt.num_triangles), "Mrays_per_s": ne / best * 1e-3, "rays": ne,
                                         "primary_hit_fraction": prim_hit,
                                         "bounce_hit_fraction": float((Tw.view(torch.int32)[:, 18] != -1).float().mean().item()),
                                         "build_ms": stt.build_ms}
        lib.rtcReleaseScene(sct)
        del T, Tw, cam, Rr, work
        lib.check(dev)
        extras["dynamic_scene_recommit"] = dynamic_leg(lib, dev, args)
        extras["dynamic_scene_two_level"] = two_level_leg(lib, dev, args)
        extras["hair_bezier"] = hair_leg(lib, dev, devt, stream, args)
        extras["hair_bezier_round"] = hair_leg(lib, dev, devt, stream, args, rnd=True)
        try:   # added at the very end of round 2: a failure here must not cost the line its other numbers
            extras["points"] = point_leg(lib, dev, devt, stream, args)
        except Exception as e:   # noqa: BLE001
            extras["points"] = {"error": repr(e)}

    # ---- parity sample + CPU baseline (rank 0, N == 1)
    cpu_baseline, parity, ref_counters = None, None, None
    if rank == 0 and world == 1 and not args.no_cpu:
        from tests.parity import api_trace_mt, compare_hits, load_oracle, load_reference
        B.copy_(A)
        trace_dev(B, n)
        torch.cuda.synchronize()
        cores, core_detail = usable_cores()
        nsample = min(n, 1 << 24)
        stride = max(1, n // nsample)
        sample_in = scenes.as_numpy_rayhits(A[::stride][:nsample].cpu())
        got = scenes.as_numpy_rayhits(B[::stride][:nsample].cpu())
        R = load_reference()
        if R is not None:
            rdev = R.new_device(None)
            rsc, rkeep, rbt = commit(R, rdev, v, t)
            log(f"reference rtcCommitScene ({cores} threads): {rbt * 1e3:.0f} ms")
            best = 1e30
            for _ in range(2):
                w = sample_in.copy()
                t0 = time.perf_counter()
                api_trace_mt(R, rsc, w, cores)
                best = min(best, time.perf_counter() - t0)
            kind, want = "reference", w
        else:
            osc = load_oracle().scene([(v, t, 0, 0xFFFFFFFF)])
            w = sample_in.copy()
            t0 = time.perf_counter()
            osc.trace(w, nthreads=cores)
            best = time.perf_counter() - t0
            kind, want, rbt = "port", w, None
        cpu_baseline = {"value": nsample / best * 1e-6, "unit": "Mrays/s", "cores": cores, "cores_detail": core_detail, "kind": kind,
                        "sample": f"{nsample} rays = every {stride}th ray of the stream, rtcIntersect1 loop on {cores} host threads (FTZ|DAZ), best of 2",
                        "commit_ms": None if rbt is None else rbt * 1e3}
        parity = compare_hits(want, got, meshes=[(v, t, 0, 0xFFFFFFFF)])
        parity["checked_against"] = kind
        ref_counters = reference_counters(args.phi, sample_in[:: max(1, nsample >> 20)], cores)

    if rank == 0:
        peaks, peak_src = measured_peaks()
        kms = float(np.mean(kernel_ms)) if kernel_ms else ms_per_step
        achieved = bytes_per_ray * n / (kms * 1e-3) * 1e-9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "ncu_traffic.json")
        if os.path.exists(tp):
            traffic = json.load(open(tp)).get("dram_bytes_per_launch")
        line = {"metric": "Mrays/s incoherent diffuse-bounce, 10M-triangle scene", "value": value, "unit": "Mrays/s", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": workload_config(args, len(t)),
                "clocks": sampler.summary(), "e2e": e2e, "gpu_launches": int(launches), "gather_verified": gather_ok, "per_rank": per_rank,
                "gather_ab": gather_ab, "numa": numa,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peaks["hbm_gbs"], "unit": "GB/s", "frac": achieved / peaks["hbm_gbs"],
                             "traffic": traffic, "peak_source": peak_src,
                             "kernel": "rtk::trace_kernel<K=1,OCCLUDED=false,STATS=false,ROBUST=false,GENERAL=0,GATHER=0,SPREAD=true>",
                             "kernel_ms": kms, "algorithmic_bytes_per_ray": bytes_per_ray,
                             "frac_with_round1_80B_nodes": (100 + nodes_per_ray * 80 + tris_per_ray * 48) * n / (kms * 1e-3) * 1e-9 / peaks["hbm_gbs"],
                             "nodes_per_ray": nodes_per_ray, "tris_per_ray": tris_per_ray, "reference_counters": ref_counters,
                             "note": "algorithmic bytes = 100 B ray/hit I/O + nodes/ray*96 B + tris/ray*48 B (device stat counters, 1 Mi-ray sample); the node "
                                     "is 96 B = three whole 32-B sectors since round 2 (round 1: 80 B, which also occupied three sectors) -- "
                                     "frac_with_round1_80B_nodes keeps the old accounting for comparison"},
                "cpu_baseline": cpu_baseline, "parity": parity, "coherent": coherent, "extras": extras,
                "build": {"device_ms": st.build_ms, "commit_wall_ms": commit_s * 1e3, "nodes": int(st.num_nodes), "sah": st.sah_cost,
                          "builder": "sah" if st.builder else "lbvh"}}
        emit(line)
    if world > 1:
        dist.destroy_process_group()


DUMP_RAYS = 1 << 18     # ~21 MB of .npy files


def dump_outputs(out_dir, rays_in, rayhits):
    """Write the RTCRayHit records the timed trace returned ([n, 24] float32 on the device) for a fixed sample of
    DUMP_RAYS ray indices (seed 0, independent of the run), together with those rays' inputs, as out_dir/<field>.npy.
    The inputs are written as well because the bounce rays start at the primary hits, i.e. they are computed too."""
    n = rayhits.shape[0]
    k = min(n, DUMP_RAYS)
    idx = np.sort(np.random.default_rng(0).choice(n, k, replace=False))
    sel = torch.from_numpy(idx).to(rayhits.device)
    hit = rayhits.index_select(0, sel).cpu().numpy()
    ray = rays_in.index_select(0, sel).cpu().numpy()
    ids = hit.view(np.uint32)
    hit_mask = ids[:, 18] != 0xFFFFFFFF
    # a miss leaves tfar at its input, +inf: the files carry hit / miss in `hit` and 0 as the tfar of a miss, so that every value is finite
    fields = {"ray_index": idx.astype(np.float64), "ray_org": ray[:, 0:3], "ray_tnear": ray[:, 3], "ray_dir": ray[:, 4:7],
              "hit": hit_mask.astype(np.float32), "tfar": np.where(hit_mask, hit[:, 8], np.float32(0)),
              "Ng": hit[:, 12:15], "u": hit[:, 15], "v": hit[:, 16],
              "primID": ids[:, 17].astype(np.float64), "geomID": ids[:, 18].astype(np.float64), "instID": ids[:, 19].astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in fields.items():
        np.save(os.path.join(out_dir, name + ".npy"), np.ascontiguousarray(a))
    log(f"wrote {len(fields)} arrays of {k} sampled rays to {out_dir}")


def emit(line):
    """The ONE JSON line of the contract goes to the process's original stdout (see _guard_stdout)."""
    _REAL_STDOUT.write(json.dumps(line) + "\n")
    _REAL_STDOUT.flush()


def _guard_stdout():
    """Libraries write to fd 1 behind our back (NCCL prints its version line there when the environment sets
    NCCL_DEBUG): keep the original stdout for the JSON line only and point fd 1 at stderr for everything else."""
    global _REAL_STDOUT
    sys.stdout.flush()
    _REAL_STDOUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)


_REAL_STDOUT = sys.stdout

if __name__ == "__main__":
    _guard_stdout()
    main()
