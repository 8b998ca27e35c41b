#!/usr/bin/env python
"""bench.py — meshlet visibility pipeline on B200 (BASELINE.json metric: meshlets culled/s + tris rasterised/s,
% of HBM roofline) with the CPU reference arm beside it.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]

A "step" is one frame of the hot path over the synthetic scene of BASELINE.json configs[1]
("1M meshlet instances, 1 camera, two-pass Hi-Z occlusion cull"): clear attachments -> cull_meshes ->
cull_meshlets(early) -> vis-buffer raster -> generate_hiz -> cull_meshlets(late) -> vis-buffer raster
(RendererInstance.cpp:842-884).  N > 1: weak scaling, 1M meshlet instances PER GPU, mesh-instance sharded,
with the real exchange steps (id-base allgather, vis-buffer max-reduce x2, survivor allgather) inside the step.

value   : whole-job meshlet instances culled / s with inputs resident in HBM (CUDA-graph replay of one frame,
          CUDA events per step on the launching stream, L2 flushed between steps, max over ranks)
e2e     : same metric through the reference-facing host API oxr_submit / oxr_wait (C++ RendererInstance mirror) with
          HOST buffers: camera + all transforms H2D from pinned memory, vis32 + survivor ids + counters D2H every frame
roofline: the late meshlet-cull kernel (cull_meshlets_hiz equivalent), algorithmic bytes of SURVEY.md §8d /
          its CUDA-event duration inside the timed loop, against MEASURED_PEAKS.json hbm_gbs
cpu_baseline / --impl reference: the oracle port of the same frame (oracle/, pthreads on all host cores) on a
          bounded sample — the reference's own Vulkan path cannot be built or run here (DESIGN.md).
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "meshlet_instances_culled_per_s"
UNIT = "meshlet instances/s"


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=100)
    ap.add_argument("--warmup", type=int, default=5)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--meshlets", type=int, default=1_000_000, help="meshlet instances per GPU")
    ap.add_argument("--width", type=int, default=1920)
    ap.add_argument("--height", type=int, default=1080)
    ap.add_argument("--no-graph", action="store_true", help="launch kernels directly instead of replaying a CUDA graph")
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="N>1: run the trailing exchange on the main stream (no overlap with the next frame)")
    ap.add_argument("--cpu-frames", type=int, default=2)
    ap.add_argument("--total-meshlets", type=int, default=0,
                    help="strong scaling: a fixed scene of this many meshlet instances split over the GPUs (BASELINE configs[4]: 50000000)")
    ap.add_argument("--unique-meshes", type=int, default=256,
                    help="256 = the contract scene (bounds L2-resident); 65536 makes bounds / vertex data stream from HBM")
    ap.add_argument("--parity-frames", type=int, default=3, help="N>1: frames of the pre-timing check N GPUs == 1 GPU (0 = skip)")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write the outputs of the last timed frame as DIR/<name>.npy (single GPU)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


# --dump-outputs: elements per array; a larger output is replaced by a fixed seeded sample of its elements, so the files stay
# under 64 MB in all (4K images, say) and hold the same positions in every run with the same arguments
DUMP_LIMITS = {"vis32": 3_000_000, "depth": 3_000_000, "visible_meshlet_instances": 2_000_000, "counters": 4}


def dump_outputs(out_dir, vis32, depth, visible, counts):
    """One frame's outputs as a caller of the path receives them (capi.Renderer.render): the R32UI vis image, the D32F depth
    image, the survivor ids (sorted: their order is atomics order) and the counters total / early / late / triangles.
    float64 holds every uint32 exactly."""
    arrays = {"vis32": vis32.astype(np.float64), "depth": depth.astype(np.float32),
              "visible_meshlet_instances": np.sort(visible).astype(np.float64),
              "counters": np.array([counts[k] for k in ("total", "early", "late", "triangles")], dtype=np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        n = DUMP_LIMITS[name]
        if a.size > n:
            a = a.ravel()[np.sort(np.random.default_rng(0).choice(a.size, n, replace=False))]
        np.save(os.path.join(out_dir, name + ".npy"), a)


def measured_peak_hbm():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index=0):
        self.gpu = gpu_index
        self.samples, self.proc, self.thread = [], None, None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None
            return
        self.thread = threading.Thread(target=self._read, daemon=True)
        self.thread.start()

    def _read(self):
        for line in self.proc.stdout:
            self.samples.append(line.strip())

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], None, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for s in self.samples:
            f = [x.strip() for x in s.split(",")]
            if len(f) < 6:
                continue
            try:
                sm.append(float(f[0]))
                mx = float(f[1])
            except ValueError:
                continue
            for n, v in zip(names, f[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(n)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": mx, "reasons": sorted(reasons),
                "samples": len(sm)}


def load_oracle():
    sys.path.insert(0, os.path.join(ROOT, "oracle"))
    import pyoracle

    pyoracle.lib()
    return pyoracle


def cpu_frames(scene, n_frames, n_threads):
    """The oracle port of the frame on the host cores (cpu_baseline / reference arm).  Returns (seconds per frame, info)."""
    orc = load_oracle()
    hs = orc.HostScene(scene)
    mask = np.zeros((scene.max_meshlet_instance_count + 31) // 32, dtype=np.uint32)
    # untimed frames bring the persistent mask to the same steady state the GPU arm is timed in
    for f in range(4):
        orc.cpu_frame(hs, scene.camera(2.0 * (f % 2)), scene.width, scene.height, mask, scene.occluder_depth, n_threads)
    times, last = [], None
    for f in range(n_frames):
        cam = scene.camera(2.0 * (f % 2))
        t0 = time.perf_counter()
        last = orc.cpu_frame(hs, cam, scene.width, scene.height, mask, scene.occluder_depth, n_threads)
        times.append(time.perf_counter() - t0)
    return float(np.mean(times)), last


def cpu_frustum_loops(scene, cam, cores):
    """BASELINE.md §3: the reference's CPU primitives looped over the meshlet bounds + draw-list build
    (engine AABB::is_on_frustum test, and the shader-equivalent cone+frustum), 1 thread and all host threads;
    plus BASELINE.json configs[0] (10 k bounds, 1 camera, scalar)."""
    orc = load_oracle()
    hs = orc.HostScene(scene)
    mi, vis, _ = orc.cull_meshes(hs, cam, 7)
    total = int(vis["total"][0])
    out = {}
    for name, mode in (("engine_aabb_is_on_frustum", 0), ("shader_equivalent_cone_frustum", 1)):
        for threads in (1, cores):
            n = total if threads > 1 else min(total, 200_000)
            best = 1e9
            for _ in range(3):
                t0 = time.perf_counter()
                surv = orc.cpu_baseline_cull(hs, mi, n, cam, mode, threads)
                best = min(best, time.perf_counter() - t0)
            out[f"{name}_{threads}t"] = {"meshlets_per_s": n / best, "meshlets": n, "survivors": int(len(surv))}
    n = min(total, 10_000)
    best = 1e9
    for _ in range(20):
        t0 = time.perf_counter()
        orc.cpu_baseline_cull(hs, mi, n, cam, 1, 1)
        best = min(best, time.perf_counter() - t0)
    out["configs0_10k_bounds_scalar_1t"] = {"meshlets_per_s": n / best, "meshlets": n}
    # configs[0], first half: "meshlet build of one mesh" — the host-side builder (oxb_build_mesh: fetch remap, quantisation,
    # scan meshlets, AABBs + normal cones, blob) on a procedural 131k-triangle torus, one thread.  Host C++ of the
    # product, no GPU involved; meshoptimizer (the reference's builder) is not available here, so this is not a comparison.
    try:
        from oxylus_b200 import capi as _capi
        nu, nv = 512, 128
        uu, vv = np.meshgrid(np.arange(nu) / nu * 2 * np.pi, np.arange(nv) / nv * 2 * np.pi, indexing="ij")
        pos = np.stack([(2 + 0.7 * np.cos(vv)) * np.cos(uu), (2 + 0.7 * np.cos(vv)) * np.sin(uu), 0.7 * np.sin(vv)], axis=2).reshape(-1, 3)
        nrm = np.stack([np.cos(vv) * np.cos(uu), np.cos(vv) * np.sin(uu), np.sin(vv)], axis=2).reshape(-1, 3)
        i, j = np.meshgrid(np.arange(nu), np.arange(nv), indexing="ij")
        a, b = i * nv + j, ((i + 1) % nu) * nv + j
        c, d = i * nv + (j + 1) % nv, ((i + 1) % nu) * nv + (j + 1) % nv
        idx = np.stack([a, b, d, a, d, c], axis=2).reshape(-1).astype(np.uint32)
        best = 1e9
        for _ in range(3):
            t0 = time.perf_counter()
            bm = _capi.BuiltMesh(pos, [(idx, 0.0)], normals=nrm)
            best = min(best, time.perf_counter() - t0)
        out["configs0_meshlet_build_1t"] = {"triangles_per_s": len(idx) / 3 / best, "triangles": int(len(idx) // 3),
                                            "meshlets": bm.lod0_meshlet_count, "ms": best * 1e3}
        bm.close()
    except Exception as e:  # the builder lives in liboxcull.so; never let a baseline extra break the bench line
        out["configs0_meshlet_build_1t"] = {"error": str(e)[:200]}
    return out


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path = the oracle port (kind "port")."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    from oxylus_b200 import synth

    cores = os.cpu_count() or 1
    scene = make_bench_scene(args, max(1, args.gpus))
    # bounded sample: every step is one full frame of the same scene on all host threads
    for _ in range(max(0, min(args.warmup, 1))):
        cpu_frames(scene, 1, cores)
    n = args.steps
    sec, last = cpu_frames(scene, n, cores)
    value = scene.max_meshlet_instance_count / sec
    if args.dump_outputs:
        v32, depth = load_oracle().resolve(last["vis64"])
        vc = last["visibility"]
        counts = dict(total=int(vc["total"][0]), early=int(vc["early"][0]), late=int(vc["late"][0]), triangles=last["triangles"])
        dump_outputs(args.dump_outputs, v32, depth, last["visible"][: counts["early"] + counts["late"]], counts)
    line = {
        "impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": n, "warmup": min(args.warmup, 1),
        "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong" if args.total_meshlets else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, scene),
        "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port",
                         "sample": f"{n} full frames of the {scene.max_meshlet_instance_count}-meshlet scene, oracle port, pthreads"},
        "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "triangles_per_s": (last["triangles"] / sec) if last else None,
    }
    print(json.dumps(line), flush=True)


def make_bench_scene(args, world):
    """The scene both arms run: configs[1] per GPU (weak scaling; instances shrunk by world^-1/2 so the screen coverage and
    with it the per-GPU share of visible work stays what one GPU sees), or a fixed scene (--total-meshlets, strong scaling)."""
    from oxylus_b200 import synth

    if args.total_meshlets:
        return synth.make_scene(args.total_meshlets, config_index=2, width=args.width, height=args.height, n_unique_meshes=args.unique_meshes)
    return synth.make_scene(args.meshlets * world, config_index=2, width=args.width, height=args.height, n_unique_meshes=args.unique_meshes,
                            instance_scale=float(world) ** -0.5)


def workload_config(args, scene):
    world = max(1, args.gpus)
    if args.total_meshlets:
        wl = (f"BASELINE.json configs[4] shape: {args.total_meshlets} meshlet instances, instance-sharded over {world} GPU(s), "
              "two-pass Hi-Z occlusion cull + vis-buffer raster, NCCL survivor allgather + vis-buffer max-reduce")
    else:
        wl = "BASELINE.json configs[1]: 1M meshlet instances per GPU, 1 camera, two-pass Hi-Z occlusion cull + vis-buffer raster"
    return {"workload": wl,
            "meshlet_instances_per_gpu": scene.max_meshlet_instance_count // world, "resolution": [args.width, args.height],
            "hiz": list(scene.hiz_extent()), "mesh_instances": scene.mesh_instance_count, "unique_meshes": len(scene.meshes),
            "instance_scale": (1.0 if args.total_meshlets else float(world) ** -0.5),
            "l2": "flushed between timed steps (256 MiB write, untimed)", "cameras": "yaw 0 / 2 deg alternating, steady-state mask",
            "parallelism": f"mesh-instance shards x{world}" if world > 1 else "single GPU"}


def main():
    args = parse_args()
    if args.impl == "reference":
        return run_reference(args)

    import torch
    import torch.distributed as dist

    from oxylus_b200 import abi, capi, dist as oxdist, pipeline, synth

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    multi = world > 1
    if multi and args.dump_outputs:
        raise SystemExit("--dump-outputs writes the outputs of one GPU: run it with --gpus 1")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if multi:
        # NCCL_DEBUG is left exactly as the launcher set it (the driver reads the communicator banner for its rank proof);
        # the JSON line is the last line rank 0 prints.  torch.distributed is plumbing here (id broadcast, timing reductions):
        # the data path is the product's own communicator + NVLink peer memory (oxc_mgpu_*).
        # gloo, not nccl: a second NCCL communicator in the process (torch's) interleaving with the product's own on other
        # streams is a documented deadlock hazard; barriers / timing reductions are host-side anyway
        dist.init_process_group("gloo")
    n_gpus = world
    args.gpus = world
    capi.load(build_if_missing=False)

    # ---------------- scene ----------------
    scene = make_bench_scene(args, world)
    wide_ids = scene.max_meshlet_instance_count > (1 << 24)
    shard, mg, cap = None, None, None
    if multi:
        lod0 = oxdist.lod0_counts_of(scene)
        parts = oxdist.partition_mesh_instances(lod0, world)
        shard = parts[rank]
        cap = max(1, max(int(lod0[f:f + c].sum()) for f, c in parts))
        uid = [capi.Context.mgpu_unique_id() if rank == 0 else None]
        dist.broadcast_object_list(uid, src=0)
    pipe = pipeline.VisibilityPipeline(scene, device=local_rank, shard=shard, auto_id_base=True, shard_capacity=cap, wide_ids=wide_ids)
    cams = [scene.camera(0.0), scene.camera(2.0)]
    if multi:
        # survivor gather segments (ncclAllGather moves whole segments, one size for all ranks): half a shard to begin with — the
        # cold frames (zeroed mask: everything that passes is a late survivor) need it; shrunk to steady state after the parity check
        pipe.mgpu = pipe.ctx.mgpu_init(rank, world, uid[0], max(4096, cap // 2))
    dev = pipe.device
    w, h = scene.width, scene.height

    def barrier():
        torch.cuda.synchronize()
        if multi:
            dist.barrier()
        torch.cuda.synchronize()

    _dbg_on = bool(os.environ.get("OXC_BENCH_DEBUG"))

    def dbg(*a):
        if _dbg_on:
            print(f"[bench r{rank} {time.perf_counter():.2f}]", *a, file=sys.stderr, flush=True)

    dbg("pipeline ready", "peer hiz" if (multi and pipe.mgpu.hiz_over_peer_memory) else "")
    # ---------------- N > 1: N GPUs == 1 GPU, bit for bit, before anything is timed ----------------
    parity = None
    if multi and args.parity_frames > 0:
        barrier()
        for f in range(args.parity_frames):
            pipe.select_buffer(0)
            pipe.frame(cams[f % 2])
            pipe.exchange_frame(slot=0)
        torch.cuda.synchronize()
        pipe.ctx.check_status()
        if rank == 0:
            cnt_g, ids_g = pipe.ctx.mgpu_gathered(0)
            ref = pipeline.VisibilityPipeline(scene, device=local_rank, wide_ids=wide_ids)
            for f in range(args.parity_frames):
                ref.frame(cams[f % 2])
            torch.cuda.synchronize()
            rc = ref.counters()
            r_ids = ref.ctx.visible_indices(rc["early"] + rc["late"])
            parity = {"image": bool(torch.equal(pipe.vis64, ref.vis64)),
                      "survivor_ids": bool(np.array_equal(np.sort(np.concatenate(ids_g)), np.sort(r_ids))),
                      "counts": bool(int(cnt_g[:, 0].sum()) == rc["total"] and int(cnt_g[:, 1].sum()) == rc["early"] and int(cnt_g[:, 2].sum()) == rc["late"]),
                      "hiz": bool(np.array_equal(np.concatenate([l.ravel() for l in pipe.ctx.hiz_levels()]).view(np.uint32),
                                                 np.concatenate([l.ravel() for l in ref.ctx.hiz_levels()]).view(np.uint32))),
                      "frames": args.parity_frames}
            parity["pass"] = all(parity[k] for k in ("image", "survivor_ids", "counts", "hiz"))
            ref.close()
            del ref
            torch.cuda.empty_cache()
        barrier()

    if multi:
        # steady-state survivor counts from real (exchanged) frames -> gather capacity = twice the largest any rank saw.  The mask is
        # NOT reset afterwards, so no cold frame follows; exceeding the capacity later is a hard error (OXC_STATUS_SURVIVOR_OVERFLOW,
        # checked after the timed region), never a silent truncation.
        seen = 0
        for f in range(6):
            pipe.select_buffer(0)
            pipe.frame(cams[f % 2])
            pipe.exchange_frame(slot=0)
            torch.cuda.synchronize()
            if f >= 4:
                cnt_w, _ = pipe.ctx.mgpu_gathered(0)
                seen = max(seen, int((cnt_w[:, 1] + cnt_w[:, 2]).max()))
        pipe.ctx.check_status()
        pipe.mgpu = pipe.ctx.mgpu_set_survivor_capacity(min(cap, max(4096, 2 * seen)))
    dbg("parity check done", parity)
    # ---------------- warm-up (also brings the visibility mask to steady state) ----------------
    W = max(4, args.warmup)  # >= 4 so the persistent visibility mask reaches its steady state
    K = args.steps
    sampler = ClockSampler(local_rank)  # samples span warm-up + timed region + per-kernel loop (all GPU-busy)
    sampler.start()
    for i in range(W):
        pipe.select_buffer(i & 1)
        pipe.frame(cams[i % 2])
        if multi:
            pipe.exchange_frame(slot=i & 1)
    torch.cuda.synchronize()

    dbg("warm-up done")
    # ---------------- CUDA graphs: one whole frame per camera / buffer ----------------
    # N > 1: the Hi-Z exchange is the product's own kernels over peer memory, so the WHOLE frame (both passes, the exchange in
    # between and the staging of the survivor list) is one graph; only the trailing NCCL calls stay outside (side stream).
    graphs = None
    if not args.no_graph:
        try:
            graphs = []
            side = torch.cuda.Stream()
            side.wait_stream(torch.cuda.current_stream())
            with torch.cuda.stream(side):
                for b, cam in enumerate(cams):
                    pipe.select_buffer(b)  # camera index == buffer index: both alternate every step
                    g = torch.cuda.CUDAGraph()
                    with torch.cuda.graph(g, stream=side):
                        pipe.use_torch_stream()
                        pipe.frame(cam)
                        if multi:
                            pipe.ctx.mgpu_stage_survivors(b)
                    graphs.append(g)
            torch.cuda.current_stream().wait_stream(side)
            pipe.use_torch_stream()
            pipe.select_buffer(0)
            torch.cuda.synchronize()
            if multi:
                barrier()
            if not multi:
                for i in range(2):
                    graphs[i % 2].replay()
                torch.cuda.synchronize()
        except Exception as e:
            sys.stderr.write(f"[bench] CUDA graph capture failed ({e!r}); timing eager launches\n")
            graphs = None
            pipe.use_torch_stream()
            pipe.select_buffer(0)
            torch.cuda.synchronize()

    # N > 1: trailing exchange (vis-buffer max-reduce, survivor allgather) on a side stream, double-buffered (vis buffer b and
    # gather slot b), so it overlaps the next frame; buffer b is reused two frames later, after its exchange has completed
    overlap = None
    if multi and not args.no_overlap:
        overlap = dict(cs=torch.cuda.Stream(), frame_done=[torch.cuda.Event() for _ in range(2)],
                       tail_done=[torch.cuda.Event() for _ in range(2)], pending=[False, False])

    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)

    def run_frame(b, mark=None):
        pipe.select_buffer(b)
        if graphs is not None and mark is None:
            graphs[b].replay()
        else:
            pipe.frame(cams[b], mark=mark)
            if multi:
                pipe.ctx.mgpu_stage_survivors(b)

    def step(i, mark=None):
        b = i & 1
        if not multi:
            return run_frame(b, mark)
        main = torch.cuda.current_stream()
        if overlap is not None and mark is None:
            o = overlap
            if o["pending"][b]:
                main.wait_event(o["tail_done"][b])  # the exchange that last used buffer / slot b (two frames ago) has finished
            run_frame(b)
            o["frame_done"][b].record(main)
            o["cs"].wait_event(o["frame_done"][b])
            pipe.exchange_frame(slot=b, stream=o["cs"], already_staged=True, vis=pipe.vis64_bufs[b])
            o["tail_done"][b].record(o["cs"])
            o["pending"][b] = True
        else:
            run_frame(b, mark)
            pipe.exchange_frame(slot=b, already_staged=True, vis=pipe.vis64_bufs[b])
            if mark:
                mark("exchange")

    def drain():
        if overlap is not None:
            torch.cuda.current_stream().wait_stream(overlap["cs"])

    dbg("graphs", graphs is not None)
    if overlap is not None:  # warm the side stream outside the timed region
        for i in range(4):
            step(i)
        drain()
        torch.cuda.synchronize()

    dbg("overlap warm-up done")
    # ---------------- timed region: exactly K steps ----------------
    launches0 = capi.kernel_launch_count()
    ev = [(torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)) for _ in range(K)]
    barrier()
    t_wall0 = time.perf_counter()
    for i in range(K):
        flush.fill_(i & 0xFF)  # L2 flush, outside the per-step event pair
        ev[i][0].record()
        step(i)
        if i == K - 1:
            drain()  # the last steps' exchanges are inside the timed region
        ev[i][1].record()
    barrier()
    t_wall = time.perf_counter() - t_wall0
    step_ms = [a.elapsed_time(b) for a, b in ev]
    ms_per_step = float(np.mean(step_ms))
    cnt = pipe.counters()
    if multi:
        pipe.ctx.check_status()  # survivor-gather overflow / peer time-out are errors, not footnotes
    if args.dump_outputs:  # before the per-kernel loop below overwrites them
        vis32 = torch.empty((h, w), dtype=torch.int32, device=dev)
        depth = torch.empty((h, w), dtype=torch.float32, device=dev)
        pipe.ctx.resolve_visbuffer(pipe.vis64_bufs[(K - 1) & 1].data_ptr(), w, h, vis32.data_ptr(), depth.data_ptr())
        dump_outputs(args.dump_outputs, vis32.cpu().numpy().view(np.uint32), depth.cpu().numpy(),
                     pipe.ctx.visible_indices(cnt["early"] + cnt["late"]), cnt)
        del vis32, depth

    dbg("timed region done", ms_per_step)
    # ---------------- per-kernel durations (same steps, eager launches, one CUDA event after every stage) ----------------
    stage_list = pipeline.STAGES + (["exchange"] if multi else [])
    stage_names = ["begin"] + stage_list
    stage_acc = {n: [] for n in stage_list}
    stage_acc["clear"] = []
    l0 = capi.kernel_launch_count()
    for i in range(K):
        flush.fill_(i & 0xFF)
        marks = {}

        def mark(name):
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            marks[name] = e

        s0 = torch.cuda.Event(enable_timing=True)
        s0.record()
        step(i, mark=mark)
        torch.cuda.synchronize()
        stage_acc["clear"].append(s0.elapsed_time(marks["begin"]))
        for a, b in zip(stage_names[:-1], stage_names[1:]):
            stage_acc[b].append(marks[a].elapsed_time(marks[b]))
    launches_per_frame = (capi.kernel_launch_count() - l0) // K
    cnt_stage = pipe.counters()  # counters of the last frame of the per-stage loop (the frame the kernel times belong to)
    # keep the GPU busy with the same steps until the sampler has a few readings, then stop it
    if multi:  # every rank must run the same number of (collective) steps: a fixed count, not a clock-driven loop
        for i in range(64):
            step(i)
        drain()
        torch.cuda.synchronize()
    else:
        t_busy = time.perf_counter()
        while len(sampler.samples) < 5 and time.perf_counter() - t_busy < 2.0:
            step(0)
            torch.cuda.synchronize()
    clocks = sampler.stop()
    stages_ms = {k: float(np.mean(v)) for k, v in stage_acc.items()}

    dbg("stage loop done")
    per_rank = None
    if multi:
        keys = sorted(stages_ms)
        t_st = torch.tensor([stages_ms[k] for k in keys] + [cnt_stage["total"], cnt_stage["early"] + cnt_stage["late"], cnt_stage["triangles"]],
                            dtype=torch.float64, device=dev)
        parts_st = [torch.empty(len(t_st), dtype=torch.float64) for _ in range(world)]
        dist.all_gather(parts_st, t_st.cpu())
        g_st = torch.stack(parts_st).numpy()
        per_rank = {"stages_ms": {k: [round(float(g_st[r, i]), 4) for r in range(world)] for i, k in enumerate(keys)},
                    "meshlet_instances": [int(g_st[r, len(keys)]) for r in range(world)],
                    "survivors": [int(g_st[r, len(keys) + 1]) for r in range(world)],
                    "triangles": [int(g_st[r, len(keys) + 2]) for r in range(world)]}
    # max over ranks
    if multi:
        t = torch.tensor([ms_per_step], dtype=torch.float64)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_per_step = float(t.item())
        tot = torch.tensor([cnt["total"], cnt["triangles"]], dtype=torch.float64)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
        job_meshlets, job_tris = float(tot[0].item()), float(tot[1].item())
    else:
        job_meshlets, job_tris = float(cnt["total"]), float(cnt["triangles"])
    value = job_meshlets / (ms_per_step * 1e-3)

    # ---------------- roofline of the dominant cull kernel (late pass: every meshlet instance fully tested) ----------------
    peak, peak_src = measured_peak_hbm()
    N_local = cnt_stage["total"]
    I_local = shard[1] if shard else scene.mesh_instance_count
    M_bits = scene.max_meshlet_instance_count // world  # mask words this rank's meshlets touch
    S_late = cnt_stage["late"]
    U = len(scene.meshes)
    # SURVEY 8d (the contract's formula: the reference's 8 B/meshlet id stream + 16 B bounds, reference tables)
    algo_survey = N_local * 24 + 2 * 4 * ((M_bits + 31) // 32) + 4 * S_late + I_local * 84 + U * 128
    # what THIS kernel has to move: no id stream any more (8 B per 32 meshlets of slab table instead), 16 B bounds, mask
    # read + write, survivors, one 272 B InstCull record per mesh instance
    algo_kernel = N_local * 16 + ((N_local + 31) // 32) * 8 + 2 * 4 * ((M_bits + 31) // 32) + 4 * S_late + I_local * 272
    t_late = stages_ms["cull_late"] * 1e-3
    achieved = algo_kernel / t_late / 1e9 if t_late > 0 else 0.0
    traffic, traffic_src = None, None
    prof = os.path.join(ROOT, "profiles", "ncu_cull_late_summary.json")
    if os.path.exists(prof):
        try:
            pj = json.load(open(prof))
            traffic, traffic_src = pj.get("dram_bytes_per_launch"), pj.get("source", "profiles/ncu_cull_late_summary.json")
        except Exception:
            traffic = None
    roofline = {"bound": "hbm", "kernel": "k_cull_meshlets<HIZ,OCC,LATE> (late pass)", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "traffic": traffic,
                "traffic_note": f"constant from a committed ncu --set full capture ({traffic_src}), not measured in this run" if traffic else None,
                "peak_source": peak_src,
                "algorithmic_bytes_per_launch": algo_kernel, "kernel_ms": stages_ms["cull_late"],
                "frac_survey_8d_formula": (algo_survey / t_late / 1e9 / peak) if t_late > 0 else None,
                "algorithmic_bytes_survey_8d_formula": algo_survey,
                "meshlets_per_s_kernel": N_local / t_late if t_late > 0 else None,
                "late_survivors_in_timed_frame": S_late,
                "note": "algorithmic bytes = N*16 + 8*ceil(N/32) + 8*ceil(M/32) + 4*S + I*272 (this kernel: slab table instead of the 8 B/meshlet "
                        "id stream, one InstCull record per mesh instance); frac_survey_8d_formula uses SURVEY 8d's N*24 + ... for comparison with "
                        f"round 1.  {U} unique meshes" + (" => bounds are L2-resident and the kernel is latency/issue-bound (DESIGN.md)" if U <= 1024 else " => bounds stream from HBM")}

    def _k(name, algo, ms):
        return {"kernel": name, "algorithmic_bytes": int(algo), "ms": ms, "achieved_gbs": algo / (ms * 1e-3) / 1e9 if ms > 0 else None,
                "frac": algo / (ms * 1e-3) / 1e9 / peak if ms > 0 else None}
    per_meshlet = 16 + 3 * 64 + 4 * 49 + 8 * 49          # Meshlet + micro indices + vertex indices + positions
    hw_, hh_ = scene.hiz_extent()
    roofline["other_kernels"] = [] if any(k not in stages_ms for k in ("cull_early", "raster_early", "hiz", "raster_late")) else [
        _k("k_cull_meshlets<HIZ,OCC,EARLY,ZERO>", ((N_local + 31) // 32) * 8 + 2 * 4 * ((M_bits + 31) // 32) + cnt_stage["early"] * 20 + I_local * 272, stages_ms["cull_early"]),
        _k("k_raster_visbuffer (early)", cnt_stage["early"] * per_meshlet + 8 * w * h, stages_ms["raster_early"]),
        _k("k_hiz_tiles + k_hiz_tail" + (" + peer exchange" if multi else ""), 4 * hw_ * hh_ + 4 * (4 * hw_ * hh_) // 3, stages_ms["hiz"]),
        _k("k_raster_visbuffer (late)", cnt_stage["late"] * per_meshlet, stages_ms["raster_late"]),
    ]

    # ---------------- e2e through the reference-facing host API with HOST buffers ----------------
    e2e = None
    if not args.no_e2e and not multi:
        r = capi.Renderer(local_rank, scene)
        pin = lambda shape, dt: torch.empty(shape, dtype=dt, pin_memory=True).numpy()  # noqa: E731
        # per-frame HOST inputs = what RendererInstance::update / render receive every frame: the camera and the (dirty)
        # transforms; the external depth (terrain stand-in) is GPU-resident in the engine, so it is uploaded once
        r.set_external_depth(scene.occluder_depth)
        xf_pinned = pin((len(scene.transforms), 16), torch.float32)
        xf_pinned[...] = scene.transforms["world"]
        # per-frame HOST outputs = the integer results of the path: the R32UI vis image, the survivor ids and the counters.
        # The D32F depth attachment only feeds GPU passes (Hi-Z, shading) and stays device-resident, as in the engine;
        # e2e_with_depth reads it back as well.
        def outbufs_for(with_depth):
            return [dict(vis32=pin((h, w), torch.int32).view(np.uint32),
                         idx=pin((max(1, scene.max_meshlet_instance_count),), torch.int32).view(np.uint32),
                         **({"depth": pin((h, w), torch.float32)} if with_depth else {})) for _ in range(2)]

        def e2e_steps(n, outbufs):
            """n pipelined frames: frame i's device->host copies overlap frame i+1's kernels (oxr_submit / oxr_wait);
            every frame still pays its own H2D (camera, transforms) and D2H (vis32, survivor ids, counters)."""
            prev, res_ = None, None
            for i in range(n):
                r.update_transforms(xf_pinned)                   # H2D: all transforms (pinned)
                t = r.submit(cams[i % 2], outbufs[i % 2])        # H2D camera; kernels; D2H enqueued on the copy stream
                if prev is not None:
                    res_ = r.wait(prev)                          # frame i-1 is now in host memory
                prev = t
            return r.wait(prev)

        def e2e_measure(with_depth):
            ob = outbufs_for(with_depth)
            e2e_steps(W, ob)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            res = e2e_steps(K, ob)
            torch.cuda.synchronize()
            sec = (time.perf_counter() - t0) / K
            d2h = ob[0]["vis32"].nbytes + ob[0]["idx"].nbytes + 12 + 8 + 8 + (ob[0]["depth"].nbytes if with_depth else 0)
            return res, sec, d2h

        res, e2e_s, d2h = e2e_measure(False)
        h2d = 96 + xf_pinned.nbytes
        e2e = {"value": res["total"] / e2e_s, "unit": UNIT, "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
               "ms_per_step": e2e_s * 1e3, "api": "oxr_update_transforms + oxr_submit / oxr_wait (C++ ox::RendererInstance mirror over the C ABI), pinned host buffers, "
                      "2 frames in flight; H2D camera + all transforms, D2H vis32 image + survivor ids + counters (depth stays on the device)"}
        res_d, e2e_d_s, d2h_d = e2e_measure(True)
        e2e["e2e_with_depth"] = {"value": res_d["total"] / e2e_d_s, "ms_per_step": e2e_d_s * 1e3, "d2h_bytes_per_step": int(d2h_d),
                                 "note": "same, plus the D32F depth attachment read back every frame"}
        r.close()

    # ---------------- CPU baseline (rank 0, N = 1 only) ----------------
    cpu_baseline = None
    if not args.no_cpu and not multi and rank == 0:
        cores = os.cpu_count() or 1
        sec, last = cpu_frames(scene, args.cpu_frames, cores)
        cpu_baseline = {"value": scene.max_meshlet_instance_count / sec, "unit": UNIT, "cores": cores, "kind": "port",
                        "sample": f"{args.cpu_frames} full frames of the same {scene.max_meshlet_instance_count}-meshlet scene "
                                  f"(oracle port of the reference shaders, pthreads x{cores}); {sec * 1e3:.0f} ms/frame",
                        "triangles_per_s": last["triangles"] / sec,
                        "frustum_cull_draw_list_loops": cpu_frustum_loops(scene, cams[0], cores)}

    dbg("reductions done")
    exchange = None
    if multi:
        def time_op(fn, n=10):
            for _ in range(2):
                fn()
            barrier()
            a, b = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a.record()
            for _ in range(n):
                fn()
            b.record()
            torch.cuda.synchronize()
            return a.elapsed_time(b) / n * 1e3  # us

        info = pipe.ctx.mgpu_info()
        pipe.select_buffer(0)
        op_us = {"oxc_mgpu_exchange_frame (vis-buffer %d MB max-reduce + count / id allgathers, %d MB ids per rank)" % (pipe.vis64.numel() * 8 >> 20, info.survivor_capacity * 4 >> 20):
                 time_op(lambda: pipe.exchange_frame(slot=0)),
                 "oxc_mgpu_exchange_hiz (mip-0 push over peer memory + flag barrier + pyramid)": time_op(lambda: pipe.ctx.mgpu_exchange_hiz(pipe.vis64.data_ptr(), w, h))}
        cnt_g, _ = pipe.ctx.mgpu_gathered(0)
        exchange = {"survivor_gather_capacity": int(info.survivor_capacity), "max_survivors_per_rank": int((cnt_g[:, 1] + cnt_g[:, 2]).max()),
                    "hiz_over_peer_memory": bool(info.hiz_over_peer_memory), "op_us_back_to_back": op_us,
                    "steps": "global ids from a local count-only replay (no exchange); Hi-Z: mip-0 texels max-reduced into every peer's buffer by the "
                             "sampling kernel over NVLink peer memory + flag barrier (inside the frame's CUDA graph); after the frame, on a side stream: "
                             "ncclAllReduce(u64 max) of the packed vis buffer, ncclAllGather of counters and survivor ids"}
        pipe.ctx.check_status()
    if rank == 0:
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": n_gpus, "steps": K, "warmup": W, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong" if args.total_meshlets else "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, scene),
            "triangles_rasterised_per_s": job_tris / (ms_per_step * 1e-3),
            "per_frame": {"meshlet_instances": job_meshlets, "early_survivors": cnt["early"], "late_survivors": cnt["late"],
                          "triangles_rasterised": job_tris},
            "stages_ms": stages_ms, "roofline": roofline, "cpu_baseline": cpu_baseline, "e2e": e2e, "clocks": clocks,
            "gpu_launches": int(launches_per_frame * K), "gpu_launches_per_step": int(launches_per_frame),
            "cuda_graph": graphs is not None, "exchange_overlapped": overlap is not None,
            "parity_vs_1gpu": (parity["pass"] if parity else None), "parity_detail": parity,
            "wall_s_timed_region": t_wall, "exchange": exchange, "per_rank": per_rank,
        }
        print(json.dumps(line), flush=True)
    pipe.close()
    if multi:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
