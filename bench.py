#!/usr/bin/env python
"""bench.py — Mrays/s of the per-pixel ray/scene hot path (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--workload c4|c3|c2|c1|c5|c5s]
                    [--dump-outputs DIR]

Workload (config.workload): BASELINE.json configs[3] "unitychan 3840x2160 64 spp", the configuration
the metric's 1/2/4/8-GPU numbers are quoted on; it fits one GPU, so it is also the N=1 workload.
"64 spp" is read as 64 camera rays per pixel = 16 reference passes x 4 jittered sub-samples
(RayTracerProgram.cpp:155-169; SURVEY.md §0.1), MaxBounceTimes 10, material as shipped
(RayTracerProgram.cpp:546-551), counter-RNG seed 0.  One STEP = one whole frame: reset the
accumulation buffer, 16 passes over every pixel, and (N > 1) the framebuffer gather to rank 0.
A ray = one nearest-hit query (FindIntersectionWithScene equivalent) or shadow query, counted on
the device; the same count comes out of the reference for the same seed (tests/).

Consecutive frames rotate through the context's frame slots (rt_gpu_set_frame_slot): frame k+1 is
enqueued while the thin last bounce rounds, the exchange and the read-back of frame k are still in flight —
the wavefront's counterpart of the reference's always-busy task queue (ThreadTaskQueue.h:84-93).  K steps are
still K whole frames, bracketed by a barrier + synchronize on both sides (--no-overlap: one slot).

N > 1: one process per GPU (torchrun), the scene replicated, 32x32-pixel tiles dealt round-robin
(tile % N == rank), no data-path collective while rendering, one NCCL gather of each rank's owned
pixels per frame.  The frame is fixed, so scaling is "strong".  e2e at N > 1: every rank writes its own
tiles of accuBuffer + bitcolor into ONE shared host frame (POSIX shared memory, registered in every
process) over its own PCIe link (rt_gpu_deliver_owned), instead of funnelling the frame through rank 0.

Meshes: the reference's Data folder where oracle/Makefile has staged it (assets/_ref/Data), else stand-ins of the
same names generated into a temporary directory (tests/standin_data.py: a textured ~22 k-triangle figure in place of
unitychan); `config.assets` of the JSON line says which, and `config.workload` marks a stand-in run.  Numbers on the
stand-ins measure the same code on other geometry: they are not comparable with the figures of BASELINE.json and
README.md, which are on the reference's meshes.  Nothing is written into the repository.

--dump-outputs DIR writes what the timed path computed in its last step, after the timing: the accumulation buffer
(accuBuffer: RGB sum + pass count) and the display buffer (bitcolor, ARGB8 as 4 floats) of a fixed, seeded sample of
2^20 pixels (every pixel of a smaller frame), their pixel indices, and the step's ray counts, as float32 / float64
.npy files (40 MB at most).  The inputs depend on the arguments only, so two builds can be compared file by file.

--impl reference times the UNMODIFIED reference (oracle/_ref/libref_oracle.so, compiled from
/root/reference by oracle/Makefile) on all host cores, same scene / camera / seed, each step one
pass (4 camera rays per pixel) over the full frame — a bounded sample of the 16-pass step; its rays are
counted by the reference itself (the instrumented twin libref_oracle_count.so).  That arm imports nothing
of the product.
"""
import argparse
import ctypes as C
import hashlib
import json
import os
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

import numpy as np  # noqa: E402

REF_DATA = os.path.join(ROOT, "assets", "_ref", "Data")
DATA = REF_DATA
ASSETS = "reference Data folder (assets/_ref/Data)"
TILE = 32
NUM_SMS = 148
DUMP_PIXELS = 1 << 20
_scratch = None


def scratch_dir():
    """A temporary directory of this process for generated inputs; removed at exit."""
    global _scratch
    if _scratch is None:
        _scratch = tempfile.TemporaryDirectory(prefix="rtb200_bench_")
    return _scratch.name


WORKLOADS = {
    # name: (scene fn name, W, H, passes, antialias, max_bounce, mode, description)
    "c4": ("c3_unitychan", 3840, 2160, 16, 1, 10, "path",
           "unitychan.obj+MTL+PNG 3840x2160, 64 camera rays/pixel (16 passes x 4 jittered), MaxBounceTimes 10"),
    "c3": ("c3_unitychan", 1920, 1080, 4, 1, 10, "path",
           "unitychan.obj+MTL+PNG 1920x1080, 16 camera rays/pixel (4 passes x 4 jittered), MaxBounceTimes 10"),
    "c2": ("c2_monkey", 1920, 1080, 1, 0, 5, "path",
           "BlenderMonkey.obj reflective + reflective ground, 1920x1080, 1 centre ray/pixel, 4 bounces"),
    "c5": ("generated:623", 3840, 2160, 4, 1, 10, "path",
           "623 translated unitychan copies = 10.0 M triangles (generated OBJ), 3840x2160, 16 camera rays/pixel, MaxBounceTimes 10"),
    "c5s": ("generated:62", 1920, 1080, 4, 1, 10, "path",
            "62 translated unitychan copies = 1.0 M triangles (generated OBJ), 1920x1080, 16 camera rays/pixel, MaxBounceTimes 10"),
    "c1": ("c1_torusknot", 640, 480, 1, 0, 1, "whitted",
           "TorusKnot.obj 640x480, 1 centre ray/pixel, primary + shadow ray to GSceneLights[0]"),
}


def peaks():
    path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(path):
        with open(path) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


class ClockSampler(threading.Thread):
    """SM clock + throttle reasons during the timed region (NVML; nvidia-smi's numbers)."""
    REASONS = {0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown",
               0x80: "hw_power_brake_slowdown", 0x2: "applications_clocks_setting", 0x10: "sync_boost"}

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.stop_flag, self.sm, self.mask, self.max_mhz, self.power = index, False, [], 0, None, []
        self.ok = False
        try:
            import pynvml
            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
            self.ok = True
        except Exception:
            self.ok = False

    def run(self):
        if not self.ok:
            return
        nv = self.nv
        while not self.stop_flag:
            try:
                self.sm.append(nv.nvmlDeviceGetClockInfo(self.h, nv.NVML_CLOCK_SM))
                try:
                    self.mask |= nv.nvmlDeviceGetCurrentClocksEventReasons(self.h)
                except Exception:
                    self.mask |= nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                self.power.append(nv.nvmlDeviceGetPowerUsage(self.h) / 1000.0)
            except Exception:
                pass
            time.sleep(0.05)

    def result(self):
        if not self.ok or not self.sm:
            return {"sm_mhz": None, "sm_max_mhz": self.max_mhz, "reasons": ["unavailable"]}
        return {"sm_mhz": float(np.median(self.sm)), "sm_max_mhz": float(self.max_mhz), "samples": len(self.sm),
                "power_w_max": float(max(self.power)) if self.power else None,
                "reasons": [n for b, n in self.REASONS.items() if self.mask & b]}


def build_spec(workload):
    import scenes
    fn, W, H, passes, aa, bounce, mode, desc = WORKLOADS[workload]
    if fn.startswith("generated:"):
        # BASELINE configs[4]: translated copies baked into an OBJ (tools/make_c5.py), written to scratch
        sys.path.insert(0, os.path.join(ROOT, "tools"))
        import make_c5
        copies = int(fn.split(":")[1])
        out_dir = os.environ.get("RT_SCRATCH") or scratch_dir()
        os.makedirs(out_dir, exist_ok=True)
        src = os.path.join(DATA, "unitychan.obj")
        out = os.path.join(out_dir, make_c5.cached_name(src, copies, W / H))
        if not os.path.exists(out):
            make_c5.main(src, out, copies, W / H)
        spec = [("mesh", out, ("blend", ("reflective", scenes.WHITE, 0.2), ("diffuse", scenes.WHITE), 1.0))]
        return spec, W, H, passes, aa, bounce, mode, desc
    return getattr(scenes, fn)(DATA), W, H, passes, aa, bounce, mode, desc


def workload_config(args, W, H, passes, aa, bounce, desc):
    """`config` of the JSON line: the workload, identical in both arms (what differs per arm is outside it)."""
    return {
        "workload": f"{args.workload}: {desc}" + ("" if DATA == REF_DATA else
                    " -- on STAND-IN meshes, not the reference's: not comparable with the figures of BASELINE.json / README.md"),
        "assets": ASSETS,
        "frame": f"{W}x{H}", "passes_per_step": passes, "camera_rays_per_pixel": passes * (4 if aa else 1), "max_bounce": bounce,
        "camera": "eye (0,0,7), dir_z -0.5 (RayTracerProgram.cpp:133,164)", "seed": 0,
        "rng": "counter RNG shared by both arms (include/rt_rng.h; interposed for rand() in the reference, lock-free)",
        "l2": "no explicit flush: every step streams its per-sample radiance buffers (GBs, written then re-read) and the path "
              "pools through L2 (126 MB); the 2 MB of geometry is resident by design",
        "parallelism": f"own arm: {TILE}x{TILE}-pixel tiles round-robin over the GPUs, scene replicated, one framebuffer gather per frame; "
                       "reference arm: all host threads pull 10-row tasks (RayTracerProgram.cpp:282-327)",
    }


# ---------------------------------------------------------------------------------------------------
# reference arm: the reference's own CPU implementation on the host cores (nothing of the product is imported)
# ---------------------------------------------------------------------------------------------------
def run_reference(args):
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    from oracle import bindings
    spec, W, H, passes, aa, bounce, mode, desc = build_spec(args.workload)
    cores = os.cpu_count() or 1
    rmode = {"path": 0, "preview": 1, "whitted": 2}[mode]
    if not bindings.ref_available():
        # (never the case where oracle/_ref travelled with the snapshot) the restatement needs the product's loader
        return run_reference_port(args, spec, W, H, passes, aa, bounce, mode, desc, cores)
    ref = bindings.RefOracle()
    ref.init_unit_vectors(0)
    scene = ref.build_scene(spec)

    def one(pass_index):
        r = ref.render(scene, W, H, mode=rmode, max_bounce=bounce, pass_begin=pass_index, pass_count=1,
                       antialias=aa, seed=0, nthreads=cores)
        return r["seconds"]

    for w in range(args.warmup):
        one(w % max(passes, 1))
    t_wall = time.perf_counter()
    for k in range(args.steps):
        one(k % max(passes, 1))
    wall = time.perf_counter() - t_wall
    # rays of exactly those passes, counted by the reference itself (instrumented twin, untimed)
    cref = bindings.RefOracle(counting=True)
    cref.init_unit_vectors(0)
    cscene = cref.build_scene(spec)
    per_pass = {}
    for k in range(args.steps):
        pi = k % max(passes, 1)
        if pi not in per_pass:
            per_pass[pi] = cref.render(cscene, W, H, mode=rmode, max_bounce=bounce, pass_begin=pi, pass_count=1,
                                       antialias=aa, seed=0, nthreads=cores)["rays"]
    rays = sum(per_pass[k % max(passes, 1)] for k in range(args.steps))
    value = rays / wall / 1e6
    sample = (f"one pass ({'4 jittered' if aa else '1 centre'} camera ray(s)/pixel) over the full {W}x{H} frame per step = 1/{passes} of the "
              f"own arm's step (all {passes} passes would take ~{passes * wall / args.steps:.0f} s per step); the metric is a rate per ray, so the ratio is like for like")
    line = {
        "impl": "reference", "metric": "Mrays/s (primary+secondary)", "value": value, "unit": "Mrays/s",
        "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": wall / args.steps * 1e3,
        "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, W, H, passes, aa, bounce, desc),
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": cores, "kind": "reference", "sample": sample},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "rays_per_step": rays / args.steps, "rays_counted_by": "oracle/_ref/libref_oracle_count.so (FindIntersectionWithScene calls of the reference itself)",
        "gpu_launches": 0,
    }
    print(json.dumps(line))
    return 0


def run_reference_port(args, spec, W, H, passes, aa, bounce, mode, desc, cores):
    from oracle import bindings
    import raytracerwin_b200 as rt
    port = bindings.PortOracle()
    hs = rt.Scene(spec)
    hs.set_unit_vectors(seed=0, count=0)
    pmode = {"path": rt.RT_MODE_PATH, "preview": rt.RT_MODE_PREVIEW, "whitted": rt.RT_MODE_WHITTED}[mode]
    rays, secs = 0, 0.0
    for k in range(args.warmup + args.steps):
        p = rt.make_params(W, H, mode=pmode, max_bounce=bounce, pass_begin=k % max(passes, 1), pass_count=1,
                           antialias=aa, seed=0, traverse=rt.RT_TRAVERSE_EXACT)
        t0 = time.perf_counter()
        o = port.render(hs.desc, p, nthreads=cores)
        if k >= args.warmup:
            secs += time.perf_counter() - t0
            rays += o["counters"]["rays"]
    value = rays / secs / 1e6
    sample = f"one pass over the full {W}x{H} frame per step = 1/{passes} of the own arm's step"
    print(json.dumps({
        "impl": "reference", "metric": "Mrays/s (primary+secondary)", "value": value, "unit": "Mrays/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs / args.steps * 1e3, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": workload_config(args, W, H, passes, aa, bounce, desc),
        "cpu_baseline": {"value": value, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample},
        "e2e": {"value": value, "unit": "Mrays/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "rays_per_step": rays / args.steps, "gpu_launches": 0}))
    return 0


# ---------------------------------------------------------------------------------------------------
# own arm
# ---------------------------------------------------------------------------------------------------
class SharedFrame:
    """One host frame (accuBuffer 16 B/px + bitcolor 4 B/px) in POSIX shared memory, mapped by every rank."""

    def __init__(self, name, npix, create):
        from multiprocessing import shared_memory
        self.header = 4096          # ready[rank] (frame number + 1 each rank has delivered) | consumed (at word 512)
        self.bytes = self.header + npix * 20
        if create:
            try:
                shared_memory.SharedMemory(name=name).unlink()
            except Exception:
                pass
            self.shm = shared_memory.SharedMemory(name=name, create=True, size=self.bytes)
        else:
            self.shm = shared_memory.SharedMemory(name=name)
            try:        # the creator unlinks it; this process's resource tracker must not try as well (Python < 3.13)
                from multiprocessing import resource_tracker
                resource_tracker.unregister(self.shm._name, "shared_memory")
            except Exception:
                pass
        self.npix = npix
        self.buf = np.frombuffer(self.shm.buf, dtype=np.uint8, count=self.bytes)
        self.addr = self.buf.ctypes.data
        self.words = self.buf[:self.header].view(np.uint32)
        if create:
            self.words[:] = 0
        self.accum = self.buf[self.header:self.header + npix * 16].view(np.float32).reshape(npix, 4)
        self.display = self.buf[self.header + npix * 16:].view(np.uint32)

    def close(self, unlink):
        self.accum = self.display = self.buf = self.words = None
        try:
            self.shm.close()
        except Exception:       # a view of the buffer is still alive somewhere: the mapping goes with the process
            pass
        if unlink:
            try:
                self.shm.unlink()
            except Exception:
                pass


def load_inst_counts(workload):
    """Thread-instruction / DRAM-byte counts per kernel class and step, from an ncu pass over this same bench.py
    command (tools/ncu_inst_counts.py -> profiles/r02_bench_inst_counts.json)."""
    path = os.path.join(ROOT, "profiles", "r02_bench_inst_counts.json")
    if not os.path.exists(path):
        return None, None
    with open(path) as f:
        d = json.load(f)
    return d.get(workload), d.get("source")


def run_own(args):
    import torch
    import torch.distributed as dist
    import raytracerwin_b200 as rt
    from raytracerwin_b200 import tiles

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if world != args.gpus and world > 1:
        raise SystemExit(f"--gpus {args.gpus} but WORLD_SIZE={world}")
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (no CPU fallback for the render path)")
    torch.cuda.set_device(local)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))

    spec, W, H, passes, aa, bounce, mode, desc = build_spec(args.workload)
    pmode = {"path": rt.RT_MODE_PATH, "preview": rt.RT_MODE_PREVIEW, "whitted": rt.RT_MODE_WHITTED}[mode]
    npix = W * H
    t0 = time.perf_counter()
    scene = rt.Scene(spec)
    if mode == "path":
        scene.set_unit_vectors(seed=0, count=0)
    t_scene = time.perf_counter() - t0
    ctx = rt.GpuContext(local)
    t0 = time.perf_counter()
    ctx.upload_scene(scene)
    ctx.synchronize()
    t_upload = time.perf_counter() - t0
    lib = rt.load_library()
    dev = torch.device("cuda", local)

    # frame slots: consecutive frames alternate, each slot with its own stream (torch sees them as external streams
    # so that the NCCL gather of a frame is ordered after that frame's passes and nothing else)
    nslots = 1 if args.no_overlap else (args.slots if args.slots > 0 else 4)
    streams = []
    for s in range(nslots):
        if nslots > 1:
            ctx.set_frame_slot(s)
        ctx.reset_accum(W, H)                       # sizes the frame buffers: their addresses are stable from here
        streams.append(torch.cuda.ExternalStream(ctx.stream, device=dev))
    torch.cuda.set_stream(streams[0])

    tile_kw = dict(tile_size=TILE, tile_count=world, tile_rank=rank) if world > 1 else {}
    params = rt.make_params(W, H, mode=pmode, max_bounce=bounce, pass_begin=0, pass_count=passes, antialias=aa,
                            seed=0, traverse=rt.RT_TRAVERSE_CULLED, **tile_kw)
    owned = [rt.owned_pixels(W, H, TILE, world, r) for r in range(world)]
    # The one exchange step: pack -> NCCL gather -> unpack (default), or RT_EXCHANGE=peer: every rank writes its
    # owned tiles straight into rank 0's frame over NVLink (rank 0's accumulation buffers mapped through CUDA IPC;
    # two 4-byte all-reduces order the ranks).  Measured on 8 B200s the gather wins (DESIGN.md §5).
    peer_frames, exchange = [None] * nslots, "none"
    if world > 1:
        ok = torch.ones(1, dtype=torch.int32, device="cuda")
        if os.environ.get("RT_EXCHANGE", "nccl") != "peer":
            ok.zero_()
        else:
            for s in range(nslots):
                if nslots > 1:
                    ctx.set_frame_slot(s)
                handle = torch.zeros(64, dtype=torch.uint8, device="cuda")
                if rank == 0:
                    handle.copy_(torch.frombuffer(bytearray(ctx.export_frame()), dtype=torch.uint8))
                dist.broadcast(handle, 0)
                if rank != 0:
                    try:
                        peer_frames[s] = ctx.open_peer_frame(bytes(handle.cpu().numpy().tobytes()))
                    except Exception as e:      # noqa: BLE001 - any refusal means "use the collective"
                        sys.stderr.write(f"[bench rank {rank}] peer frame not mapped ({e}); using NCCL gather\n")
                        ok.zero_()
        dist.all_reduce(ok, op=dist.ReduceOp.MIN)
        exchange = "peer" if int(ok.item()) == 1 else "nccl"
        if exchange == "nccl":
            for s in range(nslots):
                if peer_frames[s] is not None:
                    ctx.close_peer_frame(peer_frames[s])
                    peer_frames[s] = None
            sends = [torch.empty((max(owned), 4), dtype=torch.float32, device="cuda") for _ in range(nslots)]
        token = torch.zeros(1, dtype=torch.int32, device="cuda")

    def select(k):
        s = k % nslots
        if nslots > 1:
            ctx.set_frame_slot(s)
            torch.cuda.set_stream(streams[s])
        return s

    def render_frame(k, gather=True):
        """Frame k, enqueued on its slot: reset, all passes, (N > 1) the exchange to rank 0's device frame."""
        s = select(k)
        ctx.reset_accum(W, H)
        if exchange == "peer" and gather:
            dist.all_reduce(token)                  # rank 0 has cleared its frame: pushes may land from here on
        ctx.render_tile(params)
        if not gather:
            return s
        if exchange == "peer":
            if rank != 0:
                ctx.push_owned(params, peer_frames[s])
            dist.all_reduce(token)                  # every push has landed before rank 0 goes on
        elif exchange == "nccl":
            ctx.pack_owned(params, sends[s].data_ptr(), owned[rank] * 16)
            recv = tiles.gather_owned(dist, sends[s], owned, rank, world, dst=0)
            if rank == 0:
                for r in range(1, world):
                    ctx.unpack_owned(params, r, recv[r].data_ptr(), owned[r] * 16)
        return s

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    if args.profile_frames > 0:
        # for ncu: the scene, then N plain frames (tools/ncu_inst_counts.py divides the per-kernel sums by N)
        for k in range(args.profile_frames):
            render_frame(k)
        barrier()
        ctx.close()
        return 0

    # --- algorithmic bytes per ray: what the REFERENCE traversal evaluates (exact mode), one pass ---
    # (generated scenes: a band of rows away from the centre row — un-culled, a ray with dy == 0 has a disabled slab
    # axis and visits thousands of the 20 M nodes, RRay.cpp:105; the per-ray ratio is what is used)
    band = dict(start=(H // 4) * W, end=(H // 4 + 64) * W - 1) if WORKLOADS[args.workload][0].startswith("generated:") else {}
    exact = rt.make_params(W, H, mode=pmode, max_bounce=bounce, pass_begin=0, pass_count=1, antialias=aa, seed=0,
                           traverse=rt.RT_TRAVERSE_EXACT, **band, **tile_kw)
    select(0)
    ctx.reset_accum(W, H)
    ctx.reset_counters()
    ctx.render_tile(exact)
    ce = ctx.counters()
    textured = scene.desc.contents.num_meshes > 0 and scene.desc.contents.meshes[0].num_textures > 0
    s_hit = 128 if textured else 64
    walk_bytes = 32 * ce["node_tests"] + 48 * ce["tri_tests"]                  # the walk kernels' share
    alg_bytes = walk_bytes + s_hit * ce["mesh_hits"] + 16 * ce["camera_rays"]      # the whole step
    bytes_per_ray = alg_bytes / max(ce["rays"], 1)
    walk_bytes_per_ray = walk_bytes / max(ce["rays"], 1)

    for k in range(args.warmup):
        render_frame(k)
    barrier()
    ctx.reset_counters()
    barrier()
    launches0 = ctx.launch_count
    sampler = ClockSampler(local)
    sampler.start()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(streams[0])                      # every stream is idle here (barrier above)
    for k in range(args.steps):
        render_frame(k)
    for s in range(1, nslots):
        streams[0].wait_stream(streams[s])
    ev1.record(streams[0])                      # after the last frame of every slot
    barrier()
    sampler.stop_flag = True
    sampler.join()
    ms = ev0.elapsed_time(ev1)
    launches = ctx.launch_count - launches0
    c = ctx.counters()
    dumped = None
    if args.dump_outputs and rank == 0:
        # the last timed frame, on rank 0 the whole frame (the gather has landed: barrier above)
        select(args.steps - 1)
        dumped = (ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H).reshape(npix, 4),
                  ctx.readback(rt.RT_READ_DISPLAY_ARGB8, W, H).reshape(npix))

    # --- per-kernel-class durations: one more step with a single pipe (strictly one kernel at a time, same process,
    # same data, one CUDA event per launch on the launching stream), outside the timed region ---
    select(0)
    prev_pipes = ctx.get_pipes()
    ctx.set_pipes(1)
    ctx.time_kernels(2)
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(streams[0])
    ctx.reset_accum(W, H)
    ctx.render_tile(params)
    e1.record(streams[0])
    torch.cuda.synchronize()
    serial_step_ms = e0.elapsed_time(e1)
    classes = ctx.kernel_class_ms()
    ctx.time_kernels(0)
    ctx.set_pipes(prev_pipes)
    ctx.reset_counters()

    stats = torch.tensor([ms, float(c["rays"]), float(launches), float(c["node_visits"]), float(c["tri_visits"]),
                          float(c["camera_rays"]), float(c["mesh_walks"])], dtype=torch.float64, device="cuda")
    rank_ms = [ms / args.steps]
    if world > 1:
        every = [torch.zeros(1, dtype=torch.float64, device="cuda") for _ in range(world)]
        dist.all_gather(every, stats[:1].clone())
        rank_ms = [float(t[0]) / args.steps for t in every]
        mx = stats.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(stats, op=dist.ReduceOp.SUM)
        ms = float(mx[0])
    rays_total, launches_total = float(stats[1]), int(stats[2])
    value = rays_total / (ms * 1e-3) / 1e6

    # --- end to end through the C-ABI with host buffers: task struct in, framebuffers out -------------
    # N = 1: rt_gpu_readback of accuBuffer + bitcolor into pinned host memory.  N > 1: every rank delivers its own tiles
    # into one shared host frame over its own PCIe link; a 4-byte all-reduce per frame tells rank 0 the frame is whole.
    # Frames are enqueued ahead of the one being waited for, as many as there are slots (one host frame per slot).
    host = []
    if world == 1:
        for s in range(nslots):
            host.append((torch.empty((npix, 4), dtype=torch.float32).pin_memory(), torch.empty((npix,), dtype=torch.int32).pin_memory()))
    else:
        names = [f"rtb200_{os.environ.get('MASTER_PORT', '0')}_{s}" for s in range(nslots)]
        if rank == 0:
            frames = [SharedFrame(n, npix, True) for n in names]
        dist.barrier()
        if rank != 0:
            frames = [SharedFrame(n, npix, False) for n in names]
        frame_dev = [ctx.register_host_frame(f.addr, f.bytes) for f in frames]      # header + accuBuffer + bitcolor
        dist.barrier()

    CONSUMED = 512                              # word index of the consumer's counter in a frame's header

    def spin(cond):
        n = 0
        while not cond():
            n += 1
            if n > 200:
                time.sleep(0.00005)

    def e2e_enqueue(k):
        s = k % nslots
        if world > 1 and k >= nslots:
            # back-pressure: the consumer has taken frame k - nslots out of this host frame
            spin(lambda: int(frames[s].words[CONSUMED]) >= k - nslots + 1)
        render_frame(k, gather=(world == 1))
        if world > 1:
            ctx.deliver_owned(params, frame_dev[s] + frames[s].header, frame_dev[s] + frames[s].header + npix * 16)
            ctx.signal_host(frame_dev[s] + 4 * rank, k + 1)         # "rank has delivered frame k", after the delivery
        return s

    def e2e_wait(k):
        s = select(k)
        if world == 1:
            ctx.readback_into(rt.RT_READ_ACCUM_RGBN_F32, host[s][0].data_ptr(), npix * 16)
            ctx.readback_into(rt.RT_READ_DISPLAY_ARGB8, host[s][1].data_ptr(), npix * 4)
        elif rank == 0:
            # the consumer: frame k is whole once every rank has signalled it; no collective, nobody waits for anybody else
            spin(lambda: bool((frames[s].words[:world] >= k + 1).all()))
            frames[s].words[CONSUMED] = k + 1
        return s

    e2e_enqueue(0)
    e2e_wait(0)
    barrier()
    if world > 1:
        for f in frames:                        # frame numbering restarts for the timed run
            if rank == 0:
                f.words[:] = 0
        barrier()
    ctx.reset_counters()
    barrier()
    t0 = time.perf_counter()
    lag = max(nslots - 1, 1)                    # a slot's host frame is consumed before the slot is reused
    for k in range(args.steps):
        e2e_enqueue(k)
        if k >= lag:
            e2e_wait(k - lag)
    for k in range(max(args.steps - lag, 0), args.steps):
        last_slot = e2e_wait(k)
    barrier()
    e2e_s = time.perf_counter() - t0
    c2 = ctx.counters()
    e2e_stats = torch.tensor([e2e_s, float(c2["rays"])], dtype=torch.float64, device="cuda")
    if world > 1:
        mx = e2e_stats.clone()
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        dist.all_reduce(e2e_stats, op=dist.ReduceOp.SUM)
        e2e_s = float(mx[0])
    e2e_value = float(e2e_stats[1]) / e2e_s / 1e6
    # the frame rank 0 holds in HOST memory must carry every pass of every pixel, whoever rendered it; its hash is
    # the same for any GPU count (the frame is bit-identical by construction: RNG keyed by absolute pixel / pass)
    frame_sha = None
    if rank == 0:
        def check_frame(acc):
            if mode == "path":
                missing = int((acc[:, 3] != float(passes)).sum())
                if missing:
                    raise SystemExit(f"frame incomplete after the exchange: {missing} pixels without all {passes} passes")
            return hashlib.sha256(np.ascontiguousarray(acc).tobytes()).hexdigest()
        frame_sha = check_frame(host[last_slot][0].numpy() if world == 1 else frames[last_slot].accum)
        # and the device-resident frame the gather assembled on rank 0 (the `value` path) is that same frame
        if world > 1:
            render_frame(0)
            select(0)
            if hashlib.sha256(ctx.readback(rt.RT_READ_ACCUM_RGBN_F32, W, H).tobytes()).hexdigest() != frame_sha:
                raise SystemExit("the frame gathered on rank 0's device differs from the frame delivered to host memory")
    elif world > 1:
        render_frame(0)

    if rank == 0:
        peak, peak_src = peaks()
        clocks = sampler.result()
        sm_hz = (clocks.get("sm_mhz") or 1965.0) * 1e6
        rays_rank = c["rays"] / args.steps
        counts, counts_src = load_inst_counts(args.workload)
        total_cls_ms = sum(v[0] for v in classes.values()) or 1.0
        per_class = {}
        issue_peak = NUM_SMS * 4 * 32 * sm_hz                     # thread instructions / s at full lanes
        for name, (cms, n) in classes.items():
            e = {"ms_per_step": cms, "launches_per_step": n, "share_of_step": cms / total_cls_ms}
            if counts and name in counts.get("classes", {}) and cms > 0:
                k = counts["classes"][name]
                scale = rays_rank / counts["rays_per_step"]           # a rank's share of the profiled frame (1 at N = 1)
                e["thread_inst_per_step"] = k["thread_inst"] * scale
                e["lanes_per_warp_inst"] = k["thread_inst"] / max(k["warp_inst"], 1)
                e["issue_frac_lane_weighted"] = k["thread_inst"] * scale / (cms * 1e-3) / issue_peak
                e["issue_slot_frac"] = k["warp_inst"] * scale / (cms * 1e-3) / (NUM_SMS * 4 * sm_hz)
                e["dram_bytes_per_launch"] = k["dram_bytes"] * scale / max(n, 1)
            per_class[name] = e
        dom = "walk"                                              # rt_walk_kernel<CULL=1>: the largest share of the step
        dms, dn = classes[dom]
        walk_ms = classes["walk"][0] + classes["packet_walk"][0]
        d = per_class[dom]
        l1_peak = NUM_SMS * 128 * sm_hz / 1e9                         # GB/s: 128 B per SM per clock
        walk_alg_gbs = rays_rank * walk_bytes_per_ray / (walk_ms * 1e-3) / 1e9 if walk_ms > 0 else None
        hbm_regime = WORKLOADS[args.workload][0].startswith("generated:")      # GBs of geometry: the walk streams nodes from HBM / L2
        roofline = {
            "bound": "issue", "kernel": "rt_walk_kernel<CULL=1> (bounce / shadow rounds, a lane per walk): the largest share of the step",
            "achieved": d.get("thread_inst_per_step", 0.0) / (dms * 1e-3) / 1e12 if dms > 0 and "thread_inst_per_step" in d else None,
            "peak": issue_peak / 1e12, "unit": "T thread-instructions/s",
            "frac": d.get("issue_frac_lane_weighted"),
            "traffic": d.get("dram_bytes_per_launch"),
            "peak_source": "148 SMs x 4 schedulers x 32 lanes x the SM clock sampled during the timed region (%.0f MHz)" % (sm_hz / 1e6),
            "def": "lane-weighted issue utilisation = thread instructions executed (smsp__thread_inst_executed.sum of the kernel's launches in one "
                   "step, ncu over this same bench.py command: " + str(counts_src) + ") / the kernel's duration (live: one CUDA event per launch, "
                   "single-pipe step) / peak; SURVEY.md 8(d) names two bounds and asks for the tighter one: this is it",
            "kernel_ms_per_launch": dms / max(dn, 1), "kernel_launches_per_step": dn, "kernel_share_of_step": d["share_of_step"],
            "measured_on": "one extra step with a single pipe (kernels strictly one at a time) right after the timed region: serial step %.3f ms" % serial_step_ms,
            "classes": per_class,
            "whole_step": {
                "thread_inst": sum(e.get("thread_inst_per_step", 0.0) for e in per_class.values()) or None,
                "frac": (sum(e.get("thread_inst_per_step", 0.0) for e in per_class.values()) / (ms / args.steps * 1e-3) / issue_peak) if counts else None,
                "def": "thread instructions of every kernel of one step / the timed step (all pipes, frames in flight) / the issue peak: "
                       "how busy the machine's lanes are over the whole frame, concurrency included"},
            "memory": {
                "algorithmic_bytes_per_ray": walk_bytes_per_ray,
                "algorithmic_bytes_def": "mesh walk (packet kernel + walk kernel): 32 B x slab tests + 48 B x triangle tests the REFERENCE traversal evaluates "
                                         "for the same rays (device exact-mode counters, one pass), SURVEY.md 8(d)",
                "walk_ms_per_step": walk_ms, "achieved_GBs": walk_alg_gbs,
                "l1": {"peak_GBs": l1_peak, "frac": walk_alg_gbs / l1_peak if walk_alg_gbs else None,
                       "note": "the level the working set lives in: 2 MB of geometry, L1/L2 resident (ncu: DRAM throughput < 3 % in the walk kernels)"},
                "hbm_floor": {"peak_GBs": peak, "peak_source": peak_src, "frac": walk_alg_gbs / peak if walk_alg_gbs else None,
                              "note": "algorithmic bytes / time against the HBM peak: > 1 is expected here (resident geometry, culled walk) — a floor, not the bound"},
                "whole_step_bytes_per_ray": bytes_per_ray,
                "reference_nodes_per_ray": ce["node_tests"] / max(ce["rays"], 1), "reference_tris_per_ray": ce["tri_tests"] / max(ce["rays"], 1),
                "visited_nodes_per_ray": float(stats[3]) / max(rays_total, 1), "visited_tris_per_ray": float(stats[4]) / max(rays_total, 1),
            },
            "hbm_bound_config": "profiles/r02_bench_c5.json (bench.py --workload c5: 10 M triangles, 1.9 GB of geometry + shading records: there the walk is HBM / L2 bound)",
        }
        if hbm_regime:
            # C5 / C5s: geometry + shading records are far larger than L2, the contract's HBM bound is the one that binds
            roofline.update({
                "bound": "hbm", "kernel": "the mesh walk (rt_walk_packet_kernel + rt_walk_kernel, CULL=1)",
                "achieved": walk_alg_gbs, "peak": peak, "unit": "GB/s", "frac": walk_alg_gbs / peak if walk_alg_gbs else None,
                "traffic": None, "peak_source": peak_src,
                "def": "algorithmic bytes (32 B x slab tests + 48 B x triangle tests of the REFERENCE traversal, exact-mode counters on a band of rows) x rays / the walk kernels' duration (live, one event per launch)"})
        step_s = ms / args.steps * 1e-3
        line = {
            "metric": "Mrays/s (primary+secondary)", "value": value, "unit": "Mrays/s", "n_gpus": world,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True,
            "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": workload_config(args, W, H, passes, aa, bounce, desc),
            "run": {
                "traverse": "culled (bit-identical to exact; tests/test_gpu_parity.py)",
                "frames_in_flight": nslots, "rank_ms_per_step": rank_ms,
                "exchange": ("owned tiles written into rank 0's frame over NVLink peer memory (CUDA IPC) + two 4-byte all-reduces per frame"
                             if exchange == "peer" else "pack + NCCL gather + unpack per frame") if world > 1 else "none (1 GPU)",
                "rays_per_step": rays_total / args.steps, "camera_rays_per_step": float(stats[5]) / args.steps,
                "mesh_walks_per_step": float(stats[6]) / args.steps,
                "walks_per_s": float(stats[6]) / args.steps / step_s, "node_visits_per_s": float(stats[3]) / args.steps / step_s,
                "note": "most camera rays of this frame miss the figure's bounds and end as sky in the generate kernel: walks/s and node visits/s are the traversal throughput",
                "scene_build_host_s": t_scene, "scene_upload_s": t_upload, "scene_device_bytes": int(lib.rt_gpu_scene_bytes(ctx.handle)),
            },
            "e2e": {"value": e2e_value, "unit": "Mrays/s", "h2d_bytes_per_step": C.sizeof(rt.rt_render_params),
                    "d2h_bytes_per_step": npix * 20,
                    "note": ("per step: rt_gpu_reset_accum + rt_gpu_render_tile(host task struct) + " +
                             ("rt_gpu_readback of accuBuffer (16 B/px) and bitcolor (4 B/px) into pinned host memory" if world == 1 else
                              "rt_gpu_deliver_owned: every rank writes its own tiles of accuBuffer (16 B/px) and bitcolor (4 B/px) into one shared, registered host frame over its own PCIe link, "
                              "then rt_gpu_signal_host: a word of the frame's header; rank 0's host polls the words (no collective, no rank waits for another)") +
                             "; wall clock, max over ranks; as many frames are enqueued ahead of the one being waited for as there are frame slots; the scene is resident (uploaded once, like the reference's SetupScene)")},
            "frame_sha": frame_sha,
            "gpu_launches": launches_total,
            "clocks": clocks,
            "roofline": roofline,
        }
        if world == 1 and not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args, spec, W, H, passes, aa, bounce, mode, c["rays"] / args.steps)
        if dumped is not None:
            dump_outputs(args.dump_outputs, *dumped, stats / args.steps)
        print(json.dumps(line))
    # tear down in dependency order: collectives first (they are queued behind the context's streams),
    # then hand torch its own stream back before the context destroys the ones it borrowed
    torch.cuda.synchronize()
    if world > 1:
        dist.barrier()
        torch.cuda.synchronize()
        for f in frames:
            ctx.unregister_host_frame(f.addr)
        dist.barrier()
        for f in frames:
            f.close(unlink=(rank == 0))
    for s in range(nslots):
        if peer_frames[s] is not None:
            if nslots > 1:
                ctx.set_frame_slot(s)
            ctx.close_peer_frame(peer_frames[s])
    torch.cuda.set_stream(torch.cuda.default_stream())
    if world > 1:
        dist.destroy_process_group()
    ctx.close()
    return 0


def dump_outputs(out_dir, accum, display, stats_per_step):
    """accum (npix, 4) f32 and display (npix,) ARGB8 of one frame -> DIR/*.npy, a fixed sample of DUMP_PIXELS pixels."""
    npix = accum.shape[0]
    if npix > DUMP_PIXELS:
        index = np.sort(np.random.default_rng(0).choice(npix, DUMP_PIXELS, replace=False))
    else:
        index = np.arange(npix)
    disp = display[index].astype(np.uint32)
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "pixel_index.npy"), index.astype(np.float64))
    np.save(os.path.join(out_dir, "accum.npy"), np.ascontiguousarray(accum[index], np.float32))
    np.save(os.path.join(out_dir, "display_argb.npy"), np.stack([(disp >> s) & 255 for s in (24, 16, 8, 0)], -1).astype(np.float32))
    # rays and camera rays of one step, all ranks (node / triangle visit counts depend on how the walks were scheduled)
    np.save(os.path.join(out_dir, "counters.npy"), stats_per_step.cpu().numpy()[[1, 5]].astype(np.float64))


def cpu_baseline(args, spec, W, H, passes, aa, bounce, mode, gpu_rays_per_step):
    """The reference's CPU path on this box's host cores, bounded sample: ONE pass over the full frame."""
    from oracle import bindings
    cores = os.cpu_count() or 1
    rmode = {"path": 0, "preview": 1, "whitted": 2}[mode]
    sample = f"one pass ({'4 jittered' if aa else '1 centre'} camera ray(s)/pixel) over the full {W}x{H} frame = 1/{passes} of a step; rays = the device count of the same step / {passes} (same seed, same paths)"
    rays = gpu_rays_per_step / passes
    if bindings.ref_available():
        ref = bindings.RefOracle()
        ref.init_unit_vectors(0)
        s = ref.build_scene(spec)
        r = ref.render(s, W, H, mode=rmode, max_bounce=bounce, pass_begin=0, pass_count=1, antialias=aa, seed=0, nthreads=cores)
        out = {"value": rays / r["seconds"] / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "reference", "sample": sample,
               "seconds": r["seconds"], "rng": "counter RNG interposed for rand() (lock-free)"}
        # as shipped: glibc rand() behind its lock (SURVEY.md §6) — smaller sample, it is slow
        ref.set_libc_rand(1)
        w2, h2 = max(W // 4, 1), max(H // 4, 1)
        r2 = ref.render(s, w2, h2, mode=rmode, max_bounce=bounce, pass_begin=0, pass_count=1, antialias=aa, seed=0, nthreads=cores)
        ref.set_libc_rand(0)
        out["as_shipped_libc_rand"] = {"value": rays * (w2 * h2) / (W * H) / r2["seconds"] / 1e6, "unit": "Mrays/s", "cores": cores,
                                       "sample": f"one pass at {w2}x{h2}; ray count scaled by pixel ratio (approximate)"}
        ref.free_scene(s)
        return out
    import raytracerwin_b200 as rt
    port = bindings.PortOracle()
    hs = rt.Scene(spec)
    hs.set_unit_vectors(seed=0, count=0)
    pm = {"path": rt.RT_MODE_PATH, "preview": rt.RT_MODE_PREVIEW, "whitted": rt.RT_MODE_WHITTED}[mode]
    p = rt.make_params(W, H, mode=pm, max_bounce=bounce, pass_count=1, antialias=aa, seed=0, traverse=rt.RT_TRAVERSE_EXACT)
    t0 = time.perf_counter()
    o = port.render(hs.desc, p, nthreads=cores)
    dt = time.perf_counter() - t0
    return {"value": o["counters"]["rays"] / dt / 1e6, "unit": "Mrays/s", "cores": cores, "kind": "port", "sample": sample, "seconds": dt}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=4)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="own", choices=["own", "reference"])
    ap.add_argument("--workload", default="c4", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-overlap", action="store_true", help="one frame slot: a frame starts when the previous one has ended")
    ap.add_argument("--slots", type=int, default=0, help="frames in flight (1-4; default 4)")
    ap.add_argument("--profile-frames", type=int, default=0, help="(ncu) render this many plain frames and exit")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the last timed step's outputs (sampled frame buffers, ray counts) to DIR/*.npy")
    args = ap.parse_args()
    if args.warmup < 3 and args.impl == "own":
        args.warmup = 3                     # timing rule: at least 3 warm-up steps
    if args.steps < 1:
        raise SystemExit("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        raise SystemExit("--dump-outputs writes the outputs of the own arm; it is not available with --impl reference")
    global DATA, ASSETS
    if not os.path.isdir(DATA):
        import standin_data
        DATA = standin_data.write(os.path.join(scratch_dir(), "Data"))
        ASSETS = "generated stand-ins of the reference's meshes (tests/standin_data.py)"
    sys.exit(run_reference(args) if args.impl == "reference" else run_own(args))


if __name__ == "__main__":
    main()
