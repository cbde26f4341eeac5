#!/usr/bin/env python
"""bench.py — the hot path (camera::render's pixel x sample loop) on BASELINE.json's headline
configuration: Book-2 final scene, 800x800, 10,000 spp, max_depth 40 (config C5).

    python bench.py --gpus N --steps K --warmup W            # our arm (torchrun for N > 1)
    python bench.py --impl reference --gpus N --steps K ...  # the reference's CPU path, host cores
    python bench.py ... --dump-outputs DIR                   # + the image of the last timed step, DIR/radiance.npy

One STEP = one full render of the workload: every rank renders its shard of the sample indices
of every pixel (strong scaling: the job is fixed, N ranks split the 10,000 spp), then the exact
int64 reduce to rank 0.  `value` = W*H*spp / (max-over-ranks device time per step), scene resident
in HBM.  `e2e` = the same job through the C-ABI with HOST buffers: rt_upload_scene (H2D of the
flattened scene) + rt_render + reduce + rt_download of the RGB8 image (D2H), wall clock.
The oracle / reference harness is executed ONLY by the cpu_baseline and --impl reference legs.
"""
import argparse
import ctypes as C
import importlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

SCENE = "book2_final"
METRIC = "samples_px_per_s"
UNIT = "samples*px/s"
# flop-equivalents per unit of algorithmic work (SURVEY.md §8(d); one slab test = 12 flop + 12 cmp/sel)
F_BOX, F_SPH_MISS, F_SPH_HIT, F_QUAD_EARLY, F_QUAD_FULL, F_MEDIUM = 24, 29, 60, 12, 54, 120
F_BOXPRIM = 36  # a box() primitive: one slab test (24) + the entry/exit interval test and face pick (12)
F_SHADE = dict(lambertian=15, metal=35, dielectric=60, light=0, isotropic=15, checker=10, image=6, noise=1550, bounce=6)
# bytes per unit (fp32 device layouts): BVH2 node with both child boxes 64 B, sphere 32 B, quad 48 B
B_NODE, B_SPH, B_QUAD, B_TEXEL, B_PERLIN = 64, 32, 48, 4, 56 * 16 + 7 * 24
B_BOXPRIM = 48
# The figures bench.py cannot measure itself (DRAM traffic, issue-slot utilisation, active lanes) come from the last ncu
# capture as summarised by tools/ncu_summary.py into profiles/latest_ncu.json, which records the sha256 of csrc/ it was
# taken on: when the kernels have changed since, the figures are omitted rather than pasted.
PER_CONFIG = [  # BASELINE.json configs C1-C4 at their own size (C5 is the headline workload of the line itself)
    ("C1", "book1_final", dict(image_width=1200, samples_per_pixel=10, max_depth=50)),
    ("C2", "bouncing_spheres", dict(image_width=400, samples_per_pixel=100)),
    ("C3a", "earth", dict(image_width=400, samples_per_pixel=100)),
    ("C3b", "perlin_sphere", dict(image_width=400, samples_per_pixel=100)),
    ("C4", "cornell_smoke", dict(image_width=600, samples_per_pixel=200, max_depth=50)),
]
PER_CONFIG_CPU_SPP = {"C1": 1, "C2": 8, "C3a": 8, "C3b": 8, "C4": 2}  # bounded 1-thread reference samples (2-3 s each)
HASH_SPP = 32  # the GPU-count-invariance job: sample indices 0..31 of every pixel, seed 0


def csrc_sha():
    """sha256 of the CODE of csrc/ (comments / whitespace removed) — raytracing-practice_b200/csrc_sha.py."""
    return importlib.import_module("raytracing-practice_b200.csrc_sha").csrc_sha(ROOT)


def latest_ncu():
    p = os.path.join(ROOT, "profiles", "latest_ncu.json")
    if not os.path.exists(p):
        return None, "profiles/latest_ncu.json is missing"
    d = json.load(open(p))
    if d.get("csrc_sha") != csrc_sha():
        return None, f"profiles/latest_ncu.json was captured on csrc {d.get('csrc_sha')}, this build is {csrc_sha()}: omitted"
    return d, d.get("source", "profiles/latest_ncu.json")


def fnv1a64_words(a):
    """FNV-1a over the 64-bit words of an int64 array (the accumulator): h = (h ^ w) * prime mod 2^64."""
    h, prime, mask = 0xCBF29CE484222325, 0x100000001B3, (1 << 64) - 1
    for w in a.reshape(-1).view("uint64").tolist():
        h = ((h ^ w) * prime) & mask
    return f"{h:016x}"


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--scene", default=SCENE)
    ap.add_argument("--spp", type=int, default=0, help="override samples per pixel (0 = the config's 10,000)")
    ap.add_argument("--width", type=int, default=0)
    ap.add_argument("--cpu-spp", type=int, default=8, help="spp of the bounded CPU-baseline sample (SURVEY 8(d): >= 8)")
    ap.add_argument("--no-per-config", action="store_true", help="skip the C1-C4 block")
    ap.add_argument("--no-dropin", action="store_true", help="skip the e2e_dropin leg (build/dropin, the C++ camera::render)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--reduce", default="peer", choices=["peer", "nccl"],
                    help="N > 1: 'peer' = behind its render kernel every rank adds its accumulator into rank 0's buffer with our own "
                         "push kernel (peer memory over NVLink, CUDA IPC, no collective); 'nccl' = ncclInt64 reduce")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write the image the last one rendered (rank 0's reduced radiance, float32 H x W x 3) "
                         "to DIR/radiance.npy; above 64 MB, a fixed seeded sample of its pixels, their flat indices in DIR/pixel_index.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    return args


DUMP_LIMIT = 64 << 20  # bytes of .npy files --dump-outputs may write


def dump_outputs(out_dir, radiance):
    """radiance.npy = the H x W x 3 image, or, when that exceeds DUMP_LIMIT, the pixels at a fixed seeded sample of flat
    indices (pixel_index.npy, ascending) — the same files for the same arguments, so two builds compare output for output."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    if radiance.nbytes > DUMP_LIMIT:
        n = (DUMP_LIMIT - 4096) // (3 * radiance.itemsize + 8)
        idx = np.sort(np.random.default_rng(0).choice(radiance.shape[0] * radiance.shape[1], n, replace=False))
        np.save(os.path.join(out_dir, "pixel_index.npy"), idx.astype(np.float64))
        radiance = radiance.reshape(-1, 3)[idx]
    np.save(os.path.join(out_dir, "radiance.npy"), radiance)


# ---------------------------------------------------------------------------------------------
class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    Q = "clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], threading.Event()

    def run(self):
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:  # noqa: BLE001
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        self.stop_flag.set()
        self.join(timeout=6)
        sm = sorted(int(float(r[0])) for r in self.rows if r and r[0].replace(".", "").isdigit())
        reasons = set()
        for r in self.rows:
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        mx = [int(float(r[1])) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        pw = [float(r[2]) for r in self.rows if len(r) > 2 and r[2].replace(".", "").isdigit()]
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None, "power_w_max": max(pw) if pw else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return d.get("hbm_gbs", 6650.0), "measured", d.get("sm_max_mhz", 1965.0)
    return 6650.0, "fallback", 1965.0


# ---------------------------------------------------------------------------------------------
def cpu_reference_once(scene, width, spp, seed, native=False):
    """One process of the UNMODIFIED reference (oracle/_ref/ref_harness): camera::render, serial."""
    exe = os.path.join(ROOT, "oracle", "_ref", "ref_harness_native" if native else "ref_harness")
    env = dict(os.environ)
    rtb = importlib.import_module("raytracing-practice_b200")
    if rtb.default_image_dir():
        env["RTW_IMAGES"] = rtb.default_image_dir()
    cmd = [exe, "ppm", scene, "/dev/null", "--spp", str(spp), "--seed", str(seed)] + (["--width", str(width)] if width else [])
    return subprocess.Popen(cmd, env=env, stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)


def parse_harness(proc):
    out, _ = proc.communicate()
    line = [l for l in out.splitlines() if l.startswith("JSON ")]
    if proc.returncode != 0 or not line:
        raise RuntimeError("ref_harness failed")
    return json.loads(line[-1][5:])


def cpu_baseline(args):
    """The reference's camera::render as shipped (1 process x 1 thread) on a bounded sample."""
    if not os.path.exists(os.path.join(ROOT, "oracle", "_ref", "ref_harness")):
        return oracle_port_baseline(args, threads=1)
    j = parse_harness(cpu_reference_once(args.scene, args.width, args.cpu_spp, seed=1))
    n = j["width"] * j["height"] * j["spp"]
    return {"value": n / j["seconds"], "unit": UNIT, "cores": 1, "kind": "reference",
            "sample": f"{args.scene} {j['width']}x{j['height']} at {j['spp']} spp (of the config's 10,000), max_depth {j['max_depth']}; "
                      f"unmodified reference camera::render via oracle/_ref/ref_harness (g++ -O2), 1 process x 1 thread as shipped, "
                      f"timed by the harness around camera::render only (no process start / scene build); "
                      f"rotate_y/constant_medium/isotropic are oracle/ref_ext.hpp (absent from the reference)",
            "seconds": j["seconds"], "rays": j["rays"], "mrays_per_s": j["rays"] / j["seconds"] / 1e6, "host_cores_available": os.cpu_count()}


def oracle_port_baseline(args, threads):
    rtb = importlib.import_module("raytracing-practice_b200")
    from oracle import orc

    sc = rtb.Scene(args.scene, rand_seed=1)
    cam = sc.camera_copy(**({"image_width": args.width} if args.width else {}))
    t0 = time.time()
    _, _, rays = orc.render_linear(sc.desc, cam, spp=args.cpu_spp, seed=1, threads=threads, want_sq=False, rng="glibc")
    dt = time.time() - t0
    n = cam.image_width * rtb.image_height(cam) * args.cpu_spp
    return {"value": n / dt, "unit": UNIT, "cores": threads, "kind": "port",
            "sample": f"{args.scene} {cam.image_width}x{rtb.image_height(cam)} at {args.cpu_spp} spp, oracle/oracle.cpp restatement", "seconds": dt,
            "rays": rays, "mrays_per_s": rays / dt / 1e6, "host_cores_available": os.cpu_count()}


def dropin_leg(args, world, W, H, spp):
    """e2e through the REAL drop-in call: a C++ scene program written like the reference's main.cpp (tests/cpp/dropin_main.cpp
    -> build/dropin) from process start to its PPM closed: rt_init on every device, scene build + flatten, upload, render
    sharded over the devices, on-device reduce, download, P3 text.  camera::render's own breakdown comes from RT_B200_TIMING."""
    exe = os.path.join(ROOT, "build", "dropin")
    if not os.path.exists(exe):
        return {"unavailable": "build/dropin is not built (python __graft_entry__.py)"}
    rtb = importlib.import_module("raytracing-practice_b200")
    env = dict(os.environ, RT_B200_DEVICES=",".join(str(i) for i in range(world)), RT_B200_TIMING="1")
    if rtb.default_image_dir():
        env["RTW_IMAGES"] = rtb.default_image_dir()
    out = os.path.join("/dev/shm" if os.path.isdir("/dev/shm") else "/tmp", f"rtb200_dropin_{os.getpid()}.ppm")
    try:
        subprocess.run([exe, "quads", out, "64", "4"], env=env, capture_output=True, timeout=120)  # page the binary in
        t0 = time.time()
        r = subprocess.run([exe, args.scene, out, str(W), str(spp)], env=env, capture_output=True, text=True, timeout=600)
        wall = time.time() - t0
        size = os.path.getsize(out) if os.path.exists(out) else 0
    finally:
        if os.path.exists(out):
            os.remove(out)
    if r.returncode != 0:
        return {"error": r.stderr[-300:]}
    parts = [json.loads(l[len("RTB200_TIMING "):]) for l in r.stderr.splitlines() if l.startswith("RTB200_TIMING ")]
    return {"value": W * H * spp / wall, "unit": UNIT, "process_wall_ms": round(wall * 1e3, 1), "ppm_bytes": size, "devices": world,
            "camera_render_ms": parts[-1] if parts else None,
            "path": "process start -> scene build -> camera::render(std::ofstream, world) -> P3 file closed -> process exit (build/dropin, C++ host API)"}


def run_reference_arm(args):
    """--impl reference: the reference's own CPU implementation on all host threads.  The reference
    is serial and not re-entrant (global rand()), so 'all threads' = one process per core, each
    rendering its own bounded sample with its own srand seed; throughput is aggregated."""
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return 0
    rtb = importlib.import_module("raytracing-practice_b200")
    cores = os.cpu_count() or 1
    have_ref = os.path.exists(os.path.join(ROOT, "oracle", "_ref", "ref_harness"))
    # Timed steps render `spp_each` spp per process: 8 (SURVEY 8(d)) when K timed steps of it fit ~4 minutes, else as many
    # as fit (>= 2); the untimed warm-up steps render 1 spp.  A step's time is the harness's own clock around
    # camera::render (max over the concurrent processes): no process start, scene build or JPEG decode in it.
    sec_per_spp = 2.4  # one process, one spp of this workload with all cores busy (measured by the first warm-up below)
    times, last = [], None
    spp_each = 8
    for step in range(args.warmup + args.steps):
        timed = step >= args.warmup
        if step == args.warmup:
            spp_each = int(max(2, min(8, 240.0 / max(1, args.steps) / max(sec_per_spp, 1e-3))))
        spp_now = spp_each if timed else 1
        t0 = time.time()
        if have_ref:
            procs = [cpu_reference_once(args.scene, args.width, spp_now, seed=100 * step + c + 1) for c in range(cores)]
            res = [parse_harness(p) for p in procs]
            samples = sum(r["width"] * r["height"] * r["spp"] for r in res)
            rays = sum(r["rays"] for r in res)
            dims = (res[0]["width"], res[0]["height"], res[0]["max_depth"])
            dt = max(r["seconds"] for r in res)
        else:
            from oracle import orc

            sc = rtb.Scene(args.scene, rand_seed=1)
            cam = sc.camera_copy(**({"image_width": args.width} if args.width else {}))
            t1 = time.time()
            _, _, rays = orc.render_linear(sc.desc, cam, spp=spp_now * cores, seed=step + 1, threads=cores, want_sq=False, rng="glibc")
            dt = time.time() - t1
            samples = cam.image_width * rtb.image_height(cam) * spp_now * cores
            dims = (cam.image_width, rtb.image_height(cam), cam.max_depth)
        if not timed:
            sec_per_spp = dt / spp_now
        if timed:
            times.append(dt)
            last = (samples, rays)
    sec = sum(times) / len(times)
    value = last[0] / sec
    sample = (f"{args.scene} {dims[0]}x{dims[1]}, max_depth {dims[2]}: {cores} processes x {spp_each} spp per timed step "
              f"({'oracle/_ref/ref_harness = unmodified reference camera::render' if have_ref else 'oracle port'}), one per host core; "
              f"step time = the slowest process's own clock around camera::render (render only)")
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": sec * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": {"workload": f"{args.scene} 800x800 x 10000 spp, max_depth 40 (BASELINE config 5); each CPU step is a bounded sample of it"},
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "reference" if have_ref else "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "mrays_per_s": last[1] / sec / 1e6, "gpu_launches": 0}
    emit(line)
    return 0


# ---------------------------------------------------------------------------------------------
_REAL_STDOUT = None


def emit(line):
    """The ONE JSON line, on the real stdout (fd 1 is pointed at stderr while we run, so that
    library banners such as 'NCCL version ...' cannot end up in front of it)."""
    data = (json.dumps(line) + "\n").encode()
    if _REAL_STDOUT is None:
        sys.stdout.write(data.decode())
        sys.stdout.flush()
    else:
        os.write(_REAL_STDOUT, data)


def main():
    global _REAL_STDOUT
    args = parse()
    sys.stdout.flush()
    _REAL_STDOUT = os.dup(1)
    os.dup2(2, 1)
    if args.impl == "reference":
        return run_reference_arm(args)

    import numpy as np
    import torch

    rtb = importlib.import_module("raytracing-practice_b200")
    dist = importlib.import_module("raytracing-practice_b200.dist")
    rank, local_rank, world = dist.init_process_group()
    done_flag = f"/tmp/rtb200_bench_{os.environ.get('MASTER_PORT', '0')}.done"
    if rank == 0 and os.path.exists(done_flag):
        os.remove(done_flag)
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: there is no CPU fallback for the product path")
    torch.cuda.set_device(local_rank)
    ctx = rtb.Context(local_rank)
    sc = rtb.Scene(args.scene, rand_seed=1)
    over = {}
    if args.spp:
        over["samples_per_pixel"] = args.spp
    if args.width:
        over["image_width"] = args.width
    cam = sc.camera_copy(**over)
    W, H, spp = cam.image_width, rtb.image_height(cam), cam.samples_per_pixel
    begin, count = dist.shard_samples(spp, rank, world)
    ctx.upload_scene(sc.desc)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=f"cuda:{local_rank}")  # > 126 MB L2

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()
        ctx.synchronize()

    ev = [torch.cuda.Event(enable_timing=True) for _ in range(2)]
    peer = None
    if world > 1 and args.reduce == "peer":
        try:
            peer = dist.PeerReduce(ctx, cam)  # CUDA IPC + peer access; ships one 64-byte handle
        except Exception as e:  # noqa: BLE001  (no peer access on this box: say so and use the collective)
            sys.stderr.write(f"[bench] peer reduce unavailable ({e}); using NCCL\n")
            peer = None
        ok = torch.tensor([1 if peer is not None else 0], device=f"cuda:{local_rank}")
        torch.distributed.all_reduce(ok, op=torch.distributed.ReduceOp.MIN)
        if ok.item() == 0:
            peer = None

    def step(seed):
        """Resident-scene step: this rank's shard + reduce; returns device ms (render + reduce)."""
        flush.fill_(1)  # L2 flush between iterations (on torch's stream; finished before the render starts)
        torch.cuda.synchronize()
        if peer is not None:
            # the push kernel runs behind the render kernel inside the context's CUDA-event bracket: last_render_ms covers
            # render + push; rank 0 adds the (wall-clock) time of adopting the reduced buffer
            peer.render(seed)  # zero + barrier + render/push + barrier (+ adopt on rank 0)
            return ctx.stats().last_render_ms + (peer.adopt_ms if rank == 0 else 0.0)
        ctx.render(cam, seed=seed, sample_begin=begin, sample_count=count, clear=True)
        ms = ctx.stats().last_render_ms  # CUDA events recorded on the context's own stream
        if world > 1:
            acc = ctx.accum_tensor()
            ev[0].record()
            dist.reduce_accum_to_rank0(acc)
            ev[1].record()
            torch.cuda.synchronize()
            ms += ev[0].elapsed_time(ev[1])
        return ms

    for i in range(args.warmup):
        step(1000 + i)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = ctx.stats().kernel_launches
    t_wall0 = time.time()
    dev_ms, rays = 0.0, 0
    for i in range(args.steps):
        dev_ms += step(i)
        rays += ctx.stats().rays
    barrier()
    wall = time.time() - t_wall0
    clocks = sampler.summary()
    launches = ctx.stats().kernel_launches - launches0
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ctx.download_radiance(spp))

    # ---- e2e: the reference-facing C-ABI call sequence with host buffers ---------------------
    e2e_steps = args.steps
    scene_bytes = sum(getattr(sc.desc.contents, n) * C.sizeof(t) for n, t in
                      [("n_hittables", rtb.rt_hittable), ("n_materials", rtb.rt_material), ("n_textures", rtb.rt_texture), ("n_perlins", rtb.rt_perlin)])
    scene_bytes += 4 * sc.desc.contents.n_child_index
    for k in range(sc.desc.contents.n_images):
        scene_bytes += 3 * sc.desc.contents.images[k].width * sc.desc.contents.images[k].height
    ctx.upload_scene(sc.desc)  # untimed warm-up of the host-buffer calls (first-use module loads of the download kernels)
    ctx.render(cam, seed=99, sample_begin=begin, sample_count=min(count, 4), clear=True)
    if rank == 0:
        ctx.download_rgb8(spp)
    barrier()
    t0 = time.time()
    e2e_parts = [0.0, 0.0, 0.0, 0.0]  # upload, render, reduce, download (seconds, this rank)
    for i in range(e2e_steps):
        ta = time.time()
        ctx.upload_scene(sc.desc)  # host scene description -> device (H2D)
        tb = time.time()
        if peer is not None:
            peer.render(i)
            tc = time.time()
        else:
            ctx.render(cam, seed=i, sample_begin=begin, sample_count=count, clear=True)
            ctx.synchronize()
            tc = time.time()
            if world > 1:
                dist.reduce_accum_to_rank0(ctx.accum_tensor())
                torch.cuda.synchronize()
        td = time.time()
        if rank == 0:
            rgb = ctx.download_rgb8(spp)  # finished image -> host (D2H)
        te = time.time()
        for k, dt in enumerate((tb - ta, tc - tb, td - tc, te - td)):
            e2e_parts[k] += dt / e2e_steps
    barrier()
    e2e_sec = (time.time() - t0) / e2e_steps

    # ---- census (instrumented kernel, untimed) for the roofline's algorithmic work -------------
    census = None
    if rank == 0:
        c_spp = max(1, min(16, count))
        ctx.render(cam, seed=0, sample_begin=begin, sample_count=c_spp, clear=True, flags=rtb.RT_RENDER_COUNTERS)
        st = ctx.stats()
        cs = list(st.census)
        r = max(st.rays, 1)
        keys = ["node", "sph", "sph_hit", "quad", "quad_full", "medium", "lambertian", "metal", "dielectric", "light", "isotropic", "checker", "image", "noise", "box"]
        per_ray = {k: cs[i] / r for i, k in enumerate(keys)}
        flops = (2 * F_BOX * per_ray["node"] + F_SPH_MISS * (per_ray["sph"] - per_ray["sph_hit"]) + F_SPH_HIT * per_ray["sph_hit"]
                 + F_QUAD_EARLY * (per_ray["quad"] - per_ray["quad_full"]) + F_QUAD_FULL * per_ray["quad_full"] + F_MEDIUM * per_ray["medium"]
                 + sum(F_SHADE[k] * per_ray[k] for k in ("lambertian", "metal", "dielectric", "light", "isotropic", "checker", "image", "noise"))
                 + F_BOXPRIM * per_ray["box"] + F_SHADE["bounce"])
        nbytes = (B_NODE * per_ray["node"] + B_SPH * per_ray["sph"] + B_QUAD * per_ray["quad"] + B_BOXPRIM * per_ray["box"] + B_TEXEL * per_ray["image"]
                  + B_PERLIN * per_ray["noise"])
        census = dict(per_ray=per_ray, flops_per_ray=flops, bytes_per_ray=nbytes, rays_per_sample=st.rays / max(st.samples, 1))

    # ---- GPU-count invariance: a fixed job (seed 0, sample indices 0..HASH_SPP-1), sharded over the ranks and reduced
    # exactly like a timed step; the FNV-1a of rank 0's int64 accumulator must be the same string in every line --------
    hcam = sc.camera_copy(**dict(over, samples_per_pixel=HASH_SPP))
    if peer is not None:
        peer.render(0, cam=hcam)
    else:
        hb, hc = dist.shard_samples(HASH_SPP, rank, world)
        ctx.render(hcam, seed=0, sample_begin=hb, sample_count=hc, clear=True)
        ctx.synchronize()
        if world > 1:
            dist.reduce_accum_to_rank0(ctx.accum_tensor())
            torch.cuda.synchronize()
    accum_fnv = fnv1a64_words(ctx.download_accum()) if rank == 0 else None
    barrier()

    # ---- the other BASELINE configurations at their own size: sample-sharded over the ranks like the headline job,
    # rendered back to back until the device time exceeds 50 ms (they take 0.3 - 40 ms each) ------------------------
    per_config = []
    if not args.no_per_config:
        for tag, scene_name, cover in PER_CONFIG:
            psc = rtb.Scene(scene_name, rand_seed=1)
            pcam = psc.camera_copy(**cover)
            ctx.upload_scene(psc.desc)
            pb, pc = dist.shard_samples(pcam.samples_per_pixel, rank, world)
            ms_sum, reps, prays = 0.0, 0, 0
            if pc > 0:
                ctx.render(pcam, seed=77, sample_begin=pb, sample_count=pc, clear=True)  # warm-up (module load, clocks)
                ctx.synchronize()
            barrier()
            n_reps = 3
            while True:
                ms_round, rays_round = 0.0, 0
                for r_ in range(n_reps):
                    if pc > 0:
                        ctx.render(pcam, seed=r_, sample_begin=pb, sample_count=pc, clear=True)
                        st_ = ctx.stats()
                        ms_round += st_.last_render_ms
                        rays_round += st_.rays
                t_ = torch.tensor([ms_round, float(rays_round)], dtype=torch.float64, device=f"cuda:{local_rank}")
                if world > 1:
                    mx_ = t_.clone()
                    torch.distributed.all_reduce(mx_, op=torch.distributed.ReduceOp.MAX)
                    sm_ = t_.clone()
                    torch.distributed.all_reduce(sm_, op=torch.distributed.ReduceOp.SUM)
                    ms_round, rays_round = mx_[0].item(), sm_[1].item()
                if ms_round >= 50.0 or n_reps >= 4096:
                    ms_sum, reps, prays = ms_round, n_reps, rays_round
                    break
                n_reps = int(min(4096, max(n_reps * 2, n_reps * 60.0 / max(ms_round, 1e-3))))
            pw, ph = pcam.image_width, rtb.image_height(pcam)
            samples = pw * ph * pcam.samples_per_pixel * reps
            per_config.append({"config": tag, "scene": scene_name, "width": pw, "height": ph, "spp": pcam.samples_per_pixel, "max_depth": pcam.max_depth,
                               "renders": reps, "device_ms_total": round(ms_sum, 3), "ms_per_render": round(ms_sum / reps, 4),
                               "value": samples / (ms_sum * 1e-3), "unit": UNIT, "mrays_per_s": prays / (ms_sum * 1e-3) / 1e6,
                               "timing": "sum of the CUDA-event times of `renders` back-to-back rt_render calls of this rank's sample shard, max over ranks "
                                         "(render only: the 15 MB exchange step is in the headline line)"})
            psc.close()
        ctx.upload_scene(sc.desc)

    # ---- max over ranks -------------------------------------------------------------------------
    vals = torch.tensor([dev_ms, wall * 1e3, e2e_sec * 1e3, float(rays)], dtype=torch.float64, device=f"cuda:{local_rank}")
    if world > 1:
        mx = vals.clone()
        torch.distributed.all_reduce(mx, op=torch.distributed.ReduceOp.MAX)
        sm = vals.clone()
        torch.distributed.all_reduce(sm, op=torch.distributed.ReduceOp.SUM)
        dev_ms, wall_ms, e2e_ms, rays = mx[0].item(), mx[1].item(), mx[2].item(), sm[3].item()
    else:
        wall_ms, e2e_ms = wall * 1e3, e2e_sec * 1e3
    if rank != 0:
        # rank 0 now runs the drop-in leg on ALL devices: wait for it on the host (a NCCL barrier would spin on this GPU)
        ctx.close()
        t_wait = time.time()
        while not os.path.exists(done_flag) and time.time() - t_wait < 900:
            time.sleep(0.05)
        torch.distributed.destroy_process_group()
        return 0

    ms_per_step = dev_ms / args.steps
    total_samples = W * H * spp
    value = total_samples / (ms_per_step * 1e-3)
    rays_per_step = rays / args.steps
    mrays = rays_per_step / (ms_per_step * 1e-3) / 1e6
    hbm_peak, which, sm_max = measured_peaks()
    sm_count = torch.cuda.get_device_properties(local_rank).multi_processor_count
    fp32_peak_tflops = sm_count * 128 * 2 * sm_max * 1e6 / 1e12
    kernel_rays_s = rays_per_step / world / (ms_per_step * 1e-3)  # one launch = one rank's kernel
    ncu, ncu_src = latest_ncu()
    roofline = {"bound": "fp32",
                "bound_note": "FP32/ALU issue under divergence - neither hbm nor tensor: the whole scene is shared-memory / L1 resident and the algorithm "
                              "has no dense contraction (SURVEY.md 8(d)); the hbm view of the same launch is in roofline.hbm",
                "achieved": kernel_rays_s * census["flops_per_ray"] / 1e12, "peak": fp32_peak_tflops, "unit": "TFLOP/s",
                "frac": kernel_rays_s * census["flops_per_ray"] / 1e12 / fp32_peak_tflops,
                "traffic": ncu["dram_bytes_per_sample"] * W * H * count if ncu else None,
                "traffic_note": (f"DRAM bytes per launch = ncu dram__bytes_read+write per sample ({ncu_src}) x this launch's samples; stack/spill write-backs "
                                 "and accumulator adds, not scene data (algorithmic bytes are served by shared memory / L1)") if ncu else ncu_src,
                "simt": ({"issue_slot_utilisation": ncu["issue_slot_utilisation"], "active_lanes_per_instruction": ncu["active_lanes_per_instruction"],
                          "lane_issue_frac": ncu["issue_slot_utilisation"] * ncu["active_lanes_per_instruction"] / 32,
                          "alu_pipe_utilisation": ncu.get("alu_pipe_utilisation"), "fma_pipe_utilisation": ncu.get("fma_pipe_utilisation"),
                          "source": ncu_src} if ncu else None),
                "peak_source": f"{sm_count} SMs x 128 lanes x 2 x {sm_max:.0f} MHz (nominal max clock)",
                "flops_per_ray": census["flops_per_ray"], "bytes_per_ray": census["bytes_per_ray"], "census_per_ray": census["per_ray"],
                "hbm": {"bound": "hbm", "achieved": kernel_rays_s * census["bytes_per_ray"] / 1e9, "peak": hbm_peak, "unit": "GB/s",
                        "frac": kernel_rays_s * census["bytes_per_ray"] / 1e9 / hbm_peak, "peak_source": f"MEASURED_PEAKS.json ({which})",
                        "note": "algorithmic node/primitive/texel bytes; they are served by shared memory and L1, not DRAM"}}
    if clocks.get("sm_mhz"):
        obs = sm_count * 128 * 2 * clocks["sm_mhz"] * 1e6 / 1e12
        roofline["frac_at_observed_clock"] = roofline["achieved"] / obs
    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_per_step,
            "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
            "config": {"workload": f"{args.scene} {W}x{H} x {spp} spp, max_depth {cam.max_depth} (BASELINE config 5: 400 ground boxes, 1000-sphere cluster, "
                                   f"2 volumes, image + noise textures)", "sharding": f"sample index, {world} rank(s), exact int64 reduce to rank 0"
                                   + ("" if world == 1 else (" by our push kernel behind the render (peer red.add.u64 over NVLink, no collective)" if peer is not None else " (ncclInt64)")),
                       "l2": "256 MB device write between timed steps (flush)", "seed": "Philox key = step index"},
            "mrays_per_s": mrays, "rays_per_sample": rays_per_step / total_samples, "wall_ms_per_step": wall_ms / args.steps,
            "e2e": {"value": total_samples / (e2e_ms * 1e-3), "unit": UNIT, "h2d_bytes_per_step": int(scene_bytes), "d2h_bytes_per_step": int(W * H * 3),
                    "steps": e2e_steps, "path": "rt_upload_scene + rt_render + reduce + rt_download(RGB8) with host buffers, wall clock",
                    "rank0_ms": dict(zip(("upload", "render", "reduce", "download"), (round(1e3 * x, 2) for x in e2e_parts)))},
            "gpu_launches": int(launches), "clocks": clocks, "roofline": roofline,
            "accum_fnv": {"value": accum_fnv, "job": f"{args.scene} {W}x{H}, seed 0, sample indices 0..{HASH_SPP - 1}, sharded over {world} rank(s) and reduced like a timed "
                                                     f"step; FNV-1a over the 64-bit words of rank 0's int64 accumulator — equal across n_gpus = the image does not depend on the GPU count"},
            "per_config": per_config, "csrc_sha": csrc_sha()}
    if not args.no_cpu_baseline and world == 1:
        try:
            line["cpu_baseline"] = cpu_baseline(args)
            line["speedup_vs_cpu_baseline_1core"] = line["e2e"]["value"] / line["cpu_baseline"]["value"]
        except Exception as e:  # noqa: BLE001
            line["cpu_baseline"] = {"error": str(e)}
        # the same 1-thread reference figure for C1-C4 (bounded samples, run concurrently: 5 of the box's cores)
        if per_config and os.path.exists(os.path.join(ROOT, "oracle", "_ref", "ref_harness")):
            procs = [(pc_, cpu_reference_once(pc_["scene"], pc_["width"], PER_CONFIG_CPU_SPP[pc_["config"]], seed=1)) for pc_ in per_config]
            for pc_, pr in procs:
                try:
                    j = parse_harness(pr)
                    pc_["cpu_baseline"] = {"value": j["width"] * j["height"] * j["spp"] / j["seconds"], "unit": UNIT, "cores": 1, "kind": "reference",
                                           "sample": f"{j['spp']} spp of {pc_['spp']}, max_depth {j['max_depth']}, harness clock around camera::render"}
                    pc_["speedup_vs_cpu_baseline_1core"] = pc_["value"] / pc_["cpu_baseline"]["value"]
                except Exception as e:  # noqa: BLE001
                    pc_["cpu_baseline"] = {"error": str(e)}
    if not args.no_dropin:
        line["e2e_dropin"] = dropin_leg(args, world, W, H, spp)
    emit(line)
    ctx.close()
    if world > 1:
        open(done_flag, "w").close()
        torch.distributed.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
