"""Batch of views against a loop of single renders, on one GPU: python tools/views_bench.py DIR

Writes DIR/views_bench.json (raw numbers) and DIR/r4_views.md (the table of DESIGN §7).
  * BASELINE scenes at their BASELINE sizes and spp, V in {1, 8, 64} views on an orbit about the scene's lookat: one
    rt_render_views call against V back-to-back rt_render calls, warm, scene uploaded once.  Times: the library's CUDA
    events around the batch (rt_stats.last_render_ms), and host wall time from the first enqueue to the end of a
    stream synchronise for both forms (the loop's launch gaps are part of what a batch saves).  Median of REPS
    alternating repeats.  At V = 8 the batch's sums are compared with the loop's, bit for bit.
  * book2_final (the headline scene) at 800 x 800 and a reduced spp: a V = 1 batch against rt_render, CUDA events —
    the cost of the batch instantiation on that scene.
  * tests/cpp/views_main.cpp built like the drop-in test builds it: process wall time for 64 frames, one
    rtb200::render_views call against a loop of camera::render.
The device name and power limit are read in the same run."""
import importlib
import json
import math
import os
import statistics
import subprocess
import sys
import tempfile
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
rtb = importlib.import_module("raytracing-practice_b200")

REPS = int(os.environ.get("VIEWS_REPS", "5"))
# BASELINE.json configs: C1 book1_final, C2 bouncing_spheres, C3 earth (+ perlin_sphere, the noise path), C4 cornell_smoke
SCENES = [("earth", 400, 100), ("bouncing_spheres", 400, 100), ("perlin_sphere", 400, 100), ("book1_final", 1200, 10), ("cornell_smoke", 600, 200)]
VIEWS = [1, 8, 64]


def device_info():
    import torch

    info = {"device": torch.cuda.get_device_name(0)}
    try:
        out = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit,clocks.max.sm", "--format=csv,noheader,nounits"],
                             capture_output=True, text=True, timeout=30).stdout.strip().split(",")
        info["power_limit_w"], info["sm_max_mhz"] = float(out[0]), float(out[1])
    except Exception as e:  # recorded, not guessed
        info["power_limit_w"] = f"unavailable: {e}"
    return info


def orbit(sc, n, width, spp):
    base = sc.cam.contents
    at = np.array(base.lookat[:])
    r = np.array(base.lookfrom[:]) - at
    cams = []
    for v in range(n):
        a = 2.0 * math.pi * v / n
        c, s = math.cos(a), math.sin(a)
        cams.append(sc.camera_copy(image_width=width, samples_per_pixel=spp, lookfrom=tuple(at + np.array([c * r[0] + s * r[2], r[1], -s * r[0] + c * r[2]]))))
    return cams


def timed(fn, ctx):
    t0 = time.perf_counter()
    fn()
    ctx.synchronize()
    return (time.perf_counter() - t0) * 1e3


def scene_rows(ctx):
    rows = []
    for name, width, spp in SCENES:
        sc = rtb.Scene(name, rand_seed=1)
        ctx.upload_scene(sc.desc)
        for V in VIEWS:
            cams = orbit(sc, V, width, spp)

            def loop():
                for cam in cams:
                    ctx.render(cam, seed=1)

            def batch():
                ctx.render_views(cams, seed=1)

            loop(), ctx.synchronize(), batch(), ctx.synchronize()  # warm: modules, kernel attributes, accumulator shapes
            bw, be, lw = [], [], []
            for _ in range(REPS):
                bw.append(timed(batch, ctx))
                be.append(ctx.stats().last_render_ms)
                lw.append(timed(loop, ctx))
            row = dict(scene=name, width=width, height=rtb.image_height(cams[0]), spp=spp, views=V, batch_event_ms=statistics.median(be),
                       batch_wall_ms=statistics.median(bw), loop_wall_ms=statistics.median(lw), batch_wall_all=bw, loop_wall_all=lw)
            row["speedup_wall"] = row["loop_wall_ms"] / row["batch_wall_ms"]
            if V == 8:  # the timed sizes, bit for bit
                batch()
                acc = ctx.download_accum()
                same = True
                for v, cam in enumerate(cams):
                    ctx.render(cam, seed=1)
                    same = same and np.array_equal(ctx.download_accum(), acc[v])
                row["bit_identical"] = bool(same)
            print(json.dumps({k: v for k, v in row.items() if not k.endswith("_all")}), flush=True)
            rows.append(row)
        sc.close()
    return rows


def headline(ctx, spp=64):
    sc = rtb.Scene("book2_final", rand_seed=1)
    ctx.upload_scene(sc.desc)
    cam = sc.camera_copy(image_width=800, samples_per_pixel=spp)
    ctx.render(cam, seed=1), ctx.render_views([cam], seed=1), ctx.synchronize()
    single, batch = [], []
    for _ in range(REPS):
        ctx.render(cam, seed=1)
        single.append(ctx.stats().last_render_ms)
        ctx.render_views([cam], seed=1)
        batch.append(ctx.stats().last_render_ms)
    acc = ctx.download_accum()[0]
    ctx.render(cam, seed=1)
    row = dict(scene="book2_final", width=800, height=800, spp=spp, render_ms=statistics.median(single), views1_ms=statistics.median(batch),
               render_all=single, views1_all=batch, bit_identical=bool(np.array_equal(acc, ctx.download_accum())))
    row["ratio"] = row["views1_ms"] / row["render_ms"]
    print(json.dumps({k: v for k, v in row.items() if not k.endswith("_all")}), flush=True)
    sc.close()
    return row


def cpp_rows(frames=64, scene="bouncing_spheres", width=400, spp=100):
    host = os.path.join(ROOT, "raytracing-practice_b200", "host")
    libdir = os.path.dirname(rtb.CUDA_LIB_PATH)
    with tempfile.TemporaryDirectory() as tmp:
        exe = os.path.join(tmp, "views")
        subprocess.run(["g++", "-std=c++11", "-O1", "-I", host, "-I", os.path.join(ROOT, "include"), os.path.join(ROOT, "tests", "cpp", "views_main.cpp"),
                        "-L", libdir, "-lrt_b200", "-Wl,-rpath," + libdir, "-o", exe], check=True)
        env = dict(os.environ, RT_B200_DEVICES="0")
        times = {"loop": [], "batch": []}
        files = {}
        for _ in range(3):
            for mode in ("loop", "batch"):
                prefix = os.path.join(tmp, mode)
                t0 = time.perf_counter()
                subprocess.run([exe, scene, prefix, str(width), str(spp), str(frames), mode], check=True, env=env, stdout=subprocess.DEVNULL)
                times[mode].append(time.perf_counter() - t0)
                files[mode] = [open(f"{prefix}_{i:03d}.ppm", "rb").read() for i in range(frames)]
        row = dict(scene=scene, width=width, spp=spp, frames=frames, loop_s=statistics.median(times["loop"]), batch_s=statistics.median(times["batch"]),
                   loop_all=times["loop"], batch_all=times["batch"], files_identical=files["loop"] == files["batch"])
    print(json.dumps({k: v for k, v in row.items() if not k.endswith("_all")}), flush=True)
    return row


def table(info, rows, head, cpp):
    lines = [f"# A batch of views against a loop of single renders ({info['device']}, power limit {info.get('power_limit_w')} W)", "",
             "`python tools/views_bench.py DIR`; raw numbers in `profiles/logs/views_bench.json`.  Median of "
             f"{REPS} alternating repeats, warm, scene uploaded once.  Views orbit the scene's lookat.", "",
             "| scene | size | spp | V | batch (events) ms | batch (wall) ms | loop of V rt_render (wall) ms | loop / batch |",
             "|---|---|---|---|---|---|---|---|"]
    for r in rows:
        lines.append(f"| {r['scene']} | {r['width']}x{r['height']} | {r['spp']} | {r['views']} | {r['batch_event_ms']:.2f} | {r['batch_wall_ms']:.2f} | "
                     f"{r['loop_wall_ms']:.2f} | {r['speedup_wall']:.3f} |")
    lines += ["", "At V = 8 the batch's int64 sums equal the loop's, bit for bit: " +
              ", ".join(f"{r['scene']} {'yes' if r.get('bit_identical') else 'NO'}" for r in rows if r["views"] == 8) + ".", "",
              f"Headline scene, one view: book2_final {head['width']}x{head['height']} at {head['spp']} spp — rt_render {head['render_ms']:.2f} ms, "
              f"rt_render_views (V = 1) {head['views1_ms']:.2f} ms (ratio {head['ratio']:.3f}; same bits: {head['bit_identical']}).", "",
              f"C++ drop-in, process wall time for {cpp['frames']} frames of {cpp['scene']} {cpp['width']} px at {cpp['spp']} spp: "
              f"loop of camera::render {cpp['loop_s']:.2f} s, one rtb200::render_views {cpp['batch_s']:.2f} s "
              f"(files identical: {cpp['files_identical']})."]
    return "\n".join(lines) + "\n"


def main():
    if len(sys.argv) != 2:
        print(__doc__)
        sys.exit(2)
    out = sys.argv[1]
    os.makedirs(out, exist_ok=True)
    info = device_info()
    print(json.dumps(info), flush=True)
    ctx = rtb.Context(0)
    rows = scene_rows(ctx)
    head = headline(ctx)
    ctx.close()
    cpp = cpp_rows()
    with open(os.path.join(out, "views_bench.json"), "w") as f:
        json.dump(dict(info, reps=REPS, scenes=rows, headline=head, cpp=cpp), f, indent=1)
    with open(os.path.join(out, "r4_views.md"), "w") as f:
        f.write(table(info, rows, head, cpp))


if __name__ == "__main__":
    main()
