"""bench.py's reference arm (`--impl reference`) needs no GPU: it times the unmodified reference's camera::render
(oracle/_ref, or the oracle port where the reference was not compiled) on the host cores.  This pins the JSON line the
driver parses; the GPU arm's line carries the same keys plus roofline / clocks (checked on the GPU box by the driver)."""
import json
import os
import subprocess
import sys

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def run_arm(env_extra=None):
    env = dict(os.environ, **(env_extra or {}))
    r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), "--impl", "reference", "--steps", "1", "--warmup", "0", "--width", "40"],
                       capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    return [l for l in r.stdout.splitlines() if l.strip()]


def test_reference_arm_prints_one_json_line_with_the_contract_keys():
    lines = run_arm()
    assert len(lines) == 1
    d = json.loads(lines[0])
    assert d["impl"] == "reference" and d["metric"] == "samples_px_per_s" and d["unit"] == "samples*px/s"
    assert d["higher_is_better"] is True and d["vs_baseline"] is None and d["n_gpus"] == 1 and d["steps"] == 1 and d["warmup"] == 0
    assert d["value"] > 0 and d["ms_per_step"] > 0 and "workload" in d["config"] and "model" not in d["config"]
    cb = d["cpu_baseline"]
    assert cb["kind"] in ("reference", "port") and cb["cores"] >= 1 and cb["value"] == d["value"] and cb["sample"]
    assert d["e2e"] == {"value": d["value"], "unit": d["unit"], "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}
    assert d["gpu_launches"] == 0  # nothing of ours runs in the reference arm


def test_reference_arm_other_ranks_exit_quietly():
    assert run_arm({"RANK": "1", "WORLD_SIZE": "2"}) == []


def test_steps_and_dump_arguments_are_checked():
    for bad in (["--steps", "0"], ["--warmup", "-1"], ["--impl", "reference", "--dump-outputs", "x"]):
        r = subprocess.run([sys.executable, os.path.join(ROOT, "bench.py"), *bad], capture_output=True, text=True, timeout=60)
        assert r.returncode == 2 and r.stdout == "", (bad, r.stderr[-500:])


def test_dump_outputs_writes_the_image_or_a_fixed_sample_of_it(tmp_path, monkeypatch):
    import numpy as np

    sys.path.insert(0, ROOT)
    import bench

    img = np.random.default_rng(1).random((30, 40, 3), dtype=np.float32)
    bench.dump_outputs(str(tmp_path / "whole"), img)
    assert sorted(os.listdir(tmp_path / "whole")) == ["radiance.npy"]
    assert np.array_equal(np.load(tmp_path / "whole" / "radiance.npy"), img)
    monkeypatch.setattr(bench, "DUMP_LIMIT", 4096 + 20 * 100)  # room for 100 of the 1200 pixels
    for run in ("a", "b"):
        bench.dump_outputs(str(tmp_path / run), img)
        assert sum(os.path.getsize(tmp_path / run / f) for f in os.listdir(tmp_path / run)) <= bench.DUMP_LIMIT
    idx = np.load(tmp_path / "a" / "pixel_index.npy")
    rad = np.load(tmp_path / "a" / "radiance.npy")
    assert idx.dtype == np.float64 and rad.dtype == np.float32 and rad.shape == (100, 3) and np.all(np.diff(idx) > 0)
    assert np.array_equal(rad, img.reshape(-1, 3)[idx.astype(np.int64)])
    assert np.array_equal(idx, np.load(tmp_path / "b" / "pixel_index.npy"))


@pytest.mark.gpu
def test_dumped_image_is_the_last_timed_step(rtb, gpu_ctx, tmp_path):
    """--dump-outputs writes what the timed path computed in its last step (seed = step index, so steps - 1).  The e2e leg
    that follows renders the same seeds, so the order of the renders and the dump is recorded too: the dump must come
    straight after the warm-up and the timed renders."""
    import numpy as np

    wrapper = (
        "import importlib, json, sys\n"
        f"sys.path.insert(0, {ROOT!r})\n"
        "import bench\n"
        "rtb = importlib.import_module('raytracing-practice_b200')\n"
        "calls, render, dump = [], rtb.Context.render, bench.dump_outputs\n"
        "def rec_render(self, cam, seed=0, **kw):\n"
        "    calls.append(['render', seed])\n"
        "    return render(self, cam, seed=seed, **kw)\n"
        "def rec_dump(*a):\n"
        "    calls.append(['dump'])\n"
        "    return dump(*a)\n"
        "rtb.Context.render, bench.dump_outputs = rec_render, rec_dump\n"
        "rc = bench.main()\n"
        "sys.stderr.write('CALLS ' + json.dumps(calls) + '\\n')\n"
        "sys.exit(rc)\n")
    r = subprocess.run([sys.executable, "-c", wrapper, "--steps", "3", "--warmup", "1", "--spp", "24", "--width", "64",
                        "--no-per-config", "--no-dropin", "--no-cpu-baseline", "--dump-outputs", str(tmp_path)],
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0, r.stderr[-2000:]
    assert json.loads(r.stdout)["steps"] == 3
    calls = json.loads([l for l in r.stderr.splitlines() if l.startswith("CALLS ")][-1][6:])
    assert calls[:5] == [["render", 1000], ["render", 0], ["render", 1], ["render", 2], ["dump"]], calls[:8]
    assert ["render", 2] in calls[5:]  # the e2e leg renders seed 2 again: only the order above tells the two apart
    sc = rtb.Scene("book2_final", rand_seed=1)
    cam = sc.camera_copy(image_width=64, samples_per_pixel=24)
    gpu_ctx.upload_scene(sc.desc)
    gpu_ctx.render(cam, seed=2)
    assert np.array_equal(np.load(tmp_path / "radiance.npy"), gpu_ctx.download_radiance(24))


def test_ncu_figures_are_tied_to_the_kernel_code_not_to_its_comments(tmp_path, monkeypatch):
    """bench.py quotes DRAM traffic / issue utilisation / active lanes only from an ncu capture of THESE kernels
    (profiles/latest_ncu.json carries a hash of csrc/ with comments and whitespace removed): rewording a comment keeps the
    figures, changing a token drops them."""
    import importlib
    import sys

    sys.path.insert(0, ROOT)
    mod = importlib.import_module("raytracing-practice_b200.csrc_sha")
    a = "int f(int x) { // add one\n  return x + 1; /* here */ }\n"
    b = "int f(int x) {   // plus one, reworded\n\n  return x + 1; }\n"
    c = "int f(int x) { return x + 2; }\n"
    assert mod._code_only(a) == mod._code_only(b) != mod._code_only(c)
    assert mod._code_only('const char* s = "// not a comment";') == 'const char* s = "// not a comment";'
    import bench

    ncu, src = bench.latest_ncu()
    if ncu is not None:  # the committed capture matches the tree: its keys are the ones bench.py reads
        assert ncu["csrc_sha"] == bench.csrc_sha() and ncu["dram_bytes_per_sample"] > 0 and 0 < ncu["issue_slot_utilisation"] <= 1
    else:
        assert "omitted" in src or "missing" in src
