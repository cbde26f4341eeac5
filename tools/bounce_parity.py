"""Measures what tests/test_gpu_bounce.py gates: the start-primitive rules on adversarial start points (part a), the
render kernel's bounce segment against the oracle on every scene at full size and on the constructed scenes (part b),
and every megakernel plan against the default one (part c).  Writes DIR/bounce_parity.json and prints a summary;
profiles/r3_bounce_parity.md is the table made from it.   python tools/bounce_parity.py DIR"""
import importlib
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))
import conftest  # noqa: E402,F401  (sets RTW_IMAGES as the tests do)
import test_gpu_bounce as tb  # noqa: E402
from oracle import orc  # noqa: E402

rtb = importlib.import_module("raytracing-practice_b200")


def main(out_dir):
    os.makedirs(out_dir, exist_ok=True)
    gpu = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit", "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    res = dict(gpu=gpu, leaf={}, bounce={}, plans={})
    ctx = rtb.Context(0)
    t0 = time.time()
    for (ty, cls), r in tb.leaf_rule_table(rtb, orc, ctx).items():
        res["leaf"][f"{ty}/{cls}"] = r
        print("leaf", ty, cls, r, flush=True)
    res["leaf_seconds"] = time.time() - t0
    for name in tb.ALL_SCENES:
        t0 = time.time()
        sc = rtb.Scene(name, rand_seed=1)
        r = tb.bounce_parity(rtb, orc, ctx, sc.desc, sc.camera_copy())
        r["seconds"] = time.time() - t0
        res["bounce"][name] = r
        print("bounce", name, r, flush=True)
    for name, s, desc, cam in tb.constructed_scenes():
        t0 = time.time()
        r = tb.bounce_parity(rtb, orc, ctx, desc, cam)
        r["seconds"] = time.time() - t0
        res["bounce"][name] = r
        print("bounce", name, r, flush=True)
    ctx.close()
    for name in tb.PLAN_SCENES:
        t0 = time.time()
        out = tb.plan_outputs(rtb, name)
        ref = out["default"]
        rep = {}
        for plan, r in out.items():
            rep[plan] = dict(accum_diff=int((r["accum"] != ref["accum"]).sum()), rays=int(r["rays"]), rays_ref=int(ref["rays"]))
            if "aov" in r:
                rep[plan]["aov_diff"] = {k: int((a != ref["aov"][k]).reshape(a.shape[0], a.shape[1], -1).any(axis=2).sum()) for k, a in r["aov"].items()}
        rep["census"] = out["counters"]["census"].tolist()
        rep["seconds"] = time.time() - t0
        res["plans"][name] = rep
        print("plans", name, rep, flush=True)
    with open(os.path.join(out_dir, "bounce_parity.json"), "w") as f:
        json.dump(res, f, indent=1)


if __name__ == "__main__":
    if len(sys.argv) != 2:
        sys.exit("usage: python tools/bounce_parity.py DIR")
    main(sys.argv[1])
