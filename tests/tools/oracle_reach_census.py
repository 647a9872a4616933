"""Census of tests/test_gpu_oracle_reach.py: every case of that file rendered on the GPU and in the oracle port, one JSON line
per case with the GPU's name and power limit, the max / p99.9 / p99 of the emission, hdr and rgba differences, the TOUCHED
flag and dense_samples differences, whether the exact part held, and the wall time of both sides.  The tolerances of the
test file are set from its output (profiles/oracle_reach_census_b200.jsonl on a B200).

    python tests/tools/oracle_reach_census.py [--sections 1,2,3,4] [--out profiles/oracle_reach_census_b200.jsonl]
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]


def gpu_identity():
    import torch
    name = torch.cuda.get_device_name(0)
    try:
        limit = subprocess.run(["nvidia-smi", "-i", "0", "--query-gpu=power.limit", "--format=csv,noheader"],
                               capture_output=True, text=True, timeout=30).stdout.strip()
    except (OSError, subprocess.TimeoutExpired):
        limit = "unknown"
    return name, limit


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--sections", default="1,2,3,4")
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "oracle_reach_census_b200.jsonl"))
    args = ap.parse_args()
    want = {int(s) for s in args.sections.split(",")}

    import __graft_entry__ as g
    g.build()
    import relativisticraytracer_b200 as rrt
    import test_gpu_oracle_reach as R
    from oracle import Oracle

    gpu, ora = rrt.Renderer(0), Oracle("port")
    sky = rrt.procedural_sky(512, 256, seed=1234, stars=0)      # tests/conftest.py::sky_smooth
    name, limit = gpu_identity()
    ora_threads = ora.num_threads()
    # the oracle's share of the wall time: whole-frame renders, and the row renders (side by side) of the full-size frames
    spent = [0.0]

    def timed(fn):
        def run(*a, **k):
            t = time.perf_counter()
            try:
                return fn(*a, **k)
            finally:
                spent[0] += time.perf_counter() - t
        return run
    ora_render, R.oracle_rows = ora.render, timed(R.oracle_rows)
    ora.render = lambda *a, **k: (timed(ora_render) if threading.current_thread() is threading.main_thread() else ora_render)(*a, **k)
    with open(args.out, "w") as out:
        for c in R.all_cases():
            if c["section"] not in want:
                continue
            t0, spent[0] = time.perf_counter(), 0.0
            f, gg = R.run_case(gpu, ora, sky, c)
            wall = time.perf_counter() - t0
            m, _, _ = R.compare(c, f, gg)
            m.update({"gpu": name, "power_limit": limit, "lib": os.path.basename(rrt._capi.LIB_PATH), "host_cores": os.cpu_count(),
                      "oracle_threads": ora_threads, "wall_s": round(wall, 3), "oracle_s": round(spent[0], 3), "w": c["w"], "h": c["h"], "flags": c["flags"],
                      "fx": c["fx"], "prm": c["prm"]})
            out.write(json.dumps(m) + "\n")
            out.flush()
            print(c["id"], "exact" if not m["exact_bad"] else f"EXACT DIFFERS {m['exact_bad']}",
                  "emis max %.2e" % m["emis_rel"]["max"], "hdr max %.2e" % m["hdr_rel"]["max"], "rgba max %d" % m["rgba_diff"]["max"],
                  "flips", m["touched_flips"], "%.1fs" % wall, flush=True)


if __name__ == "__main__":
    main()
