"""Census of tests/test_gpu_params.py: every (regime, camera, tracer) case of that file rendered on the GPU and in the
oracle port, one JSON line per case with the GPU's name and power limit and the comparison numbers of
test_gpu_oracle_reach.compare (whether the exact part held, max / p99.9 / p99 of the emission, hdr and rgba differences,
TOUCHED flips, dense_samples difference).  A regime whose numbers exceed the tolerances of test_gpu_oracle_reach.py gets
its own bound in test_gpu_params.py from this output (profiles/params_census_b200.jsonl on a B200).

    python tests/tools/params_census.py [--out profiles/params_census_b200.jsonl]
"""
import argparse
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests"), HERE]


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "params_census_b200.jsonl"))
    args = ap.parse_args()

    import __graft_entry__ as g
    g.build()
    import relativisticraytracer_b200 as rrt
    import test_gpu_params as P
    from oracle import Oracle
    from oracle_reach_census import gpu_identity
    from test_gpu_dof import _renderer
    from test_gpu_oracle_reach import _frame_dicts, compare

    ora = Oracle("port")
    sky_np = rrt.procedural_sky(512, 256, seed=1234, stars=0)      # tests/conftest.py::sky_smooth
    ctxs = {"auto": _renderer("auto"), "scalar": _renderer("scalar")}
    skies = {k: r.create_sky(sky_np) for k, r in ctxs.items()}
    name, limit = gpu_identity()
    with open(args.out, "w") as out:
        for regime, k in P.cases():
            frames = {}
            for tracer, (_, _, flags, _) in P.TRACERS.items():
                if flags not in frames:
                    frames[flags] = P.oracle_frame(ora, sky_np, regime, k, flags)
                gd, _ = P.render_tracer(ctxs, skies, tracer, regime, k)
                cid = f"{P.case_id(regime, k)} {tracer}"
                m, _, _ = compare(P.case_dict(cid), *_frame_dicts(frames[flags], gd))
                m.update({"gpu": name, "power_limit": limit, "regime": regime, "prm": P.REGIMES[regime][0], "tracer": tracer,
                          "flags": flags, "w": P.W, "h": P.H})
                out.write(json.dumps(m) + "\n")
                out.flush()
                print(cid, "exact" if not m["exact_bad"] else f"EXACT DIFFERS {m['exact_bad']}",
                      "emis max %.2e p999 %.2e p99 %.2e" % tuple(m["emis_rel"][q] for q in ("max", "p999", "p99")),
                      "hdr max %.2e p999 %.2e p99 %.2e" % tuple(m["hdr_rel"][q] for q in ("max", "p999", "p99")),
                      "rgba max %d" % m["rgba_diff"]["max"], "flips", m["touched_flips"], "dense", m["dense_samples_diff"], flush=True)


if __name__ == "__main__":
    main()
