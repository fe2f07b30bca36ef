"""Appending training points (GPR.add_points -> gprc_gpr_append) against refitting the concatenated data, on the C4
generator (d = 8, sqrexp l = 1, noise 0.01).

For n in {8192, 50000} and batches k in {1, 32, 128, 1024, 20000}: one warm-up append of the same shapes on a fresh model,
then the timed append on another fresh model (CUDA events on the library's stream around the call, which ends in a
device synchronise), and a warm-up + timed refit of all n + k points.  The appended model is checked against the refit
(logp, alpha).  At n = 8192 also a loop of 100 single-point appends (ms per append).  The card's name, power limit and
max SM clock are read in the same process.  Writes one JSON file (default profiles/append_probe.json).

    python tools/append_probe.py [--out PATH] [--n 8192 50000] [--k 1 32 128 1024 20000]
"""
import argparse
import json
import math
import os
import subprocess
import sys
import time

import numpy as np

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import gprc_b200 as g  # noqa: E402


def c4(n):
    rng = np.random.default_rng(4)
    X = rng.uniform(-1, 1, size=(8, n))
    y = np.sum(np.sin(math.pi * X), axis=0) + rng.normal(0, 0.1, n)
    return X, y


def card():
    out = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv"],
                         capture_output=True, text=True).stdout.strip().splitlines()
    return out[1] if len(out) > 1 else "unknown"


def timed(ctx, fn):
    """device time (ms) of fn() between two events on the library's stream, and the host wall time (ms)"""
    ctx.sync()
    t0 = time.perf_counter()
    ctx.mark(0)
    out = fn()
    ctx.mark(1)
    ctx.sync()
    wall = (time.perf_counter() - t0) * 1e3
    return out, ctx.elapsed_ms(0, 1), wall


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join("profiles", "append_probe.json"))
    ap.add_argument("--n", type=int, nargs="+", default=[8192, 50000])
    ap.add_argument("--k", type=int, nargs="+", default=[1, 32, 128, 1024, 20000])
    ap.add_argument("--loop", type=int, default=100, help="single-point appends at the smallest n")
    args = ap.parse_args()
    ctx = g.default_context()
    kern = g.cov_func(g.sqrexp, l=1.0)
    noise = 0.01
    X, y = c4(max(args.n) + max(args.k) + args.loop)
    rows = []
    result = dict(card=card(), generator="C4: d = 8, sqrexp l = 1, noise 0.01", rows=rows)
    print("card:", result["card"], flush=True)
    for n in args.n:
        for k in args.k:
            Xa, ya = X[:, :n + k], y[:n + k]
            for rep in range(2):  # rep 0 warms up the shapes
                m = g.GPR(Xa[:, :n], ya[:n], noise, kern, ctx=ctx)
                ctx.reset_timers()
                _, ms, wall = timed(ctx, lambda: m.add_points(Xa[:, n:], ya[n:]))
                phases, _ = ctx.timers()
                lp, alpha = m.logp[0, 0], m.alpha.copy()
                del m
            for rep in range(2):
                ref, ms_refit, wall_refit = timed(ctx, lambda: g.GPR(Xa, ya, noise, kern, ctx=ctx))
                lp_ref, alpha_ref = ref.logp[0, 0], ref.alpha.copy()
                del ref
            row = dict(n=n, k=k, append_ms=ms, append_wall_ms=wall, refit_ms=ms_refit, refit_wall_ms=wall_refit,
                       speedup=ms_refit / ms, append_phases_ms=dict(build_k=phases["build_k"], chol=phases["chol"],
                                                                  solve=phases["solve"]),
                       logp_rel_diff=abs(lp - lp_ref) / abs(lp_ref),
                       alpha_rel_diff=float(np.max(np.abs(alpha - alpha_ref)) / np.max(np.abs(alpha_ref))))
            rows.append(row)
            print(json.dumps(row), flush=True)
            assert row["logp_rel_diff"] <= 1e-10 and row["alpha_rel_diff"] <= 1e-8, row
    n = min(args.n)
    for rep in range(2):  # rep 0 warms up
        m = g.GPR(X[:, :n], y[:n], noise, kern, ctx=ctx)

        def loop():
            for i in range(n, n + args.loop):
                m.add_points(X[:, i], y[i:i + 1])

        _, ms, wall = timed(ctx, loop)
        lp, alpha = m.logp[0, 0], m.alpha.copy()
        del m
    ref = g.GPR(X[:, :n + args.loop], y[:n + args.loop], noise, kern, ctx=ctx)
    loop_row = dict(n=n, appends=args.loop, ms_per_append=ms / args.loop, wall_ms_per_append=wall / args.loop,
                    logp_rel_diff=abs(lp - ref.logp[0, 0]) / abs(ref.logp[0, 0]),
                    alpha_rel_diff=float(np.max(np.abs(alpha - ref.alpha)) / np.max(np.abs(ref.alpha))))
    result["single_point_loop"] = loop_row
    print(json.dumps(loop_row), flush=True)
    assert loop_row["logp_rel_diff"] <= 1e-10 and loop_row["alpha_rel_diff"] <= 1e-8, loop_row
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    with open(args.out, "w") as f:
        json.dump(result, f, indent=1)
    print("wrote", args.out)


if __name__ == "__main__":
    main()
