#!/usr/bin/env python3
"""Compressible against plain witness slots, alternated: each pair runs bench.py with the shipped library (compressible slots) and
then the same bench.py through the TUNING library with POB_PLAIN_SLOTS=1 (plain slots; otherwise the same code).  Extra arguments
go to bench.py.  Prints each run's JSON line tagged with its arm, then the per-pair ratios and the spread of each arm.

    python tools/slots_ab.py --pairs 3 -- --no-cpu-baseline
"""
import argparse, json, os, subprocess, sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
TUNING = os.path.join(ROOT, "proof-of-burn_b200", "pob_b200", "libpob_b200_tuning.so")
# bench.py unchanged, only the library it loads is the tuning build
PLAIN = ("import runpy, sys; sys.path.insert(0, %r); import pob_b200; pob_b200.LIB_PATH = %r; sys.argv = ['bench.py'] + sys.argv[1:]; "
         "runpy.run_path(%r, run_name='__main__')" % (os.path.join(ROOT, "proof-of-burn_b200"), TUNING, os.path.join(ROOT, "bench.py")))


def run(arm, extra):
    env = dict(os.environ)
    if arm == "compressible":
        cmd = [sys.executable, os.path.join(ROOT, "bench.py")] + extra
    else:
        cmd, env["POB_PLAIN_SLOTS"] = [sys.executable, "-c", PLAIN] + extra, "1"
    out = subprocess.run(cmd, cwd=ROOT, env=env, capture_output=True, text=True, timeout=1800)
    lines = [l for l in out.stdout.splitlines() if l.startswith("{")]
    if out.returncode != 0 or not lines:
        sys.stderr.write(out.stderr[-3000:])
        raise SystemExit("%s arm failed (rc %d)" % (arm, out.returncode))
    r = json.loads(lines[-1])
    print(json.dumps({"arm": arm, **r}), flush=True)
    return r


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=3)
    ap.add_argument("extra", nargs="*", help="arguments for bench.py (after --)")
    a = ap.parse_args()
    vals = {"compressible": [], "plain": []}
    for _ in range(a.pairs):
        for arm in ("compressible", "plain"):
            vals[arm].append(run(arm, a.extra)["value"])
    ratios = [c / p for c, p in zip(vals["compressible"], vals["plain"])]
    print(json.dumps({"summary": {arm: {"values": v, "min": min(v), "max": max(v), "spread": (max(v) - min(v)) / min(v)} for arm, v in vals.items()},
                      "ratio_per_pair": ratios, "compressible_faster_in_every_pair": all(r > 1 for r in ratios)}))


if __name__ == "__main__":
    main()
