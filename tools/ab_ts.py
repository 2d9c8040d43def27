"""Same-box A/B of InfoNCE kernel builds at the headline shape (B = 64, D = 512, 256 x 256, K = 256): each arm is a library and
the rc_infonce_bf16 flags it is called with, timed in a fresh process by tools/ablate_pair.py's child (7 single-launch CUDA
event timings after 3 warm-up launches); the arms alternate for ROUNDS rounds so that clock and neighbour drift spread over all
of them.

    python tools/ab_ts.py ROUNDS NAME=LIB[:FLAGS] ...      # e.g. ss=old.so:0 ts=new.so:8
"""
import json
import os
import statistics
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def main():
    rounds = int(sys.argv[1])
    arms = []
    for a in sys.argv[2:]:
        name, spec = a.split("=", 1)
        lib, _, flags = spec.partition(":")
        arms.append((name, os.path.abspath(lib), flags or "0"))
    res = {n: [] for n, _, _ in arms}
    for r in range(rounds):
        for name, lib, flags in arms:
            p = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "ablate_pair.py"), "child"], capture_output=True, text=True,
                               timeout=600, env=dict(os.environ, RC_AB_LIB=lib, RC_AB_FLAGS=flags, RANGECLIP_B200_ABLATE="0"))
            if p.returncode != 0:
                raise SystemExit(f"{name}: {p.stderr[-800:]}")
            line = json.loads(p.stdout.strip().splitlines()[-1])
            res[name].append(line["ms_med"])
            print(json.dumps({"round": r, "arm": name, "flags": int(flags), **line}), flush=True)
    summary = {n: {"ms_median": statistics.median(v), "ms_min": min(v), "ms_max": max(v), "spread_ms": max(v) - min(v), "runs": v}
               for n, v in res.items()}
    print(json.dumps({"summary": summary}))


if __name__ == "__main__":
    main()
