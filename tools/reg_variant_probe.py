"""Times the condensed register-kernel builds (reg_variant 4 and 5) on the C2 batch, 4096 LPs of 64 x 128,
alternating them, and writes the result as JSON (run on a B200):

    python tools/reg_variant_probe.py OUT.json [rounds]

CUDA events around `reps` back-to-back launches per round; the card's name, power limit and max SM clock are
read in the same run and stored with the numbers."""
import json
import os
import subprocess
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tools"))
import gpu_probe as G  # noqa: E402


def main():
    out = sys.argv[1]
    rounds = int(sys.argv[2]) if len(sys.argv) > 2 else 5
    card = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                          capture_output=True, text=True).stdout.strip()
    runs = []
    for rnd in range(rounds):
        for rv in (4, 5):
            r = G.time_batched(G.F.KERNEL_CTA_REG, reg_variant=rv, reps=20)
            r["round"] = rnd
            runs.append(r)
            print(json.dumps(r), flush=True)
    summary = {}
    for rv in (4, 5):
        ms = sorted(r["ms"] for r in runs if r["reg_variant"] == rv)
        summary[f"reg_variant_{rv}"] = dict(ms_median=ms[len(ms) // 2], ms_min=ms[0], ms_max=ms[-1],
                                            pivots_per_batch=runs[0]["pivots"])
    doc = dict(what="reg_simplex_kernel, condensed builds, C2 batch (4096 LPs, 64 x 128, seed 1), ms per batch",
               card=card, reps_per_round=20, summary=summary, runs=runs)
    with open(out, "w") as f:
        json.dump(doc, f, indent=1)
    print(json.dumps(summary), flush=True)


if __name__ == "__main__":
    main()
