"""Semi-global mode on the config-2 batch, timed against global mode in the same process.

For each scoring (1/-1/-1 and 2/-3/-4) the 1 M-pair config-2 batch (workload.config2, seed 481) runs in two ways, global and
semi-global alternating, `--reps` times each:
  device-resident  b2a_batch_upload once, then b2a_batch_run: CUDA-event fill and traceback times (kernels only);
  end to end       b2a_align_batch from host memory with the op lists kept on the device (copies included).
A seeded sample of 2 000 semi-global pairs is checked against the semi-global oracle (tests/semiglobal_oracle.c) in the same run.
Prints one JSON document (GPU name and power limit included) and writes it to --out if given.

    python scripts/semiglobal_bench.py [--pairs 1000000] [--reps 5] [--out FILE]
"""
import argparse
import json
import os
import random
import statistics
import subprocess
import sys
import time

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path[:0] = [ROOT, os.path.join(ROOT, "tests")]

from __graft_entry__ import load_package  # noqa: E402

pkg = load_package()
from bioinformatics_algorithms_b200 import workload  # noqa: E402
import semiglobal_oracle as sg  # noqa: E402


def gpu_info():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader", "-i", "0"],
                       capture_output=True, text=True)
    name, power, clk = ([x.strip() for x in q.stdout.strip().split(",")] + ["?", "?", "?"])[:3]
    return {"gpu": name, "power_limit": power, "max_sm_clock": clk}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--pairs", type=int, default=1_000_000)
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--sample", type=int, default=2000)
    ap.add_argument("--out")
    a = ap.parse_args()
    eng = pkg.Engine(0)
    pat, po, txt, to = workload.config2(a.pairs, seed=481)
    cells = int(((po[1:] - po[:-1]).astype("int64") * (to[1:] - to[:-1]).astype("int64")).sum())
    out = dict(gpu_info(), pairs=a.pairs, cells=cells, reps=a.reps, workload="config2 seed 481 (150 x 1000)", runs={})
    modes = {"global": pkg.GLOBAL, "semiglobal": pkg.SEMIGLOBAL}
    for s in ((1, -1, -1), (2, -3, -4)):
        key = "%d/%d/%d" % s
        t = {m: {"fill_ms": [], "tb_ms": [], "device_ms": [], "e2e_ms": []} for m in modes}
        for m, md in modes.items():                                  # warm-up of every shape and kernel the timed window uses
            eng.upload(md, pat, po, txt, to, *s, want_ops=True); eng.run()
            eng.align_packed(md, pat, po, txt, to, *s, want_ops=True)
        for _ in range(a.reps):
            for m, md in modes.items():
                eng.upload(md, pat, po, txt, to, *s, want_ops=True)
                eng.run()
                f, tb, tot = eng.times()
                t[m]["fill_ms"].append(f); t[m]["tb_ms"].append(tb); t[m]["device_ms"].append(tot)
            for m, md in modes.items():
                t0 = time.perf_counter()
                eng.align_packed(md, pat, po, txt, to, *s, want_ops=True)          # returns after the results are on the host
                t[m]["e2e_ms"].append((time.perf_counter() - t0) * 1e3)
        run = {}
        for m in modes:
            d = {k: round(statistics.median(v), 3) for k, v in t[m].items()}
            d.update({k + "_spread": round(max(v) - min(v), 3) for k, v in t[m].items()})
            d["gcups_device"] = round(cells / (d["device_ms"] * 1e-3) / 1e9, 1)
            d["gcups_e2e"] = round(cells / (d["e2e_ms"] * 1e-3) / 1e9, 1)
            run[m] = d
        # oracle check of a seeded sample of the semi-global results (this run's records and op lists)
        res = eng.align_packed(pkg.SEMIGLOBAL, pat, po, txt, to, *s, want_ops=True)
        words, off = eng.copy_ops(a.pairs)
        rng = random.Random(481)
        bad = 0
        for k in rng.sample(range(a.pairs), min(a.sample, a.pairs)):
            p, tt = bytes(pat[po[k]:po[k + 1]]), bytes(txt[to[k]:to[k + 1]])
            w = sg.align(p, tt, *s)
            got = tuple(int(res[f][k]) for f in ("score", "end_i", "end_j", "start_i", "start_j", "overlap"))
            if got != (w.score, w.end_i, w.end_j, w.start_i, w.start_j, w.overlap) or pkg.unpack_ops(words, off, k, res["n_ops"][k]) != w.ops:
                bad += 1
        run["oracle_sample"] = {"pairs": min(a.sample, a.pairs), "mismatches": bad}
        run["paths"] = {"short16": int((res["path"] == 1).sum()), "wide32": int((res["path"] == 2).sum())}
        out["runs"][key] = run
        if bad:
            raise SystemExit(f"semi-global results differ from the oracle on {bad} sampled pairs (scoring {key})")
    eng.close()
    text = json.dumps(out, indent=1)
    print(text)
    if a.out:
        with open(a.out, "w") as f:
            f.write(text + "\n")


if __name__ == "__main__":
    main()
