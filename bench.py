#!/usr/bin/env python3
"""bench.py -- GCUPS of the NW/SW fill+traceback hot path (BASELINE.json metric) on N B200s.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--impl reference] [--config c2|c4|c5] [--pairs P] [--dump-outputs DIR]

--config c2 (default, the bench line): BASELINE.json configs[1] -- a synthetic batch of P (default 1 M) pairs,
150 bp pattern x 1 kb text DNA, seed 481, scoring 1/-1/-1, global AND local, score + traceback.  One "step" =
one pass of the hot path over the batch in both modes.

  value      = cells / device time of the fill+traceback kernels, inputs already resident in HBM (CUDA events
               recorded by the library on its launching streams), max over ranks.  N > 1: every rank holds its
               own P-pair batch (seed 481+rank): WEAK scaling, no data-path collective.
  e2e        = the same metric through b2a_align_batch_multi with HOST (pinned) buffers: ONE H2D of the
               sequences serving both modes, all kernels, D2H of both modes' result records, every step.
  e2e_seq2   = e2e over compact host buffers (b2a_align_batch_multi_seq2: 2-bit codes + exception list, packed
               once outside the timed region): a quarter of the H2D bytes, identical records.  The headline
               e2e stays the byte-string call, since bytes are what the reference program holds.
  e2e_all_ops = e2e with every pair's traceback op list of both modes delivered to pinned host memory as well
               (b2a_set_ops_sink), i.e. all of struct AlignmentResult for all pairs, not only the records.
  strong     = BASELINE.json configs[2]: the ONE seed-481 P-pair batch pair-sharded over the N ranks
               (rank r takes pairs [r P/N, (r+1) P/N)), device-resident and end to end.  The end-to-end
               figure includes the HOST GATHER and the winner selection (hw2.cpp:340-357): every rank's
               result records land by DMA in its slice of one shared host array, every rank selects over
               its slice, a barrier, rank 0 merges the N candidates -- all inside the timed region.
  roofline   = integer-ALU roofline: algorithmic int16 lane-ops (5 per NW cell, 6 per SW cell, SURVEY.md 8d)
               against 2 x the VIADDMNMX.S16x2 issue rate microbenchmarked on this GPU in this run.
               frac = frac_step uses fill + traceback kernel time (SURVEY.md 8d metric 1), frac_fill the
               fill kernels alone; mix_ceiling is what the kernels' own arithmetic instruction mix can
               reach with no loads/shuffles/stores (microbenchmarked), so "1.00" is interpretable.
  cpu_baseline / --impl reference = the UNMODIFIED reference binary (oracle/_ref/hw2) on a bounded
               sample of the same batch on all host cores.
--config c4: one 100 kb x 100 kb pair, local, score + traceback (configs[3]).  --config c5: the reference's own
16 x 100 kb input, all-vs-all score-only, hw3's affine scoring and hw2's linear scoring (configs[4]), pairs
sharded over the ranks.  Same JSON shape; rooflines against the int32 lines.

--dump-outputs DIR: after the timed steps, rank 0 writes what the headline (device-resident) path returned in its last
step as DIR/<name>.npy (float32 where every value is exact in it, else float64; at most DUMP_BYTES in all), so that two
builds can be compared output for output on identical seeded inputs.  c2/c4: per mode the record fields <mode>_<field>
of the pairs in pair_index (every pair when they fit, else a fixed seeded sample), and <mode>_ops: the op lists of the
pairs in ops_pair_index as ASCII codes (M 77, D 68, I 73) in traceback order, one row per pair, zero-padded.
c5: affine_pair_scores, affine_star_sums, affine_centre of all 120 pairs (with N > 1 the ranks' shards are summed into
rank 0 after the timed steps).  c2 and c4 dump rank 0's own batch, which does not depend on N either.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

M, N_TXT = 150, 1000
SCORING = (1, -1, -1)
OPS_PER_CELL = {0: 5, 1: 6}          # SURVEY.md 8(d): NW 5, SW 6 integer ops per cell; hw3 affine 10
METRIC = "GCUPS (cell updates/s) NW/SW fill+traceback"


def env_int(name, default):
    try:
        return int(os.environ.get(name, default))
    except ValueError:
        return default


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons sampled DURING the timed region."""
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        super().__init__(daemon=True)
        self.index, self.rows, self.stop_flag = index, [], False

    def run(self):
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q,
                                      "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout
                self.rows.append([x.strip() for x in out.strip().split(",")])
            except Exception:
                pass
            time.sleep(0.02)

    def summary(self):
        self.stop_flag = True
        self.join(timeout=6)
        sm = [float(r[0]) for r in self.rows if len(r) >= 7 and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) >= 7 and r[1].replace(".", "").isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 7:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[3:7]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(self.rows)}


def bind_to_gpu_numa_node(index):
    """Best effort: run this rank (and allocate its pinned host buffers) on the CPUs next to its GPU."""
    try:
        bus = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip().lower()
        if bus.startswith("0000"):
            bus = bus[4:]                                  # sysfs uses a 4-digit PCI domain
        cpus = open(f"/sys/bus/pci/devices/{bus}/local_cpulist").read().strip()
        ids = set()
        for part in cpus.split(","):
            lo, _, hi = part.partition("-")
            ids.update(range(int(lo), int(hi or lo) + 1))
        ids &= os.sched_getaffinity(0)
        if ids:
            os.sched_setaffinity(0, ids)
            return cpus
    except Exception:
        pass
    return None


DUMP_BYTES = 64_000_000
DUMP_OPS_PAIRS = 256                    # op lists per mode in a dump
RECORD_FIELDS = ("score", "end_i", "end_j", "start_i", "start_j", "overlap", "n_ops")    # "path" names the kernel family, not a result


def dump_pairs(n_pairs, n_txt_max):
    """(pair_index, ops_pair_index) of a dump: every pair whose record fits the budget left by the op lists, else a fixed seeded
    sample; the op lists of a fixed seeded sample of those."""
    ops_bytes = 2 * DUMP_OPS_PAIRS * (M + n_txt_max) * 4
    per_pair = 2 * len(RECORD_FIELDS) * 4 + (4 if n_pairs <= 1 << 24 else 8)
    keep = (DUMP_BYTES - ops_bytes - 4096) // per_pair
    rng = np.random.default_rng(0)
    idx = np.arange(n_pairs) if n_pairs <= keep else np.sort(rng.choice(n_pairs, size=keep, replace=False))
    ops_idx = np.sort(rng.choice(idx, size=min(DUMP_OPS_PAIRS, len(idx)), replace=False))
    return idx, ops_idx


def alignment_arrays(name, records, idx, ops):
    """<name>_<field> of the records at idx, and <name>_ops: one zero-padded row of ASCII op codes per op list"""
    out = {f"{name}_{f}": records[f][idx] for f in RECORD_FIELDS}
    rows = np.zeros((len(ops), max([len(o) for o in ops] + [1])), dtype=np.uint8)
    for r, o in enumerate(ops):
        rows[r, :len(o)] = np.frombuffer(o, dtype=np.uint8)
    out[f"{name}_ops"] = rows
    return out


def write_dump(out_dir, arrays):
    os.makedirs(out_dir, exist_ok=True)
    total = 0
    for name, a in arrays.items():
        a = np.asarray(a)
        v = a.astype(np.float32)
        if not np.array_equal(v, a):
            v = a.astype(np.float64)
        path = os.path.join(out_dir, name + ".npy")
        np.save(path, v)
        total += os.path.getsize(path)
    if total > DUMP_BYTES:
        raise RuntimeError(f"--dump-outputs wrote {total} bytes, more than {DUMP_BYTES}")


def load_peaks():
    try:
        return json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        return {}


# ------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline
# ------------------------------------------------------------------------------------------------------------
def reference_run_c2(pairs_per_proc, seed):
    """Times oracle/_ref/hw2 (the unmodified reference) on a bounded sample: one process per host core, each on its
    own pairs_per_proc-pair shard of the same synthetic workload, -g then -l.  Returns aggregate GCUPS + details."""
    import oracle_binding as ob
    from __graft_entry__ import load_package
    load_package()
    from bioinformatics_algorithms_b200 import workload
    if not ob.have_ref():
        return None
    cores = os.cpu_count() or 1
    out = {}
    with tempfile.TemporaryDirectory() as td:
        for c in range(cores):
            pat, po, txt, to = workload.config2(pairs_per_proc, seed=seed + 1000 + c)
            workload.write_fasta(os.path.join(td, f"p{c}.fa"), pat, po, b"p")
            workload.write_fasta(os.path.join(td, f"t{c}.fa"), txt, to, b"t")
        cells = cores * pairs_per_proc * M * N_TXT
        total = 0.0
        for flag in ("-g", "-l"):
            t0 = time.perf_counter()
            procs = [subprocess.Popen([ob.REF_HW2, flag, "-p", os.path.join(td, f"p{c}.fa"), "-t", os.path.join(td, f"t{c}.fa"),
                                       "-o", os.path.join(td, f"o{c}.txt"), "-s", *map(str, SCORING)]) for c in range(cores)]
            for p in procs:
                if p.wait() != 0:
                    raise RuntimeError("reference hw2 failed")
            dt = time.perf_counter() - t0
            out[flag] = cells / dt / 1e9
            total += dt
    return {"value": 2 * cells / total / 1e9, "unit": "GCUPS", "cores": cores, "kind": "reference",
            "sample": f"{cores} processes x {pairs_per_proc} pairs 150x1000 each, -g then -l, oracle/_ref/hw2 (g++ -O2, 1 thread/process)",
            "gcups_global": out["-g"], "gcups_local": out["-l"], "seconds": total}


def reference_run_c4(side):
    """The unmodified hw2 -l on the side x side prefix of the seed-482 pair (the full pair needs 49 GB and minutes): 1 core."""
    import oracle_binding as ob
    from __graft_entry__ import load_package
    load_package()
    from bioinformatics_algorithms_b200 import workload
    if not ob.have_ref():
        return None
    p, t = workload.config4(100_000, seed=482)
    p, t = p[:side], t[:side]
    with tempfile.TemporaryDirectory() as td:
        for name, seq in (("p.fa", p), ("t.fa", t)):
            with open(os.path.join(td, name), "wb") as f:
                f.write(b">s\n" + seq.tobytes() + b"\n")
        t0 = time.perf_counter()
        subprocess.check_call([ob.REF_HW2, "-l", "-p", os.path.join(td, "p.fa"), "-t", os.path.join(td, "t.fa"),
                               "-o", os.path.join(td, "o.txt"), "-s", "1", "-1", "-1"])
        dt = time.perf_counter() - t0
    return {"value": len(p) * len(t) / dt / 1e9, "unit": "GCUPS", "cores": 1, "kind": "reference", "seconds": dt,
            "sample": f"oracle/_ref/hw2 -l on the {len(p)} x {len(t)} prefix of the seed-482 pair (quadratic memory: the full pair needs 49 GB)"}


def reference_run_c5(side):
    """hw3 itself cannot run 100 kb (240 GB per pair, hw3.cpp:28-37); the oracle's linear-memory restatement of its score path
    (oracle/hw2_oracle.c orc_affine_score) is timed on side x side prefixes of the shipped sequences, one pair per host core."""
    import oracle_binding as ob
    from __graft_entry__ import load_package
    load_package()
    from bioinformatics_algorithms_b200 import workload
    seqs = [s for _, s in workload.config5_shipped()]
    cores = os.cpu_count() or 1
    ij = [(i, j) for i in range(len(seqs)) for j in range(i + 1, len(seqs))]
    jobs = [ij[k % len(ij)] for k in range(cores)]
    ob.lib()
    t0 = time.perf_counter()
    th = [threading.Thread(target=ob.affine_score, args=(seqs[i][:side], seqs[j][:side], 5, -4, -16, -4)) for i, j in jobs]
    for x in th:
        x.start()
    for x in th:
        x.join()
    dt = time.perf_counter() - t0
    return {"value": cores * side * side / dt / 1e9, "unit": "GCUPS", "cores": cores, "kind": "port", "seconds": dt,
            "sample": f"{cores} threads x one {side} x {side} prefix pair of input16100000.fasta, orc_affine_score (linear-memory C restatement of hw3.cpp:23-98)"}


def print_reference_line(args, cb, workload_name):
    if cb is None:
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/hw2 was not built (reference sources absent at build time)"}))
        return
    print(json.dumps({"impl": "reference", "metric": METRIC, "value": cb["value"], "unit": "GCUPS",
                      "n_gpus": args.gpus, "steps": max(1, args.steps), "warmup": args.warmup, "ms_per_step": cb["seconds"] * 1e3,
                      "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32", "data": "synthetic",
                      "config": {"workload": workload_name, "reference_sample": cb["sample"]},
                      "cpu_baseline": cb,
                      "e2e": {"value": cb["value"], "unit": "GCUPS", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))


# ------------------------------------------------------------------------------------------------------------
# distributed plumbing (barrier + max/sum over ranks; no data-path collective)
# ------------------------------------------------------------------------------------------------------------
class Dist:
    def __init__(self):
        import torch
        self.torch = torch
        self.rank, self.world, self.local_rank = env_int("RANK", 0), env_int("WORLD_SIZE", 1), env_int("LOCAL_RANK", 0)
        self.numa_cpus = bind_to_gpu_numa_node(self.local_rank) if self.world > 1 else None
        torch.cuda.set_device(self.local_rank)
        if self.world > 1:
            import torch.distributed as dist
            self.dist = dist
            # NCCL prints its version banner on stdout at the first communicator; stdout must carry the JSON line only
            sys.stdout.flush()
            saved = os.dup(1)
            os.dup2(2, 1)
            try:
                dist.init_process_group("nccl", device_id=torch.device("cuda", self.local_rank))
                dist.barrier()
                torch.cuda.synchronize()
            finally:
                sys.stdout.flush()
                os.dup2(saved, 1)
                os.close(saved)

    def barrier(self):
        if self.world > 1:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def close(self):
        if self.world > 1:
            self.dist.barrier()
            self.dist.destroy_process_group()


def pinned_copy(pkg, arr):
    out = pkg.pinned_empty(len(arr), arr.dtype)
    out[:] = arr
    return out


def shm_path(tag):
    """files all ranks of the box map: POSIX shared memory when it has room (1.2 GB of sequences + 64 MB of records), else the temp dir"""
    base = "/dev/shm"
    try:
        import shutil
        if shutil.disk_usage(base).free < (3 << 30):
            base = tempfile.gettempdir()
    except OSError:
        base = tempfile.gettempdir()
    return os.path.join(base, f"b2a_bench_{os.environ.get('MASTER_PORT', '0')}_{tag}")


# ------------------------------------------------------------------------------------------------------------
# config 2 / 3
# ------------------------------------------------------------------------------------------------------------
def device_arm(pkg, dev, pat, po, txt, to, steps, warmup, local_rank, seg_pairs=0, ops_pairs=()):
    """inputs resident in HBM; returns per-mode kernel times (sums over `steps`), the launches, the result arrays for checking and the op
    lists of ops_pairs, all of the last step.
    The two modes run one after the other, each with its own engine: a 1 M-pair record is 55 GB per mode (110 GB with 4-bit deltas)."""
    fill_ms = {0: 0.0, 1: 0.0}; tb_ms = {0: 0.0, 1: 0.0}; tot_ms = {0: 0.0, 1: 0.0}
    check, ops, launches, wall, fill_bytes = {}, {}, 0, 0.0, 0
    n = len(po) - 1
    sampler = ClockSampler(local_rank)
    for mode in (pkg.GLOBAL, pkg.LOCAL):
        eng = pkg.Engine(local_rank)
        if seg_pairs:
            eng.set_option(pkg.OPT_SEG_PAIRS, seg_pairs)
        eng.upload(mode, pat, po, txt, to, *SCORING, want_ops=True)
        for _ in range(warmup):
            eng.run()
        dev.barrier()
        if mode == pkg.GLOBAL:
            sampler.start()
        l0 = eng.stats()["launches"]
        t0 = time.perf_counter()
        for _ in range(steps):
            eng.run()
            f, t, tot = eng.times()             # CUDA events on the launching streams: per kernel, and first start -> last end
            fill_ms[mode] += f; tb_ms[mode] += t; tot_ms[mode] += tot
        dev.barrier()
        wall += time.perf_counter() - t0
        launches += eng.stats()["launches"] - l0
        check[mode] = eng.download(n)
        ops[mode] = [eng.fetch_ops(int(q), check[mode]["n_ops"][q]) for q in ops_pairs]
        if mode == pkg.GLOBAL:
            fill_bytes = eng.stats()["fill_bytes"]
        eng.close()
    clocks = sampler.summary()
    return {"fill_ms": fill_ms, "tb_ms": tb_ms, "tot_ms": tot_ms, "wall": wall, "clocks": clocks, "launches": launches,
            "check": check, "ops": ops, "fill_bytes": fill_bytes}


def bench_c2(args):
    global SCORING
    SCORING = tuple(int(x) for x in args.scoring.split(","))
    from __graft_entry__ import load_package
    pkg = load_package()
    from bioinformatics_algorithms_b200 import workload
    from bioinformatics_algorithms_b200.sharding import max_over_ranks, sum_over_ranks, pair_range, merge_best, first_strict_max
    dev = Dist()
    rank, world, local_rank = dev.rank, dev.world, dev.local_rank
    n_pairs = args.pairs
    workload_name = (f"config2: {n_pairs} pairs/GPU, 150 bp x 1 kb DNA, seed 481+rank, -s {' '.join(map(str, SCORING))}, "
                     "global+local, score+traceback")

    pat_np, po_np, txt_np, to_np = workload.config2(n_pairs, seed=481 + rank, n_rate=args.n_rate)
    if args.n_rate:
        workload_name += f", {args.n_rate:g} of the pattern bases replaced by 'N' (robustness variant, not the BASELINE config)"
    if world > 1 and rank == 0:                                  # rank 0's batch IS the seed-481 batch of the strong arm
        np.save(shm_path("pat.npy"), pat_np); np.save(shm_path("txt.npy"), txt_np)
    pat, txt, po, to = (pinned_copy(pkg, a) for a in (pat_np, txt_np, po_np, to_np))
    del pat_np, txt_np
    cells_mode = n_pairs * M * N_TXT

    # ---- weak, device-resident: W warm-up steps, then exactly K timed steps ----
    dump_idx, dump_ops_idx = dump_pairs(n_pairs, N_TXT) if args.dump_outputs and rank == 0 else (None, ())
    d = device_arm(pkg, dev, pat, po, txt, to, args.steps, args.warmup, local_rank, args.resident_seg_pairs, dump_ops_idx)
    fill_ms, tb_ms, tot_ms = d["fill_ms"], d["tb_ms"], d["tot_ms"]
    dev_s = max_over_ranks(sum(tot_ms.values()) * 1e-3)
    wall_dev = max_over_ranks(d["wall"])
    total_cells = sum_over_ranks(2.0 * cells_mode * args.steps)
    value = total_cells / dev_s / 1e9

    # ---- weak, end to end: host buffers in (ONE upload for both modes), both modes' result records out, every step ----
    eng = pkg.Engine(local_rank)
    res_host = [pkg.pinned_empty(n_pairs, pkg.RESULT_DTYPE) for _ in range(2)]
    modes = [pkg.GLOBAL, pkg.LOCAL]
    for _ in range(max(1, min(args.warmup, 2))):
        eng.align_packed_multi(modes, pat, po, txt, to, *SCORING, want_ops=True, results=res_host)
    dev.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.align_packed_multi(modes, pat, po, txt, to, *SCORING, want_ops=True, results=res_host)
    dev.barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    e2e_value = total_cells / e2e_s / 1e9
    st = eng.stats()
    h2d, d2h, e2e_launches = st["h2d_bytes"], st["d2h_bytes"], st["launches"]
    for k, mode in enumerate(modes):
        assert np.array_equal(res_host[k], d["check"][mode]), "e2e and device-resident arms disagree"
    winners = [pkg.select_best(mode, res_host[k]) for k, mode in enumerate(modes)]

    # ---- end to end with EVERY pair's op list delivered to pinned host memory too (b2a_set_ops_sink: copied per segment under the kernels) ----
    off_all, ops_total = eng.ops_offsets(n_pairs)
    sinks = [pkg.pinned_empty(ops_total, np.uint32) for _ in range(2)]
    eng.set_ops_sink(sinks)
    for _ in range(max(1, min(args.warmup, 2))):
        eng.align_packed_multi(modes, pat, po, txt, to, *SCORING, want_ops=True, results=res_host)
    dev.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.align_packed_multi(modes, pat, po, txt, to, *SCORING, want_ops=True, results=res_host)
    dev.barrier()
    ops_s = max_over_ranks(time.perf_counter() - t0)
    st_ops = eng.stats()
    eng.set_ops_sink(None)
    for k, mode in enumerate(modes):                             # a sampled op list re-scores to the reported score
        for q in range(0, n_pairs, max(1, n_pairs // 50)):
            o = np.frombuffer(pkg.unpack_ops(sinks[k], off_all, q, res_host[k]["n_ops"][q]), np.uint8)
            nm = int((o == 0x4D).sum())
            assert len(o) == int(res_host[k]["n_ops"][q]) and int(res_host[k]["end_i"][q]) - int(res_host[k]["start_i"][q]) == nm + int((o == 0x44).sum())
    e2e_all_ops = {"value": total_cells / ops_s / 1e9, "unit": "GCUPS", "ms_per_step": ops_s * 1e3 / args.steps,
                   "h2d_bytes_per_step": st_ops["h2d_bytes"], "d2h_bytes_per_step": st_ops["d2h_bytes"],
                   "what": "e2e + the op lists of ALL pairs of both modes copied to pinned host memory per segment (b2a_set_ops_sink)"}
    del sinks

    # ---- the same end to end over COMPACT host buffers (b2a_seq2: 2-bit codes + exception list, packed once outside the timed region) ----
    t0 = time.perf_counter()
    pat2, txt2 = pkg.PackedSeq(pat, pinned=True), pkg.PackedSeq(txt, pinned=True)
    pack_s = time.perf_counter() - t0
    for r in res_host:
        r["score"] = -7
    for _ in range(max(1, min(args.warmup, 2))):
        eng.align_seq2_multi(modes, pat2, po, txt2, to, *SCORING, want_ops=True, results=res_host)
    dev.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.align_seq2_multi(modes, pat2, po, txt2, to, *SCORING, want_ops=True, results=res_host)
    dev.barrier()
    seq2_s = max_over_ranks(time.perf_counter() - t0)
    st2 = eng.stats()
    for k, mode in enumerate(modes):
        assert np.array_equal(res_host[k], d["check"][mode]), "the compact-input arm and the device-resident arm disagree"
    e2e_seq2 = {"value": total_cells / seq2_s / 1e9, "unit": "GCUPS", "ms_per_step": seq2_s * 1e3 / args.steps,
                "h2d_bytes_per_step": st2["h2d_bytes"], "d2h_bytes_per_step": st2["d2h_bytes"], "gpu_launches_per_step": st2["launches"],
                "exceptions": pat2.n_exc + txt2.n_exc, "pack_ms_once": pack_s * 1e3,
                "what": "b2a_align_batch_multi_seq2: 2-bit codes + exception list in pinned host memory (packed once, outside the timed "
                        "region), expanded on the device per segment; records identical"}
    del pat2, txt2
    eng.close()

    # ---- strong (BASELINE configs[2]): the ONE seed-481 batch pair-sharded over the ranks, host gather + selection timed ----
    strong = None
    if world == 1:
        strong = {"value": value, "e2e": e2e_value, "ms_per_step": dev_s * 1e3 / args.steps, "e2e_ms_per_step": e2e_s * 1e3 / args.steps,
                  "e2e_seq2": e2e_seq2["value"], "e2e_seq2_ms_per_step": e2e_seq2["ms_per_step"],
                  "pairs_total": n_pairs, "winners": winners, "note": "n_gpus = 1: the strong and the weak arm are the same run"}
    else:
        first, count = pair_range(n_pairs, rank, world)
        dev.barrier()                                            # rank 0's .npy files are complete
        sp = np.load(shm_path("pat.npy"), mmap_mode="r"); stx = np.load(shm_path("txt.npy"), mmap_mode="r")
        spat = pinned_copy(pkg, np.ascontiguousarray(sp[first * M:(first + count) * M]))
        stxt = pinned_copy(pkg, np.ascontiguousarray(stx[first * N_TXT:(first + count) * N_TXT]))
        spo = pinned_copy(pkg, np.arange(count + 1, dtype=np.uint64) * np.uint64(M))
        sto = pinned_copy(pkg, np.arange(count + 1, dtype=np.uint64) * np.uint64(N_TXT))
        del sp, stx
        # one host array for all ranks' records (POSIX shared memory, pinned by every rank): the gather IS the D2H copies
        rec_path, cand_path = shm_path("records"), shm_path("cand")
        if rank == 0:
            np.lib.format.open_memmap(rec_path, mode="w+", dtype=pkg.RESULT_DTYPE, shape=(2, n_pairs)).flush()
            np.lib.format.open_memmap(cand_path, mode="w+", dtype=np.int64, shape=(world, 2, 2)).flush()
        dev.barrier()
        shared = np.lib.format.open_memmap(rec_path, mode="r+")
        cand = np.lib.format.open_memmap(cand_path, mode="r+")              # per rank and mode: (key, global pair index) of the slice's winner
        dma_into_shared = True
        try:
            pkg.host_register(shared)
        except Exception:
            dma_into_shared = False                              # cannot pin the mapping here: stage through a private pinned array
        mine = [shared[k, first:first + count] for k in range(2)] if dma_into_shared else \
               [pkg.pinned_empty(count, pkg.RESULT_DTYPE) for _ in range(2)]
        sd = device_arm(pkg, dev, spat, spo, stxt, sto, args.steps, args.warmup, local_rank)
        s_dev_s = max_over_ranks(sum(sd["tot_ms"].values()) * 1e-3)
        eng = pkg.Engine(local_rank)
        s_winners = None
        spat2, stxt2 = pkg.PackedSeq(spat, pinned=True), pkg.PackedSeq(stxt, pinned=True)

        def strong_step(compact=False):
            nonlocal s_winners
            if compact:
                eng.align_seq2_multi(modes, spat2, spo, stxt2, sto, *SCORING, want_ops=True, results=mine)
            else:
                eng.align_packed_multi(modes, spat, spo, stxt, sto, *SCORING, want_ops=True, results=mine)
            if not dma_into_shared:
                for k in range(2):
                    shared[k, first:first + count] = mine[k]
            # hw2.cpp:340-357: first strict maximum.  Every rank scans its own slice (in parallel); the ranks own ascending index
            # ranges, so the batch winner is the first strict maximum of the N slice winners taken in rank order.
            for k, mode in enumerate(modes):
                b = pkg.select_best(mode, mine[k])
                key = int(mine[k]["overlap" if mode == pkg.GLOBAL else "score"][b]) if b >= 0 else -1000000
                cand[rank, k] = (key, first + b if b >= 0 else -1)
            dev.barrier()                                        # every rank's records are in the one host array, every candidate is posted
            if rank == 0:
                s_winners = [first_strict_max(cand[:, k, :]) for k in range(2)]

        for _ in range(max(1, min(args.warmup, 2))):
            strong_step()
        dev.barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            strong_step()
        dev.barrier()
        s_e2e_s = max_over_ranks(time.perf_counter() - t0)
        sst = eng.stats()
        byte_winners = s_winners
        for _ in range(max(1, min(args.warmup, 2))):
            strong_step(True)
        dev.barrier()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            strong_step(True)
        dev.barrier()
        s_seq2_s = max_over_ranks(time.perf_counter() - t0)
        sst2 = eng.stats()
        assert rank != 0 or s_winners == byte_winners, "compact and byte inputs pick different winners"
        # cross-check the gathered winner against the collective-free merge of per-rank winners (sharding.merge_best)
        merged = [merge_best(mode, mine[k], first)[0] for k, mode in enumerate(modes)]
        if rank == 0:
            assert merged == s_winners, (merged, s_winners)
            assert s_winners == winners, "strong and weak arms pick different winners for the seed-481 batch"
            assert s_winners == [pkg.select_best(mode, shared[k]) for k, mode in enumerate(modes)], "serial scan of the gathered records disagrees"
        eng.close()
        if dma_into_shared:
            pkg.host_unregister(shared)
        del mine, shared, cand
        dev.barrier()
        if rank == 0:
            for tag in ("pat.npy", "txt.npy", "records", "cand"):
                try:
                    os.unlink(shm_path(tag))
                except OSError:
                    pass
        scells = 2.0 * cells_mode * args.steps
        strong = {"value": scells / s_dev_s / 1e9, "e2e": scells / s_e2e_s / 1e9, "ms_per_step": s_dev_s * 1e3 / args.steps,
                  "e2e_ms_per_step": s_e2e_s * 1e3 / args.steps, "pairs_total": n_pairs, "pairs_per_gpu": count, "winners": s_winners,
                  "h2d_bytes_per_step_per_gpu": sst["h2d_bytes"], "d2h_bytes_per_step_per_gpu": sst["d2h_bytes"],
                  "e2e_seq2": scells / s_seq2_s / 1e9, "e2e_seq2_ms_per_step": s_seq2_s * 1e3 / args.steps,
                  "e2e_seq2_h2d_bytes_per_step_per_gpu": sst2["h2d_bytes"],
                  "gather": ("every rank's D2H lands in its slice of one POSIX-shm host array pinned with b2a_host_register; every rank runs "
                             "b2a_select_best over its slice and posts (key, index); barrier; rank 0 takes the first strict maximum of the N "
                             "candidates in rank order -- all inside the timed region (checked afterwards against one serial scan of all records)")
                            if dma_into_shared else "private pinned array -> memcpy into the shared host array; per-rank select; barrier; rank 0 merges"}

    line = None
    if rank == 0:
        eng = pkg.Engine(local_rank)
        gops = {k: eng.microbench(k)[0] for k in (0, 1, 2, 10, 11)}
        eng.close()
        peak_cellops = gops[0] * 2.0                     # two int16 cells per 32-bit lane instruction
        alg_ops = sum(cells_mode * args.steps * OPS_PER_CELL[m] for m in (0, 1))
        fill_s = (fill_ms[0] + fill_ms[1]) * 1e-3
        step_s = sum(tot_ms.values()) * 1e-3             # rank 0's own fill + traceback device time
        peaks = load_peaks()
        hbm_peak = peaks.get("hbm_gbs", 6650.0)
        traffic, traffic_src = None, None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "r02_fill_traffic.json")))
            per_pair = sum(tr[m]["dram_read_bytes"] + tr[m]["dram_write_bytes"] for m in ("global", "local")) / 2.0 / tr["pairs_per_launch"]
            traffic, traffic_src = per_pair * n_pairs, tr["source"]
        except Exception:
            pass
        gc = lambda ms: cells_mode * args.steps / (ms * 1e-3) / 1e9
        nw_ceiling, sw_ceiling = gops[10] * 2.0, gops[11] * 2.0       # cell pairs/s -> cells/s
        roofline = {"bound": "int_alu", "achieved": alg_ops / step_s / 1e9, "peak": peak_cellops, "unit": "G int16-cell-ops/s",
                    "frac": alg_ops / step_s / 1e9 / peak_cellops,
                    "frac_step": alg_ops / step_s / 1e9 / peak_cellops, "frac_fill": alg_ops / fill_s / 1e9 / peak_cellops,
                    "achieved_fill": alg_ops / fill_s / 1e9,
                    "definition": "frac = frac_step: algorithmic ops / (fill + traceback kernel time) (SURVEY 8d metric 1); frac_fill: fill kernels alone",
                    "traffic": traffic, "traffic_unit": "DRAM bytes per fill launch (mean of NW and SW)", "traffic_source": traffic_src,
                    "algorithmic_bytes_per_launch": d["fill_bytes"],
                    "peak_source": "b2a_microbench_int16x2 kind 0 (VIADDMNMX.S16x2, 8-way ILP, all SMs) measured in this run, x2 cells/lane",
                    "ops_per_cell": {"global": 5, "local": 6},
                    "mix_ceiling": {"nw_gcups": nw_ceiling, "sw_gcups": sw_ceiling,
                                    "nw_fill_frac_of_mix": gc(fill_ms[0]) / nw_ceiling, "sw_fill_frac_of_mix": gc(fill_ms[1]) / sw_ceiling,
                                    "what": "microbenchmarked rate of the kernels' own arithmetic per cell pair (NW: PRMT, VIADDMNMX.S16x2, VIMNMX.S16x2, "
                                            "IMAD; SW: PRMT, VIADD.16x2, 2 VIADDMNMX, VIMNMX, IMAD), 8 independent chains, no loads/shuffles/stores"},
                    "hbm_fill_write_gbs": d["fill_bytes"] * 2 * args.steps / fill_s / 1e9, "hbm_peak_gbs": hbm_peak,
                    "hbm_peak_source": "MEASURED_PEAKS.json" if peaks else "fallback"}
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            cpu = reference_run_c2(args.ref_pairs, 481)
        line = {"metric": METRIC, "value": value, "unit": "GCUPS", "n_gpus": world,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_s * 1e3 / args.steps,
                "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int16x2", "data": "synthetic",
                "config": {"workload": workload_name, "pairs_per_gpu": n_pairs, "l2": "inputs+record (>50 GB/mode) far larger than L2",
                           "timing": "library CUDA events on the launching streams (first kernel start -> last kernel end per mode), max over ranks",
                           "e2e_pipeline": "b2a_align_batch_multi: segments of 16k pairs doubling to 128k; per segment ONE H2D copy, then the NW and the SW "
                                           "kernels; the copy of segment k+1 overlaps the kernels of segment k",
                           "wall_ms_per_step_device_arm": wall_dev * 1e3 / args.steps, "rank0_cpu_binding": dev.numa_cpus},
                "e2e": {"value": e2e_value, "unit": "GCUPS", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                        "ms_per_step": e2e_s * 1e3 / args.steps, "gpu_launches_per_step": e2e_launches,
                        "returns": "32-byte result records of both modes (score, end/start cell, overlap, n_ops); the 2-bit op lists stay "
                                   "on the device for b2a_fetch_ops / b2a_copy_ops (about 0.3 GB per mode if all are fetched)"},
                "e2e_seq2": e2e_seq2, "e2e_all_ops": e2e_all_ops, "strong": strong,
                "nw_fill_ms": fill_ms[0] / args.steps, "nw_tb_ms": tb_ms[0] / args.steps, "sw_fill_ms": fill_ms[1] / args.steps,
                "sw_tb_ms": tb_ms[1] / args.steps, "nw_gcups": gc(tot_ms[0]), "sw_gcups": gc(tot_ms[1]),
                "frac_fill": roofline["frac_fill"], "frac_step": roofline["frac_step"],
                "gpu_launches": d["launches"], "clocks": d["clocks"], "roofline": roofline, "cpu_baseline": cpu}
        if args.dump_outputs:
            arrays = {"pair_index": dump_idx, "ops_pair_index": dump_ops_idx}
            for mode, name in ((pkg.GLOBAL, "global"), (pkg.LOCAL, "local")):
                arrays.update(alignment_arrays(name, d["check"][mode], dump_idx, d["ops"][mode]))
            write_dump(args.dump_outputs, arrays)
    dev.close()
    if rank == 0:
        print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------------------
# config 4: one 100 kb x 100 kb pair, local, score + traceback
# ------------------------------------------------------------------------------------------------------------
def bench_c4(args):
    from __graft_entry__ import load_package
    pkg = load_package()
    from bioinformatics_algorithms_b200 import workload
    from bioinformatics_algorithms_b200.sharding import max_over_ranks, sum_over_ranks
    import oracle_binding as ob
    dev = Dist()
    rank, world, local_rank = dev.rank, dev.world, dev.local_rank
    p, t = workload.config4(args.len, seed=482)
    s = (1, -1, -1)
    cells = len(p) * len(t)
    pat, po = pkg.pack([p.tobytes()]); txt, to = pkg.pack([t.tobytes()])
    pat, po, txt, to = (pinned_copy(pkg, a) for a in (pat, po, txt, to))
    eng = pkg.Engine(local_rank)
    eng.upload(pkg.LOCAL, pat, po, txt, to, *s, want_ops=True)
    for _ in range(args.warmup):
        eng.run()
    dev.barrier()
    sampler = ClockSampler(local_rank); sampler.start()
    fill = tb = tot = 0.0
    l0 = eng.stats()["launches"]
    for _ in range(args.steps):
        eng.run()
        f, b, x = eng.times()
        fill += f; tb += b; tot += x
    dev.barrier()
    clocks = sampler.summary()
    launches = eng.stats()["launches"] - l0
    res = eng.download(1)
    res_ops = [eng.fetch_ops(0, res["n_ops"][0])] if args.dump_outputs else []
    res_host = pkg.pinned_empty(1, pkg.RESULT_DTYPE)
    eng.align_packed(pkg.LOCAL, pat, po, txt, to, *s, want_ops=True, results=res_host)
    dev.barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        eng.align_packed(pkg.LOCAL, pat, po, txt, to, *s, want_ops=True, results=res_host)
    dev.barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    st = eng.stats()
    dev_s = max_over_ranks(tot * 1e-3)
    total_cells = sum_over_ranks(float(cells) * args.steps)
    line = None
    if rank == 0:
        gops0 = eng.microbench(0)[0]
        peak = gops0                                     # one int32 cell per lane instruction
        want = ob.score_only(pkg.LOCAL, p.tobytes(), t.tobytes(), *s)
        ok = (int(res["score"][0]), int(res["end_i"][0]), int(res["end_j"][0])) == want and res_host[0] == res[0]
        cpu = None if args.no_cpu_baseline else reference_run_c4(args.ref_side)
        alg = cells * args.steps * 6.0
        line = {"metric": METRIC, "value": total_cells / dev_s / 1e9, "unit": "GCUPS", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": dev_s * 1e3 / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "int32",
                "data": "synthetic",
                "config": {"workload": f"config4: one {len(p)} x {len(t)} pair (seed 482), -l -s 1 -1 -1, score + traceback; N > 1 = replicas only",
                           "l2": "5 GB record per launch, far larger than L2", "timing": "library CUDA events, max over ranks"},
                "e2e": {"value": total_cells / e2e_s / 1e9, "unit": "GCUPS", "h2d_bytes_per_step": st["h2d_bytes"], "d2h_bytes_per_step": st["d2h_bytes"],
                        "ms_per_step": e2e_s * 1e3 / args.steps},
                "fill_ms": fill / args.steps, "traceback_ms": tb / args.steps, "score": int(res["score"][0]), "n_ops": int(res["n_ops"][0]),
                "check": "score + end cell equal the linear-memory oracle" if ok else "MISMATCH against the oracle",
                "gpu_launches": launches, "clocks": clocks,
                "roofline": {"bound": "int_alu", "achieved": alg / (tot * 1e-3) / 1e9, "peak": peak, "unit": "G int32-cell-ops/s",
                             "frac": alg / (tot * 1e-3) / 1e9 / peak, "frac_step": alg / (tot * 1e-3) / 1e9 / peak,
                             "frac_fill": alg / (fill * 1e-3) / 1e9 / peak, "ops_per_cell": {"local": 6}, "traffic": None,
                             "peak_source": "b2a_microbench_int16x2 kind 0 lane-instruction rate measured in this run, one int32 cell per lane (SURVEY 8d: half the s16x2 line)"},
                "cpu_baseline": cpu}
        assert ok, "config 4 result differs from the oracle"
        if args.dump_outputs:
            write_dump(args.dump_outputs, {"pair_index": [0], "ops_pair_index": [0], **alignment_arrays("local", res, [0], res_ops)})
    eng.close()
    dev.close()
    if rank == 0:
        print(json.dumps(line))
    return 0


# ------------------------------------------------------------------------------------------------------------
# config 5: 16 x 100 kb all-vs-all, score only, pairs sharded over the ranks
# ------------------------------------------------------------------------------------------------------------
def bench_c5(args):
    from __graft_entry__ import load_package
    pkg = load_package()
    from bioinformatics_algorithms_b200 import workload
    from bioinformatics_algorithms_b200.sharding import max_over_ranks, sum_over_ranks, star_pair_range, reduce_star_sums
    dev = Dist()
    rank, world, local_rank = dev.rank, dev.world, dev.local_rank
    seqs = [x for _, x in workload.config5_shipped()]
    ij = [(i, j) for i in range(len(seqs)) for j in range(i + 1, len(seqs))]
    first, count = star_pair_range(len(seqs), rank, world)
    mine = ij[first:first + count]
    cells = float(sum(len(seqs[i]) * len(seqs[j]) for i, j in mine))
    eng = pkg.Engine(local_rank)
    aff = (5, -4, -16, -4)
    for _ in range(args.warmup):
        eng.affine_star_scores(seqs, *aff, pair_first=first, pair_count=count)
    dev.barrier()
    sampler = ClockSampler(local_rank); sampler.start()
    k_ms = 0.0
    t0 = time.perf_counter()
    for _ in range(args.steps):
        ps, sums, centre = eng.affine_star_scores(seqs, *aff, pair_first=first, pair_count=count)
        k_ms += eng.times()[2]
    dev.barrier()
    e2e_s = max_over_ranks(time.perf_counter() - t0)
    clocks = sampler.summary()
    st = eng.stats()
    dev_s = max_over_ranks(k_ms * 1e-3)
    total_cells = sum_over_ranks(cells * args.steps)
    if args.dump_outputs and world > 1:             # every rank: the dump holds all pairs' scores and the full sums whatever the GPU count
        all_ps = np.zeros(len(ij), dtype=np.int64)
        all_ps[first:first + count] = ps
        ps, _ = reduce_star_sums(all_ps)
        sums, centre = reduce_star_sums(sums)
    # hw2's linear scoring over the same pairs, score only
    pat, po = pkg.pack([seqs[i] for i, _ in mine]); txt, to = pkg.pack([seqs[j] for _, j in mine])
    eng.upload(pkg.GLOBAL, pat, po, txt, to, 1, -1, -1, score_only=True)
    eng.run()
    lin_ms = 0.0
    for _ in range(args.steps):
        eng.run()
        lin_ms += eng.times()[2]
    lin_s = max_over_ranks(lin_ms * 1e-3)
    line = None
    if rank == 0:
        gops0 = eng.microbench(0)[0]
        cpu = None if args.no_cpu_baseline else reference_run_c5(args.ref_side)
        alg = cells * args.steps * 10.0
        line = {"metric": METRIC, "value": total_cells / dev_s / 1e9, "unit": "GCUPS", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": dev_s * 1e3 / args.steps, "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "int32",
                "data": "the reference's own input16100000.fasta (tests/golden/input16100000.fasta.gz)",
                "config": {"workload": "config5: all-vs-all of the shipped 16 x 100 kb sequences (120 pairs), hw3 affine scoring 5:-4:-16:-4, score only, "
                                       "pairs sharded over the ranks (hw3.cpp:231-241)", "pairs_this_rank": count,
                           "l2": "boundary exchange of the concurrent pairs exceeds L2", "timing": "library CUDA events, max over ranks"},
                "e2e": {"value": total_cells / e2e_s / 1e9, "unit": "GCUPS", "h2d_bytes_per_step": st["h2d_bytes"], "d2h_bytes_per_step": st["d2h_bytes"],
                        "ms_per_step": e2e_s * 1e3 / args.steps},
                "linear_gcups": total_cells / lin_s / 1e9, "linear_ms_per_step": lin_s * 1e3 / args.steps,
                "gpu_launches": st["launches"], "clocks": clocks,
                "roofline": {"bound": "int_alu", "achieved": alg / (k_ms * 1e-3) / 1e9, "peak": gops0, "unit": "G int32-cell-ops/s",
                             "frac": alg / (k_ms * 1e-3) / 1e9 / gops0, "ops_per_cell": {"affine": 10}, "traffic": None,
                             "note": "the kernel spends 6 instructions on the 10 nominal ops of a cell, so frac can exceed 1",
                             "linear_frac": cells * args.steps * 5.0 / (lin_ms * 1e-3) / 1e9 / gops0,
                             "peak_source": "b2a_microbench_int16x2 kind 0 lane-instruction rate measured in this run, one int32 cell per lane"},
                "cpu_baseline": cpu}
        if args.dump_outputs:
            write_dump(args.dump_outputs, {"affine_pair_scores": ps, "affine_star_sums": sums, "affine_centre": [centre]})
    eng.close()
    dev.close()
    if rank == 0:
        print(json.dumps(line))
    return 0


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200")
    ap.add_argument("--config", default="c2", choices=("c2", "c4", "c5"))
    ap.add_argument("--pairs", type=int, default=1_000_000, help="c2: pairs per GPU (weak arm) = pairs of the one strong-arm batch")
    ap.add_argument("--ref-pairs", type=int, default=1500, help="c2 reference sample: pairs per host process and mode")
    ap.add_argument("--ref-side", type=int, default=20000, help="c4/c5 reference sample: prefix length")
    ap.add_argument("--len", type=int, default=100_000, help="c4: sequence length")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--resident-seg-pairs", type=int, default=0, help="experiment: pairs per segment of the device-resident arm")
    ap.add_argument("--n-rate", type=float, default=0.0, help="c2 variant: fraction of pattern bases turned into 'N' (pairs holding one leave the 4-symbol s16x2 path)")
    ap.add_argument("--scoring", default="1,-1,-1", help="c2: match,mismatch,gap (SURVEY 8d also names 2,-3,-4: 4-bit deltas, twice the record)")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the outputs of the last timed step as DIR/<name>.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of the B200 path; the reference arm has none to dump")

    if args.impl == "reference":
        if env_int("RANK", 0) != 0:
            return 0
        global SCORING
        SCORING = tuple(int(x) for x in args.scoring.split(","))
        steps = max(1, args.steps)
        if args.config == "c2":
            if args.warmup:
                reference_run_c2(max(200, args.ref_pairs // 2), 480)                 # one short warm-up pass
            vals = [reference_run_c2(args.ref_pairs, 481 + 10 * s) for s in range(steps)]
            name = f"config2: {args.pairs} pairs/GPU, 150 bp x 1 kb DNA, seed 481+rank, -s {' '.join(map(str, SCORING))}, global+local, score+traceback"
        elif args.config == "c4":
            vals = [reference_run_c4(args.ref_side) for _ in range(steps)]
            name = "config4: one 100 kb x 100 kb pair, -l"
        else:
            vals = [reference_run_c5(args.ref_side) for _ in range(steps)]
            name = "config5: 16 x 100 kb all-vs-all, hw3 affine scoring, score only"
        if vals[0] is None:
            print_reference_line(args, None, name)
            return 0
        cb = dict(vals[-1])
        cb["value"] = float(np.mean([x["value"] for x in vals]))
        cb["seconds"] = float(np.mean([x["seconds"] for x in vals]))
        print_reference_line(args, cb, name)
        return 0
    return {"c2": bench_c2, "c4": bench_c4, "c5": bench_c5}[args.config](args)


if __name__ == "__main__":
    sys.exit(main())
