#!/usr/bin/env python
"""bench.py — HiFi Gbp overlapped/sec of the WHOLE overlap + error-correction stage (BASELINE.json metric, SURVEY.md §8d).

Workload (BASELINE.json configs[1]): synthetic 100 Mb diploid genome (0.1 % SNPs, 5 % of it in 50-copy 5 kb repeat families), 30x HiFi reads of
15 kb (sd 2 kb) with 0.2 % errors (sub / ins / del 35 / 30 / 35 %), k = 51, w = 51: 200 k reads, 3.0 Gbp (tools/simgen.c, seeded).

A step = the stage hifiasm runs between reading the reads and building the string graph (Assembly.cpp:2076-2108), as ONE C-ABI call on the raw reads:
hb_stage_run = ha_ft_gen, 3 x (ha_pt_gen + cal_ec_r), ha_pt_gen + cal_ov_r -> the final R_INF.paf[] / reverse_paf[] of every read in host memory and the
corrected reads in HBM.  Every step starts from the RAW reads (the EC rounds rewrite the store), so each step uploads them again:
  value : bases / device time of hb_stage_run (CUDA events on the engine's stream, max over ranks), raw reads resident in HBM when the region starts;
  e2e   : bases / wall time of {hb_reads_upload from pinned host buffers + hb_stage_run + the lists read on the host}, max over ranks.
Multi-GPU (torchrun, one process per GPU): STRONG scaling — the same 100 Mb read set at every N; reads + index replicated, the query reads of every pass
sharded over the ranks, one NCCL all-gather of edit scripts + overlap lists per EC round (and of the final lists).
--impl reference: the UNMODIFIED hifiasm binary (oracle/_ref/hifiasm, built from /root/reference) running the same stage on the host cores, timed by its own
stage stamp ("found overlaps for the final round", BASELINE.md §3), on a bounded sample of the workload (same generator, smaller genome).
"""
import argparse
import hashlib
import json
import os
import re
import statistics
import subprocess
import sys
import tempfile
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tools"))
sys.dont_write_bytecode = True   # the benchmark leaves the tree it runs from as it found it

GENOME_MB = float(os.environ.get("HB_BENCH_GENOME_MB", "100"))
REF_SAMPLE_MB = float(os.environ.get("HB_BENCH_REF_MB", "4"))
COV = float(os.environ.get("HB_BENCH_COV", "30"))
SEED = 20260923
METRIC = "HiFi Gbp overlapped/sec"
DUMP_READS = 128              # --dump-outputs: reads whose overlap records and corrected bases are written
DUMP_PER_READ_MAX = 800000    # --dump-outputs: reads whose per-read values are written (every read of a set up to this size)


def workload_name(mb):
    return ("whole overlap + EC stage (ha_ft_gen, 3 x (ha_pt_gen + cal_ec_r), ha_pt_gen + cal_ov_r) on synthetic %g Mb diploid, %gx HiFi, 15 kb reads, 0.2 %% errors, "
            "5 %% of the genome in 50-copy 5 kb repeats, k=51 w=51") % (mb, COV)


class ClockSampler:
    Q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"

    def __init__(self, dev):
        self.dev, self.rows, self.stop, self.t = dev, [], False, None

    def _run(self):
        while not self.stop:
            try:
                o = subprocess.run(["nvidia-smi", "-i", str(self.dev), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits"], capture_output=True, text=True, timeout=5).stdout.strip()
                if o:
                    self.rows.append([x.strip() for x in o.split(",")])
            except Exception:
                pass
            time.sleep(0.5)

    def __enter__(self):
        self.t = threading.Thread(target=self._run, daemon=True); self.t.start(); return self

    def __exit__(self, *a):
        self.stop = True; self.t.join(timeout=6)

    def summary(self):
        sm = [int(r[0]) for r in self.rows if r[0].isdigit()]; mx = [int(r[1]) for r in self.rows if r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[j] for r in self.rows for j in range(4) if len(r) > 2 + j and r[2 + j].lower().startswith("active")})
        return {"sm_mhz": int(statistics.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons, "samples": len(sm)}


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


# ---- the reference on the host cores ----------------------------------------------------------------------------------------------------------
def run_reference_stage(genome_mb, threads, reps=1):
    """-> list of dicts (one per repetition): stage seconds from the binary's own stamp, bases"""
    import simgen
    ref = os.path.join(ROOT, "oracle", "_ref", "hifiasm")
    if not os.path.exists(ref):
        return None, "oracle/_ref/hifiasm is missing (it is built where /root/reference exists: make -C oracle ref)"
    out = []
    with tempfile.TemporaryDirectory() as td:
        fa = os.path.join(td, "reads.fa")
        rs = simgen.make(genome_mb, COV, seed=SEED, fasta=fa)
        for rep in range(reps):
            t = time.time()
            # (a prefix of its own per repetition: hifiasm reloads <prefix>.ec.bin / .ovlp.*.bin of an earlier run instead of computing the stage again)
            p = subprocess.run([ref, "-o", os.path.join(td, "ref%d" % rep), "-t%d" % threads, "-f0", "--bin-only", fa], capture_output=True, text=True)
            wall = time.time() - t
            m = re.search(r"\[M::ha_assemble::([0-9.]+)\*[0-9.]+@[0-9.]+GB\] ==> found overlaps for the final round", p.stderr)
            if p.returncode != 0 or not m:
                return None, "the reference binary failed: %s" % p.stderr[-300:]
            out.append({"stage_s": float(m.group(1)), "wall_s": wall, "bases": rs.bases, "reads": rs.n,
                        "pec_s": [float(x) for x in re.findall(r"\[M::pec::([0-9.]+)\]", p.stderr)]})
    return out, None


def reference_sample_text(r, threads):
    return ("unmodified hifiasm binary, same generator and seed at %g Mb (%d reads, %.3f Gbp), whole stage from FASTA (parsing runs inside its first counting pass), -t%d -f0; "
            "time = its own stamp at 'found overlaps for the final round'") % (REF_SAMPLE_MB, r["reads"], r["bases"] / 1e9, threads)


# ---- algorithmic bytes of the kernels that can top the stage (DESIGN.md §4; SURVEY.md §8d) -----------------------------------------------------
def algorithmic_bytes(kernel, c, bases):
    """bytes the kernel has to move for the whole stage, from the stage's counters (sums over its 4 passes)"""
    mz, an, win, ov, seg = c["minimizers"], c["anchors"], c["windows"], c["ec_overlaps"], c["ec_segments"]
    f = {
        "k_expand": mz * 28 + an * 24,
        "k_group": an * 16 * 2 + an * 4,                       # anchors in (keys once more) and out
        "k_group_big": an * 16 * 2 + an * 4,
        "k_chain": an * 16 + c["chain_slots"] * 48,
        "k_windows": win * ((775 + 837) // 4 + 40),            # the two packed substrings + the record
        "k_sketch_events": bases * 8 // 4 // 4 + bases * 16 * 8,   # 8 sketch passes (4 index + 4 query): packed reads in, 16-byte events out
        "k_sketch_select": bases * 16 * 8 + mz * 16 * 2,
        "k_ec_overlap": win * 40 + ov * 32,
        "k_ec_overlap_fast": win * 40 + ov * 32,
        "k_ecb_seg_fast": seg * 32 + bases * 60 // 4,         # one record per segment + both substrings (about 2 x coverage x bases / 4 per pass)
        "k_ecb_seg": seg * 0.15 * (2 * 100 // 4 + 32 + 100 * 24),  # queued segments (~15 %): substrings, record, 24-byte trace rows
        "k_ecb_seg_tier1": seg * 0.01 * (2 * 400 // 4 + 32 + 400 * 24),
        "k_ph_decide": ov * 48 + win * 32,
        "k_ph_count": win * 32 + ov * 48,
        "k_ec_cns": win * 32 + bases // 4,
        "k_post": c["chain_slots"] * 48 * 2,
        "k_ecb_merge": seg * 32 + win * 32,
    }
    return float(f.get(kernel, 0))


def dump_outputs(d, eng, r):
    """What the last timed step computed, as d/<name>.npy (float64; 0/1 flags and bases float32), at most 64 MB in all so that two builds can be compared
    output for output: per-read values of every read (of a seeded sample above DUMP_PER_READ_MAX reads) — the overlap counts of both final lists, the two
    read flags, the corrected lengths — and, for a seeded sample of DUMP_READS reads, every field of their final overlap records and their corrected
    bases (0-3, 4 = N); the coverage peaks and corrected bases per round in stage_scalars."""
    n = eng.n_reads
    rng = np.random.default_rng(SEED)
    per = np.arange(n) if n <= DUMP_PER_READ_MAX else np.sort(rng.choice(n, DUMP_PER_READ_MAX, replace=False))
    pick = np.sort(rng.choice(n, min(n, DUMP_READS), replace=False))
    rs = eng.download_reads()
    out = {"per_read_ids": per, "sample_read_ids": pick, "stage_scalars": np.array([r["hom_cov"], r["het_cov"]] + r["corrected_bases"]),
           "corrected_length": rs.length[per], "is_fully_corrected": r["is_fully_corrected"][per].astype(np.float32),
           "is_abnormal": r["is_abnormal"][per].astype(np.float32),
           "sample_corrected_bases": np.concatenate([rs.decode(int(i)) for i in pick]).astype(np.float32)}
    for lst in ("src", "rev"):
        off = r[lst + "_off"].astype(np.int64)
        out[lst + "_per_read"] = np.diff(off)[per]
        rec = np.concatenate([r[lst][off[i]:off[i + 1]] for i in pick])
        # columns: qn, qs (the two halves of qns), qe, tn, ts, te, ml, rev, bl, del, el, no_l_indel
        out["sample_" + lst + "_records"] = np.stack([rec["qns"] >> np.uint64(32), rec["qns"] & np.uint64(0xffffffff)] +
                                                     [rec[f] for f in ("qe", "tn", "ts", "te", "ml", "rev", "bl", "del", "el", "no_l_indel")], axis=1)
    out = {k: (a if a.dtype == np.float32 else a.astype(np.float64)) for k, a in out.items()}
    total = sum(a.nbytes for a in out.values())
    if total > 64 << 20:
        raise RuntimeError("--dump-outputs: %d bytes would exceed 64 MB" % total)
    os.makedirs(d, exist_ok=True)
    for k, a in out.items():
        np.save(os.path.join(d, k + ".npy"), a)
    return total


_JSON_OUT = None


def emit(obj):
    _JSON_OUT.write(json.dumps(obj) + "\n"); _JSON_OUT.flush()


def main():
    # stdout carries the ONE JSON line and nothing else: libraries that print there (NCCL's version banner) go to stderr
    global _JSON_OUT
    sys.stdout.flush()
    _JSON_OUT = os.fdopen(os.dup(1), "w")
    os.dup2(2, 1)
    try:
        return _main()
    except Exception:
        import traceback
        traceback.print_exc()
        return 1


def _main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=2)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write what the last one computed as DIR/<name>.npy (see dump_outputs)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes what this project's stage computed; the reference binary keeps its own files")
    rank = int(os.environ.get("RANK", "0")); world = int(os.environ.get("WORLD_SIZE", "1")); local = int(os.environ.get("LOCAL_RANK", "0"))
    threads = len(os.sched_getaffinity(0))
    dtype = "u8/u64/f64 (2-bit bases, 64-bit bit-vectors, double chain scores)"

    if args.impl == "reference":
        if rank != 0:
            return 0
        runs, why = run_reference_stage(REF_SAMPLE_MB, threads, reps=max(1, min(args.warmup, 1)) + args.steps)  # one untimed run (page cache, CPU clocks), then the timed steps
        if runs is None:
            emit({"impl": "reference", "unavailable": why}); return 0
        timed = runs[-args.steps:]
        secs = sum(r["stage_s"] for r in timed); v = sum(r["bases"] for r in timed) / secs / 1e9
        sample = reference_sample_text(timed[0], threads)
        emit({"impl": "reference", "metric": METRIC, "value": v, "unit": "Gbp/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup, "ms_per_step": secs / args.steps * 1e3,
              "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
              "config": {"workload": workload_name(GENOME_MB), "sample": sample, "stage_s_per_step": [r["stage_s"] for r in timed], "ec_round_s": timed[0]["pec_s"]},
              "cpu_baseline": {"value": v, "unit": "Gbp/s", "cores": threads, "kind": "reference", "sample": sample},
              "e2e": {"value": v, "unit": "Gbp/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}})
        return 0

    import torch
    import torch.distributed as dist
    import hifiasm_b200
    from hifiasm_b200 import dist as hdist
    from hifiasm_b200.engine import torch_allgather
    import simgen
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local))
    torch.cuda.set_device(local)
    tdev = torch.device("cuda", local)

    t0 = time.time()
    rs = simgen.make(GENOME_MB, COV, seed=SEED)
    # pinned host copies: the e2e region uploads from these
    pin = {k: torch.from_numpy(np.ascontiguousarray(v)).pin_memory() for k, v in (("len", rs.length), ("flat", rs.flat), ("boff", rs.byte_off))}
    h_len, h_flat, h_boff = pin["len"].numpy(), pin["flat"].numpy(), pin["boff"].numpy()
    t_gen = time.time() - t0
    n = rs.n; bases = rs.bases
    eng = hifiasm_b200.Engine(local)
    cb = torch_allgather(tdev) if world > 1 else None

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def step():
        torch.cuda.synchronize(); ta = time.time()
        eng.upload_reads(h_len, h_flat, h_boff)
        torch.cuda.synchronize(); tb = time.time()
        r = eng.stage_run(3, rank, world, cb, copy=False)
        n_src, n_rev = int(r["src"].shape[0]), int(r["rev"].shape[0])
        # the result is read on the host: totals of the two lists' records (touches every record)
        chk = int(r["src"]["qe"].astype(np.uint64).sum() + r["rev"]["qe"].astype(np.uint64).sum())
        tc = time.time()
        return r, (tb - ta), (tc - tb), (tc - ta), n_src, n_rev, chk

    def summarize(r):
        if r["n_unfinished"]:
            raise RuntimeError("%d reads could not be finished on the device" % r["n_unfinished"])
        h = hashlib.blake2b(digest_size=8)
        for f in ("qns", "qe", "tn", "ts", "te", "el", "no_l_indel", "ml", "rev", "bl"):
            h.update(np.ascontiguousarray(r["src"][f]).tobytes()); h.update(np.ascontiguousarray(r["rev"][f]).tobytes())
        h.update(r["src_off"].tobytes()); h.update(r["rev_off"].tobytes())
        return h.hexdigest(), r["corrected_bases"], r["hom_cov"]

    digest = None
    for w in range(args.warmup):
        r, t_up, t_st, t_all, n_src, n_rev, chk = step()
        if w == 0:
            digest, corrected, hom = summarize(r)
        sys.stderr.write("[bench] rank %d warm-up %d: upload %.3f s, stage %.3f s (device %.3f s; exchange %.3f s)\n" % (rank, w, t_up, t_st, r["device_ms"] / 1e3, r["ms"]["exchange"] / 1e3))
    barrier()
    dev_ms = 0.0; e2e_s = 0.0; up_s = 0.0; ex_ms = 0.0; kms = {}; counters = None; step_ms = []
    with ClockSampler(local) as cs:
        for _ in range(args.steps):
            r, t_up, t_st, t_all, n_src, n_rev, chk = step()
            dev_ms += r["device_ms"]; e2e_s += t_all; up_s += t_up; ex_ms += r["ms"]["exchange"]; step_ms.append(round(r["device_ms"], 1))
            if digest is None:
                digest, corrected, hom = summarize(r)
            pk, counters = eng.stage_profile()
            for k, v in pk.items():
                a = kms.setdefault(k, [0, 0.0]); a[0] += v[0]; a[1] += v[1]
            last_ms = r["ms"]
    barrier()
    if args.dump_outputs and rank == 0:
        nb = dump_outputs(args.dump_outputs, eng, r)
        sys.stderr.write("[bench] outputs of the last timed step: %d bytes in %s\n" % (nb, args.dump_outputs))
    clocks = cs.summary()
    dev_ms_max, _ = hdist.reduce_time_and_units(dev_ms, 0.0, device="cuda")
    e2e_max, _ = hdist.reduce_time_and_units(e2e_s, 0.0, device="cuda")
    tot_bases = float(bases) * args.steps
    value = tot_bases / (dev_ms_max / 1e3) / 1e9
    h2d = int(h_flat.nbytes + h_boff.nbytes + h_len.size * 4)
    d2h = int((n_src + n_rev) * 48 + 2 * (n + 1) * 8)
    e2e = {"value": tot_bases / e2e_max / 1e9, "unit": "Gbp/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
           "note": "hb_reads_upload from pinned host buffers + hb_stage_run + the final lists read on the host; the EC rounds move their lists through host memory inside the call (the reference's structures are host arrays)"}

    if rank != 0:
        dist.barrier(); dist.destroy_process_group()   # stay alive until rank 0 has printed
        return 0

    # ---- roofline of the kernel with the largest share of the step
    peak, peak_src = measured_peak_gbs()
    per_step = {k: v[1] / args.steps for k, v in kms.items()}
    top = max(per_step.items(), key=lambda kv: kv[1]) if per_step else (None, 0.0)
    launches = kms[top[0]][0] // args.steps if top[0] else 0
    alg = algorithmic_bytes(top[0], counters, bases) if top[0] else 0.0
    achieved = (alg / (top[1] / 1e3) / 1e9) if top[1] > 0 and alg > 0 else None
    roofline = {"bound": "hbm", "kernel": top[0], "kernel_ms_per_step": round(top[1], 2), "share_of_step": round(top[1] / (dev_ms / args.steps), 3) if dev_ms else None,
                "launches_per_step": launches, "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None, "traffic": None,
                "algorithmic_bytes_per_launch": (alg / launches) if launches else None, "peak_source": peak_src,
                "note": "achieved = algorithmic bytes of all its launches in a step (DESIGN.md §4) / their summed CUDA-event time; the kernel is latency / integer-issue bound, not byte bound (SURVEY.md §8d)",
                "kernels_ms_per_step": {k: round(v, 2) for k, v in sorted(per_step.items(), key=lambda kv: -kv[1])}}
    lanes = int(os.environ.get("HB_LANES", "3"))
    roofline["lanes"] = lanes
    if lanes > 1:
        roofline["note"] += "; the batches of a pass run on %d lanes (streams), so a kernel's event time includes what ran beside it and the per-kernel times add up to more than the step: HB_LANES=1 gives exclusive times" % lanes
    # the one kernel of the stage that IS byte bound (the seed-hash probe): its own line, from the same run
    if "k_expand" in per_step and per_step["k_expand"] > 0:
        xb = algorithmic_bytes("k_expand", counters, bases)
        roofline["byte_bound_kernel"] = {"kernel": "k_expand", "kernel_ms_per_step": round(per_step["k_expand"], 2), "achieved": xb / (per_step["k_expand"] / 1e3) / 1e9, "unit": "GB/s",
                                         "frac": xb / (per_step["k_expand"] / 1e3) / 1e9 / peak, "algorithmic_bytes_per_launch": xb / max(1, kms["k_expand"][0] // args.steps)}
    cpu = None
    if not args.no_cpu_baseline and world == 1:
        runs, why = run_reference_stage(REF_SAMPLE_MB, threads, reps=1)
        if runs:
            v = runs[0]["bases"] / runs[0]["stage_s"] / 1e9
            cpu = {"value": v, "unit": "Gbp/s", "cores": threads, "kind": "reference", "sample": reference_sample_text(runs[0], threads), "stage_s": runs[0]["stage_s"], "ec_round_s": runs[0]["pec_s"]}
        else:
            cpu = {"value": None, "unit": "Gbp/s", "cores": threads, "kind": "reference", "sample": why}
    out = {"metric": METRIC, "value": value, "unit": "Gbp/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup, "ms_per_step": dev_ms_max / args.steps,
           "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": dtype, "data": "synthetic",
           "config": {"workload": workload_name(GENOME_MB), "reads": n, "bases": bases, "parallelism": "query reads of every pass sharded x%d; reads + index replicated; one all-gather of edit scripts + lists per EC round" % world,
                      "l2": "inputs larger than L2 (packed reads %.2f GB + index + %.0f M anchors per pass)" % (h_flat.nbytes / 1e9, counters["anchors"] / 4e6),
                      "lanes": int(os.environ.get("HB_LANES", "3")), "hom_cov": hom, "corrected_bases_per_round": corrected, "overlaps_src": n_src, "overlaps_rev": n_rev, "result_digest": digest,
                      "step_device_ms": step_ms, "last_step_host_ms": {k: (round(v, 1) if not isinstance(v, list) else [round(x, 1) for x in v]) for k, v in last_ms.items()},
                      "upload_s_per_step": round(up_s / args.steps, 3), "exchange_ms_per_step": round(ex_ms / args.steps, 1), "setup_s": {"generate": round(t_gen, 1)}, "counters": counters},
           "clocks": clocks, "e2e": e2e, "gpu_launches": int(sum(v[0] for v in kms.values())), "roofline": roofline, "cpu_baseline": cpu}
    emit(out)
    if world > 1:
        dist.barrier(); dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
