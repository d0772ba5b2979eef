#!/usr/bin/env python
"""Benchmark of the string_grouper hot path on B200 — one JSON line on stdout (rank 0).

    python bench.py --gpus 1 --steps 3 --warmup 3
    python -m torch.distributed.run --nnodes=1 --nproc-per-node N --master-addr 127.0.0.1 --master-port P \
        bench.py --gpus N --steps K --warmup W
    python bench.py --impl reference ...        # the reference's CPU path (oracle port) on this box's cores

Workload (BASELINE.json metric / configs[2]): match_strings self-match of a 663 000-name sec__edgar-shaped
synthetic corpus (synth_corpus.make_names(seed=0)), 3-grams, min_similarity 0.8, max_n_matches 20, float64.
One step = one pass of the hot path: K1 vectorise -> K2 top-n cosine product -> K4 symmetrise.

  value        matched pairs / s with the packed strings already resident in HBM (CUDA events around K1..K4)
  e2e          same metric through string_grouper_b200.StringGrouper(series).fit().get_matches(): host buffers in,
               DataFrame out, H2D / D2H inside the timed region
  roofline     the dominant kernel chain (K2 candidates: pack + block-max filter + tile kernel): bytes it really
               streams / CUDA-event time, against the measured HBM peak; the bytes of the full Gustavson traversal
               (SURVEY.md §8d) are reported beside it as `algorithmic`
  parity       ALL pairs of the step's result against the CPU port's whole-job result (N=1)
  cpu_baseline the CPU port's measured whole job on this box's usable cores (N=1)

--dump-outputs DIR writes the match list of the last timed step as .npy files (see dump_outputs) so that two builds
can be compared output for output; the input corpus depends on --rows alone.  The benchmark writes nothing into the
source tree (it may be read-only): the CPU whole-job cache lives in the system temp directory.
"""
import argparse
import atexit
import hashlib
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

METRIC = "match_strings matched pairs/sec (663k names self-match @0.8, top 20, 3-gram)"
UNIT = "pairs/s"
TOP_N, MIN_SIM = 20, 0.8


# ----------------------------------------------------------------------------- clocks
class ClockSampler:
    """nvidia-smi sampled every 200 ms while the timed region runs (B200_PROFILING.md recipe).

    start() launches the process early (its NVML initialisation enumerates every GPU of the box and was seen to
    stall rank 0 for 10-15 ms when it fell into a timed step of an 8-GPU run); arm() marks the beginning of the timed
    region: only samples from then on (and the one just before) are reported."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index):
        self.gpu, self.rows, self.proc, self.t_arm = gpu_index, [], None, None

    def arm(self):
        if self.proc is None:
            self.start()
        self.t_arm = time.time()

    def start(self):
        if self.proc is not None:
            return
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + self.Q,
                                          "--format=csv,noheader,nounits", "-lms", "200"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            atexit.register(self._kill)          # never leave the sampler behind, whatever ends the run
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _kill(self):
        try:
            if self.proc is not None and self.proc.poll() is None:
                self.proc.terminate()
        except Exception:
            pass

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append((time.time(), [x.strip() for x in line.split(",")]))

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm, mx, power, reasons = [], [], [], set()
        rows = list(self.rows)
        if self.t_arm is not None:
            before = [r for t, r in rows if t < self.t_arm][-1:]
            rows = before + [r for t, r in rows if t >= self.t_arm]
        else:
            rows = [r for _, r in rows]
        for r in rows:
            try:
                sm.append(float(r[1])); mx.append(float(r[2])); power.append(float(r[3]))
            except Exception:
                continue
            for name, v in zip(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"], r[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        busy = [s for s, p in zip(sm, power) if p > 250] or sm
        return {"sm_mhz": float(np.median(busy)) if busy else None, "sm_max_mhz": max(mx) if mx else None,
                "power_w_max": max(power) if power else None, "samples": len(sm), "reasons": sorted(reasons)}


def workload_config(n, gpus, sha):
    """Identical in both arms (the driver compares the `config` of the reference line with ours)."""
    return {"workload": "match_strings self-match, %d synthetic sec__edgar-shaped names (synth_corpus seed 0), "
                        "ngram 3, min_similarity %.1f, max_n_matches %d, tfidf float64" % (n, MIN_SIM, TOP_N),
            "rows": n, "corpus_sha256": sha,
            "parallelism": "left-row shards x%d, right matrix replicated" % gpus,
            "l2": "256 MiB memset between steps (untimed); tile blobs + survivor masks exceed what stays L2-resident "
                  "across steps"}


# ----------------------------------------------------------------------------- CPU reference arm
def run_reference_arm(args, names, sha):
    """--impl reference: the reference's CPU implementation of the path (the oracle port: the reference tree has
    no native code and its Python cannot travel to this box) on all usable host threads.

    The WHOLE job is run and timed once (bench_cpu.whole_job: vectorise x3 passes, block product, LIL symmetrise,
    match list, get_matches frame) — `value`, `ms_per_step` and the pair count come from that measured run.  The
    K + W steps the driver asks for are bounded samples (bench_cpu.sample_model); their extrapolation to the whole
    job is printed next to the measurement with its error (`model`)."""
    import bench_cpu as C
    from oracle import pipeline as P
    from oracle import sdt
    sdt.build()
    t0 = time.perf_counter()
    full, _, _ = P.tf_idf_matrices(names[:60000])       # thread probe on a slice (untimed)
    cores, probe = C.best_thread_count(full)
    setup = time.perf_counter() - t0
    job = C.whole_job(names, cores)
    full = job["matrix"]
    ests, walls, last = [], [], None
    for step in range(args.warmup + args.steps):
        t0 = time.perf_counter()
        est, est_pairs, detail = C.sample_model(names, full, cores)
        wall = time.perf_counter() - t0
        if step >= args.warmup:
            ests.append((est, est_pairs))
            walls.append(wall)
        last = detail
    value = job["pairs"] / job["wall_s"]
    est_s = float(np.mean([e[0] for e in ests])) if ests else None
    est_pairs = float(np.mean([e[1] for e in ests])) if ests else None
    model = None
    if ests:
        model = {"est_whole_job_s": est_s, "est_pairs": est_pairs,
                 "error_vs_measured_s": est_s / job["wall_s"] - 1.0,
                 "error_vs_measured_pairs": est_pairs / job["pairs"] - 1.0,
                 "sample_wall_s_per_step": float(np.mean(walls)), "detail": last}
    sample = ("whole job measured once in this run: %d names, n_blocks=%s, %d OpenMP threads (fastest of %s; "
              "os.cpu_count() = %s, usable = %d), phases %s; the %d+%d steps are bounded samples (20000-name fit + "
              "block products of %s left rows x all right rows) whose extrapolation is reported under `model`"
              % (len(names), job["n_blocks"], cores, probe, os.cpu_count(), C.usable_cores(), job["phases"],
                 args.warmup, args.steps, last["left_rows_s1_s2"] if last else None))
    line = {"impl": "reference", "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": job["wall_s"] * 1e3,
            "timed_whole_jobs": 1, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(len(names), args.gpus, sha),
            "whole_job": C.public(job), "model": model,
            "cpu_baseline": {"value": value, "unit": UNIT, "cores": cores, "kind": "port", "sample": sample},
            "e2e": {"value": value, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
            "setup_s": setup}
    print(json.dumps(line), flush=True)


def triples_digest(r, c, s):
    """Order-independent digest of a match list (sorted by (row, col) first)."""
    r, c, s = np.asarray(r, dtype=np.int64), np.asarray(c, dtype=np.int64), np.asarray(s, dtype=np.float64)
    o = np.lexsort((c, r))
    h = hashlib.sha256()
    h.update(r[o].tobytes()); h.update(c[o].tobytes()); h.update(s[o].tobytes())
    return h.hexdigest()[:32]


DUMP_BYTES = 64_000_000
DUMP_SAMPLE_ROWS = 1 << 18


def dump_outputs(out_dir, triples, n, seed=0):
    """Write a match list (row, col, score triples) as float64 .npy files under `out_dir`:

      pairs_per_row  (n,)  pairs of every row
      sample_rows    sorted rows of a fixed sample: the first DUMP_SAMPLE_ROWS of a permutation seeded by `seed`,
                     fewer only if their pairs would take the files past DUMP_BYTES
      row, col, score  every pair of the sampled rows, sorted by (row, col)

    Row and column indices are exact in float64."""
    r = np.asarray(triples[0]).astype(np.int64)
    c = np.asarray(triples[1]).astype(np.int64)
    s = np.asarray(triples[2]).astype(np.float64)
    counts = np.bincount(r, minlength=n)
    order = np.random.default_rng(seed).permutation(n)[:DUMP_SAMPLE_ROWS]
    budget = DUMP_BYTES // 8 - n - 5 * 16             # float64 elements left (pairs_per_row, .npy headers)
    cost = np.cumsum(1 + 3 * counts[order])           # one sample_rows entry + row, col, score per pair
    rows = np.sort(order[:int(np.searchsorted(cost, budget, side="right"))])
    sel = np.zeros(n, dtype=bool)
    sel[rows] = True
    sel = sel[r]
    o = np.lexsort((c[sel], r[sel]))
    arrays = {"pairs_per_row": counts, "sample_rows": rows, "row": r[sel][o], "col": c[sel][o], "score": s[sel][o]}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a.astype(np.float64))


# ----------------------------------------------------------------------------- B200 arm
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--rows", type=int, default=663_000)
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU whole job (parity + cpu_baseline)")
    ap.add_argument("--no-aux", action="store_true", help="multi-GPU: skip the two-Series sharded-K1 run")
    ap.add_argument("--aux-master", type=int, default=2_000_000)
    ap.add_argument("--aux-duplicates", type=int, default=400_000)
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the match list of the last timed step under DIR as .npy files (B200 arm, rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs applies to --impl b200")
    sys.dont_write_bytecode = True          # no __pycache__ in the source tree for the project modules imported below

    if os.environ.get("NCCL_DEBUG", "").upper() == "VERSION":
        os.environ["NCCL_DEBUG"] = "WARN"           # keep stdout to the one JSON line
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))

    from synth_corpus import corpus_sha256, make_names
    if args.impl == "reference":
        if rank != 0:
            return 0
        names = make_names(args.rows, seed=0)
        run_reference_arm(args, names, corpus_sha256(names))
        return 0

    import pandas as pd
    import torch
    import torch.distributed as dist

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (B200); use --impl reference for the CPU arm")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()          # long before the timed region, see ClockSampler
    if world > 1:
        os.environ.setdefault("SG_B200_DISTRIBUTED", "1")     # the library shards only when told to (ADVICE r1)
        dist.init_process_group("nccl", device_id=dev)
    import string_grouper_b200 as api
    from string_grouper_b200 import _device as D
    from string_grouper_b200 import _dist, _ingest, _lib
    _lib.load()

    names = make_names(args.rows, seed=0)
    n = len(names)
    sha = corpus_sha256(names)
    series = pd.Series(names)
    data, offsets, flags, _ = _ingest.pack_strings([series])
    d_bytes, d_off, total = D.upload_strings(data, offsets, dev)
    flush = torch.empty(256 << 20, dtype=torch.uint8, device=dev)
    lo, hi = _dist.shard_range(n, rank, world)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    info = {}

    def resident_step(stats, row_lo=lo, row_hi=hi, gather=True):
        D.mark(stats, "start")
        A, _, _ = D.tfidf_resident(d_bytes, d_off, n, total, n, 3, flags, np.float64, stats=stats)
        D.mark(stats, "k1")
        M = D.cossim_topn(A, A, TOP_N, MIN_SIM, row_begin=row_lo, row_end=row_hi, stats=stats)
        info["k2_nnz_local"] = M.nnz
        info["M"] = M
        if world > 1 and gather:
            M = D.gather_shards(M)
            D.mark(stats, "gather")
        S = D.symmetrize(M)
        D.mark(stats, "k4")
        info["A"] = A
        return S

    # ---- device-resident throughput ("value") ----
    step_ms, cand_ms, pairs = [], [], 0
    launches0 = None
    S = None
    for step in range(args.warmup + args.steps):
        flush.zero_()
        barrier()
        timed = step >= args.warmup
        if timed and launches0 is None:
            launches0 = dict(D.LAUNCH_COUNTS)
            if rank == 0:
                sampler.arm()
        stats = {"time_kernels": True}
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        S = resident_step(stats)
        e1.record()
        barrier()
        if timed:
            step_ms.append(e0.elapsed_time(e1))
            cand_ms.append(sum(a.elapsed_time(b) for a, b in stats["candidate_events"]))
            pairs = S.nnz
            info["stats"] = stats
    launches = sum(D.LAUNCH_COUNTS.values()) - sum(launches0.values())
    t_local = torch.tensor([sum(step_ms)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_local, op=dist.ReduceOp.MAX)
    total_ms = float(t_local.item())
    ms_per_step = total_ms / args.steps
    value = pairs / (ms_per_step / 1e3)
    phases = {k: round(v, 3) for k, v in D.phases_ms(info["stats"]).items()}
    phases_all = [phases]
    if world > 1:
        phases_all = [None] * world
        dist.all_gather_object(phases_all, phases)
    final_triples = S.host_triples()
    pre_triples = info["M"].host_triples() if world == 1 else None

    # ---- multi-GPU: the gathered result must equal the unsharded one (untimed) ----
    shard_check = None
    if world > 1:
        S1 = resident_step({}, 0, n, gather=False)
        ok = triples_digest(*S1.host_triples()) == triples_digest(*final_triples)
        flag = torch.tensor([0 if ok else 1], dtype=torch.int64, device=dev)
        dist.all_reduce(flag, op=dist.ReduceOp.SUM)
        shard_check = {"gathered_equals_unsharded": int(flag.item()) == 0, "ranks_checked": world,
                       "pairs": int(S1.nnz)}
        if int(flag.item()) != 0:
            raise SystemExit("bench.py: the gathered multi-GPU match list differs from the unsharded result on %d "
                             "rank(s)" % int(flag.item()))
        del S1

    # ---- multi-GPU only: one two-Series run that takes the sharded-K1 path (BASELINE.json configs[3] shape) ----
    aux_two_series = None
    if world > 1 and not args.no_aux:
        n_m, n_d = args.aux_master, args.aux_duplicates
        base = make_names(n_m + int(0.6 * n_d), seed=1)
        master2 = pd.Series(base[:n_m])
        dupes2 = pd.Series(base[n_m - (n_d - int(0.6 * n_d)):])          # 40 % of the duplicates are master rows
        del base
        os.environ["SG_B200_SHARD_VECTORISE"] = "1"      # K1 sharded: df all-reduce + all-gather of the duplicate CSR
        D.TIME_KERNELS = True
        walls = []
        for rep in range(2):                             # warm-up + one timed run
            barrier()
            t0 = time.perf_counter()
            sg2 = api.StringGrouper(master2, dupes2, min_similarity=0.7)
            sg2.fit()
            out2 = sg2.get_matches()
            torch.cuda.synchronize()
            walls.append(time.perf_counter() - t0)
        D.TIME_KERNELS = False
        os.environ.pop("SG_B200_SHARD_VECTORISE", None)
        st2 = sg2._last_stats
        mine = {"wall_s": walls[-1], "k2_candidates_ms": sum(a.elapsed_time(b) for a, b in st2.get("candidate_events", [])),
                "phases_ms": {k: round(v, 2) for k, v in D.phases_ms(st2).items()},
                "sharded_vectorise": bool(st2.get("sharded_vectorise")), "local_nnz": int(st2.get("nnz", 0))}
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)
        t_aux = torch.tensor([walls[-1]], dtype=torch.float64, device=dev)
        dist.all_reduce(t_aux, op=dist.ReduceOp.MAX)
        n_match = len(sg2._matches_list)
        aux_two_series = {
            "workload": "match_strings(master %d, duplicates %d) min_similarity 0.7, K1 sharded over the ranks (df table "
                        "all-reduce, duplicate-matrix CSR all-gather over NVLink), left rows = this rank's master block"
                        % (n_m, n_d),
            "wall_s_max_over_ranks": float(t_aux.item()), "matches": int(n_match),
            "pairs_per_s": n_match / float(t_aux.item()),
            "nccl_bytes_per_rank": {"df_allreduce": 4 * (1 << 21),
                                    "duplicate_csr_allgather": int(16 * sum(p["local_nnz"] for p in per_rank) * n_d / (n_m + n_d)),
                                    "match_list_allgather": 16 * int(n_match)},
            "per_rank": per_rank}
        del sg2, out2, master2, dupes2

    # ---- end to end through the public API ("e2e") ----
    e2e_s, e2e_rows, h2d, d2h = [], 0, 0, 0
    e2e_parts = {}
    if world > 1:
        os.environ["SG_B200_RESULT"] = "rank0"       # the match list / DataFrame is materialised on rank 0 only
    for step in range(args.warmup + args.steps):
        flush.zero_()
        barrier()
        d2h0 = D.TRANSFER_BYTES["d2h"]
        t0 = time.perf_counter()
        sg = api.StringGrouper(series)
        t1 = time.perf_counter()
        sg.fit()
        t2 = time.perf_counter()
        out = sg.get_matches()
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if step >= args.warmup:
            e2e_s.append(dt)
            e2e_parts = {"validate_s": t1 - t0, "fit_s": t2 - t1, "get_matches_s": t0 + dt - t2}
            e2e_rows = len(out)
            h2d = int(sg._last_stats.get("h2d_bytes", 0))
            d2h = int(D.TRANSFER_BYTES["d2h"] - d2h0)      # match list + gathered strings (small read-backs not counted)
    t_e2e = torch.tensor([sum(e2e_s)], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(t_e2e, op=dist.ReduceOp.MAX)
    e2e_value = e2e_rows / (float(t_e2e.item()) / args.steps)
    # the same call on an object-dtype Series (pandas < 3 users): ingest converts to Arrow first (one extra pass)
    obj_series = series.astype(object)
    barrier()
    t0 = time.perf_counter()
    api.StringGrouper(obj_series).fit().get_matches()
    torch.cuda.synchronize()
    e2e_object_s = time.perf_counter() - t0
    del obj_series
    clocks = sampler.stop() if rank == 0 else None

    # ---- roofline of the dominant kernel chain (K2 candidates) ----
    A = info["A"]
    st = info["stats"]
    idx = A.d_indices[:A.nnz].long()
    df = torch.bincount(idx, minlength=A.shape[1])
    ip = A.d_indptr
    nnz_a_local = int((ip[hi] - ip[lo]).item())
    macs_local = int(df[A.d_indices[int(ip[lo].item()):int(ip[hi].item())].long()].sum().item())
    macs_total = int((df * df).sum().item())
    alg_bytes = 8 * macs_local + 8 * nnz_a_local + 4 * (hi - lo + 1) + 8 * info["k2_nnz_local"] + 4 * (hi - lo + 1)
    k2_ms = float(np.mean(cand_ms))
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "MEASURED_PEAKS.json hbm_gbs (measured)"
    else:
        peak, peak_src = 6650.0, "B200_PROFILING.md fallback"
    # what the launches really read and write: the (row, tile) pairs that survive the block-max test and the postings of
    # their buckets are COUNTED by the tile formulation's kernel on the same input (one untimed run; both formulations
    # apply the same pruning and the same block-max test), the rest follows from the array shapes
    n_loc = hi - lo
    st_walk = {}
    D.cossim_topn(A, A, TOP_N, MIN_SIM, row_begin=lo, row_end=hi, stats=st_walk, kernel="tiles")
    streamed = None
    if st_walk.get("kernel") == "tiles" and st_walk.get("pairs_walked"):
        T = int(st["n_tiles"])
        Tp = (T + 63) // 64 * 64
        pairs_w, post_w = int(st_walk["pairs_walked"]), int(st_walk["postings_walked"])
        feats_per_row = nnz_a_local / max(n_loc, 1)              # upper bound of the kept features per row
        if st.get("kernel") == "tiles":
            streamed = {
                "postings_bytes": 4 * post_w,                          # shared-memory reads of the TMA-staged tile blobs
                "left_rows_bytes": int(pairs_w * (16 + 8 * feats_per_row)),   # row record + {feature, weight} per pair
                "survivor_mask_bytes": 4 * (Tp // 32) * n_loc + 4 * int(st_walk["n_tiles"]) * n_loc,
                "filter_block_maxima_bytes": 2 * Tp * nnz_a_local,     # fp16 block maximum per (kept feature, tile)
                "pack_left_bytes": 24 * nnz_a_local,
                "candidate_bytes": 8 * int(st["n_candidates"])}
        else:
            streamed = {
                "postings_bytes": 4 * post_w,                          # 4-byte postings of the surviving buckets (L2)
                "directory_bytes": int(8 * pairs_w * feats_per_row),   # one 8-byte bucket entry per kept feature and pair
                "filter_block_maxima_bytes": 2 * Tp * nnz_a_local,     # fp16 block maximum per (kept feature, tile) (L2)
                "left_rows_bytes": 12 * nnz_a_local * max(1, (T + int(st.get("tiles_per_group") or T) - 1)
                                                          // int(st.get("tiles_per_group") or T)),
                # row, column and (when the grouped bound re-tests them, `n_refined`) the partial score
                "candidate_bytes": (12 if st.get("n_refined") is not None else 8) * int(st["n_candidates"])}
        streamed["total"] = int(sum(streamed.values()))
        streamed["pairs_walked"], streamed["postings_walked"] = pairs_w, post_w
        streamed["note"] = ("pairs / postings counted by sg::tile_candidates_kernel on the same input; upper bounds where "
                            "the kept-feature count is needed (the pruned rows hold fewer features)")
    traffic = pipe = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and world == 1:      # the ncu capture is a 1-GPU launch over all rows
        traffic = json.load(open(tpath)).get("%d" % n)
    ppath = os.path.join(ROOT, "profiles", "pipe.json")
    if os.path.exists(ppath) and world == 1:
        pipe = json.load(open(ppath)).get("%d" % n)
    bytes_real = streamed["total"] if streamed else None
    achieved = (bytes_real / (k2_ms / 1e3) / 1e9) if bytes_real else None
    alg_gbps = alg_bytes / (k2_ms / 1e3) / 1e9
    roofline = {"bound": "hbm", "kernel": "K2 candidates chain: sg::pack_left + sg::tile_filter + sg::tile_candidates"
                if st.get("kernel") == "tiles" else "sg::cossim_candidates_kernel",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": (achieved / peak) if achieved else None,
                "traffic": traffic, "peak_source": peak_src, "kernel_ms": k2_ms,
                "kernel_share_of_step": k2_ms / float(np.mean(step_ms)),
                "streamed": streamed,
                "note": "achieved/frac = bytes the launches really stream (kernel-counted postings and pairs, array "
                        "sizes for the rest; served by shared memory / L2, DRAM traffic is `traffic`) / CUDA-event time / "
                        "measured HBM copy peak.  The kernel is bound by instruction issue and shared-memory atomics, not by "
                        "HBM: `limiter` holds the ncu pipe utilisation.  `algorithmic` = SURVEY.md §8d bytes of the FULL "
                        "Gustavson traversal over the same time: an algorithmic gain (exact pruning + block-max skipping), "
                        "not a utilisation.",
                "algorithmic": {"bytes_per_launch": alg_bytes, "macs_per_launch": macs_local, "macs_total": macs_total,
                                "GBps_equivalent": alg_gbps, "frac_equivalent": alg_gbps / peak,
                                "gain_vs_streamed": (alg_bytes / bytes_real) if bytes_real else None},
                "limiter": pipe,
                "tile": {k: st.get(k) for k in ("kernel", "tile_w", "warps", "n_tiles", "stage_bytes", "n_candidates",
                                                "n_refined", "n_above_threshold", "prune", "acc")}}

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return 0
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, final_triples, n)

    # ---- CPU port on this box: measured whole job -> cpu_baseline + parity of ALL pairs (N=1 only) ----
    cpu_baseline = parity = None
    if world == 1 and not args.no_cpu_baseline:
        import bench_cpu as C
        job = C.load_cached_job(names)
        if job is None:
            from oracle import pipeline as P
            from oracle import sdt
            sdt.build()
            probe_m, _, _ = P.tf_idf_matrices(names[:60000])
            cores, probe = C.best_thread_count(probe_m)
            job = C.whole_job(names, cores)
        parity = C.compare(job, pre_triples, final_triples)
        parity["cpu_job"] = "measured by this process" if not job.get("from_cache") else \
            "measured by `bench.py --impl reference` on this box earlier in this boot (bench_cpu.CACHE_DIR)"
        cpu_baseline = {"value": job["pairs"] / job["wall_s"], "unit": UNIT, "cores": job["threads"], "kind": "port",
                        "sample": "the WHOLE job, measured once on this box (%d names, n_blocks=%s, %d OpenMP threads; "
                                  "os.cpu_count() = %s, usable = %d): %.1f s, phases %s"
                                  % (n, job["n_blocks"], job["threads"], os.cpu_count(), C.usable_cores(),
                                     job["wall_s"], job["phases"]),
                        "whole_job": C.public(job)}

    line = {"metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "strong",
            "vs_baseline": None, "dtype": "f64", "data": "synthetic",
            "config": workload_config(n, world, sha),
            "workload_stats": {"pairs_per_step": pairs, "nnz": A.nnz, "vocab": A.shape[1]},
            "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                    "s_per_step": float(np.mean(e2e_s)), "s_each_step": [round(x, 4) for x in e2e_s],
                    "rows": e2e_rows, "last_step_parts": e2e_parts,
                    "input": "Arrow-backed pandas `str` Series (zero-copy ingest); object dtype: `object_dtype_s`",
                    "object_dtype_s": e2e_object_s,
                    "result": "every rank" if world == 1 else "rank 0 only (SG_B200_RESULT=rank0)"},
            "gpu_launches": launches // args.steps,
            "phases_ms": {"rank%d" % r: p for r, p in enumerate(phases_all)},
            "shard_check": shard_check, "aux_two_series": aux_two_series,
            "roofline": roofline, "parity": parity, "cpu_baseline": cpu_baseline}
    print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
