"""CPU arm of bench.py / bench_configs.py: the reference's CPU implementation of the hot path (the oracle port —
the reference tree holds no native code and `sparse_dot_topn` cannot be installed here, DESIGN.md §2) timed on
this box's host cores.  BENCH / TEST INFRASTRUCTURE: this is the only module besides tests/ and
__graft_entry__.smoke() that executes anything under oracle/, and only as the baseline / the checker.

  whole_job()      ONE measured pass of the reference's match_strings self-match on the whole corpus, phase by
                   phase (/root/reference/string_grouper/string_grouper.py: __init__ :267, fit :380-431,
                   get_matches :443-518), with the true pair count and the match lists for the parity check
  sample_model()   the bounded per-step sample (a 20 000-name fit + two left-row slices against all right rows)
                   and the whole-job estimate it extrapolates to; calibrated against whole_job() by the caller
  compare()        all pairs of the CUDA result against the CPU result (SURVEY.md §8c parity definition)
"""
import hashlib
import json
import os
import socket
import tempfile
import time

import numpy as np

# whole-job results handed from `bench.py --impl reference` to a later bench.py on the same box; kept outside the
# source tree, which the benchmark must leave untouched (it may be read-only)
CACHE_DIR = os.path.join(tempfile.gettempdir(), "string_grouper_b200_cpu_jobs")
TOP_N, MIN_SIM = 20, 0.8


def usable_cores():
    """Host threads this process may really use: affinity mask capped by the cgroup CPU quota (os.cpu_count()
    reports the machine, and OpenMP threads beyond the quota only spin against each other)."""
    try:
        n = len(os.sched_getaffinity(0))
    except AttributeError:
        n = os.cpu_count() or 1
    for path, parse in (("/sys/fs/cgroup/cpu.max", lambda txt: txt.split()),
                        ("/sys/fs/cgroup/cpu/cpu.cfs_quota_us", None)):
        try:
            if parse:
                q, per = parse(open(path).read())
                if q != "max":
                    n = min(n, max(1, int(float(q) / float(per))))
            else:
                q = int(open(path).read())
                per = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, q // per))
        except Exception:
            pass
    return max(1, n)


_THREADS = {}


def best_thread_count(full_matrix, top_n=TOP_N, min_sim=MIN_SIM):
    """The OpenMP thread count at which the oracle's block product runs fastest on this box (probed once on
    8000 left rows x 48000 right rows; candidates: the usable cores and a few fractions of them)."""
    if "n" in _THREADS:
        return _THREADS["n"], _THREADS["probe"]
    from oracle import pipeline as P
    cores = usable_cores()
    cand = sorted({cores, max(1, cores // 2), max(1, cores // 4), min(cores, 32), min(cores, 16), min(cores, 8)})
    nl, nr = min(8000, full_matrix.shape[0]), min(48000, full_matrix.shape[0])
    left, right = full_matrix[:nl], full_matrix[:nr]
    probe = {}
    for c in cand:
        best = 1e30
        for _ in range(2):
            t0 = time.perf_counter()
            P.build_matches(left, right, (1, 12), top_n, min_sim, c)
            best = min(best, time.perf_counter() - t0)
        probe[c] = round(best, 4)
    _THREADS["n"] = min(probe, key=probe.get)
    _THREADS["probe"] = probe
    return _THREADS["n"], probe


def box_id():
    try:
        boot = open("/proc/sys/kernel/random/boot_id").read().strip()
    except Exception:
        boot = "?"
    return "%s/%s" % (socket.gethostname(), boot)


def _cache_path(names, top_n, min_sim):
    h = hashlib.sha256(("\n".join(names[:1000]) + "|%d|%d|%r" % (len(names), top_n, min_sim)).encode()).hexdigest()[:16]
    return os.path.join(CACHE_DIR, "job_%s.npz" % h)


def load_cached_job(names, top_n=TOP_N, min_sim=MIN_SIM, max_age_s=6 * 3600):
    """The whole-job result another bench.py process measured on THIS box (same boot) a short while ago, or None."""
    path = _cache_path(names, top_n, min_sim)
    try:
        z = np.load(path, allow_pickle=False)
        meta = json.loads(str(z["meta"]))
        if meta.get("box") != box_id() or time.time() - meta.get("when", 0) > max_age_s:
            return None
        job = dict(meta)
        job["from_cache"] = True
        for k in ("c_indptr", "c_indices", "c_data", "row", "col", "score"):
            job[k] = z[k]
        return job
    except Exception:
        return None


def whole_job(names, n_threads, top_n=TOP_N, min_sim=MIN_SIM, save=True):
    """ONE measured pass of the reference's `match_strings(series)` on the CPU port, every phase timed.

    Phases follow the reference call stack (SURVEY.md §3.1): the vectoriser is fitted in __init__ (:267 -> :305-308),
    re-fitted and applied in fit() (:687-689) — three analyzer passes; block product with the reference's own block
    guess (:387-394, :709-752); LIL fix-diagonal + symmetrise (:419-427); match list (:755-763); get_matches frame
    (:443-518).  Returns the timings, the pre-symmetrisation product (CSR) and the final match list."""
    import pandas as pd
    from sklearn.feature_extraction.text import TfidfVectorizer
    from oracle import pipeline as P
    from oracle import sdt
    sdt.build()
    n = len(names)
    ph = {}
    t_all = time.perf_counter()
    t0 = time.perf_counter()
    series = pd.Series(names)
    TfidfVectorizer(min_df=1, analyzer=P.n_grams, dtype=np.float64).fit(series)      # __init__ :267
    m, d, _ = P.tf_idf_matrices(names)                                                 # fit() :385 -> :687-689
    ph["vectorise_s"] = time.perf_counter() - t0
    blocks = P.guess_blocks(n, n)
    t0 = time.perf_counter()
    C = P.build_matches(m, d, blocks, top_n, min_sim, n_threads)
    ph["product_s"] = time.perf_counter() - t0
    true_max = int(np.diff(C.indptr).max()) if n else 0
    t0 = time.perf_counter()
    S = P.fix_diagonal_and_symmetrize(C)
    ph["symmetrise_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    ml = P.matches_list(S)
    ph["matches_list_s"] = time.perf_counter() - t0
    t0 = time.perf_counter()
    frame = P.get_matches_frame(series, ml)
    ph["get_matches_s"] = time.perf_counter() - t0
    wall = time.perf_counter() - t_all
    job = {"wall_s": wall, "phases": {k: round(v, 3) for k, v in ph.items()}, "pairs": int(len(frame)),
           "pairs_product": int(C.nnz), "true_max_n_matches": true_max, "threads": int(n_threads),
           "n_blocks": list(blocks), "rows": n, "nnz": int(m.nnz), "vocab": int(m.shape[1]),
           "macs": int(P.hot_path_macs(m, d)), "box": box_id(), "when": time.time(), "from_cache": False}
    arrays = {"c_indptr": C.indptr.astype(np.int64), "c_indices": C.indices.astype(np.int32),
              "c_data": C.data.astype(np.float64), "row": ml.master_side.to_numpy().astype(np.int64),
              "col": ml.dupe_side.to_numpy().astype(np.int64), "score": ml.similarity.to_numpy().astype(np.float64)}
    if save:
        try:
            os.makedirs(CACHE_DIR, exist_ok=True)
            meta = {k: v for k, v in job.items() if k != "from_cache"}
            np.savez(_cache_path(names, top_n, min_sim), meta=np.array(json.dumps(meta)), **arrays)
        except Exception:
            pass
    job.update(arrays)
    job["matrix"] = m
    return job


def public(job):
    """The JSON-able part of a whole_job() result."""
    return {k: job[k] for k in ("wall_s", "phases", "pairs", "pairs_product", "true_max_n_matches", "threads",
                                "n_blocks", "rows", "nnz", "vocab", "macs", "from_cache") if k in job}


def compare(job, pre, final, top_n=TOP_N, min_sim=MIN_SIM, tol=1e-5):
    """All pairs of the CUDA result against the CPU port (SURVEY.md §8c): `pre` = (row, col, score) of the top-n
    product before symmetrisation, `final` = the match list.  A pair held by one side only counts as a boundary tie
    when its score lies within `tol` of min_similarity or of the top-n cut-off of a full row (there the reference's own
    choice depends on heap order and n_blocks); anything else is a mismatch."""
    n = int(job["rows"])
    out = {"tolerance": tol}

    def one(rr, rc, rs, gr, gc, gs, cut_r, cut_c, label):
        rk = rr.astype(np.int64) * n + rc.astype(np.int64)
        gk = np.asarray(gr).astype(np.int64) * n + np.asarray(gc).astype(np.int64)
        ro, go = np.argsort(rk, kind="stable"), np.argsort(gk, kind="stable")
        rk, rs_, rr_, rc_ = rk[ro], rs[ro], rr[ro], rc[ro]
        gk, gs_, gr_, gc_ = gk[go], np.asarray(gs)[go], np.asarray(gr)[go], np.asarray(gc)[go]
        common, ri, gi = np.intersect1d(rk, gk, assume_unique=True, return_indices=True)
        err = float(np.abs(rs_[ri] - gs_[gi]).max()) if len(common) else 0.0

        def exempt(rows, cols, scores):
            ok = np.abs(scores - min_sim) <= tol
            ok |= np.abs(scores - cut_r[rows]) <= tol
            if cut_c is not None:
                ok |= np.abs(scores - cut_c[cols]) <= tol
            return ok

        only_r = np.setdiff1d(np.arange(len(rk)), ri)
        only_g = np.setdiff1d(np.arange(len(gk)), gi)
        ex_r = exempt(rr_[only_r], rc_[only_r], rs_[only_r])
        ex_g = exempt(gr_[only_g], gc_[only_g], gs_[only_g])
        return {"pairs_ref": int(len(rk)), "pairs_gpu": int(len(gk)), "common": int(len(common)),
                "only_ref": int(len(only_r)), "only_gpu": int(len(only_g)),
                "boundary_ties": int(ex_r.sum() + ex_g.sum()),
                "mismatches": int((~ex_r).sum() + (~ex_g).sum()), "max_abs_err": err}

    indptr, data = job["c_indptr"], job["c_data"]
    cnt = np.diff(indptr)
    cut = np.full(n, -np.inf)          # top-n cut-off score of the rows that are full
    nonempty = np.nonzero(cnt > 0)[0]
    if len(nonempty):
        cut[nonempty] = np.minimum.reduceat(data, indptr[:-1][nonempty])   # non-empty rows partition `data` exactly
    cut[cnt < top_n] = -np.inf
    full = np.nonzero(cnt >= top_n)[0]
    rr = np.repeat(np.arange(n, dtype=np.int64), cnt)
    out["product"] = one(rr, job["c_indices"].astype(np.int64), data, pre[0], pre[1], pre[2], cut, None, "product")
    out["match_list"] = one(job["row"], job["col"], job["score"], final[0], final[1], final[2], cut, cut, "final")
    out["rows_at_top_n"] = int(len(full))
    out["ok"] = bool(out["product"]["mismatches"] == 0 and out["match_list"]["mismatches"] == 0
                     and out["product"]["max_abs_err"] <= tol and out["match_list"]["max_abs_err"] <= tol)
    return out


def sample_model(names, full_matrix, n_threads, sample_left=(6000, 30000), sample_self=20000, top_n=TOP_N,
                 min_sim=MIN_SIM):
    """Bounded sample of the reference CPU path, extrapolated to the whole job (the per-step figure of the
    reference arm; bench.py prints its error against the measured whole_job()).

    (a) the oracle's fit() on the first `sample_self` names: analyzer + TfidfVectorizer (2 of the reference's 3
        analyzer passes), block product, LIL symmetrise, match list -> per-string and per-match host costs;
    (b) the block product of the first s1 and the first s2 left rows against ALL right rows with the reference's
        own block heuristic (string_grouper.py:387-389): t(s) = fixed + per_row * s.
    Returns (estimated seconds for the full job, estimated pairs, detail dict)."""
    from oracle import pipeline as P
    n = len(names)
    sample_self = min(sample_self, n)
    t0 = time.perf_counter()
    m, d, _ = P.tf_idf_matrices(names[:sample_self])
    t_vec = time.perf_counter() - t0
    t0 = time.perf_counter()
    C = P.build_matches(m, d, P.guess_blocks(sample_self, sample_self), top_n, min_sim, n_threads)
    t_mm_small = time.perf_counter() - t0
    t0 = time.perf_counter()
    S = P.fix_diagonal_and_symmetrize(C)
    ml = P.matches_list(S)
    t_post = time.perf_counter() - t0
    per_string = 1.5 * t_vec / sample_self            # fit + transform measured; the reference also fits in __init__
    per_match = t_post / max(len(ml), 1)
    blocks = (1, P.guess_blocks(n, n)[1])
    s1, s2 = (min(x, n) for x in sample_left)
    times, nnz_s2 = [], 0
    for sl in (s1, s2):
        t0 = time.perf_counter()
        Cs = P.build_matches(full_matrix[:sl], full_matrix, blocks, top_n, min_sim, n_threads)
        times.append(time.perf_counter() - t0)
        nnz_s2 = Cs.nnz
    if s2 > s1:
        per_row = max((times[1] - times[0]) / (s2 - s1), 0.0)
        fixed = max(times[0] - per_row * s1, 0.0)
    else:
        per_row, fixed = times[0] / max(s1, 1), 0.0
    t_product = fixed + per_row * n
    est_pairs = (nnz_s2 / s2) * n * (len(ml) / max(C.nnz, 1))      # symmetrisation growth from (a)
    est = per_string * n + t_product + per_match * est_pairs
    detail = {"t_vectorise_sample_s": round(t_vec, 3), "t_product_s1_s2_s": [round(x, 3) for x in times],
              "left_rows_s1_s2": [s1, s2], "product_fixed_s": round(fixed, 3),
              "product_per_left_row_us": round(per_row * 1e6, 3), "est_product_s": round(t_product, 2),
              "t_post_sample_s": round(t_post, 3), "t_product_small_s": round(t_mm_small, 3),
              "est_vectorise_s": round(per_string * n, 2), "est_post_s": round(per_match * est_pairs, 2),
              "est_total_s": round(est, 2), "est_pairs": int(est_pairs), "n_blocks": list(blocks),
              "threads": n_threads}
    return est, est_pairs, detail
