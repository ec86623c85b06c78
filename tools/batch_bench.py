"""Batched fits against the loop of ordinary fits (DESIGN.md §4d), one GPU, everything in one process.

    python tools/batch_bench.py --out profiles/r03_batch.jsonl

W1  B = 1024 distinct configs[0]-shaped problems (20x8x6, M=1, R=3, fp64, synthetic seeds 0..1023):
    fit_batch against a loop of tPLS.fit, fits per second.
W2  leave-one-out Q2Y of one 200x22x6 fp64 problem (M=4, R=5, 200 folds): q2y_sweep with algorithm="batch"
    against "covariance" and "stream".
W3  B = 148 problems (one per SM) of n x 32 x 16 fp64 whose per-problem working set is about 0.1, 1, 4, 16 and
    64 MB, through the batch kernel (TPLS_BATCH_MB raised so that it takes all of them) and through the loop: where
    the default TPLS_BATCH_MB threshold comes from.
Every timed configuration is warmed up first and every clock is read after a device synchronise; outputs of the
batch path are compared with the loop's (max aligned error, equal trips).  One JSON line per measurement, the card's
name and power limit in every line.
"""

import argparse
import json
import os
import subprocess
import sys
import time

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))


def card():
    q = subprocess.run(["nvidia-smi", "--query-gpu=name,power.limit,clocks.max.sm", "--format=csv,noheader"],
                       capture_output=True, text=True).stdout.strip().splitlines()
    name, power, clk = [s.strip() for s in q[0].split(",")]
    return dict(gpu=name, power_limit=power, max_sm_clock=clk)


def state(est):
    if hasattr(est, "Xs_factors"):
        return dict(T=est.factor_T, W=[f[1:] for f in est.Xs_factors], U=est.Y_factors[0], Q=est.Y_factors[1],
                    coef=est.coef_, R2X=est.R2Xs, R2Y=est.R2Y)
    return dict(T=est.X_factors[0], W=[est.X_factors[1:]], U=est.Y_factors[0], Q=est.Y_factors[1],
                coef=est.coef_, R2X=[est.R2X], R2Y=est.R2Y)


def parity(batch_models, loop_models):
    from cmtf_pls_b200.selfcheck import aligned_errors
    worst, same_trips = 0.0, True
    for a, b in zip(batch_models, loop_models):
        same_trips &= a.n_iter_.tolist() == b.n_iter_.tolist()
        worst = max(worst, max(aligned_errors(state(a), state(b)).values()))
    return dict(max_aligned_err=worst, equal_trips=bool(same_trips))


def timed(fn, sync, reps):
    out, best = None, float("inf")
    for _ in range(reps):
        sync()
        t0 = time.perf_counter()
        out = fn()
        sync()
        best = min(best, time.perf_counter() - t0)
    return out, best


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--out", default=os.path.join(ROOT, "profiles", "r03_batch.jsonl"))
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--w3-sizes", default="0.1,1,4,16,64")
    args = ap.parse_args()
    import torch
    from cmtf_pls_b200 import fit_batch, q2y_sweep, tPLS
    from oracle import tpls_oracle as orc
    if not torch.cuda.is_available():
        raise SystemExit("no GPU: nothing to measure")
    info = card()
    sync = torch.cuda.synchronize
    os.makedirs(os.path.dirname(os.path.abspath(args.out)), exist_ok=True)
    f = open(args.out, "w")

    def emit(rec):
        rec.update(info)
        line = json.dumps(rec)
        print(line, flush=True)
        f.write(line + "\n")
        f.flush()

    # ---- W1 ----
    B = 1024
    Xs, Ys = [], []
    for s in range(B):
        X, Y, _ = orc.synthetic((20, 8, 6), 1, 3, error=1.0, seed=s)
        Xs.append(X)
        Ys.append(Y)
    Xb, Yb = np.stack(Xs), np.stack(Ys)
    fit_batch(Xb[:8], Yb[:8], 3)
    tPLS(3).fit(Xs[0], Ys[0])

    def loop():
        ms = []
        for X, Y in zip(Xs, Ys):
            m = tPLS(3)
            m.fit(X, Y)
            ms.append(m)
        return ms
    bm, tb = timed(lambda: fit_batch(Xb, Yb, 3), sync, args.reps)
    lm, tl = timed(loop, sync, args.reps)
    emit(dict(workload="W1", B=B, shape=[20, 8, 6], M=1, R=3, dtype="float64", path=bm[0].stats_["batch"],
              batch_s=tb, loop_s=tl, batch_fits_per_s=B / tb, loop_fits_per_s=B / tl, speedup=tl / tb,
              batch_kernel_ms=bm[0].stats_.get("batch_fit_ms"), **parity(bm, lm)))

    # ---- W2 ----
    X, Y, _ = orc.synthetic((200, 22, 6), 4, 5, error=1.0, seed=7)
    res = {}
    for alg in ("batch", "covariance", "stream"):
        q2y_sweep(X[:40], Y[:40], 5, n_splits=None, algorithm=alg)   # warm-up (a smaller sweep)
        res[alg] = timed(lambda: q2y_sweep(X, Y, 5, n_splits=None, algorithm=alg), sync, args.reps)
    emit(dict(workload="W2", folds=200, shape=[200, 22, 6], M=4, R=5, dtype="float64",
              batch_s=res["batch"][1], covariance_s=res["covariance"][1], stream_s=res["stream"][1],
              speedup_vs_covariance=res["covariance"][1] / res["batch"][1],
              speedup_vs_stream=res["stream"][1] / res["batch"][1],
              max_q2_diff_vs_covariance=float(np.max(np.abs(res["batch"][0] - res["covariance"][0]))),
              max_q2_diff_vs_stream=float(np.max(np.abs(res["batch"][0] - res["stream"][0])))))

    # ---- W3 ----
    G = torch.Generator(device="cuda")
    for mb in [float(v) for v in args.w3_sizes.split(",")]:
        n = max(8, int(round(mb * 1048576 / (32 * 16 * 8))))
        G.manual_seed(int(mb * 1000) + 3)
        P = 148
        T = torch.randn(P, n, 3, device="cuda", dtype=torch.float64, generator=G)
        A = torch.randn(P, 32, 3, device="cuda", dtype=torch.float64, generator=G)
        C = torch.randn(P, 16, 3, device="cuda", dtype=torch.float64, generator=G)
        Xd = torch.einsum("bnr,bjr,bkr->bnjk", T, A, C) + torch.randn(P, n, 32, 16, device="cuda", dtype=torch.float64,
                                                                         generator=G)
        Yd = T @ torch.randn(P, 3, 2, device="cuda", dtype=torch.float64, generator=G) + \
            0.5 * torch.randn(P, n, 2, device="cuda", dtype=torch.float64, generator=G)
        os.environ["TPLS_BATCH_MB"] = "100000"
        fit_batch(Xd[:2], Yd[:2], 3)
        bm, tb = timed(lambda: fit_batch(Xd, Yd, 3), sync, args.reps)
        os.environ.pop("TPLS_BATCH_MB")

        def loop3():
            ms = []
            for b in range(P):
                m = tPLS(3)
                m.fit(Xd[b], Yd[b])
                ms.append(m)
            return ms
        tPLS(3).fit(Xd[0], Yd[0])
        lm, tl = timed(loop3, sync, max(1, args.reps - 1))
        emit(dict(workload="W3", B=P, shape=[n, 32, 16], M=2, R=3, dtype="float64", working_set_mb=mb,
                  path=bm[0].stats_["batch"], batch_s=tb, loop_s=tl, speedup=tl / tb,
                  batch_kernel_ms=bm[0].stats_.get("batch_fit_ms"), **parity(bm, lm)))
        del Xd, Yd, T, A, C, bm, lm
        torch.cuda.empty_cache()
    f.close()


if __name__ == "__main__":
    main()
