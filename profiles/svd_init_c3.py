#!/usr/bin/env python
"""The SVD initialisers on the device (Engine.init_svd, Engine.init_svd2; csrc/svd_init.cuh) at
C2 size (20k genes x 100k cells, ~1.6e8 nonzeros, rank 10) and C3 size (20k x 1.3M, ~2.07e9,
rank 20), both generated on the GPU by synth.tenx_like_device.  Times each call end to end (host
clock around a synchronised call, after one warm-up call) and counts, in a torch.profiler pass of
its own, the SpMM passes over the matrix (spmm_x_kernel: Y = X Z, spmm_xt_kernel: Z = X^T Y)
and the subspace iterations: every pass of the loop starts with one X^T Y, and one more closes
it, so iterations = X^T Y passes - 1 (a retry without oversampling would show as a second
gauss_fill_kernel).  For comparison, the host path vb_init(..., 'svd') (scipy ARPACK svds on a
float64 copy) at C2 size in a child process stopped after --host-cap-s seconds.  The card's name
and power limit are read in the same run.  Prints one JSON line and writes it to --out.

    python profiles/svd_init_c3.py [--reps 3] [--skip-c3] [--host-cap-s 600] [--out FILE]"""
import argparse, json, multiprocessing as mp, os, sys, time
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..")))
sys.path.insert(0, HERE)
import numpy as np, scipy.sparse as sp, torch
import bench
from ccfindr_b200 import api, synth
from ccfindr_b200.engine import Engine, trim_pool
from qc_c3 import gpu_facts, timed

HYPER = dict(aw=1.0, bw=1.0, ah=1.0, bh=1.0)


def kernel_counts(fn):
    """Launches of the SVD kernels in one call, from torch.profiler."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        fn()
        torch.cuda.synchronize()
    names = ("spmm_x_kernel", "spmm_xt_kernel", "gauss_fill_kernel", "gram_part_kernel")
    cnt = {k: 0 for k in names}
    ms = {k: 0.0 for k in names}
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        for k in names:
            if k + "<" in e.name or e.name.endswith(k) or (k + "(") in e.name:
                cnt[k] += 1
                ms[k] += e.time_range.elapsed_us() / 1e3
    return dict(x_passes=cnt["spmm_x_kernel"], xt_passes=cnt["spmm_xt_kernel"],
                sketches=cnt["gauss_fill_kernel"], gram_launches=cnt["gram_part_kernel"],
                subspace_iterations=cnt["spmm_xt_kernel"] - cnt["gauss_fill_kernel"],
                spmm_x_ms=ms["spmm_x_kernel"], spmm_xt_ms=ms["spmm_xt_kernel"])


def device_case(wl, m, rank, dev, reps):
    n = wl["n"]
    trim_pool(dev.index)
    torch.cuda.empty_cache()
    colptr, rowidx, values, _ = synth.tenx_like_device(n, m, wl["r_true"], wl["density"],
                                                       wl["seed"], dev)
    torch.cuda.synchronize()
    nnz = int(rowidx.numel())
    out = dict(n=n, m=m, nnz=nnz, rank=rank)
    with Engine.from_device_csc(n, m, nnz, colptr, rowidx, values) as eng:
        calls = dict(init_svd=lambda: eng.init_svd(rank, seed=1),
                     init_svd2=lambda: eng.init_svd2(rank, HYPER, seed=1))
        for name, fn in calls.items():
            ts = timed(fn, reps)
            out[name] = dict(seconds=ts, best_s=min(ts), **kernel_counts(fn))
        eng.init_svd(rank, seed=1)             # the last call was init_svd2
        st = eng.get_state(("lw", "lh"))
        out["init_svd_finite"] = bool(np.isfinite(st["lw"]).all() and np.isfinite(st["lh"]).all())
        out["init_svd_nonneg_k_ge_1"] = bool((st["lw"][:, 1:] >= 0).all() and (st["lh"][1:] >= 0).all())
    host = None
    if m == wl.get("m_per_gpu"):
        host = sp.csc_matrix((values.cpu().numpy().astype(np.float64), rowidx.cpu().numpy(),
                              colptr.cpu().numpy()), shape=(n, m))
    del colptr, rowidx, values
    torch.cuda.empty_cache()
    return out, host


def _host_svd(X, rank, q):
    t0 = time.perf_counter()
    w, h = api.vb_init(X.shape[0], X.shape[1], X, rank, HYPER, "svd", seed=1)
    q.put(dict(seconds=time.perf_counter() - t0, finite=bool(np.isfinite(w).all() and np.isfinite(h).all())))


def host_case(X, rank, cap_s):
    """api.vb_init(..., 'svd') in a forked child (it uses no CUDA) stopped after cap_s seconds."""
    ctx = mp.get_context("fork")
    q = ctx.Queue()
    p = ctx.Process(target=_host_svd, args=(X, rank, q))
    t0 = time.perf_counter()
    p.start()
    p.join(cap_s)
    if p.is_alive():
        p.terminate()
        p.join()
        return dict(finished=False, cap_s=cap_s, elapsed_s=time.perf_counter() - t0,
                    host_cpus=os.cpu_count())
    res = q.get() if not q.empty() else {}
    return dict(finished=p.exitcode == 0 and bool(res), cap_s=cap_s, host_cpus=os.cpu_count(), **res)


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--skip-c3", action="store_true")
    ap.add_argument("--host-cap-s", type=float, default=600.0, help="0: no host comparison")
    ap.add_argument("--out", default=os.path.join(HERE, "svd_init_c3_1gpu.json"))
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    c2, c3 = bench.WORKLOADS["c2"], bench.WORKLOADS["c3"]
    res = dict(workload="Engine.init_svd / Engine.init_svd2 (vb_init 'svd' / 'svd2' on the device)",
               gpu=gpu_facts(dev))
    res["c2"], X = device_case(c2, c2["m_per_gpu"], c2["rank"], dev, a.reps)
    if not a.skip_c3:
        res["c3"], _ = device_case(c3, c3["m_total"], c3["rank"], dev, max(1, a.reps - 1))
    if a.host_cap_s > 0:
        res["c2_host_vb_init_svd"] = host_case(X, c2["rank"], a.host_cap_s)
    line = json.dumps(res)
    print(line)
    with open(a.out, "w") as f:
        f.write(line + "\n")


if __name__ == "__main__":
    main()
