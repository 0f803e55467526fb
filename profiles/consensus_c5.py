#!/usr/bin/env python
"""Consensus measures on the device (engine.consensus, csrc/consensus.cuh): dispersion and the
cophenetic correlation of factorize(device_consensus=True).

On planted labels (nrun 20, K 15, each cell relabelled at random with probability p; the
generator of tests/test_api_cpu.py) at 100k and 1.3M cells: the moments-only call and the tree
call end to end (host clock around synchronised calls, after a warm-up call), the kernel times of
the tree call split into grouping (the radix sorts and group_* kernels), IP fill, initial row
cache and merge loop from a torch.profiler pass of its own; G, the triangle's bytes, rescans per
merge and the merge loop's time per merge; the device memory in use after repeated calls; and the
host dispersion_from_labels time where it finishes in reasonable time.  Then one
factorize(ranks=[15], nrun=20, device_consensus=True) on the C5 matrix (20k genes x 100k cells):
the G its restarts produced and its time split between the runs and the consensus calls.
Prints one JSON line (and writes it to --out when given).

    python profiles/consensus_c5.py [--reps 3] [--skip-factorize] [--itmax 200] [--out FILE]"""
import argparse, json, os, sys, time
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..")))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..", "tests")))
import numpy as np, scipy.sparse as sp, torch
import bench
from ccfindr_b200 import api, engine, synth
from qc_c3 import gpu_facts, used_bytes
from test_api_cpu import _label_runs

GROUPING = ("group_", "RadixSort", "DeviceScan")


def kernel_ms(L):
    """Device time per phase of one tree call (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        engine.consensus(L)
        torch.cuda.synchronize()
    out = dict(moments=0.0, grouping=0.0, ip_fill=0.0, row_cache=0.0, merge_loop=0.0)
    for e in prof.events():
        if e.device_type.name != "CUDA":
            continue
        ms = e.time_range.elapsed_us() / 1e3
        if "pair_contingency_kernel" in e.name:
            out["moments"] += ms
        elif any(g in e.name for g in GROUPING):
            out["grouping"] += ms
        elif "ip_fill_kernel" in e.name:
            out["ip_fill"] += ms
        elif "row_best_kernel" in e.name:
            out["row_cache"] += ms
        elif "merge_loop_kernel" in e.name:
            out["merge_loop"] += ms
    return out


def timed(fn, reps):
    fn()
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize(); ts.append(time.perf_counter() - t0)
    return ts


def labels_case(m, p, seed, dev, reps, host):
    L = (np.stack(_label_runs(np.random.default_rng(seed), m, 20, 15, p)) - 1).astype(np.int32)
    out = dict(m=m, nrun=20, K=15, p=p)
    out["moments_s"] = timed(lambda: engine.consensus(L, tree=False), reps)
    res = {}
    out["tree_s"] = timed(lambda: res.update(engine.consensus(L)), reps)
    G = res["ngroups"]
    out.update(G=G, triangle_bytes=8 * G * (G - 1) // 2, rescans=res["rescans"],
               rescans_per_merge=res["rescans"] / max(G - 1, 1))
    out["kernel_ms"] = kernel_ms(L)
    out["merge_loop_us_per_merge"] = out["kernel_ms"]["merge_loop"] * 1e3 / max(G - 1, 1)
    ub = []
    for _ in range(3):
        engine.consensus(L)
        torch.cuda.synchronize()
        ub.append(used_bytes(dev))
    out["used_bytes_after_calls"] = ub
    d, c = api.consensus_from_labels(list(L + 1))
    out.update(dispersion=d, cophenetic=c)
    if host:
        t0 = time.perf_counter()
        out["host_dispersion"] = api.dispersion_from_labels(list(L + 1))
        out["host_dispersion_s"] = time.perf_counter() - t0
    return out


def factorize_c5(wl, dev, itmax):
    n, m = wl["n"], wl["m_per_gpu"]
    colptr, rowidx, values, _ = synth.tenx_like_device(n, m, wl["r_true"], wl["density"],
                                                       wl["seed"], dev)
    X = sp.csc_matrix((values.cpu().numpy().astype(np.float64), rowidx.cpu().numpy(),
                       colptr.cpu().numpy()), shape=(n, m))
    del colptr, rowidx, values
    torch.cuda.empty_cache()
    spent = dict(tree=0.0, moments=0.0, calls=0)
    inner = api.consensus_from_labels

    def timed_consensus(label_runs, tree=True, device=0, max_groups=0):
        t0 = time.perf_counter()
        r = inner(label_runs, tree=tree, device=device, max_groups=max_groups)
        spent["tree" if tree else "moments"] += time.perf_counter() - t0
        spent["calls"] += 1
        return r
    api.consensus_from_labels = timed_consensus
    try:
        obj = api.scNMFSet(X)
        t0 = time.perf_counter()
        api.factorize(obj, ranks=[15], nrun=20, Itmax=itmax, verbose=0, device_consensus=True,
                      store_connectivity=True)
        torch.cuda.synchronize()
        total = time.perf_counter() - t0
    finally:
        api.consensus_from_labels = inner
    L = np.stack(obj.metadata["labels"]) - 1
    G = engine.consensus(L)["ngroups"]
    return dict(n=n, m=m, nnz=int(X.nnz), call="factorize(ranks=[15], nrun=20, Itmax=%d, "
                "device_consensus=True)" % itmax, seconds=total,
                consensus_tree_s=spent["tree"], consensus_moments_s=spent["moments"],
                runs_s=total - spent["tree"] - spent["moments"], G=G,
                measure={k: [float(x) for x in v] for k, v in obj.measure.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--itmax", type=int, default=200)
    ap.add_argument("--skip-factorize", action="store_true")
    ap.add_argument("--out")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    res = dict(workload="engine.consensus (dispersion / cophenetic of factorize)",
               gpu=gpu_facts(dev))
    res["cases"] = [labels_case(100000, 0.01, 3, dev, a.reps, host=True),
                    labels_case(100000, 0.05, 3, dev, a.reps, host=False),
                    labels_case(1300000, 0.01, 7, dev, a.reps, host=False),
                    labels_case(1300000, 0.02, 7, dev, a.reps, host=False)]
    if not a.skip_factorize:
        res["c5_factorize"] = factorize_c5(bench.WORKLOADS["c2"], dev, a.itmax)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
