#!/usr/bin/env python
"""Column shuffle on the device (Engine.shuffle, csrc/shuffle.cuh): the null matrices of
factorize(randomize=True, device_shuffle=True).

Times Engine.shuffle end to end (kernel + scan_matrix + allocation, host clock around a
synchronised call, after one warm-up call) on the C2/C5 matrix (20k genes x 100k cells, ~1.6e8
nonzeros) and on a C3-sized one (20k x 1.3M, ~2.07e9), both generated on the GPU by
synth.tenx_like_device; the shuffle kernel alone from a torch.profiler pass of its own.  Reports
bytes per nonzero over time as a share of HBM bandwidth, the device memory the source and the
shuffled handle hold at C3, and one factorize(randomize=True, device_shuffle=True, ranks=[15],
nrun=1, nsmpl=2, Itmax=50) at C5.  Prints one JSON line (and writes it to --out when given).

    python profiles/shuffle_c5.py [--reps 5] [--skip-c3] [--skip-factorize] [--out FILE]"""
import argparse, json, os, sys, time
HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.abspath(os.path.join(HERE, "..")))
sys.path.insert(0, HERE)
import numpy as np, scipy.sparse as sp, torch
import bench
from ccfindr_b200 import api, synth
from ccfindr_b200.engine import Engine, trim_pool
from qc_c3 import gpu_facts, used_bytes


def traffic_bytes(nnz, m, val_bytes=4):
    """The kernel's bytes: values read and written, s_t written and read back, rows written (the
    rows of the source are not read), colptr read; plus the colptr copy."""
    return nnz * (2 * val_bytes + 4 + 4 + 4) + 8 * (m + 1) * 3


def kernel_ms(eng, seed):
    """Device time of the shuffle kernel in one Engine.shuffle call (torch.profiler)."""
    from torch.profiler import ProfilerActivity, profile
    with profile(activities=[ProfilerActivity.CUDA]) as prof:
        eng.shuffle(seed).close()
        torch.cuda.synchronize()
    ev = [e for e in prof.events() if "shuffle_columns_kernel" in e.name]
    assert len(ev) == 1, [e.name for e in prof.events()]
    return ev[0].time_range.elapsed_us() / 1e3


def shuffle_case(n, m, wl, dev, reps, hbm_gbs, memory=False):
    trim_pool(dev.index)
    torch.cuda.empty_cache()
    base = used_bytes(dev)
    colptr, rowidx, values, _ = synth.tenx_like_device(n, m, wl["r_true"], wl["density"],
                                                       wl["seed"], dev)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()
    nnz = int(rowidx.numel())
    out = dict(n=n, m=m, nnz=nnz)
    with Engine.from_device_csc(n, m, nnz, colptr, rowidx, values) as src:
        ts = []
        src.shuffle(1).close()   # warm-up
        for i in range(reps):
            torch.cuda.synchronize(); t0 = time.perf_counter()
            sh = src.shuffle(100 + i)
            torch.cuda.synchronize(); ts.append(time.perf_counter() - t0)
            sh.close()
        out["shuffle_s"] = ts
        out["kernel_ms"] = kernel_ms(src, 7)
        if memory:
            trim_pool(dev.index)
            with_src = used_bytes(dev)
            with src.shuffle(8) as sh:
                trim_pool(dev.index)
                out["shuffled_handle_bytes"] = used_bytes(dev) - with_src
            out["source_bytes"] = with_src - base   # CSC tensors + the source handle's own arrays
            out["both_handles_bytes"] = out["source_bytes"] + out["shuffled_handle_bytes"]
    b = traffic_bytes(nnz, m)
    out["kernel_bytes"] = b
    out["kernel_bytes_per_nnz"] = b / nnz
    out["kernel_share_of_hbm"] = b / (out["kernel_ms"] / 1e3) / (hbm_gbs * 1e9)
    out["end_to_end_share_of_hbm"] = b / min(ts) / (hbm_gbs * 1e9)
    del colptr, rowidx, values
    torch.cuda.empty_cache()
    return out


def factorize_c5(wl, dev):
    n, m = wl["n"], wl["m_per_gpu"]
    colptr, rowidx, values, _ = synth.tenx_like_device(n, m, wl["r_true"], wl["density"],
                                                       wl["seed"], dev)
    X = sp.csc_matrix((values.cpu().numpy().astype(np.float64), rowidx.cpu().numpy(),
                       colptr.cpu().numpy()), shape=(n, m))
    del colptr, rowidx, values
    torch.cuda.empty_cache()
    obj = api.scNMFSet(X)
    t0 = time.perf_counter()
    api.factorize(obj, ranks=[15], nrun=1, randomize=True, nsmpl=2, Itmax=50, verbose=0,
                  device_shuffle=True)
    torch.cuda.synchronize()
    return dict(n=n, m=m, nnz=int(X.nnz), call="factorize(ranks=[15], nrun=1, randomize=True, "
                "nsmpl=2, Itmax=50, device_shuffle=True)", seconds=time.perf_counter() - t0,
                measure={k: [float(x) for x in v] for k, v in obj.measure.items()})


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=5)
    ap.add_argument("--skip-c3", action="store_true")
    ap.add_argument("--skip-factorize", action="store_true")
    ap.add_argument("--out")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    c2, c3 = bench.WORKLOADS["c2"], bench.WORKLOADS["c3"]
    facts = gpu_facts(dev)
    hbm = facts["hbm_gbs_device_attributes"]   # shares of peak are taken against this
    res = dict(workload="Engine.shuffle (column shuffle of factorize(randomize=True))", gpu=facts)
    res["c5_shuffle"] = shuffle_case(c2["n"], c2["m_per_gpu"], c2, dev, a.reps, hbm)
    if not a.skip_c3:
        res["c3_shuffle"] = shuffle_case(c3["n"], c3["m_total"], c3, dev, a.reps, hbm, memory=True)
    if not a.skip_factorize:
        res["c5_factorize"] = factorize_c5(c2, dev)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
