#!/usr/bin/env python
"""Cell / gene QC on the device at C3 size (20k genes x 1.3M cells, ~2.07e9 nonzeros, built on
the GPU by synth.tenx_like_device): times Engine.qc_stats and Engine.subset (keep ~90 % of the
cells and genes) with the host clock around synchronised calls, after one warm-up call each.
Also records the device memory the subset handle adds next to its source, and, for comparison,
the same QC steps with scipy on the host cores at C2 size (20k x 100k, ~1.6e8 nonzeros).
Prints one JSON line (and writes it to --out when given).

    python profiles/qc_c3.py [--reps 3] [--skip-host] [--out FILE]"""
import argparse, json, os, subprocess, sys, time
sys.path.insert(0, os.path.abspath(os.path.join(os.path.dirname(__file__), "..")))
import numpy as np, scipy.sparse as sp, torch
import bench
from ccfindr_b200 import synth
from ccfindr_b200.engine import Engine, trim_pool

DATASHEET_HBM_GBS = 7700.0  # HGX B200 data sheet, one GPU


def gpu_facts(dev):
    p = torch.cuda.get_device_properties(dev)
    q = subprocess.run(["nvidia-smi", "-i", str(dev.index), "--query-gpu=name,power.limit,clocks.max.sm",
                        "--format=csv,noheader"], capture_output=True, text=True).stdout.strip()
    # 2 transfers per memory clock (kHz) x bus width (bits) / 8
    attr_gbs = 2.0 * p.memory_clock_rate * 1e3 * p.memory_bus_width / 8 / 1e9
    return dict(name=p.name, nvidia_smi=q, hbm_gbs_device_attributes=attr_gbs,
                hbm_gbs_datasheet=DATASHEET_HBM_GBS)


def used_bytes(dev):
    free, total = torch.cuda.mem_get_info(dev)
    return total - free


def timed(fn, reps):
    fn()  # warm-up
    ts = []
    for _ in range(reps):
        torch.cuda.synchronize(); t0 = time.perf_counter()
        fn()
        torch.cuda.synchronize(); ts.append(time.perf_counter() - t0)
    return ts


def device_qc(n, m, wl, dev, reps, keep=0.9):
    colptr, rowidx, values, _ = synth.tenx_like_device(n, m, wl["r_true"], wl["density"],
                                                       wl["seed"], dev)
    nnz = int(rowidx.numel())
    rng = np.random.default_rng(1)
    rows, cols = rng.random(n) < keep, rng.random(m) < keep
    out = dict(n=n, m=m, nnz=nnz)
    with Engine.from_device_csc(n, m, nnz, colptr, rowidx, values) as eng:
        t_stats = timed(eng.qc_stats, reps)

        def sub():
            eng.subset(rows, cols).close()
        t_sub = timed(sub, reps)
        # the engine's memory pool keeps freed blocks: trim it so that the difference in device
        # memory in use is what the subset handle holds (before the second trim: plus the
        # temporaries of its creation)
        trim_pool(dev.index)
        before = used_bytes(dev)
        with eng.subset(rows, cols) as s:
            peak = used_bytes(dev) - before
            trim_pool(dev.index)
            held = used_bytes(dev) - before
            out["subset_nnz"] = s.nnz
        out.update(stats_s=t_stats, subset_s=t_sub, subset_bytes_held=held,
                   subset_bytes_with_creation_temporaries=peak,
                   device_bytes_in_use_before_subset=before)
    b_stats = 8 * nnz + 8 * (m + 1)  # rowidx + fp32 values + colptr, one pass
    out["stats_bytes_per_pass"] = b_stats
    out["stats_gbs"] = b_stats / min(t_stats) / 1e9
    del colptr, rowidx, values
    torch.cuda.empty_cache()
    return out


def host_qc_c2(wl, dev):
    n, m = wl["n"], wl["m_per_gpu"]
    colptr, rowidx, values, _ = synth.tenx_like_device(n, m, wl["r_true"], wl["density"],
                                                       wl["seed"], dev)
    X = sp.csc_matrix((values.cpu().numpy().astype(np.float64), rowidx.cpu().numpy(),
                       colptr.cpu().numpy()), shape=(n, m))
    del colptr, rowidx, values
    torch.cuda.empty_cache()
    t = {}

    def tm(name, f):
        t0 = time.perf_counter(); r = f(); t[name] = time.perf_counter() - t0
        return r
    umi = tm("cell_sums", lambda: np.asarray(X.sum(axis=0)).ravel())
    tm("gene_sums", lambda: np.asarray(X.sum(axis=1)).ravel())
    tm("gene_sumsq", lambda: np.asarray(X.multiply(X).sum(axis=1)).ravel())
    tm("cells_expressed", lambda: np.diff((X > 0).tocsr().indptr))
    rng = np.random.default_rng(1)
    gi, ci = np.flatnonzero(rng.random(n) < 0.9), np.flatnonzero(rng.random(m) < 0.9)
    tm("subset", lambda: X[gi][:, ci])
    tm("scale_columns", lambda: X @ sp.diags(np.median(umi) / umi))
    return dict(n=n, m=m, nnz=int(X.nnz), seconds=t, total_s=sum(t.values()),
                host_cores=os.cpu_count(), threads="one (scipy.sparse is single-threaded)")


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--reps", type=int, default=3)
    ap.add_argument("--skip-host", action="store_true")
    ap.add_argument("--out")
    a = ap.parse_args()
    assert torch.cuda.is_available(), "needs a CUDA device"
    dev = torch.device("cuda", 0)
    facts = gpu_facts(dev)
    c3, c2 = bench.WORKLOADS["c3"], bench.WORKLOADS["c2"]
    res = dict(workload="QC: qc_stats + subset(~90% of genes and cells)", gpu=facts)
    res["c2_device"] = device_qc(c2["n"], c2["m_per_gpu"], c2, dev, a.reps)
    res["c3_device"] = device_qc(c3["n"], c3["m_total"], c3, dev, a.reps)
    for k in ("c2_device", "c3_device"):
        res[k]["stats_share_of_hbm_attr"] = res[k]["stats_gbs"] / facts["hbm_gbs_device_attributes"]
    if not a.skip_host:
        res["c2_host_scipy"] = host_qc_c2(c2, dev)
    line = json.dumps(res)
    print(line)
    if a.out:
        with open(a.out, "w") as f:
            f.write(line + "\n")


if __name__ == "__main__":
    main()
