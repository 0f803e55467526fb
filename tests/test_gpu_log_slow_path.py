"""The bound term of the fp64 cell-owner pass takes the low three bits of every count through
products and the rest of a larger count through a log, after p is formed again from the tile row
and the owner row.  These tests put counts up to 65535 through that slow path where the kernel
differs from the r = 10 case of test_gpu_parity.py: the split layout with 4-lane groups (r = 18,
20) and two lanes per nonzero (r = 30), with small tiles so that several slabs are walked."""
import numpy as np
import pytest
import scipy.sparse as sp

from conftest import relerr

pytestmark = pytest.mark.gpu
FACT = ("lw", "lh", "ew", "eh", "dw", "dh")
TOL = 1e-9
COUNTS = [1, 2, 3, 7, 8, 9, 15, 16, 255, 4096, 65535]


@pytest.mark.parametrize("r", [18, 20, 30])
def test_large_counts_take_the_log_slow_path(monkeypatch, r):
    import torch
    assert torch.cuda.is_available(), "this test needs a CUDA device"
    from ccfindr_b200 import synth
    from ccfindr_b200.engine import Engine
    from oracle import bindings as ob
    from oracle import oracle_dense as od
    monkeypatch.setenv("VBNMF_TILE_ROWS", "160")
    rng = np.random.default_rng(90 + r)
    n, m = 700, 900
    X = sp.random(n, m, density=0.08, random_state=rng, format="csc",
                  data_rvs=lambda k: rng.choice(COUNTS, size=k).astype(float))
    X = synth.fix_empty(X, r)
    w0 = rng.gamma(1.0, 1.0, size=(n, r)) + 1e-3
    h0 = rng.gamma(1.0, 1.0, size=(r, m)) + 1e-3
    hyper = dict(aw=0.9, bw=1.1, ah=1.2, bh=0.8)
    ref = od.vb_init_from(w0, h0)
    with Engine(X) as eng:
        eng.set_state(w0, h0)
        info = eng.layout_info()
        assert info["format"] == "p16"
        assert info["tile_rows"] == 160 and info["gene_slabs"] == 5 and info["cell_slabs"] == 6
        assert info["nonzeros_per_group_step"] == 4
        for it in range(3):
            ref = ob.sparse_vb_step(X, ref, hyper, od.EPS)
            assert relerr(eng.step(hyper, od.EPS), ref["lkh"]) < TOL, it
        st = eng.get_state()
        cid = eng.cluster_id()
    for k in FACT:
        assert relerr(st[k], ref[k]) < TOL, k
    assert np.array_equal(cid, od.cluster_id(ref["eh"]))
