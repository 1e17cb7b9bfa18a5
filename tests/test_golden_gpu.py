"""CUDA path vs the committed golden fixtures (answers produced by the reference itself,
tests/golden/make_golden.py) — runs on the GPU box where /root/reference does not exist."""
import os

import numpy as np
import pytest

from knowhere_b200 import datagen
from tests.test_oracle_cpu import _lists
from tests.util import assert_topk_parity

pytestmark = pytest.mark.gpu
G = os.path.join(os.path.dirname(__file__), "golden")


def test_golden_flat_gpu(kb):
    z = np.load(os.path.join(G, "flat_1000x128.npz"))
    xb, xq = datagen.uniform(1000, 128, 42), datagen.uniform(10, 128, 43)
    for metric, name in (("L2", "l2"), ("IP", "ip")):
        ids, dist = kb.brute_force_search(xb, xq, 10, metric)
        assert np.array_equal(ids, z[f"flat_{name}_ids"])       # bit-exact labels
        assert np.array_equal(ids, z[f"bf_{name}_ids"])
        np.testing.assert_allclose(dist, z[f"flat_{name}_dist"], rtol=1e-5)


@pytest.mark.parametrize("name,metric", [("l2", "L2"), ("ip", "IP")])
def test_golden_ivf_gpu(kb, name, metric):
    z = np.load(os.path.join(G, f"ivf_4000x64_{name}.npz"))
    nb, d, nq, k, nprobe, m = 4000, 64, 20, 10, 4, 8
    xb, xq = datagen.clustered(nb, d, 42), datagen.clustered(nq, d, 43)
    ix = kb.Index("IVF_FLAT", metric, d, {"nlist": 16})
    L = _lists(z, "ivf_flat", d * 4, xb)
    ix.ivf_import(z["ivf_flat_centroids"], None, [(l,) + L[l] for l in sorted(L)])
    ids, dist = ix.search(xq, k, {"nprobe": nprobe})
    assert_topk_parity(ids, dist, z["ivf_flat_ids"], z["ivf_flat_dist"], what="golden IVF_FLAT")
    ix = kb.Index("IVF_PQ", metric, d, {"nlist": 16, "m": m, "refine": True, "refine_type": "flat"})
    L = _lists(z, "ivf_pq", m)
    ix.ivf_import(z["ivf_pq_centroids"], z["ivf_pq_pq"], [(l,) + L[l] for l in sorted(L)], raw=xb)
    ids, dist = ix.search(xq, k, {"nprobe": nprobe, "refine_k": 4})
    assert_topk_parity(ids, dist, z["ivf_pq_refine4_ids"], z["ivf_pq_refine4_dist"], what="golden IVF_PQ refine")
    ix2 = kb.Index("IVF_PQ", metric, d, {"nlist": 16, "m": m})
    ix2.ivf_import(z["ivf_pq_centroids"], z["ivf_pq_pq"], [(l,) + L[l] for l in sorted(L)])
    ids, dist = ix2.search(xq, k, {"nprobe": nprobe})
    assert_topk_parity(ids, dist, z["ivf_pq_ids"], z["ivf_pq_dist"], rtol=1e-4, atol=1e-3, what="golden IVF_PQ",
                       max_tie_rows=nq // 4)


@pytest.mark.parametrize("name,metric", [("l2", "L2"), ("ip", "IP")])
def test_golden_hnsw_gpu(kb, name, metric):
    z = np.load(os.path.join(G, f"hnsw_3000x32_{name}.npz"))
    xb, xq = datagen.clustered(3000, 32, 42), datagen.clustered(20, 32, 43)
    ix = kb.Index("HNSW", metric, 32, {"M": 8})
    ix.hnsw_import(xb, z["levels"], z["offsets"], z["neighbors"], z["cum"], int(z["entry_point"]), int(z["max_level"]))
    ids, dist = ix.search(xq, 10, {"ef": 32})
    assert (ids == z["ids"]).mean() > 0.98
    eq = ids == z["ids"]
    np.testing.assert_allclose(dist[eq], z["dist"][eq], rtol=1e-4, atol=1e-4)
