"""Generates tests/golden/*.npz from the REFERENCE itself (oracle/_ref, compiled by oracle/build_ref.py).
Run where the reference sources exist:  python tests/golden/make_golden.py
Inputs are regenerated from seeds by knowhere_b200.datagen; fixtures hold the reference's trained
state and its answers, so the GPU box can check both the numpy oracle and the CUDA path without
/root/reference."""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from knowhere_b200 import datagen  # noqa: E402
from oracle import ref  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))


def flat():
    # shape of the reference's own integration test (tests/ut/test_search.cc:57-80: nb=1000 nq=10 dim=128)
    xb, xq = datagen.uniform(1000, 128, 42), datagen.uniform(10, 128, 43)
    out = {}
    for metric, name in ((0, "l2"), (1, "ip")):
        I, D = ref.flat_search(xb, xq, 10, metric)
        I2, D2 = ref.bruteforce_search(xb, xq, 10, metric)
        out[f"flat_{name}_ids"], out[f"flat_{name}_dist"] = I, D
        out[f"bf_{name}_ids"], out[f"bf_{name}_dist"] = I2, D2
    lims, ids, dis = ref.flat_range_search(xb, xq, float(np.median(out["flat_l2_dist"][:, 5])), 0)
    out.update(range_radius=np.float32(np.median(out["flat_l2_dist"][:, 5])), range_lims=lims, range_ids=ids,
               range_dist=dis)
    np.savez_compressed(os.path.join(OUT, "flat_1000x128.npz"), **out)


def ivf():
    nb, d, nlist, m, nq, k, nprobe = 4000, 64, 16, 8, 20, 10, 4
    xb, xq = datagen.clustered(nb, d, 42), datagen.clustered(nq, d, 43)
    for metric, name in ((0, "l2"), (1, "ip")):
        out = {}
        for kind in ("IVF_FLAT", "IVF_PQ"):
            r = ref.RefIvf(kind, d, metric, nlist, m if kind == "IVF_PQ" else 0, 8, refine=(kind == "IVF_PQ"))
            r.train(xb)
            r.add(xb)
            tag = kind.lower()
            out[f"{tag}_centroids"] = r.centroids()
            if kind == "IVF_PQ":
                out[f"{tag}_pq"] = r.pq_centroids()
                out[f"{tag}_use_precomputed_table"] = np.int32(r.use_precomputed_table())
            sizes, ids_all, codes_all = [], [], []
            for l, ids, codes in r.lists():
                sizes.append(len(ids))
                ids_all.append(ids)
                codes_all.append(codes.reshape(-1))
            out[f"{tag}_list_sizes"] = np.array(sizes, np.int64)
            out[f"{tag}_list_ids"] = np.concatenate(ids_all)
            codes_all = np.concatenate(codes_all)
            if kind == "IVF_FLAT":
                # IVF_FLAT codes are the base rows: the tests rebuild them from xb (keeps the fixture small)
                assert np.array_equal(codes_all, xb[out[f"{tag}_list_ids"]].view(np.uint8).reshape(-1))
            else:
                out[f"{tag}_list_codes"] = codes_all
            I, D = r.search(xq, k, nprobe)
            out[f"{tag}_ids"], out[f"{tag}_dist"] = I, D
            CI, CD = r.coarse(xq, nprobe)
            out[f"{tag}_coarse_ids"], out[f"{tag}_coarse_dist"] = CI, CD
            if kind == "IVF_PQ":
                I, D = r.search(xq, k, nprobe, refine_k=4.0)
                out[f"{tag}_refine4_ids"], out[f"{tag}_refine4_dist"] = I, D
        np.savez_compressed(os.path.join(OUT, f"ivf_4000x64_{name}.npz"), **out)


def hnsw():
    n, d, M, nq, k, ef = 3000, 32, 8, 20, 10, 32
    xb, xq = datagen.clustered(n, d, 42), datagen.clustered(nq, d, 43)
    for metric, name in ((0, "l2"), (1, "ip")):
        h = ref.RefHnsw(d, M, metric, 40)
        h.add(xb)
        g = h.export()
        I, D, st = h.search(xq, k, ef, nthreads=1)
        np.savez_compressed(os.path.join(OUT, f"hnsw_3000x32_{name}.npz"), ids=I, dist=D, stats=np.array(st, np.int64),
                            levels=g["levels"], offsets=g["offsets"], neighbors=g["neighbors"], cum=g["cum"],
                            entry_point=np.int32(g["entry_point"]), max_level=np.int32(g["max_level"]))


if __name__ == "__main__":
    flat()
    ivf()
    hnsw()
    print("golden fixtures written to", OUT)
