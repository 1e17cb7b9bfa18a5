#!/usr/bin/env python3
"""bench.py — queries/sec at recall@10 >= 0.95 on IVF_PQ L2 10M x 128 (m=16 nbits=8 nlist=4096 nprobe=64,
batch=10000): BASELINE.json's metric on BASELINE.json configs[2].

  python bench.py --gpus N --steps K --warmup W            our arm (CUDA path through the C ABI)
  python bench.py --impl reference --gpus N ...           the reference's CPU implementation (oracle/_ref =
                                                          the unmodified faiss/knowhere sources) on the host cores

A "step" = one Search() of the whole 10000-query batch.  `value` times the search with queries and
outputs resident in HBM; `e2e` times the same call with pinned HOST buffers (H2D of the queries and
D2H of ids+distances inside the timed region).  Inputs (200 MB of codes, 5 GB of refine vectors) are
larger than L2, so no explicit flush is needed between iterations.
N>1: inverted lists are packed onto the ranks by size; the SAME search call is a collective inside the library
(NCCL communicator owned by libknowhere_b200.so): every rank ranks the centroids for 1/N of the batch (probe
all-gather), bounds are min-reduced, every rank scans its own lists for the full batch, one all-gather of the
per-shard top-k + merge kernel ("strong" scaling: fixed index and batch).  The N>1 line carries the proof that the
merged result equals the unsharded one.  torch is plumbing here (device buffers, RNG, events, torch.distributed).

--dump-outputs DIR writes what the last timed step returned (rank 0): DIR/ids.npy (float64, exact for int64 labels) and
DIR/distances.npy (float32), nq x k each.  Inputs come from fixed seeds, so two builds run with the same arguments can be
compared output for output.
"""
import argparse
import json
import os
import statistics
import subprocess
import sys
import tempfile
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

WORKLOADS = {
    # name: (index, metric, n, d, params, nq, k)
    "ivf_pq_10m": dict(index="IVF_PQ", metric="L2", n=10_000_000, d=128, nq=10000, k=10,
                       build={"nlist": 4096, "m": 16, "nbits": 8, "refine": True, "refine_type": "flat"},
                       search={"nprobe": 64}),
    "ivf_pq_1m": dict(index="IVF_PQ", metric="L2", n=1_000_000, d=128, nq=10000, k=10,
                      build={"nlist": 1024, "m": 16, "nbits": 8, "refine": True, "refine_type": "flat"},
                      search={"nprobe": 64}),
    "ivf_flat_1m": dict(index="IVF_FLAT", metric="L2", n=1_000_000, d=128, nq=1000, k=10,
                        build={"nlist": 1024}, search={"nprobe": 32}),
    # BASELINE configs[3] (C4).  The graph is built on the host cores (OpenMP; SURVEY 8f rank 3) -- minutes at 1M x 768.
    "hnsw_1m": dict(index="HNSW", metric="IP", n=1_000_000, d=768, nq=1000, k=10,
                    build={"M": 16, "efConstruction": 200}, search={"ef": 128}),
    "hnsw_100k": dict(index="HNSW", metric="IP", n=100_000, d=768, nq=1000, k=10,
                      build={"M": 16, "efConstruction": 200}, search={"ef": 128}),
}
METRIC_NAME = "queries/sec at recall@10>=0.95, 10Mx128 f32 IVF_PQ"
TARGET_RECALL = 0.95


def l2_policy(wl, n, d):
    """what makes the timed region independent of the 126 MB L2 (bench contract: inputs larger than L2, or a flush)"""
    if wl["index"] == "IVF_PQ":
        return (f"inputs larger than L2: every step streams the probed lists' codes (the whole {n * wl['build']['m'] / 1e6:.0f} MB "
                f"code array is touched at this nprobe) and gathers refine rows from a {n * d * 4 / 1e9:.1f} GB store")
    if wl["index"] == "IVF_FLAT":
        return f"inputs larger than L2: every step streams the probed lists' fp32 rows (store of {n * d * 4 / 1e6:.0f} MB)"
    return f"inputs larger than L2: random rows of a {n * d * 4 / 1e9:.2f} GB vector store + {n * 4 * 2 * wl['build'].get('M', 16) / 1e6:.0f} MB of links"


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def peaks_tensor():
    """dense bf16 tensor peak: the burst figure (the filter kernel is timed alone with CUDA events)."""
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        j = json.load(open(p))
        if "bf16_tflops" in j:
            return float(j["bf16_tflops"]), "measured (MEASURED_PEAKS.json bf16_tflops, burst)"
    return 1590.0, "fallback (B200_PROFILING.md 1.59 PFLOP/s dense bf16)"


class ClockSampler:
    """nvidia-smi clock / throttle sampling DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, gpu_index):
        self.f = tempfile.NamedTemporaryFile("w+", suffix=".csv", delete=False)
        q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,"
             "clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20",
                                       "-i", str(gpu_index)], stdout=self.f, stderr=subprocess.DEVNULL)
        except Exception:
            self.p = None
        # nvidia-smi needs a few hundred ms to start: wait for its first line so that the (tens of ms long) timed region is
        # sampled from its first step on
        t0 = time.time()
        while self.p and time.time() - t0 < 3.0:
            try:
                if os.path.getsize(self.f.name) > 0:
                    break
            except OSError:
                pass
            time.sleep(0.02)

    def stop(self):
        out = {"sm_mhz": None, "sm_max_mhz": None, "reasons": []}
        if not self.p:
            return out
        self.p.terminate()
        try:
            self.p.wait(timeout=5)
        except Exception:
            self.p.kill()
        self.f.flush()
        rows = [r.split(",") for r in open(self.f.name).read().strip().splitlines() if r.count(",") >= 8]
        os.unlink(self.f.name)
        if not rows:
            return out
        sm = [float(r[1]) for r in rows if r[1].strip().replace(".", "").isdigit()]
        out["sm_mhz"] = statistics.median(sm) if sm else None
        out["sm_max_mhz"] = float(rows[0][2]) if rows[0][2].strip().replace(".", "").isdigit() else None
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for i, nm in enumerate(names):
            if any("Active" == r[5 + i].strip() for r in rows):
                out["reasons"].append(nm)
        out["samples"] = len(rows)
        return out


def host_cores():
    """Threads the CPU arm may actually use: the affinity mask, capped by the cgroup CPU quota (a 128-thread box leased
    with a 16-CPU quota runs 128 OpenMP threads 8x oversubscribed: that was the 6x CPU-arm swing in round 1)."""
    try:
        aff = len(os.sched_getaffinity(0))
    except Exception:
        aff = os.cpu_count() or 1
    quota = None
    try:
        txt = open("/sys/fs/cgroup/cpu.max").read().split()
        if txt and txt[0] != "max":
            quota = float(txt[0]) / float(txt[1])
    except Exception:
        pass
    use = aff
    if quota:
        use = max(1, min(aff, int(quota + 0.5)))
    return {"threads_used": use, "affinity": aff, "cgroup_cpu_quota": quota, "os_cpu_count": os.cpu_count()}


def ground_truth(kb, torch, xb, xq_sub, k, metric):
    ids, _ = kb.brute_force_search(xb, xq_sub, k, metric, device=xb.device.index or 0,
                                   stream=torch.cuda.current_stream().cuda_stream)
    return ids.cpu().numpy()


def recall_of(gt, ids):
    hit = 0
    for a, b in zip(gt, ids):
        hit += len(set(a.tolist()) & set(b.tolist()) - {-1})
    return hit / float(gt.shape[0] * gt.shape[1])


def dump_outputs(path, ids, dist):
    os.makedirs(path, exist_ok=True)
    np.save(os.path.join(path, "ids.npy"), np.asarray(ids).astype(np.float64))
    np.save(os.path.join(path, "distances.npy"), np.asarray(dist).astype(np.float32))


def make_comm(kb, dist, rank, world, device_index):
    """library-owned NCCL communicator; torch.distributed only ships rank 0's 128-byte id"""
    def bcast(b):
        box = [b]
        dist.broadcast_object_list(box, src=0)
        return box[0]
    return kb.Comm(rank, world, device_index, bcast)


def build_index(kb, torch, dist, wl, xb, rank, world, stream, comm=None, build_cfg=None):
    """GPU build; for world>1 rank 0 trains and broadcasts centroids/codebooks so that every rank
    encodes against the same quantizers, then each rank keeps the lists l % world == rank."""
    d = wl["d"]
    dev_i = xb.device.index or 0
    cfgb = build_cfg or wl["build"]
    ix = kb.Index(wl["index"], wl["metric"], d, cfgb, device=dev_i)
    ix.set_stream(stream)
    m = cfgb.get("m", 0)
    if world == 1:
        ix.train(xb)
        return_q = None
    else:
        ix.set_shard(rank, world)
        nlist = cfgb["nlist"]
        cent = torch.empty((nlist, d), dtype=torch.float32, device=xb.device)
        pq = torch.empty((max(m, 1), 256, d // max(m, 1)), dtype=torch.float32, device=xb.device)
        if rank == 0:
            t = kb.Index(wl["index"], wl["metric"], d, cfgb, device=dev_i)
            t.set_stream(stream)
            t.train(xb)
            c_h, pq_h = t.ivf_export_centroids(m)
            cent.copy_(torch.from_numpy(c_h))
            if m:
                pq.copy_(torch.from_numpy(pq_h))
            del t
        dist.broadcast(cent, 0)
        dist.broadcast(pq, 0)
        torch.cuda.synchronize()
        kb._check(kb.lib().kb2_ivf_import_begin(ix.h, nlist, cent.data_ptr(), pq.data_ptr() if m else None))
        return_q = (cent, pq)
    ix.add(xb)
    if comm is not None:
        ix.set_comm(comm)
    ix._quantizers = return_q
    return ix


def multi_gpu_parity(kb, torch, wl, xb, xq, k, rank, world, stream, comm, quantizers):
    """merged == unsharded, proven inside the run: a sharded and (rank 0) an unsharded PURE-ADC index (no refine, same
    quantizers) answer the whole batch; the merged collective result must equal the unsharded one id for id (refine
    would only ADD candidates on the sharded side, so pure ADC is the exact comparison)."""
    d, m = wl["d"], wl["build"].get("m", 0)
    nlist = wl["build"]["nlist"]
    cfgb = {kk: v for kk, v in wl["build"].items() if kk not in ("refine", "refine_type")}
    cent, pq = quantizers
    dev_i = xb.device.index or 0
    sh = kb.Index(wl["index"], wl["metric"], d, cfgb, device=dev_i)
    sh.set_stream(stream)
    sh.set_shard(rank, world)
    kb._check(kb.lib().kb2_ivf_import_begin(sh.h, nlist, cent.data_ptr(), pq.data_ptr() if m else None))
    sh.add(xb)
    sh.set_comm(comm)
    cfg = dict(wl["search"])
    mi, md = sh.search(xq, k, cfg)           # collective
    torch.cuda.synchronize()
    del sh
    out = None
    if rank == 0:
        full = kb.Index(wl["index"], wl["metric"], d, cfgb, device=dev_i)
        full.set_stream(stream)
        kb._check(kb.lib().kb2_ivf_import_begin(full.h, nlist, cent.data_ptr(), pq.data_ptr() if m else None))
        full.add(xb)
        fi, fd = full.search(xq, k, cfg)
        torch.cuda.synchronize()
        a, b = mi.cpu().numpy(), fi.cpu().numpy()
        da, db = md.cpu().numpy(), fd.cpu().numpy()
        rows = (a == b).all(axis=1)
        sets = np.array([set(x.tolist()) == set(y.tolist()) for x, y in zip(a, b)])
        out = {"queries": int(a.shape[0]), "rows_identical": int(rows.sum()), "id_sets_identical": int(sets.sum()),
               "distances_bit_identical_rows": int((da.view(np.uint32) == db.view(np.uint32)).all(axis=1).sum()),
               "what": "sharded pure-ADC search (collective, merged inside the library) vs unsharded pure-ADC search, "
                       "same quantizers, whole batch"}
        del full
    return out


def run_ours(args):
    import torch
    import torch.distributed as dist

    import knowhere_b200 as kb
    from knowhere_b200 import datagen

    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        os.environ.setdefault("NCCL_DEBUG", "WARN")   # keep NCCL's version banner off stdout: one JSON line only
        dist.init_process_group("nccl", device_id=dev)
    wl = WORKLOADS[args.workload]
    n, d, nq, k = wl["n"], wl["d"], wl["nq"], wl["k"]
    stream = torch.cuda.current_stream().cuda_stream

    t0 = time.time()
    xb = datagen.clustered_torch(n, d, 42, dev)
    xq = datagen.clustered_torch(nq, d, 43, dev)
    torch.cuda.synchronize()
    t_gen = time.time() - t0
    comm = make_comm(kb, dist, rank, world, local_rank) if world > 1 else None
    t0 = time.time()
    ix = build_index(kb, torch, dist, wl, xb, rank, world, stream, comm=comm)
    torch.cuda.synchronize()
    t_build = time.time() - t0

    # ---- search closure (device-resident I/O).  world > 1: the SAME call is a collective inside the library (probe
    #      all-gather, bound all-reduce, ONE all-gather of the per-shard top-k + merge kernel) and returns the merged result.
    ids = torch.empty((nq, k), dtype=torch.int64, device=dev)
    dis = torch.empty((nq, k), dtype=torch.float32, device=dev)

    def search_dev(cfg, q=None):
        ix.search(xq if q is None else q, k, cfg, out=(ids, dis))
        return ids, dis

    # ---- recall calibration: smallest refine_k reaching the target (benchmark_float_qps.cpp:80-108 method)
    cfg = dict(wl["search"])
    recall = None
    n_gt = nq   # recall over the WHOLE batch (round 1 sampled 1000 queries)
    gt = ground_truth(kb, torch, xb, xq[:n_gt].contiguous(), k, wl["metric"])
    if wl["index"] == "IVF_PQ":
        for rk in (1, 2, 4, 8, 16, 32):
            cfg["refine_k"] = rk
            r_ids, _ = search_dev(cfg)
            recall = recall_of(gt, r_ids[:n_gt].cpu().numpy())
            if recall >= TARGET_RECALL:
                break
    else:
        r_ids, _ = search_dev(cfg)
        recall = recall_of(gt, r_ids[:n_gt].cpu().numpy())

    # ---- timed region: device-resident
    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # clocks are sampled from the warm-up steps on (same load as the timed steps; the timed region alone lasts ~50 ms)
    sampler = ClockSampler(local_rank) if rank == 0 else None
    for _ in range(args.warmup):
        search_dev(cfg)
    ix.enable_kernel_timing(True)
    kernel_ms, stage_ms, stage_info = [], [], None
    barrier()
    if os.environ.get("KB2_PROFILE"):       # ncu --profile-from-start off: capture only the timed steps
        torch.cuda.cudart().cudaProfilerStart()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    launches = 0
    for _ in range(args.steps):
        search_dev(cfg)
        kernel_ms.append(ix.last_kernel_ms())
        stage_info = ix.last_stage_info()
        stage_ms.append(stage_info["stage_ms"])
        launches += ix.last_counters()["launches"]
    e1.record()
    barrier()
    if os.environ.get("KB2_PROFILE"):
        torch.cuda.cudart().cudaProfilerStop()
    clocks = sampler.stop() if sampler else None
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, ids.cpu().numpy(), dis.cpu().numpy())
    ms_total = e0.elapsed_time(e1)
    if world > 1:
        t = torch.tensor([ms_total], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ctr = ix.last_counters()
    ix.enable_kernel_timing(False)
    breakdown = None
    parity = None
    if world > 1:
        # where the N>1 step goes (device events inside the library, this rank): list-scan stage, collectives + merge
        ix.enable_kernel_timing(True)
        ts, tm, tk = [], [], []
        ea, eb = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        for _ in range(5):
            ea.record()
            search_dev(cfg)
            eb.record()
            torch.cuda.synchronize()
            info = ix.last_stage_info()
            ts.append(ea.elapsed_time(eb))
            tm.append(info["comm_ms"])
            tk.append(info["stage_ms"])
        ix.enable_kernel_timing(False)
        breakdown = {"step_ms": statistics.median(ts), "collectives_and_merge_ms": statistics.median(tm),
                     "list_scan_stage_ms": statistics.median(tk),
                     "collectives": "all-gather(probes) + min-all-reduce(bounds) + all-gather(top-k) + merge, NCCL inside the library"}
        parity = multi_gpu_parity(kb, torch, wl, xb, xq, k, rank, world, stream, comm, ix._quantizers)

    # ---- end to end: pinned host queries in, host results out, through the same public call
    xq_h = torch.empty((nq, d), dtype=torch.float32).pin_memory()
    xq_h.copy_(xq.cpu())
    ids_h = torch.empty((nq, k), dtype=torch.int64).pin_memory()
    dis_h = torch.empty((nq, k), dtype=torch.float32).pin_memory()
    xq_np, ids_np, dis_np = xq_h.numpy(), ids_h.numpy(), dis_h.numpy()

    def search_e2e():
        # host buffers straight through the public call on every rank (H2D, collectives, D2H inside the library)
        ix.search(xq_np, k, cfg, out=(ids_np, dis_np))

    for _ in range(max(1, args.warmup)):
        search_e2e()
    barrier()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        search_e2e()
    barrier()
    e2e_s = time.perf_counter() - t0
    if world > 1:
        t = torch.tensor([e2e_s], device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        e2e_s = float(t.item())
    e2e_ok = bool(np.array_equal(ids_np, ids.cpu().numpy()))

    if rank != 0:
        if world > 1:
            dist.barrier()
            dist.destroy_process_group()
        return

    qps = nq * args.steps / (ms_total / 1e3)
    e2e_qps = nq * args.steps / e2e_s
    peak, peak_src = peaks()
    # roofline of the dominant kernel, live CUDA-event duration (kb2_index_last_kernel_ms):
    #  * query-major scan kernels (ivfpq_scan / ivfflat_scan): HBM view, algorithmic bytes per launch = codes scanned x
    #    code_size (SURVEY §8d: 16 B per PQ code, ids excluded);
    #  * list-major tensor-core engine (ivfpq_tc_filter_kernel): tensor view, algorithmic flops per launch =
    #    (query, code) pairs x 2 x d — the bf16 contraction the kernel issues on tcgen05 — against the measured dense
    #    bf16 peak; the HBM view of the same launch is reported beside it.
    k_ms = statistics.mean(kernel_ms)
    st_ms = statistics.mean(stage_ms)
    engine = stage_info["engine"] if stage_info else "scan"
    alg_bytes = ctr["code_bytes"]
    traffic = None
    tp = os.path.join(ROOT, "profiles", "scan_kernel_traffic.json")
    if os.path.exists(tp):
        try:
            traffic = json.load(open(tp)).get(args.workload + ("_tc" if engine == "tc" else ""))
        except Exception:
            traffic = None
    if engine == "tc" and wl["index"] == "IVF_FLAT":
        # list-major tcgen05 IVF_FLAT engine: HBM view on SURVEY 8(d)'s algorithmic bytes (rows scanned x d x 4 per (query, list)
        # pair); every list is physically read once per batch, so the algorithmic figure exceeds the HBM peak by design
        achieved = alg_bytes / (k_ms / 1e3) / 1e9
        tpeak, tsrc = peaks_tensor()
        flops = ctr["codes"] * 2.0 * d * 3.0       # 3 x TF32 MMAs per product
        roofline = {"bound": "hbm", "kernel": "ivfflat_tc_kernel", "achieved": achieved, "peak": peak, "unit": "GB/s",
                    "frac": achieved / peak, "peak_source": peak_src, "traffic": traffic, "kernel_ms": k_ms,
                    "traffic_source": "constant from profiles/scan_kernel_traffic.json (ncu --set full of this kernel at this "
                                      "workload), not measured in this run",
                    "algorithmic_bytes_per_launch": alg_bytes, "rows_scanned_per_launch": ctr["codes"],
                    "physical_index_bytes": n * d * 4, "physical_frac_of_hbm_peak": n * d * 4 / (k_ms / 1e3) / 1e9 / peak,
                    "tf32_tflops_issued": flops / (k_ms / 1e3) / 1e12,
                    "kernel_share_of_step": k_ms / (ms_total / args.steps), "scan_stage_ms": st_ms,
                    "note": "each list is read once per batch (list-major), so the SURVEY 8(d) algorithmic figure exceeds 1.0"}
    elif engine == "tc":
        alg_flops = ctr["codes"] * 2.0 * d
        achieved = alg_flops / (k_ms / 1e3) / 1e12
        tpeak, tsrc = peaks_tensor()
        roofline = {"bound": "tensor", "kernel": "ivfpq_tc_filter_kernel", "achieved": achieved, "peak": tpeak,
                    "unit": "TFLOP/s", "frac": achieved / tpeak, "peak_source": tsrc, "traffic": traffic,
                    "kernel_ms": k_ms, "algorithmic_flops_per_launch": alg_flops,
                    "codes_scanned_per_launch": ctr["codes"], "kernel_share_of_step": k_ms / (ms_total / args.steps),
                    "scan_stage_ms": st_ms, "survivors_re_evaluated": ctr["survivors"], "queries_redone": ctr["flagged"],
                    "traffic_source": "constant from profiles/scan_kernel_traffic.json (ncu --set full of this kernel at this "
                                      "workload), not measured in this run",
                    "hbm_algorithmic": {"bytes_per_launch": alg_bytes, "achieved_gbs": alg_bytes / (k_ms / 1e3) / 1e9,
                                        "frac_of_hbm_peak": alg_bytes / (k_ms / 1e3) / 1e9 / peak,
                                        "frac_whole_step": alg_bytes / (ms_total / args.steps / 1e3) / 1e9 / peak,
                                        "peak_gbs": peak, "peak_source": peak_src,
                                        "note": "SURVEY 8(d) figure (codes x 16 B / time); list-major reuse reads each "
                                                "list once per batch, so this exceeds 1.0 by design"}}
    else:
        achieved = alg_bytes / (k_ms / 1e3) / 1e9
        kname = {"IVF_PQ": "ivfpq_scan_kernel", "IVF_FLAT": "ivfflat_scan_kernel", "HNSW": "hnsw_search_kernel"}.get(wl["index"], "?")
        roofline = {"bound": "hbm", "kernel": kname,
                    "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                    "peak_source": peak_src, "traffic": traffic, "kernel_ms": k_ms,
                    "algorithmic_bytes_per_launch": alg_bytes, "codes_scanned_per_launch": ctr["codes"],
                    "kernel_share_of_step": k_ms / (ms_total / args.steps)}
    out = {
        "metric": METRIC_NAME if args.workload == "ivf_pq_10m" else f"queries/sec, {args.workload}",
        "value": qps, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
        "ms_per_step": ms_total / args.steps, "higher_is_better": True,
        "scaling": "strong", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
        "config": {"workload": f"{wl['index']} {wl['metric']} {n}x{d} f32, " +
                               ", ".join(f"{a}={b}" for a, b in {**wl['build'], **cfg}.items()) +
                               f", batch={nq}, k={k}",
                   "recall_at_10": recall, "recall_queries": n_gt, "refine_k": cfg.get("refine_k"),
                   "data": "clustered low-rank gaussian mixture, seeds base 42 / query 43 (SURVEY 8d)",
                   "l2_policy": l2_policy(wl, n, d),
                   "sharding": ("inverted lists packed onto the ranks by size, collectives inside libknowhere_b200.so (kb2_comm_*): probe "
                                "all-gather, bound all-reduce, one all-gather of per-shard top-k + merge kernel")
                   if world > 1 else "single GPU",
                   "build_s": round(t_build, 2), "datagen_s": round(t_gen, 2)},
        "e2e": {"value": e2e_qps, "unit": "queries/s", "h2d_bytes_per_step": nq * d * 4,
                "d2h_bytes_per_step": nq * k * 12, "results_equal_device_path": e2e_ok},
        "gpu_launches": launches,
        "multi_gpu_breakdown": breakdown,
        "multi_gpu_parity": parity,
        "clocks": clocks,
        "roofline": roofline,
    }

    if isinstance(roofline.get("hbm_algorithmic"), dict):
        # SURVEY 8(d)'s HBM view of the same launch at top level too (per kernel and over the whole step)
        out["roofline_hbm_algorithmic"] = roofline["hbm_algorithmic"]
    # ---- CPU baseline beside it (rank 0, N=1 only): the reference's own CPU code on the host cores
    if world == 1 and not args.no_cpu_baseline and wl["index"] in ("IVF_PQ", "IVF_FLAT"):
        try:
            out["cpu_baseline"] = cpu_baseline(kb, wl, ix, xb, xq_np, cfg, gt, n_gt, k, gpu_ids=ids_np.copy(),
                                               gpu_dist=dis_np.copy())
        except Exception as e:  # the baseline is a reported extra; never lose the GPU line over it
            out["cpu_baseline"] = {"error": str(e)[:200]}
    print(json.dumps(out))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def export_to_reference(kb, wl, ix, xb):
    """hand the GPU-built index to the reference classes so both sides search the same index"""
    from oracle import ref
    d = wl["d"]
    m = wl["build"].get("m", 0)
    nlist = ix.ivf_nlist()
    refine = bool(wl["build"].get("refine"))
    r = ref.RefIvf(wl["index"], d, 0 if wl["metric"] == "L2" else 1, nlist, m, 8, refine=refine)
    cent, pq = ix.ivf_export_centroids(m)
    cs = m if m else d * 4
    raw = xb.cpu().numpy() if refine else None
    r.import_state(cent, pq, ((l,) + ix.ivf_export_list(l, cs) for l in range(nlist)), raw=raw)
    return r


def time_reference(r, xq_np, k, cfg, min_seconds=10.0, max_reps=5):
    nthreads = host_cores()["threads_used"]
    rk = float(cfg.get("refine_k", 0) or 0)
    r.search(xq_np[:256], k, cfg["nprobe"], refine_k=rk, nthreads=nthreads)  # warm-up
    times = []
    t_all = time.perf_counter()
    I = None
    while len(times) < max_reps and (time.perf_counter() - t_all < min_seconds or len(times) < 3):
        t0 = time.perf_counter()
        I, _ = r.search(xq_np, k, cfg["nprobe"], refine_k=rk, nthreads=nthreads)
        times.append(time.perf_counter() - t0)
    return I, times, nthreads


def cpu_baseline(kb, wl, ix, xb, xq_np, cfg, gt, n_gt, k, gpu_ids=None, gpu_dist=None):
    r = export_to_reference(kb, wl, ix, xb)
    I, times, nthreads = time_reference(r, xq_np, k, cfg)
    med = statistics.median(times)
    out = {"value": len(xq_np) / med, "unit": "queries/s", "cores": nthreads, "host": host_cores(), "kind": "reference",
           "sample": f"full {len(xq_np)}-query batch x {len(times)} reps (median), one query per OpenMP task "
                     f"(= Knowhere's one task per query), same index exported from the GPU build",
           "recall_at_10": recall_of(gt, I[:n_gt])}
    if gpu_ids is not None:
        # id-level parity of the timed GPU batch against the reference's answer on the same index
        rk = float(cfg.get("refine_k", 0) or 0)
        _, D = r.search(xq_np, k, cfg["nprobe"], refine_k=rk, nthreads=nthreads)
        rows_equal = (gpu_ids == I).all(axis=1)
        sets_equal = np.array([set(a.tolist()) == set(b.tolist()) for a, b in zip(gpu_ids, I)])
        eq = gpu_ids == I
        rel = np.abs(gpu_dist[eq] - D[eq]) / np.maximum(np.abs(D[eq]), 1e-12)
        out["parity_vs_gpu"] = {"queries": int(len(I)), "rows_identical": int(rows_equal.sum()),
                                "id_sets_identical": int(sets_equal.sum()),
                                "ids_equal_fraction": float(eq.mean()),
                                "max_rel_dist_err_on_equal_ids": float(rel.max()) if rel.size else None}
    return out


def run_reference(args):
    """--impl reference: the reference's CPU implementation of the path (oracle/_ref) on the host cores."""
    world = int(os.environ.get("WORLD_SIZE", "1"))
    rank = int(os.environ.get("RANK", "0"))
    if rank != 0:
        return
    import torch

    import knowhere_b200 as kb
    from knowhere_b200 import datagen
    wl = WORKLOADS[args.workload]
    n, d, nq, k = wl["n"], wl["d"], wl["nq"], wl["k"]
    dev = torch.device("cuda", 0)
    xb = datagen.clustered_torch(n, d, 42, dev)
    xq = datagen.clustered_torch(nq, d, 43, dev)
    # the index is built once on the GPU and exported; the TIMED path below is 100% reference CPU code
    ix = kb.Index(wl["index"], wl["metric"], d, wl["build"])
    ix.build(xb)
    cfg = dict(wl["search"])
    gt = ground_truth(kb, torch, xb, xq, k, wl["metric"])
    r = export_to_reference(kb, wl, ix, xb)
    xq_np = xq.cpu().numpy()
    del ix
    recall = None
    if wl["index"] == "IVF_PQ":
        for rk in (1, 2, 4, 8, 16, 32):
            cfg["refine_k"] = rk
            I, _ = r.search(xq_np, k, cfg["nprobe"], refine_k=float(rk), nthreads=host_cores()["threads_used"])
            recall = recall_of(gt, I)
            if recall >= TARGET_RECALL:
                break
    nthreads = host_cores()["threads_used"]
    rk = float(cfg.get("refine_k", 0) or 0)
    for _ in range(args.warmup):
        r.search(xq_np, k, cfg["nprobe"], refine_k=rk, nthreads=nthreads)
    t0 = time.perf_counter()
    I = D = None
    for _ in range(args.steps):
        I, D = r.search(xq_np, k, cfg["nprobe"], refine_k=rk, nthreads=nthreads)
    el = time.perf_counter() - t0
    if args.dump_outputs and I is not None:
        dump_outputs(args.dump_outputs, I, D)
    qps = nq * args.steps / el
    out = {"impl": "reference", "metric": METRIC_NAME if args.workload == "ivf_pq_10m" else f"queries/sec, {args.workload}",
           "value": qps, "unit": "queries/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": el / args.steps * 1e3, "higher_is_better": True, "scaling": "strong", "vs_baseline": None,
           "dtype": "f32", "data": "synthetic",
           "config": {"workload": f"{wl['index']} {wl['metric']} {n}x{d} f32, " +
                                  ", ".join(f"{a}={b}" for a, b in {**wl['build'], **cfg}.items()) + f", batch={nq}, k={k}",
                      "recall_at_10": recall, "refine_k": cfg.get("refine_k")},
           "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": nthreads, "host": host_cores(), "kind": "reference",
                            "sample": f"full {nq}-query batch per step, faiss IndexIVFPQ+IndexRefine via oracle/_ref, "
                                      f"one query per OpenMP task"},
           "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(out))


def main():
    # stdout carries exactly ONE JSON line: anything a library prints to fd 1 meanwhile (e.g. NCCL's version banner at
    # communicator creation) is sent to stderr; the line itself goes to the saved descriptor
    saved = os.dup(1)
    os.dup2(2, 1)
    sys.stdout = os.fdopen(saved, "w", buffering=1)
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default="ivf_pq_10m", choices=sorted(WORKLOADS))
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the last timed step's ids and distances to DIR/*.npy")
    args = ap.parse_args()
    args.warmup = max(args.warmup, 3) if args.impl == "ours" else args.warmup
    if args.impl == "reference":
        run_reference(args)
    else:
        run_ours(args)


if __name__ == "__main__":
    main()
