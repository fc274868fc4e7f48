#!/usr/bin/env python
"""bench.py -- headline benchmark of the query -> top-k hot path (BASELINE.json metric):

    queries/sec @ top-k=100 on a 100M x 768 IVF-PQ index (nlist=16384, M=64, nbits=8, nprobe=32), 1/2/4/8 B200,
    plus the list-scan kernel's achieved HBM GB/s against the measured peak.

One "step" = one pass of the hot path (coarse scan -> LUT -> ADC list scan -> top-k [-> all-gather + merge])
over one batch of `--nq` synthetic queries.  `value` = queries/s with the queries already resident in HBM;
`e2e` = the same through the public API with pinned HOST query buffers and host result buffers, H2D/D2H inside
the timed region.  At N GPUs the 100M datastore is statically partitioned (strong scaling: total work fixed),
every rank scans its slice for every query and the per-shard top-k are all-gathered over NCCL and merged
(reference semantics: src/search.py:357-367).

    python bench.py [--gpus N] [--steps K] [--warmup W]            # this framework
    python bench.py --impl reference ...                           # the reference's CPU path (oracle port of
                                                                    # faiss-cpu 1.8.0 semantics) on the host cores
The default line also carries: `parity` (tie-aware comparison of the timed GPU results with the CPU oracle's over
the queries the cpu_baseline leg searched -- all of them at N=1, a 256-query sample at N>1 -- plus a float64
re-score of every returned (id, score) pair), `recall` (recall@k against exact search over the same corpus),
`sweep` (full-sweep HBM micro-benchmark, N=1), `encoder` + `c5_encode_plus_search` (BASELINE config 5).
Extra knobs (development only; the defaults are the BASELINE configuration): --n --nq --nlist --m --nprobe --k
--no-sweep --no-recall --no-encoder --no-cpu-baseline --e2e-transfer.
`--steps` / `--warmup` set the timed / untimed passes of every timed block (search arms, sweep, encoder, config 5).
`--dump-outputs DIR` writes the (ids, scores) of the last timed search step as DIR/*.npy: the queries and corpus come
from fixed seeds and the index training is reproducible (ReproducibleTrainingOps), so the same arguments give the same
outputs and two builds can be compared output for output.
"""
from __future__ import annotations

import argparse
import json
import math
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import numpy as np
import torch

CHUNK_ROWS = 1_000_000


def log(*a):
    print("[bench]", *a, file=sys.stderr, flush=True)


def parse():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--n", type=int, default=int(os.environ.get("RSB_BENCH_N", 100_000_000)))
    ap.add_argument("--nq", type=int, default=10_000)
    ap.add_argument("--nlist", type=int, default=int(os.environ.get("RSB_BENCH_NLIST", 16384)))
    ap.add_argument("--m", type=int, default=64)
    ap.add_argument("--nprobe", type=int, default=32)
    ap.add_argument("--k", type=int, default=100)
    ap.add_argument("--d", type=int, default=768)
    ap.add_argument("--train-per-centroid", type=int, default=64)
    ap.add_argument("--no-sweep", action="store_true", help="skip the full-sweep HBM micro-benchmark (N=1)")
    ap.add_argument("--no-cpu-baseline", action="store_true", help="skip the CPU oracle leg (and with it the parity block)")
    ap.add_argument("--no-recall", action="store_true", help="skip recall@k vs exact search over the same corpus")
    ap.add_argument("--recall-queries", type=int, default=1000)
    ap.add_argument("--no-encoder", action="store_true", help="skip the BERT-base query-encoder timing / BASELINE config 5 block")
    ap.add_argument("--parity-queries", type=int, default=256, help="queries of the N>1 parity sample (N=1 checks every query the CPU leg searched)")
    ap.add_argument("--encoder-batch", type=int, default=2048)
    ap.add_argument("--encoder-only", action="store_true")
    ap.add_argument("--gather", default="fused", choices=["fused", "fused-full", "nccl"],
                    help="multi-GPU reduction: merge kernel over peer memory (query-sliced, results stored to every "
                         "GPU), the same with every GPU merging all queries, or NCCL all-gather + merge")
    ap.add_argument("--e2e-transfer", default="sliced", choices=["replicated", "sliced"],
                    help="end-to-end arm at N > 1: 'sliced' (default) = every rank uploads its 1/N slice of the host queries "
                         "(slices all-gathered over NVLink) and downloads the 1/N of the merged result it produced, so each "
                         "byte crosses PCIe once per job; 'replicated' = every rank uploads all queries and downloads the "
                         "full result")
    ap.add_argument("--share-tau", type=int, default=1, help="N > 1, fused gather: exchange the running top-k thresholds "
                    "between the GPUs during the scan (rsb_search_preassigned_shared); 0 = every GPU filters with its own")
    ap.add_argument("--peer-coarse", type=int, default=1, help="N > 1, fused gather: publish the sharded coarse tables with "
                    "P2P stores + one barrier; 0 = two NCCL all-gathers")
    ap.add_argument("--e2e-pipeline", type=int, default=1, help="end-to-end arm: 1 (default) = dist.HostPipeline, the copies of "
                    "neighbouring batches overlap the search (every batch is still uploaded and downloaded in full); 0 = one "
                    "batch at a time, copies and search serialised")
    ap.add_argument("--partition", default="list", choices=["list", "vector"],
                    help="static datastore partition across GPUs: whole inverted lists per GPU, or 1/G of every list")
    ap.add_argument("--cpu-seconds", type=float, default=15.0, help="CPU-baseline time budget")
    ap.add_argument("--dump-outputs", metavar="DIR", help="after the timed steps, write the ids and scores the last timed "
                    "search step returned to DIR/ids.npy (float64) and DIR/scores.npy (float32); above 64 MB a fixed "
                    "seeded sample of query rows is written, with their row numbers in DIR/rows.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and (args.impl != "b200" or args.encoder_only):
        ap.error("--dump-outputs writes the results of the GPU search arm: not with --impl reference or --encoder-only")
    return args


# ----------------------------------------------------------------------------------------------------------
# clocks sampling (B200_PROFILING.md recipe)
# ----------------------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.gpu = gpu_index
        self.proc = None
        self.lines = []
        self.nvml = None
        self.samples = []
        self._stop = False

    def sample_now(self):
        if self.nvml is None:
            return
        import pynvml as N
        h = self.nvml
        try:
            sm = N.nvmlDeviceGetClockInfo(h, N.NVML_CLOCK_SM)
            mx = N.nvmlDeviceGetMaxClockInfo(h, N.NVML_CLOCK_SM)
            pw = N.nvmlDeviceGetPowerUsage(h) / 1000.0
            rs = N.nvmlDeviceGetCurrentClocksEventReasons(h)
            self.samples.append((sm, mx, pw, rs))
        except Exception:
            pass

    def _nvml_loop(self):
        while not self._stop:
            self.sample_now()
            time.sleep(0.005)

    def start(self):
        # in-process NVML polling every 5 ms (short timed regions at 8 GPUs last < 100 ms); nvidia-smi as fallback
        try:
            import pynvml as N
            N.nvmlInit()
            vis = os.environ.get("CUDA_VISIBLE_DEVICES")
            phys = int(vis.split(",")[self.gpu]) if vis and vis.split(",")[self.gpu].strip().isdigit() else self.gpu
            self.nvml = N.nvmlDeviceGetHandleByIndex(phys)
            self.thread = threading.Thread(target=self._nvml_loop, daemon=True)
            self.thread.start()
            return
        except Exception:
            self.nvml = None
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", f"--id={self.gpu}", f"--query-gpu={self.FIELDS}", "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.thread = threading.Thread(target=self._pump, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _pump(self):
        for line in self.proc.stdout:
            self.lines.append(line.strip())

    def stop(self):
        if self.nvml is not None:
            import pynvml as N
            self._stop = True
            self.thread.join(timeout=1)
            if not self.samples:
                return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
            bits = {"hw_slowdown": N.nvmlClocksEventReasonHwSlowdown, "hw_thermal_slowdown": N.nvmlClocksEventReasonHwThermalSlowdown,
                    "sw_thermal_slowdown": N.nvmlClocksEventReasonSwThermalSlowdown, "sw_power_cap": N.nvmlClocksEventReasonSwPowerCap}
            reasons = sorted(nm for nm, b in bits.items() if any(s[3] & b for s in self.samples))
            return {"sm_mhz": float(np.median([s[0] for s in self.samples])), "sm_max_mhz": float(max(s[1] for s in self.samples)),
                    "power_w_max": float(max(s[2] for s in self.samples)), "power_w_median": float(np.median([s[2] for s in self.samples])),
                    "samples": len(self.samples), "reasons": reasons,
                    "source": "nvml, 5 ms period, during the timed region"}
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            self.proc.kill()
        sm, mx, pw, reasons = [], [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            parts = [p.strip() for p in ln.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0])); mx.append(float(parts[1])); pw.append(float(parts[2]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["no samples"]}
        return {"sm_mhz": float(np.median(sm)), "sm_max_mhz": float(max(mx)), "power_w_max": float(max(pw)),
                "samples": len(sm), "reasons": sorted(reasons)}


# ----------------------------------------------------------------------------------------------------------
# index construction (setup; not timed).  Build side = SURVEY §8f-1, through librsb: k-means / PQ training
# (`train.py` with librsb's assignment kernels; member sums in fixed point, see ReproducibleTrainingOps), list
# assignment by the tensor-core coarse quantizer (`index.assign`), residual PQ encoding and the interleaved list
# layout (`rsb_add_preassigned`, `rsb_finalize`).
# While the corpus streams through, the exact top-k of a query sample is accumulated (librsb Flat kernels) as the
# ground truth of the recall figure -- the 307 GB fp32 corpus never materialises.
# ----------------------------------------------------------------------------------------------------------
def fixed_point_sums(x: torch.Tensor, seg: torch.Tensor, k: int, chunk_elems: int = 1 << 26) -> torch.Tensor:
    """Sums of the rows of x [n, d] per segment id seg [n] in [0, k), as float32 [k, d].  Every value is rounded to a
    multiple of 2**-s, with s as fine as the bound n * max|x| < 2**62 allows, and added as an int64: integer addition
    is exact, so the sums do not depend on the order in which the GPU's atomics add the rows."""
    n, d = x.shape
    bound = float(x.abs().max()) * n if n else 0.0
    scale = 2.0 ** (62 - math.ceil(math.log2(bound))) if bound > 0 else 1.0
    acc = torch.zeros(k, d, dtype=torch.int64, device=x.device)
    rows = max(1, chunk_elems // d)                       # bounds the float64 / int64 copies of a chunk
    for i in range(0, n, rows):
        acc.index_add_(0, seg[i:i + rows], torch.round(x[i:i + rows].double() * scale).long())
    return (acc.double() / scale).float()


class ReproducibleTrainingOps:
    """The operations `train.kmeans` / `train.train_pq` run, with the assignments from `assign_ops` (librsb's kernels
    in the bench) and the member sums from fixed_point_sums.  librsb's accumulate kernels add floats atomically in
    arrival order, so their sums, the trained index and every search result change a little from run to run; with
    these the same arguments give the same index, and --dump-outputs compares like with like."""

    def __init__(self, assign_ops):
        self.assign_ops = assign_ops

    def assign_ip(self, x, c):
        return self.assign_ops.assign_ip(x, c)

    def pq_assign(self, r, cb):
        return self.assign_ops.pq_assign(r, cb)

    def accumulate(self, x, a, k):
        return fixed_point_sums(x, a, k), torch.bincount(a, minlength=k).float()

    def pq_accumulate(self, r, codes, M, ksub):
        n, d = r.shape
        entry = (codes.long() + torch.arange(M, device=r.device) * ksub).flatten()    # codebook entry of each sub-vector
        sums = fixed_point_sums(r.reshape(n * M, d // M), entry, M * ksub)
        return sums.view(M, ksub, d // M), torch.bincount(entry, minlength=M * ksub).float().view(M, ksub)


def build_index(args, rank: int, world: int, device, gt_queries=None):
    import retrieval_scaling_b200 as rsb
    from retrieval_scaling_b200 import synth, train

    t0 = time.time()
    n_centres = max(16, args.nlist // 4)
    corpus = synth.Corpus(d=args.d, mode="gmm", n_centres=n_centres, device=device)
    index = rsb.IndexIVFPQ(args.d, args.nlist, args.m, 8, device=device)
    index.nprobe = args.nprobe

    # ---- train on rank 0, broadcast (identical centroids/codebooks on every shard => G-GPU ids == 1-GPU ids)
    cent = torch.empty(args.nlist, args.d, device=device)
    cb = torch.empty(args.m, 256, args.d // args.m, device=device)
    if rank == 0:
        ops = ReproducibleTrainingOps(train.LibrsbOps())
        ntrain = min(args.n, args.nlist * args.train_per_centroid)
        xt = corpus.train_sample(ntrain)
        cent.copy_(train.kmeans(xt, args.nlist, niter=10, metric="ip", spherical=True, seed=1234, ops=ops))
        xs = xt[: 256 * 256]
        a = train.assign_ip(xs, cent, ops=ops)
        cb.copy_(train.train_pq(xs - cent[a], args.m, 256, niter=25, seed=1234, ops=ops))
        del xt, xs, a, ops
    if world > 1:
        torch.distributed.broadcast(cent, 0)
        torch.distributed.broadcast(cb, 0)
    index.set_centroids(cent)
    index.set_codebook(cb)
    torch.cuda.synchronize()
    t_train = time.time() - t0

    # ---- add this rank's static shard; ids are global row numbers.
    #   partition "list"  : rank r owns whole inverted lists.  Every (query, list) pair is scanned by exactly one
    #                       GPU at full list length, so the scan scales ~1/G (default).
    #   partition "vector": chunk c (1M rows) belongs to rank c % world: every rank holds 1/G of every list (the
    #                       reference's per-passage-shard layout); per-(query, list) overheads do not shrink with G.
    nchunks = (args.n + CHUNK_ROWS - 1) // CHUNK_ROWS
    by_list = args.partition == "list" and world > 1
    owner = None
    if by_list:
        # balanced static list -> GPU map: rank 0 estimates list sizes from chunk 0 and probe frequencies from a
        # calibration query sample, assigns lists to GPUs by expected scan work with the longest-processing-time
        # greedy rule and broadcasts the map (one map for all ranks by construction)
        owner = torch.empty(args.nlist, dtype=torch.int32, device=device)
        if rank == 0:
            x0 = corpus.chunk(0, CHUNK_ROWS)[: min(CHUNK_ROWS, args.n)]
            est = torch.bincount(index.assign(x0).long(), minlength=args.nlist)
            del x0
            # scan work of a list = its length x how often it is probed: estimate the probe frequency from an
            # independent calibration sample of the query distribution (not the queries that are searched)
            qc = corpus.calibration_queries(16384)
            top, _ = index.coarse(qc, min(args.nprobe, args.nlist))
            probes = torch.bincount(top.flatten(), minlength=args.nlist)
            del qc, top
            est_h = (est.double() + 1.0).mul_(probes.double() + 1.0).cpu().numpy()
            load = np.zeros(world, dtype=np.float64)
            owner_h = np.empty(args.nlist, dtype=np.int32)
            for l in np.argsort(-est_h, kind="stable"):
                r = int(np.argmin(load))
                owner_h[l] = r
                load[r] += est_h[l]
            owner.copy_(torch.from_numpy(owner_h))
        torch.distributed.broadcast(owner, 0)
    gt = None
    if gt_queries is not None:
        gt = {"D": None, "I": None, "pD": [], "pI": []}
    for c in (range(nchunks) if by_list else range(rank, nchunks, world)):
        rows = min(CHUNK_ROWS, args.n - c * CHUNK_ROWS)
        x = corpus.chunk(c, CHUNK_ROWS)[:rows]
        if gt is not None and c % world == rank:     # exact top-k of the recall sample over the chunks this rank owns
            D, I = rsb.knn_ip(gt_queries, x, args.k, id_offset=c * CHUNK_ROWS)
            gt["pD"].append(D); gt["pI"].append(I)
            if len(gt["pD"]) == 15:
                _fold_gt(gt, args.k)
        lists = index.assign(x)
        ids = torch.arange(c * CHUNK_ROWS, c * CHUNK_ROWS + rows, dtype=torch.int64, device=device)
        if by_list:
            mine = torch.nonzero(owner[lists.long()] == rank).flatten()
            x, lists, ids = x[mine], lists[mine], ids[mine]
        index.add_preassigned(x, lists, ids)
        del x, lists, ids
        if (c if by_list else c // world) % 10 == 9:
            log(f"rank {rank}: added chunk {c + 1}/{nchunks} ({time.time() - t0:.1f}s)")
    index.finalize()
    torch.cuda.synchronize()
    gt_I = None
    if gt is not None:
        _fold_gt(gt, args.k)
        gD, gI = gt["D"], gt["I"]
        if gD is None:                               # a rank that owned no chunk
            gD = torch.full((gt_queries.shape[0], args.k), float(np.finfo(np.float32).min), device=device)
            gI = torch.full((gt_queries.shape[0], args.k), -1, dtype=torch.int64, device=device)
        if world > 1:
            aD = torch.empty((world,) + tuple(gD.shape), dtype=gD.dtype, device=device)
            aI = torch.empty((world,) + tuple(gI.shape), dtype=gI.dtype, device=device)
            torch.distributed.all_gather_into_tensor(aD, gD.contiguous())
            torch.distributed.all_gather_into_tensor(aI, gI.contiguous())
            gD, gI = rsb.merge_topk(aD, aI, args.k)
        gt_I = gI
    build_s = time.time() - t0
    log(f"rank {rank}: built IVF-PQ shard ntotal={index.ntotal} ({index.index_bytes / 1e9:.2f} GB) "
        f"train {t_train:.1f}s total {build_s:.1f}s")
    return index, corpus, cent, gt_I, {"train_s": t_train, "total_s": build_s}


def _fold_gt(gt, k):
    import retrieval_scaling_b200 as rsb
    if not gt["pD"]:
        return
    if gt["D"] is not None:
        gt["pD"].append(gt["D"]); gt["pI"].append(gt["I"])
    gt["D"], gt["I"] = rsb.merge_topk(torch.stack(gt["pD"]), torch.stack(gt["pI"]), k)
    gt["pD"], gt["pI"] = [], []


def recall_block(I_pq: torch.Tensor, gt_I: torch.Tensor, k: int):
    """recall@k = |returned top-k  intersect  exact top-k| / k, averaged over the sample; plus how often the exact
    best / the exact top-10 are inside the returned k."""
    a = I_pq.cpu().numpy()
    b = gt_I.cpu().numpy()
    nq = b.shape[0]
    hits = top1 = top10 = 0
    for i in range(nq):
        sa = set(a[i].tolist())
        hits += len(sa & set(b[i].tolist()))
        top1 += int(b[i, 0]) in sa
        top10 += len(sa & set(b[i, :10].tolist()))
    return {"queries": nq, "k": k, f"recall@{k}": hits / (nq * k), f"top1_in_top{k}": top1 / nq,
            f"top10_in_top{k}": top10 / (nq * min(10, k)),
            "ground_truth": "exact inner-product search (librsb Flat kernels) over the same synthetic corpus, "
                            "accumulated chunk by chunk during the build"}


def sweep_microbench(index, args, cent, device):
    """Full-sweep HBM micro-benchmark (SURVEY §8d): nlist/nprobe queries whose probe sets partition all lists
    exactly once => pair-bytes == unique bytes == the whole code array, nothing is re-read from L2."""
    nprobe = args.nprobe
    nq = args.nlist // nprobe
    g = torch.Generator(device=device).manual_seed(99)
    q = torch.randn(nq, args.d, generator=g, device=device)
    lists = torch.randperm(args.nlist, generator=g, device=device)[: nq * nprobe].reshape(nq, nprobe).contiguous()
    dis = torch.einsum("qd,qpd->qp", q, cent[lists])
    index.set_profiling(True)
    try:
        index.profile()
    except Exception:
        pass
    ms, nbytes = [], 0
    for it in range(args.warmup + args.steps):
        index.search_preassigned(q, args.k, lists, dis)
        torch.cuda.synchronize()
        p = index.profile()
        if it >= args.warmup:
            ms.append(p["scan_ms"]); nbytes = p["scan_bytes"]
    t = float(np.mean(ms))
    return {"queries": nq, "scan_ms": t, "bytes": nbytes, "gbs": nbytes / t / 1e6 if t > 0 else None,
            "what": "every inverted list scanned exactly once per launch: pair-bytes == unique bytes == DRAM bytes"}


# ----------------------------------------------------------------------------------------------------------
# query encoder (BASELINE config 5): BERT-base fp16 forward over NQ-length token batches
# ----------------------------------------------------------------------------------------------------------
def encoder_setup(args, device, rank: int, world: int):
    """Seeded random-init Contriever-architecture weights (no checkpoint offline) + this rank's slice of `nq`
    synthetic queries whose token counts follow examples/nq_open.jsonl (tests/golden/nq_open_token_lengths.npy),
    as pinned HOST token batches of `--encoder-batch` sequences."""
    from retrieval_scaling_b200.encoder import BERT_BASE, B200Contriever, random_state_dict
    model = B200Contriever(BERT_BASE, "average", device=device)
    model.load_state_dict(random_state_dict(BERT_BASE, 0))
    lens_fix = np.load(os.path.join(ROOT, "tests", "golden", "nq_open_token_lengths.npy")).astype(np.int64)
    lens = np.resize(lens_fix, args.nq)
    per = (args.nq + world - 1) // world
    lo, hi = min(args.nq, rank * per), min(args.nq, (rank + 1) * per)
    g = torch.Generator(device="cpu").manual_seed(1000 + rank)

    def batches_of(bs):
        out = []
        for b0 in range(lo, hi, bs):
            l = torch.from_numpy(lens[b0:min(hi, b0 + bs)]).int()
            cu = torch.zeros(len(l) + 1, dtype=torch.int32)
            cu[1:] = torch.cumsum(l, 0)
            T = int(cu[-1])
            ids = torch.randint(1000, 30000, (T,), generator=g, dtype=torch.int32)
            out.append((ids.pin_memory(), cu.pin_memory(), int(l.max()), T))
        return out
    return model, batches_of, (lo, hi)


def encoder_bench(args, device):
    """Device-resident timing of the forward at the reference's batch size (64, `per_gpu_batch_size`) and at the
    grouped batch this framework uses (`encode_group`)."""
    model, batches_of, _ = encoder_setup(args, device, 0, 1)
    out = {}
    for bs in ([args.encoder_batch] if os.environ.get("RSB_ENC_ONLY_BATCH") else sorted({64, args.encoder_batch})):
        batches = [(i.to(device), c.to(device), mx, T) for i, c, mx, T in batches_of(bs)]
        total_tokens = sum(b[3] for b in batches)

        def run():
            return torch.cat([model.forward_varlen(ids, cu, mx, None, T) for ids, cu, mx, T in batches], 0)

        for _ in range(args.warmup):
            run()
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        sampler = ClockSampler(device.index or 0)
        sampler.start()
        e0.record()
        for _ in range(args.steps):
            run()
        e1.record()
        torch.cuda.synchronize()
        clocks = sampler.stop()
        ms = e0.elapsed_time(e1) / args.steps
        flops = 169.9e6 * total_tokens
        out[f"batch_{bs}"] = {"queries": args.nq, "tokens": total_tokens, "ms": ms, "queries_per_s": args.nq / ms * 1e3,
                              "gemm_tflops": flops / ms / 1e9, "launches": model.launches * len(batches), "clocks": clocks}
    peaks = os.path.join(ROOT, "MEASURED_PEAKS.json")
    sustained = 1469.3
    if os.path.exists(peaks):
        sustained = json.load(open(peaks)).get("bf16_tflops_sustained", sustained)
    for v in out.values():
        v["frac_of_measured_bf16_sustained"] = v["gemm_tflops"] / sustained
    out["peak_tflops"] = sustained
    out["note"] = ("fp16 tcgen05 GEMMs (72 per forward), un-padded token stream, 169.9 MFLOP/token counted (Linear layers "
                   "only), seeded random-init BERT-base weights, token counts of examples/nq_open.jsonl")
    return out


def c5_encode_plus_search(args, device, rank, world, searcher, xq, steps, warmup):
    """BASELINE config 5 end to end: host token ids -> encoder forward (queries sharded across ranks) -> embeddings
    all-gathered -> IVF-PQ search of the sharded datastore -> host (ids, scores).  Offline there are no pretrained
    weights, so the embeddings of the random-init encoder are unrelated to the synthetic datastore; they are computed,
    converted and all-gathered (so every byte and FLOP of the step is paid) but the search consumes the synthetic gmm
    queries -- the same workload as the headline line, for which recall@k is known."""
    model, batches_of, (lo, hi) = encoder_setup(args, device, rank, world)
    batches = batches_of(args.encoder_batch)
    per = (args.nq + world - 1) // world
    I_host = torch.empty((per if world > 1 else args.nq, args.k), dtype=torch.int64).pin_memory()
    D_host = torch.empty((per if world > 1 else args.nq, args.k), dtype=torch.float32).pin_memory()
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(3)]
    enc_ms = []

    def step(timed):
        if timed:
            ev[0].record()
        embs = []
        for ids, cu, mx, T in batches:
            embs.append(model.forward_varlen(ids.to(device, non_blocking=True), cu.to(device, non_blocking=True), mx, None, T))
        emb = torch.cat(embs, 0).float() if embs else torch.zeros((0, args.d), device=device)
        if world > 1:
            pad = torch.zeros((per, args.d), device=device)
            pad[: emb.shape[0]] = emb
            allq = torch.empty((world * per, args.d), device=device)
            torch.distributed.all_gather_into_tensor(allq, pad)
            emb = allq[: args.nq]
        if timed:
            ev[1].record()
        searcher.search_to_host(xq, args.k, out=(I_host, D_host))     # synchronises the D2H copy
        if timed:
            ev[2].record()
            torch.cuda.synchronize()
            enc_ms.append(ev[0].elapsed_time(ev[1]))
        return emb

    for _ in range(warmup):
        step(False)
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    for _ in range(steps):
        step(True)
    if world > 1:
        torch.distributed.barrier()
    torch.cuda.synchronize()
    t = torch.tensor([time.perf_counter() - t0], device=device, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    total_ms = float(t.item()) / steps * 1e3
    tokens = sum(b[3] for b in batches)
    return {"queries": args.nq, "value": args.nq / total_ms * 1e3, "unit": "queries/s", "ms_per_step": total_ms,
            "encode_ms_rank0": float(np.mean(enc_ms)) if enc_ms else None,
            "search_and_copy_ms_rank0": (total_ms - float(np.mean(enc_ms))) if enc_ms else None,
            "h2d_bytes_per_step_per_rank": int(tokens * 4 + sum(b[1].numel() for b in batches) * 4),
            "d2h_bytes_per_step_per_rank": int(I_host.numel() * 8 + D_host.numel() * 4),
            "encoder_queries_per_rank": hi - lo, "encoder_batch": args.encoder_batch,
            "note": "host token ids in, host (ids, scores) out; encoder sharded by query across the ranks, embeddings "
                    "all-gathered; random-init weights (no checkpoint offline) => the search consumes the synthetic gmm "
                    "queries (same workload as the headline), see bench.py:c5_encode_plus_search"}


# ----------------------------------------------------------------------------------------------------------
# CPU baseline: the oracle's C/OpenMP port of the reference's faiss-cpu IVF-PQ search, on host cores
# ----------------------------------------------------------------------------------------------------------
def export_host(index):
    off, codes, ids = index.export_lists()
    out = (off.cpu().numpy(), codes.cpu().numpy(), ids.cpu().numpy())
    del off, codes, ids
    torch.cuda.empty_cache()
    return out


def cpu_threads_setup(share: int = 1):
    """OpenMP team of the CPU arm = every core of this process's affinity mask (divided by `share` when several ranks
    run the oracle at once).  Set explicitly: torchrun exports OMP_NUM_THREADS=1 to its workers."""
    from oracle import c_oracle as C
    C.build()
    cores = C.host_cores()
    threads = C.set_num_threads(max(1, cores // max(1, share)))
    return threads, {"cpu_model": C.cpu_model(), "host_cores": cores, "os_cpu_count": os.cpu_count(),
                     "omp_num_threads_env": os.environ.get("OMP_NUM_THREADS")}


def cpu_search_rate(host_index, cent_np, cb_np, xq_np, args, seconds: float):
    """Times oracle.c_oracle.ivfpq_search on a bounded sample of the workload's queries; returns the (D, I) of the
    timed call as well (the parity block compares the GPU result with it)."""
    from oracle import c_oracle as C
    off, codes, ids = host_index
    threads, info = cpu_threads_setup()
    fa = faiss_search_fn(host_index, cent_np, cb_np, args)
    info["kind"] = "reference" if fa is not None else "port"
    info["implementation"] = ("faiss IndexIVFPQ.search (the reference's own arithmetic) on the same index" if fa is not None else
                              "oracle/ann_oracle.c: C/OpenMP restatement of faiss-cpu 1.8.0 IndexIVFPQ.search (faiss is not installable offline)")

    def run(x):
        return fa(x) if fa is not None else C.ivfpq_search(x, cent_np, cb_np, off, codes, ids, args.nprobe, args.k)
    n0 = min(xq_np.shape[0], max(threads, 16))
    t0 = time.perf_counter()
    run(xq_np[:n0])
    dt0 = time.perf_counter() - t0
    rate0 = n0 / dt0
    n1 = int(min(xq_np.shape[0], max(n0, rate0 * seconds)))
    t0 = time.perf_counter()
    D, I = run(xq_np[:n1])
    dt = time.perf_counter() - t0
    info["_run"] = run
    return n1 / dt, threads, n1, dt, (D, I), info


def faiss_search_fn(host_index, cent_np, cb_np, args):
    """The reference's own arithmetic, if it is there: `faiss.IndexIVFPQ.search` on the SAME index (written in faiss'
    file layout by retrieval_scaling_b200.faiss_io and loaded with faiss.read_index), all host cores.  faiss is not
    installable in the build image (no wheel, no network), so this normally returns None and the oracle port is timed."""
    try:
        import faiss  # noqa: F401
    except Exception:
        return None
    try:
        import tempfile
        from retrieval_scaling_b200 import faiss_io
        off, codes, ids = host_index
        d = "/dev/shm" if os.path.isdir("/dev/shm") else None
        with tempfile.NamedTemporaryFile(suffix=".faiss", dir=d, delete=False) as f:
            path = f.name
        try:
            faiss_io.write_faiss(path, {"kind": "IVFPQ", "centroids": cent_np, "codebook": cb_np, "offsets": off, "codes": codes,
                                        "ids": ids, "nprobe": args.nprobe})
            index = faiss.read_index(path)
        finally:
            os.remove(path)
        index.nprobe = args.nprobe
        from oracle import c_oracle as C
        faiss.omp_set_num_threads(C.host_cores())

        def search(xq):
            return index.search(np.ascontiguousarray(xq, dtype=np.float32), args.k)
        return search
    except Exception as e:  # a faiss that cannot take the file must not take the bench line down
        log(f"faiss is importable but could not be used as the CPU arm ({type(e).__name__}: {e}); timing the oracle port")
        return None


PARITY_RTOL, PARITY_ATOL = 1e-5, 2e-4


def parity_block(host_index, cent_np, cb_np, xq_np, D_gpu, I_gpu, D_ref, I_ref):
    """GPU (timed run) vs oracle on the same queries: tie-aware id comparison + fp64 re-score of every returned pair."""
    from oracle import parity as P
    n = D_ref.shape[0]
    out = P.topk_parity(D_gpu[:n], I_gpu[:n], D_ref, I_ref, rtol=PARITY_RTOL, atol=PARITY_ATOL)
    H = P.HostIVFPQ(cent_np, cb_np, *host_index)
    out.update(H.verify_pairs(xq_np[:n], D_gpu[:n], I_gpu[:n], rtol=PARITY_RTOL, atol=PARITY_ATOL))
    out["oracle"] = "the cpu_baseline leg's results (see cpu_baseline.implementation; the oracle port is 'parity unpinned': no faiss offline)"
    out["ok"] = bool(out["non_tie_mismatches"] == 0 and out["scores_out_of_tol"] == 0 and out["padding_mismatches"] == 0
                     and out["rescore_out_of_tol"] == 0 and out["unknown_ids"] == 0)
    return out


def parity_block_sharded(index, cent, xq, I_gpu, D_gpu, args, rank, world, device):
    """N > 1: every rank runs the oracle on ITS exported shard for a query sample, the per-shard results are merged
    with the reference's rule (oracle merge_topk: concat in shard order, stable sort desc, keep k) and compared with
    the N-GPU result; every rank re-scores in float64 the returned pairs whose ids it holds."""
    from oracle import ann_oracle as O
    from oracle import c_oracle as C
    from oracle import parity as P
    ns = min(args.parity_queries, args.nq)
    threads, _ = cpu_threads_setup(share=world)
    host = export_host(index)
    cent_np, cb_np = cent.cpu().numpy(), index.get_codebook().cpu().numpy()
    xq_np = xq[:ns].cpu().numpy()
    Dr, Ir = C.ivfpq_search(xq_np, cent_np, cb_np, *host, args.nprobe, args.k)
    aD = torch.empty((world, ns, args.k), dtype=torch.float32, device=device)
    aI = torch.empty((world, ns, args.k), dtype=torch.int64, device=device)
    torch.distributed.all_gather_into_tensor(aD, torch.from_numpy(Dr).to(device))
    torch.distributed.all_gather_into_tensor(aI, torch.from_numpy(Ir).to(device))
    Dg, Ig = D_gpu[:ns].cpu().numpy(), I_gpu[:ns].cpu().numpy()
    H = P.HostIVFPQ(cent_np, cb_np, *host)
    v = H.verify_pairs(xq_np, Dg, Ig, rtol=PARITY_RTOL, atol=PARITY_ATOL)
    acc = torch.tensor([v["rescored_pairs"], v["rescore_out_of_tol"]], dtype=torch.float64, device=device)
    mx = torch.tensor([v["rescore_max_rel_err"]], dtype=torch.float64, device=device)
    torch.distributed.all_reduce(acc)
    torch.distributed.all_reduce(mx, op=torch.distributed.ReduceOp.MAX)
    del host
    if rank != 0:
        return None
    aD, aI = aD.cpu().numpy(), aI.cpu().numpy()
    Dm, Im = O.merge_topk([aD[r] for r in range(world)], [aI[r] for r in range(world)], args.k)
    out = P.topk_parity(Dg, Ig, Dm, Im, rtol=PARITY_RTOL, atol=PARITY_ATOL)
    nvalid = int((Ig >= 0).sum())
    out.update({"rescored_pairs": int(acc[0].item()), "rescore_out_of_tol": int(acc[1].item()),
                "rescore_max_rel_err": float(mx.item()), "unknown_ids": nvalid - int(acc[0].item()),
                "oracle": f"oracle/ann_oracle.c on each of the {world} exported shards ({threads} threads per rank), merged with "
                          "the reference's rule (src/search.py:357-367); parity unpinned: no faiss offline"})
    out["ok"] = bool(out["non_tie_mismatches"] == 0 and out["scores_out_of_tol"] == 0 and out["padding_mismatches"] == 0
                     and out["rescore_out_of_tol"] == 0 and out["unknown_ids"] == 0)
    return out


def measured_peak_gbs():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


def scan_source_hash() -> str:
    """Hash of the scan kernel's source text -- the region of rsb_ivf.cu that holds `raise_tau` and everything from the
    look-up helpers to `ivfpq_scan_kernel`, plus the headers it is built from: stamps profiles/scan_traffic.json, so a
    DRAM-traffic figure captured on another version of the kernel is never reported (other code in the same file --
    work list, LUT builders, the generic-M path -- may change without invalidating the capture)."""
    import hashlib
    csrc = os.path.join(ROOT, "retrieval_scaling_b200", "csrc")
    text = open(os.path.join(csrc, "rsb_ivf.cu")).read()
    h = hashlib.sha256()
    try:
        a0 = text.index("// Raise the running threshold of query")
        a1 = text.index("// IVF-Flat list scan", a0)
        b0 = text.index("// IVF-PQ ADC list scan -- the hot kernel")
        b1 = text.index("// Generic-M path", b0)
        h.update(text[a0:a1].encode())
        h.update(text[b0:b1].encode())
    except ValueError:          # markers moved: fall back to the whole file
        h.update(text.encode())
    for f in ("rsb_common.cuh", "rsb_layout.h", "rsb_tc.cuh"):
        with open(os.path.join(csrc, f), "rb") as fh:
            h.update(fh.read())
    return h.hexdigest()[:16]


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(out_dir: str, I: torch.Tensor, D: torch.Tensor, limit: int = DUMP_LIMIT_BYTES) -> dict:
    """Writes what a caller of the timed search received: ids as float64 (exact below 2**53) and scores as float32.
    When both together would pass `limit` bytes, the same rows of each are written for a sample of queries drawn with
    a fixed seed, and the row numbers go to rows.npy, so runs with the same arguments always write the same rows."""
    ids = I.cpu().numpy().astype(np.float64)
    scores = D.cpu().numpy().astype(np.float32)
    arrays = {"ids": ids, "scores": scores}
    nq = ids.shape[0]
    max_rows = (limit - 4096) // (ids.shape[1] * (8 + 4) + 8)     # 4 KB leaves room for the three .npy headers
    if nq > max_rows:
        rows = np.sort(np.random.default_rng(0).choice(nq, max_rows, replace=False))
        arrays = {"ids": ids[rows], "scores": scores[rows], "rows": rows.astype(np.float64)}
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)
    return {name: list(a.shape) for name, a in arrays.items()}


def workload_name(args):
    return (f"IVF-PQ nlist={args.nlist} M={args.m} nbits=8 nprobe={args.nprobe}, {args.n}x{args.d} synthetic gmm, "
            f"top-k={args.k}, batch of {args.nq} queries")


def make_config(args, world):
    """Identical in both arms (`--impl reference` runs under the same launcher, so it sees the same world size)."""
    return {"workload": workload_name(args), "index": "IVFPQ", "n": args.n, "d": args.d, "nlist": args.nlist,
            "M": args.m, "nbits": 8, "nprobe": args.nprobe, "k": args.k, "nq_per_step": args.nq, "n_gpus": world,
            "sharding": (f"datastore statically partitioned over {world} GPU(s) by {args.partition}; coarse scan sharded "
                         f"by query; per-shard top-k combined over NVLink"),
            "l2": "index (>= 6.4 GB of PQ codes at 100M) is far larger than the 126 MB L2; every step re-reads it"}


# ----------------------------------------------------------------------------------------------------------
def main():
    sys.dont_write_bytecode = True   # the tree may be read-only: the project modules imported below leave no __pycache__
    args = parse()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))

    if args.impl == "reference" and rank != 0:
        return 0  # the CPU arm runs on rank 0 alone
    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    device = torch.device("cuda", local_rank)

    metric = f"queries/sec @ top-k={args.k}, {args.n // 1_000_000}M x {args.d} IVF-PQ"
    config = make_config(args, world)

    # ------------------------------------------------------------------ reference arm (CPU, rank 0 only)
    if args.impl == "reference":
        a1 = argparse.Namespace(**vars(args))
        index, corpus, cent, _, _ = build_index(a1, 0, 1, device)   # setup only: same index, built on the GPU
        xq = corpus.queries(args.nq).cpu().numpy()
        host = export_host(index)
        cent_np, cb_np = cent.cpu().numpy(), index.get_codebook().cpu().numpy()
        del index
        torch.cuda.empty_cache()
        rate, threads, nsample, _, _, cpu_info = cpu_search_rate(host, cent_np, cb_np, xq, args, args.cpu_seconds / 3)
        per_step = int(max(threads, min(args.nq, rate * max(1.0, args.cpu_seconds / max(1, args.steps)))))
        run = cpu_info.pop("_run")
        for _ in range(args.warmup):
            run(xq[:per_step])
        t0 = time.perf_counter()
        for s in range(args.steps):
            run(xq[:per_step])
        dt = time.perf_counter() - t0
        v = per_step * args.steps / dt
        sample = f"{per_step} of the workload's {args.nq} queries per step, full {args.n}-vector index on the host"
        out = {"impl": "reference", "metric": metric, "value": v, "unit": "queries/s", "n_gpus": args.gpus,
               "steps": args.steps, "warmup": args.warmup, "ms_per_step": dt / args.steps * 1e3,
               "higher_is_better": True, "scaling": "strong", "vs_baseline": None, "dtype": "u8 codes / f32 LUT+accumulate",
               "data": "synthetic", "config": config,
               "cpu_baseline": {"value": v, "unit": "queries/s", "cores": threads, "sample": sample, **cpu_info},
               "e2e": {"value": v, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(out), flush=True)
        return 0

    if args.encoder_only:   # development aid: encoder timing without building the 100M index
        if rank == 0:
            print(json.dumps({"encoder": encoder_bench(args, device)}), flush=True)
        return 0

    # ------------------------------------------------------------------ this framework
    run_env = {}
    if world > 1:
        t_init = time.time()
        # NVLS (in-switch multicast) set-up took ~140 s at 8 ranks on this pool and buys nothing for the few-MB
        # gathers of this path; communicator creation takes ~4 s without it.  Override with NCCL_NVLS_ENABLE=1.
        os.environ.setdefault("NCCL_NVLS_ENABLE", "0")
        run_env["NCCL_NVLS_ENABLE"] = os.environ["NCCL_NVLS_ENABLE"]
        torch.distributed.init_process_group("nccl", device_id=device)
        warm = torch.zeros(1, device=device)
        torch.distributed.all_reduce(warm)           # forces communicator creation here, so it shows up in the log
        torch.cuda.synchronize()
        log(f"rank {rank}: NCCL communicator ready after {time.time() - t_init:.1f}s")
    import retrieval_scaling_b200 as rsb
    from retrieval_scaling_b200 import dist as rdist

    xq_all = None
    do_recall = not args.no_recall
    corpus_probe = None
    if do_recall:
        from retrieval_scaling_b200 import synth
        corpus_probe = synth.Corpus(d=args.d, mode="gmm", n_centres=max(16, args.nlist // 4), device=device)
        xq_all = corpus_probe.queries(args.nq)
    n_gt = min(args.recall_queries, args.nq)
    index, corpus, cent, gt_I, build_info = build_index(args, rank, world, device,
                                                        gt_queries=xq_all[:n_gt].contiguous() if do_recall else None)
    del corpus_probe
    xq = xq_all if xq_all is not None else corpus.queries(args.nq)
    index.set_profiling(True)
    searcher = rdist.ShardedSearcher(index, world, rank, fused_gather=args.gather.startswith("fused"),
                                     sliced_merge=(args.gather == "fused"), share_tau=bool(args.share_tau),
                                     peer_coarse=bool(args.peer_coarse))

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    # ---- kernel-resident arm: queries already in HBM
    for _ in range(args.warmup):
        searcher.search(xq, args.k)
    barrier()
    try:
        index.profile()                          # drop the warm-up searches from the per-stage averages
    except Exception:
        pass
    sampler = ClockSampler(local_rank)
    sampler.start()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    searcher.timing = world > 1                  # event records only; read back after the timed region
    barrier()
    e0.record()
    for _ in range(args.steps):
        I, D = searcher.search(xq, args.k)       # no host sync (and no NVML call: it stalls the launch thread) in here
    e1.record()
    barrier()
    ms_total = e0.elapsed_time(e1)
    clocks = sampler.stop()
    searcher.timing = False
    phase_ms = searcher.pop_timing()
    prof_acc = {kk: vv * args.steps for kk, vv in index.profile().items()}   # library averages its per-search events
    t = torch.tensor([ms_total], device=device, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
    ms_step = float(t.item()) / args.steps
    value = args.nq / (ms_step / 1e3)
    gather_desc = {"none": "single GPU", "nccl": "NCCL all_gather_into_tensor + rsb_merge_topk",
                   "fused-p2p": "fused: rsb_merge_topk_peers reads every shard's top-k in place over NVLink "
                                "(symmetric memory) after one device-side barrier",
                   "fused-p2p-sliced": "fused: rsb_merge_topk_peers_scatter -- each GPU merges its 1/G of the queries "
                                       "from every shard's top-k in place (P2P loads) and stores the rows into all "
                                       "GPUs' result buffers (P2P stores); two device-side barriers, no NCCL"
                   }[searcher.gather_mode]
    prof = {kk: vv / args.steps for kk, vv in prof_acc.items()}
    I_keep, D_keep = I.clone(), D.clone()        # result of the last timed step: what the parity block checks

    # ---- end-to-end arm: pinned host queries in, host (ids, scores) out, copies inside the timed region
    sliced = world > 1 and args.e2e_transfer == "sliced"
    per = (args.nq + world - 1) // world
    xq_host = xq.cpu().pin_memory()
    out_rows = per if sliced else args.nq
    I_host = torch.empty((out_rows, args.k), dtype=torch.int64).pin_memory()
    D_host = torch.empty((out_rows, args.k), dtype=torch.float32).pin_memory()

    pipelined = bool(args.e2e_pipeline) and (world == 1 or sliced)
    I_host2 = torch.empty_like(I_host).pin_memory()
    D_host2 = torch.empty_like(D_host).pin_memory()
    host_out = [(I_host, D_host), (I_host2, D_host2)]
    pipe = rdist.HostPipeline(searcher, device, out_slice=sliced) if pipelined else None

    def e2e_step(i=0):
        if pipe is not None:   # upload of batch i+1 / download of batch i-1 overlap the search of batch i
            pipe.submit(xq_host, args.k, host_out[i & 1])
            return
        if sliced:     # each rank uploads 1/G of the queries (all-gathered over NVLink) and downloads the 1/G it merged
            searcher.search_host(xq_host, args.k, device=device, out=(I_host, D_host), out_slice=True)
            return
        q = xq_host.to(device, non_blocking=True)
        I, D = searcher.search(q, args.k)
        I_host.copy_(I, non_blocking=True)
        D_host.copy_(D, non_blocking=True)
        torch.cuda.current_stream().synchronize()

    for i in range(args.warmup):
        e2e_step(i)
    if pipe is not None:
        pipe.drain()
    barrier()
    try:
        index.profile()                          # per-stage averages of the end-to-end searches only
    except Exception:
        pass
    t0 = time.perf_counter()
    for i in range(args.steps):
        e2e_step(i)
    if pipe is not None:
        pipe.drain()
        if (args.steps - 1) & 1:             # the last batch's results are what the equality check below reads
            I_host, D_host = I_host2, D_host2
    barrier()
    t_e2e = torch.tensor([time.perf_counter() - t0], device=device, dtype=torch.float64)
    if world > 1:
        torch.distributed.all_reduce(t_e2e, op=torch.distributed.ReduceOp.MAX)
    e2e_value = args.nq * args.steps / float(t_e2e.item())
    try:                                         # stage times of the searches inside the end-to-end arm, every rank's
        pe = index.profile()
        mine_e = torch.tensor([float(pe.get(nm, 0.0)) for nm in ("scan_ms", "lut_ms", "merge_ms")], device=device, dtype=torch.float64)
        if world > 1:
            all_e = torch.empty(world * 3, device=device, dtype=torch.float64)
            torch.distributed.all_gather_into_tensor(all_e, mine_e)
            all_e = all_e.view(world, 3).cpu().numpy()
        else:
            all_e = mine_e.view(1, 3).cpu().numpy()
        e2e_stage = {nm: [round(float(v), 4) for v in all_e[:, j]] for j, nm in enumerate(("scan_ms", "lut_ms", "merge_ms"))}
    except Exception:
        e2e_stage = None
    # bytes over PCIe per step, summed over the ranks of the job
    h2d = (min(args.nq, per * world) if sliced else args.nq * world) * args.d * 4
    d2h = (I_host.numel() * 8 + D_host.numel() * 4) * world
    # what landed on the host must be the rows of the device-resident result of the timed arm
    if sliced:
        lo = min(args.nq, rank * per)
        nmine = min(args.nq, lo + per) - lo
        e2e_ok = bool(torch.equal(I_host[:nmine], I_keep[lo:lo + nmine].cpu()))
    else:
        e2e_ok = bool(torch.equal(I_host, I_keep.cpu()))

    # ---- roofline of the dominant kernel (ADC list scan): algorithmic bytes = sum over probed (q,list) pairs
    #      of len(list) * M (code bytes only), measured per launch with CUDA events on the launching stream
    peak, peak_src = measured_peak_gbs()
    scan_gbs = prof["scan_bytes"] / prof["scan_ms"] / 1e6 if prof.get("scan_ms", 0) > 0 else None
    roofline = {"bound": "hbm", "kernel": "ivfpq_scan_kernel<K=M/16>", "achieved": scan_gbs, "peak": peak,
                "unit": "GB/s", "frac": (scan_gbs / peak) if scan_gbs else None, "traffic": None,
                "peak_source": peak_src, "bytes_per_launch": prof.get("scan_bytes"),
                "ms_per_launch": prof.get("scan_ms"),
                "note": "algorithmic pair-bytes (sum over probed (query, list) pairs of len x M) against the measured HBM "
                        "peak; batched queries share lists through L2, so DRAM traffic is lower, and ncu shows the "
                        "kernel's binding resource is the L1/shared-memory data pipe, see profiles/"}
    # DRAM traffic of the scan kernel comes from an `ncu --set full` capture of this exact configuration AND this
    # exact kernel source (a number printed under the profiler is never a bench value, so it is read from the
    # committed summary, not measured here; a summary of another kernel version is refused)
    tpath = os.path.join(ROOT, "profiles", "scan_traffic.json")
    if os.path.exists(tpath) and world == 1:
        try:
            tj = json.load(open(tpath))
            c = tj.get("config", {})
            same_cfg = all(c.get(kk) == vv for kk, vv in (("n", args.n), ("nq", args.nq), ("nlist", args.nlist), ("M", args.m),
                                                          ("nprobe", args.nprobe), ("k", args.k)))
            if same_cfg and tj.get("kernel_source_sha16") == scan_source_hash():
                roofline["traffic"] = tj["dram_bytes_per_launch"]
                roofline["traffic_source"] = tj.get("source")
            elif same_cfg:
                roofline["traffic_stale"] = ("profiles/scan_traffic.json was captured on another version of the scan "
                                             "kernel (source hash differs); not reported")
        except Exception:
            pass
    stage_ms = {kk: prof[kk] for kk in ("coarse_ms", "setup_ms", "lut_ms", "scan_ms", "merge_ms") if kk in prof}
    ranks_out = None
    if world > 1:
        # per-rank view: load balance of the list partition (scan time / bytes) and the phases of the sharded search
        names = ["scan_ms", "lut_ms", "merge_ms", "scan_bytes", "coarse_gather_ms", "local_search_ms", "combine_ms"]
        mine = torch.tensor([float(prof.get(nm, phase_ms.get(nm, 0.0))) for nm in names], device=device,
                            dtype=torch.float64)
        allr = torch.empty(world * len(names), device=device, dtype=torch.float64)
        torch.distributed.all_gather_into_tensor(allr, mine)
        allr = allr.view(world, len(names)).cpu().numpy()
        ranks_out = {nm: [round(float(v), 4) for v in allr[:, j]] for j, nm in enumerate(names)}
    from retrieval_scaling_b200 import _lib as _rl
    roofline["scan_path"] = {1: "literal-offset LDS", 2: "generic addressing"}.get(int(round(prof.get("scan_path", 0))), "n/a")
    roofline["dynamic_smem_base"] = int(_rl.lib().rsb_debug_smem_base())

    extra = {}
    if not args.no_sweep and rank == 0 and world == 1:     # right after the search arms: same clock / thermal state
        extra["sweep"] = sweep_microbench(index, args, cent, device)
        if extra["sweep"]["gbs"]:
            extra["sweep"]["frac_of_peak"] = extra["sweep"]["gbs"] / peak
    index.set_profiling(False)
    if do_recall and gt_I is not None and rank == 0:
        extra["recall"] = recall_block(I_keep[:n_gt], gt_I, args.k)
        log("recall:", extra["recall"])
    if not args.no_encoder:
        c5 = c5_encode_plus_search(args, device, rank, world, searcher, xq, steps=args.steps, warmup=args.warmup)
        if rank == 0:
            extra["c5_encode_plus_search"] = c5
            if "recall" in extra:
                c5[f"recall@{args.k}"] = extra["recall"][f"recall@{args.k}"]
            log("c5:", c5)
    if not args.no_encoder and rank == 0:
        extra["encoder"] = encoder_bench(args, device)
        log("encoder:", extra["encoder"])
    if world > 1:
        torch.distributed.barrier()

    cpu_baseline, parity = None, None
    if not args.no_cpu_baseline:
        if world == 1:
            try:
                xq_np = xq.cpu().numpy()
                host = export_host(index)
                cent_np, cb_np = cent.cpu().numpy(), index.get_codebook().cpu().numpy()
                rate, threads, nsample, dt, (D_ref, I_ref), cpu_info = cpu_search_rate(host, cent_np, cb_np, xq_np, args,
                                                                                   args.cpu_seconds)
                cpu_info.pop("_run", None)
                cpu_baseline = {"value": rate, "unit": "queries/s", "cores": threads,
                                "sample": f"{nsample} of the workload's {args.nq} queries against the full {args.n}-vector index ({dt:.1f} s of CPU work)",
                                **cpu_info}
                try:
                    parity = parity_block(host, cent_np, cb_np, xq_np, D_keep.cpu().numpy(), I_keep.cpu().numpy(), D_ref, I_ref)
                except Exception as e:
                    parity = {"ok": False, "error": f"{type(e).__name__}: {e}"}
                del host
            except Exception as e:  # the baseline must never take the bench line down
                cpu_baseline = {"value": None, "unit": "queries/s", "cores": os.cpu_count(), "kind": "port",
                                "sample": f"failed: {type(e).__name__}: {e}"}
        else:
            try:
                parity = parity_block_sharded(index, cent, xq, I_keep, D_keep, args, rank, world, device)
            except Exception as e:
                parity = {"ok": False, "error": f"{type(e).__name__}: {e}"}

    if rank == 0:
        launches = int(round(prof.get("launches", 0))) + (1 if world > 1 else 0)
        out = {"metric": metric, "value": value, "unit": "queries/s", "n_gpus": world, "steps": args.steps,
               "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "strong",
               "vs_baseline": None, "dtype": "u8 codes / f32 LUT+accumulate", "data": "synthetic", "config": config,
               "clocks": clocks,
               "e2e": {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": h2d, "d2h_bytes_per_step": d2h,
                       "transfer": ("sliced: each rank uploads 1/N of the queries and downloads the 1/N of the merged result "
                                    "it produced (bytes are job totals)" if sliced else
                                    "every rank uploads all queries and downloads the full result (bytes are job totals)"),
                       "pipelined": ("dist.HostPipeline: the upload of batch i+1 and the download of batch i-1 overlap the search of "
                                     "batch i (own copy streams, <= 2 batches in flight); every batch is uploaded, searched "
                                     "and downloaded in full" if pipelined else False),
                       "host_result_equals_device_result": e2e_ok, "stage_ms_per_rank": e2e_stage,
                       "ms_per_step": 1e3 * args.nq / e2e_value},
               "gpu_launches": launches * args.steps, "gpu_launches_per_step": launches,
               "roofline": roofline, "stage_ms": stage_ms, "cpu_baseline": cpu_baseline, "parity": parity,
               "gather": gather_desc,
               "multi_gpu": ({"threshold_exchange": bool(args.share_tau and searcher.gather_mode.startswith("fused")),
                              "coarse_tables": ("P2P stores into symmetric memory + barrier" if (args.peer_coarse and searcher.gather_mode.startswith("fused"))
                                                else "2 NCCL all_gather_into_tensor")} if world > 1 else None),
               "build": build_info,
               "run_env": {**run_env, "torch_allow_tf32": bool(torch.backends.cuda.matmul.allow_tf32),
                           "build_gemms": "librsb (3xTF32 tcgen05 + exact fp32 re-score); no cuBLAS in build or search"}}
        if ranks_out is not None:
            out["per_rank"] = ranks_out
        out.update(extra)
        if args.dump_outputs:
            log(f"outputs of the last timed step -> {args.dump_outputs}:", dump_outputs(args.dump_outputs, I_keep, D_keep))
        print(json.dumps(out), flush=True)
    if world > 1:
        torch.distributed.barrier()
        torch.distributed.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
