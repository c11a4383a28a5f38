#!/usr/bin/env python
"""bench.py -- QPS of the batched search hot path (BASELINE.json metric) on N B200s of one node.

A "step" is one pass of the hot path over one batch of synthetic queries:
    VectorIndex::SearchIndex(batch of 10 000 queries, k = 10)  over a device-resident BKT + RNG index.

Workload at N=1 = BASELINE.json configs[1]: SPTAG-BKT, 1M x 768 float32, cosine, batch 10k queries
(`--n/--dim/--metric/--nq` override it for experiments; the JSON always names what ran).

JSON line keys (bench contract): metric/value/unit = whole-job QPS with inputs resident in HBM;
`e2e` = the same metric through the C-ABI entry point with HOST buffers (H2D of the queries and D2H of
the results inside the timed region); `roofline` = achieved algorithmic GB/s of the search kernel
(sum over queries of D_q*row_bytes + E_q*degree*4 + Tn_q*12, SURVEY.md 8d) / CUDA-event time vs
MEASURED_PEAKS.json; `cpu_baseline` = the reference's own CPU search (oracle/_ref, all host threads)
on a bounded sample of the same batch on the same index files.

--impl reference times the UNMODIFIED reference CPU implementation (oracle/_ref/libsptag_ref.so,
VectorIndex::LoadIndex + SearchIndex(batch)) on the same index folder.  The reference/oracle is only
ever executed in that leg and in the cpu_baseline leg -- never on the product path.

Multi-GPU (`--gpus N` under torchrun, one rank per GPU).  Default `--mode auto` runs BOTH forms and says which is which:
  replica leg -> `value`: every rank holds the C2 index and searches its OWN 10k-query batch; no data-path collective
        (queries are the independent units); weak scaling; this is the aggregate-QPS figure of the north star.
  shard leg -> key `shard`: BASELINE config 5's form (SURVEY.md 8e): rank r holds an independent index over vector
        partition r (2.5M x 768 per GPU, ids offset), every rank searches the SAME batch, the per-shard top-k lists are
        exchanged with ONE NCCL all-gather and merged on the GPU (sptag_b200/sharded.py ShardedSearch).  Its parity is
        checked against the REFERENCE searched shard by shard (each rank runs oracle/_ref on its own shard, the lists
        are host-merged by (Dist, VID), QueryResultSet.h:17-26) -- ids and distance bits.
  `--mode replica` / `--mode shard` run one form only (shard: `value` is the shard-mode QPS over the N-shard corpus).
"""
import argparse
import contextlib
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
# the index build runs with torch's deterministic algorithms (deterministic_build), which require a fixed cuBLAS
# workspace configuration; cuBLAS reads it when its first handle is created, so it is set before torch is imported
os.environ.setdefault("CUBLAS_WORKSPACE_CONFIG", ":4096:8")

BUILDER_VERSION = 4   # 4: deterministic index build
L2_BYTES = 126 * 1000 * 1000  # B200 L2 (B200_PROFILING.md)


def l2_policy_text(row_bytes_total):
    gb = row_bytes_total / 1e9
    if row_bytes_total > 4 * L2_BYTES:
        return "index (%.2f GB of vector rows) and per-step traffic are larger than L2; no explicit flush" % gb
    if row_bytes_total > L2_BYTES:
        return ("index (%.2f GB of vector rows) is only %.1fx the L2: rows are partly L2-resident between steps, no explicit "
                "flush -- this line is not an HBM-roofline measurement" % (gb, row_bytes_total / L2_BYTES))
    return ("index (%.3f GB of vector rows) fits the L2: rows are L2-resident, no explicit flush -- this line is not an "
            "HBM-roofline measurement" % gb)


def log(*a):
    if int(os.environ.get("RANK", "0")) == 0:
        print("[bench]", *a, file=sys.stderr, flush=True)


REFERENCE_DUMP_QUERIES = 256   # the least the reference arm's timed sample holds


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=20)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--mode", default="auto", choices=["auto", "replica", "shard"])
    ap.add_argument("--shard-n", type=int, default=2500000, help="vectors per GPU in the shard leg of --mode auto (config C5: 20M / 8)")
    ap.add_argument("--shard-parity-sample", type=int, default=256, help="queries the reference searches shard by shard")
    ap.add_argument("--in-flight", type=int, default=1, choices=[1, 2],
                    help="2: consecutive batches alternate between two CUDA streams (and two output buffers), so batch i+1 starts "
                         "on the SMs batch i's tail has vacated; reported as the extra key `pipelined` -- `value` stays one batch at a time")
    ap.add_argument("--builder", default="gpu", choices=["gpu", "reference"],
                    help="reference: the index is built by the unmodified reference (oracle/_ref BuildIndex) on the host cores")
    # (--num-vectors: under `python -m torch.distributed.run` a bare --n is swallowed by torchrun's own
    #  abbreviation matching (--nnodes / --nproc-per-node), so multi-GPU launches must use the long name)
    ap.add_argument("--n", "--num-vectors", dest="n", type=int, default=1000000)
    ap.add_argument("--dim", type=int, default=768)
    ap.add_argument("--metric", default="Cosine", choices=["Cosine", "L2"])
    ap.add_argument("--nq", type=int, default=10000)
    ap.add_argument("--k", type=int, default=10)
    ap.add_argument("--maxcheck", type=int, default=8192)
    ap.add_argument("--data", default="lowrank", choices=["lowrank", "iid"])
    ap.add_argument("--rank-dim", type=int, default=32, help="latent rank of the low-rank synthetic set")
    ap.add_argument("--seed", type=int, default=1234)
    ap.add_argument("--cache", default=os.environ.get("SPTAG_B200_CACHE", "/tmp/sptag_b200_cache"))
    ap.add_argument("--cpu-sample", type=int, default=0, help="queries in the cpu_baseline sample (0 = auto)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-clocks", action="store_true", help="debug: do not sample nvidia-smi during the timed region")
    ap.add_argument("--param", action="append", default=[], help="Name=Value passed to sptag_b200_set_param")
    ap.add_argument("--tpt-above", type=int, default=2500000,
                    help="builder: above this many vectors use partition-tree kNN candidates instead of brute force")
    ap.add_argument("--algo", default="bkt", choices=["bkt", "kdt"], help="space-partition tree of the index")
    ap.add_argument("--quantizer", default="none", choices=["none", "pq", "opq"],
                    help="index holds uint8 PQ codes (BASELINE config 4 shape: --quantizer opq --raw-type int8 --dim 100 --pq-m 50)")
    ap.add_argument("--pq-m", type=int, default=50, help="number of PQ sub-vectors")
    ap.add_argument("--raw-type", default="float", choices=["float", "int8"], help="element type of raw vectors/queries")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the result lists of the last timed step as DIR/ids.npy (float64) and DIR/dists.npy (float32); "
                         "--impl reference writes its first %d queries (its per-step sample is sized by timing)" % REFERENCE_DUMP_QUERIES)
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    return args


DUMP_LIMIT_BYTES = 64 << 20


def dump_outputs(folder, ids, dists):
    """What a caller of the timed path receives: ids [nq, k] as float64 (exact for int32 ids) and dists [nq, k] as
    float32.  Above DUMP_LIMIT_BYTES a fixed, seeded sample of query rows is written, with its row numbers in rows.npy."""
    import numpy as np
    ids = np.asarray(ids).astype(np.float64)
    dists = np.asarray(dists, dtype=np.float32)
    row_bytes = ids.shape[1] * 8 + dists.shape[1] * 4 + 8
    os.makedirs(folder, exist_ok=True)
    if ids.shape[0] * row_bytes > DUMP_LIMIT_BYTES:
        rows = np.sort(np.random.default_rng(0).choice(ids.shape[0], DUMP_LIMIT_BYTES // row_bytes, replace=False))
        ids, dists = ids[rows], dists[rows]
        np.save(os.path.join(folder, "rows.npy"), rows.astype(np.float64))
    np.save(os.path.join(folder, "ids.npy"), ids)
    np.save(os.path.join(folder, "dists.npy"), dists)
    log("outputs of the last timed step written to %s" % folder)


# ---------------------------------------------------------------------------------------------
# synthetic data + index folder (built on the GPU once per box, cached under --cache)
# ---------------------------------------------------------------------------------------------
def gen_data(args, n, seed, device):
    """Synthetic vectors [n, dim] (float32 values; int8-valued when --raw-type int8).  Generated in 10M-row pieces so
    that 100M-point sets never need more than the result plus one piece of temporaries."""
    import torch
    piece = 10000000
    if n > piece:
        out = torch.empty((n, args.dim), dtype=torch.float32, device=device)
        for i, s in enumerate(range(0, n, piece)):
            e = min(n, s + piece)
            out[s:e] = gen_data(args, e - s, seed * 1000003 + i + 1, device)
        return out
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    if args.data == "iid":
        x = torch.randn((n, args.dim), generator=g, device=device, dtype=torch.float32)
    else:
        # BASELINE.md "low-rank synthetic": x = z.A + 0.1*eps, A entries N(0,1)/sqrt(r)
        # the mixing matrix is shared by base vectors, shards and queries -- and by indexes prepared on another machine
        # (build/bench_cache: the reference-built folder is built on the CPU container), so it always comes from the CPU
        # generator, whatever device the rest is drawn on
        ga = torch.Generator(device="cpu")
        ga.manual_seed(args.seed)
        r = args.rank_dim
        A = (torch.randn((r, args.dim), generator=ga, device="cpu", dtype=torch.float32) / (r ** 0.5)).to(device)
        z = torch.randn((n, r), generator=g, device=device, dtype=torch.float32)
        x = z @ A
        x += 0.1 * torch.randn((n, args.dim), generator=g, device=device, dtype=torch.float32)
    if args.raw_type == "int8":
        # SPACEV-style int8 raw vectors (SURVEY.md 8d): clamp(round(32 x), -127, 127), kept as float values here
        x = torch.clamp(torch.round(32.0 * x), -127, 127)
    if args.metric == "Cosine":
        # the reference normalises base vectors at build time (BKTIndex.cpp:749-756) and expects
        # unit-norm queries from the caller
        x = x / x.norm(dim=1, keepdim=True).clamp_min(1e-30)
    return x.contiguous()


@contextlib.contextmanager
def deterministic_build():
    """The index is an input of every timed step: build it with torch's deterministic kernels (index_add_ without float
    atomics in the k-means) so that the same arguments give the same index, and the same outputs, on every run.  An op
    without a deterministic implementation raises instead of building a different index."""
    import torch
    prev = torch.are_deterministic_algorithms_enabled()
    torch.use_deterministic_algorithms(True)
    try:
        yield
    finally:
        torch.use_deterministic_algorithms(prev)


def index_folder(args, shard):
    key = "%s_%s_%dx%d_%s_r%d_s%d_shard%d_v%d" % (args.algo, args.metric, args.n, args.dim, args.data, args.rank_dim,
                                                   args.seed, shard, BUILDER_VERSION)
    if args.tpt_above != 2500000:
        key += "_tpt%d" % args.tpt_above
    if args.quantizer != "none":
        key += "_%s%d_%s" % (args.quantizer, args.pq_m, args.raw_type)
    elif args.raw_type != "float":
        key += "_" + args.raw_type
    if getattr(args, "builder", "gpu") == "reference":
        key += "_refbuilt"
    return os.path.join(args.cache, key)


def ensure_index(args, shard, device):
    """Build (GPU, torch) and save the reference-format folder unless it is cached. Returns folder."""
    import numpy as np
    import torch
    from tools import gpu_index_builder as B
    folder = index_folder(args, shard)
    done = os.path.join(folder, "DONE")
    if os.path.exists(done):
        return folder
    t0 = time.time()
    if getattr(args, "builder", "gpu") == "reference":
        # the index SPTAG itself produces: the unmodified reference's BuildIndex (k-means BKT / KD-tree, TP-tree initial
        # graph, RefineGraph passes) on the host cores, then its own SaveIndex
        if args.quantizer != "none" or args.raw_type != "float":
            raise SystemExit("--builder reference: float un-quantized indexes only")
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import reflib
        x = gen_data(args, args.n, args.seed + 1000 * (shard + 1), device).cpu().numpy()
        ridx = reflib.RefIndex.build(args.algo.upper(), x, args.metric, threads=os.cpu_count() or 1)
        ridx.save(folder)
        del ridx
        with open(done, "w") as f:
            f.write("ok\n")
        log("index built by the reference in %.1fs -> %s" % (time.time() - t0, folder))
        return folder
    torch.backends.cuda.matmul.allow_tf32 = True
    x = gen_data(args, args.n, args.seed + 1000 * (shard + 1), device)
    with deterministic_build():
        nodes, starts, graph = B.build_index(x, args.metric, seed=args.seed + shard, log=log, algo=args.algo.upper(),
                                             tpt_above=args.tpt_above)
    if args.quantizer != "none":
        with deterministic_build():
            cb, rot = B.train_quantizer_gpu(x, args.pq_m, opq=(args.quantizer == "opq"), seed=args.seed)
            codes = B.encode_gpu(x, cb, rot)
        blob = B.quantizer_blob(cb, rot, 0 if args.raw_type == "int8" else 3)
        B.save_index_folder(folder, codes.cpu().numpy(), graph, nodes, starts, args.metric, quantizer=blob)
    elif args.raw_type == "int8":   # unquantized int8 rows (DistanceUtils int8 variants), e.g. SPACEV / PerfTest.cpp shape
        B.save_index_folder(folder, x.cpu().numpy().astype(np.int8), graph, nodes, starts, args.metric,
                            algo=args.algo.upper(), value_type="Int8")
    else:
        B.save_index_folder(folder, x.cpu().numpy(), graph, nodes, starts, args.metric, algo=args.algo.upper())
    torch.backends.cuda.matmul.allow_tf32 = False
    with open(done, "w") as f:
        f.write("ok\n")
    del x
    torch.cuda.empty_cache()
    log("index shard %d built and saved in %.1fs -> %s" % (shard, time.time() - t0, folder))
    return folder


class _InMemoryIndex:
    """What bench needs from reflib.IndexFiles, for an index that is built and handed to the device without touching
    the disk (shard mode on many GPUs: eight 8-GB folders would not fit the box's scratch disk)."""

    def __init__(self, vectors, graph, nodes, tree_starts, metric_name):
        self.vectors, self.graph, self.nodes, self.tree_starts = vectors, graph, nodes, tree_starts
        self.value_type = 3
        self.metric = {"L2": 0, "Cosine": 1}[metric_name]
        self.n, self.dim = vectors.shape
        self.degree = graph.shape[1]
        self.quantizer = None


def build_in_memory(args, shard, device):
    import numpy as np
    import torch
    from tools import gpu_index_builder as B
    t0 = time.time()
    torch.backends.cuda.matmul.allow_tf32 = True
    x = gen_data(args, args.n, args.seed + 1000 * (shard + 1), device)
    with deterministic_build():
        nodes, starts, graph = B.build_index(x, args.metric, seed=args.seed + shard, log=log, algo=args.algo.upper(),
                                             tpt_above=args.tpt_above)
    torch.backends.cuda.matmul.allow_tf32 = False
    files = _InMemoryIndex(x.cpu().numpy(), graph, nodes, starts, args.metric)
    del x
    torch.cuda.empty_cache()
    log("index shard %d built in memory in %.1fs" % (shard, time.time() - t0))
    return files


def load_folder_arrays(folder):
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import reflib
    return reflib.IndexFiles(folder)


# ---------------------------------------------------------------------------------------------
# clocks sampler (profiling recipe's nvidia-smi line)
# ---------------------------------------------------------------------------------------------
class ClockSampler:
    FIELDS = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
              "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
              "clocks_event_reasons.sw_power_cap")

    def __init__(self, device):
        self.device = device
        self.lines = []
        self.proc = None

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.device), "--query-gpu=" + self.FIELDS,
                 "--format=csv,noheader,nounits", "-lms", "100"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL,
                text=True)
            self.thread = threading.Thread(target=self._read, daemon=True)
            self.thread.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.lines.append((time.time(), line.strip()))

    def mark(self):
        return time.time()

    def stop(self):
        if self.proc:
            self.proc.terminate()
            try:
                self.proc.wait(timeout=2)
            except Exception:
                self.proc.kill()

    def summary(self, t0, t1):
        sm, mx, reasons = [], 0.0, set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ts, line in self.lines:
            if ts < t0 - 0.05 or ts > t1 + 0.15:
                continue
            parts = [p.strip() for p in line.split(",")]
            if len(parts) < 7:
                continue
            try:
                sm.append(float(parts[0]))
                mx = max(mx, float(parts[1]))
            except ValueError:
                continue
            for nm, v in zip(names, parts[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        if not sm:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": [], "samples": 0}
        sm.sort()
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": mx, "reasons": sorted(reasons), "samples": len(sm)}


# ---------------------------------------------------------------------------------------------
# reference / cpu baseline leg (the ONLY place the oracle is executed by bench.py)
# ---------------------------------------------------------------------------------------------
def cpu_search_leg(folder, queries_np, k, maxcheck, threads, sample, repeats=1, each=False):
    """Times the reference's CPU SearchIndex(batch) on `sample` queries. Returns dict + ids for a parity check."""
    import numpy as np
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import reflib
    q = np.ascontiguousarray(queries_np[:sample])
    if reflib.have_ref():
        kind = "reference"
        idx = reflib.RefIndex.load(folder)
        idx.set_param("MaxCheck", maxcheck)
        # quantized indexes: the per-query overload on raw queries, as IndexSearcher does (SURVEY.md 8b)
        run = idx.search_each if each else idx.search
        run(q[:min(256, sample)], k, threads=threads)  # creates the per-thread work spaces
        best = None
        for _ in range(repeats):
            ids, dists, sec = run(q, k, threads=threads)
            best = sec if best is None else min(best, sec)
        isa = reflib.ref().ref_isa()
    else:
        kind = "port"
        files = reflib.IndexFiles(folder)
        o = reflib.OracleIndex(files)
        o.max_check = maxcheck
        best = None
        for _ in range(repeats):
            t = time.time()
            ids, dists, _ = o.search(q, k, threads=threads, want_stats=False)
            sec = time.time() - t
            best = sec if best is None else min(best, sec)
        isa = 512
    return {"value": sample / best, "unit": "queries/s", "cores": threads, "kind": kind,
            "sample": "%d of the %d-query batch, MaxCheck %d, %d OpenMP threads, ISA %d, best of %d"
                      % (sample, queries_np.shape[0], maxcheck, threads, isa, repeats),
            "seconds": best}, ids, dists


def best_cpu_threads(folder, queries_np, k, maxcheck, each=False):
    """The reference gets every host thread it can use; on SMT boxes one thread per physical core is
    sometimes faster for this DRAM-bound loop, so probe both and keep the faster."""
    n = os.cpu_count() or 1
    cands = sorted({n, max(1, n // 2)}, reverse=True)
    best_t, best_v = n, -1.0
    for t in cands:
        r, _, _ = cpu_search_leg(folder, queries_np, k, maxcheck, t, min(queries_np.shape[0], 1024), each=each)
        if r["value"] > best_v:
            best_t, best_v = t, r["value"]
    return best_t


def recall_at_k(ids, truth, k):
    import numpy as np
    hit = 0
    for i in range(ids.shape[0]):
        hit += len(set(ids[i, :k].tolist()) & set(truth[i, :k].tolist()))
    return hit / float(ids.shape[0] * k)


# ---------------------------------------------------------------------------------------------
def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    if world != args.gpus and world > 1:
        args.gpus = world

    quantized = args.quantizer != "none"
    if quantized or args.raw_type == "int8":
        # the reference's quantizers have no cosine distance (PQQuantizer.h:130-136); int8 cosine needs base-127
        # normalised rows, which this synthetic generator does not produce
        args.metric = "L2"
    workload = "SPTAG-%s, %dx%d %s %s, batch %d queries, k=%d, MaxCheck=%d, %s synthetic" % (
        args.algo.upper(), args.n, args.dim, "float32" if args.raw_type == "float" else "int8", args.metric.lower(), args.nq, args.k,
        args.maxcheck, args.data)
    if quantized:
        workload += ", %s uint8 codes M=%d Ks=256 (SDC)" % (args.quantizer.upper(), args.pq_m)
    config = {"workload": workload, "index": "%s+RNG(degree 32)" % args.algo.upper(), "n": args.n, "dim": args.dim,
              "metric": args.metric, "batch": args.nq, "k": args.k, "max_check": args.maxcheck,
              "parallelism": ("%s x%d" % (args.mode, args.gpus)) if args.gpus > 1 else "single GPU",
              "l2_policy": l2_policy_text(args.n * (args.pq_m if quantized else args.dim * 4))}

    # ------------------------------ reference arm ------------------------------
    if args.impl == "reference":
        if rank != 0:
            return 0
        import numpy as np
        import torch
        dev = torch.device("cuda", 0) if torch.cuda.is_available() else None
        if dev is None and not os.path.exists(os.path.join(index_folder(args, 0), "DONE")):
            print(json.dumps({"impl": "reference", "unavailable": "index folder not cached and no GPU to build it"}))
            return 0
        folder = ensure_index(args, 0, dev) if dev is not None else index_folder(args, 0)
        q = gen_data(args, args.nq, args.seed + 7, dev if dev is not None else "cpu").cpu().numpy()
        if args.raw_type == "int8":
            q = q.astype(np.int8)
        threads = best_cpu_threads(folder, q, args.k, args.maxcheck, each=quantized)
        # bounded sample per step: probe the speed, then size a step to ~3 s of CPU work
        probe, _, _ = cpu_search_leg(folder, q, args.k, args.maxcheck, threads, min(args.nq, 512), each=quantized)
        sample = int(max(256, min(args.nq, probe["value"] * 3.0)))
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import reflib
        idx = reflib.RefIndex.load(folder) if reflib.have_ref() else None
        secs = []
        if idx is not None:
            idx.set_param("MaxCheck", args.maxcheck)
            kind = "reference"
            for s in range(args.warmup + args.steps):
                ids, dists, sec = (idx.search_each if quantized else idx.search)(q[:sample], args.k, threads=threads)
                if s >= args.warmup:
                    secs.append(sec)
        else:
            kind = "port"
            o = reflib.OracleIndex(reflib.IndexFiles(folder))
            o.max_check = args.maxcheck
            for s in range(args.warmup + args.steps):
                t = time.time()
                ids, dists, _ = o.search(q[:sample], args.k, threads=threads, want_stats=False)
                if s >= args.warmup:
                    secs.append(time.time() - t)
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, ids[:REFERENCE_DUMP_QUERIES], dists[:REFERENCE_DUMP_QUERIES])
        total = sum(secs)
        qps = sample * len(secs) / total
        line = {"impl": "reference", "metric": "queries_per_second", "value": qps, "unit": "queries/s",
                "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": 1000.0 * total / len(secs), "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": qps, "unit": "queries/s", "cores": threads, "kind": kind,
                                 "sample": "%d of the %d-query batch per step, MaxCheck %d, %d OpenMP threads"
                                           % (sample, args.nq, args.maxcheck, threads)},
                "e2e": {"value": qps, "unit": "queries/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return 0

    # ------------------------------ B200 arm ------------------------------
    return b200_arm(args, rank, local_rank, world, quantized, config)



def host_info():
    """What the reference arm's number depends on (VERDICT r1: 1 745 QPS at 64 threads on one box, 5 319 at 128 on another)."""
    info = {"cpu_count": os.cpu_count()}
    try:
        info["affinity_cpus"] = len(os.sched_getaffinity(0))
    except Exception:
        info["affinity_cpus"] = None
    try:
        info["numa_nodes"] = len([d for d in os.listdir("/sys/devices/system/node") if d.startswith("node")])
    except Exception:
        info["numa_nodes"] = None
    try:
        for ln in open("/proc/cpuinfo"):
            if ln.startswith("model name"):
                info["cpu_model"] = ln.split(":", 1)[1].strip()
                break
    except Exception:
        pass
    return info


def kept_traffic(workload_key, alg_bytes):
    """roofline.traffic: dram__bytes_read.sum + dram__bytes_write.sum of one launch of the dominant kernel from a kept
    `ncu --set full` capture of the same workload (profiles/r02_ncu_traffic.json, written from the .ncu-rep by
    tools/ncu_traffic.py); None when no capture of this workload is kept."""
    path = os.path.join(ROOT, "profiles", "r02_ncu_traffic.json")
    if not os.path.exists(path):
        return None, None
    try:
        rec = json.load(open(path)).get(workload_key)
    except Exception:
        return None, None
    if not rec:
        return None, None
    # the capture may have been taken with a different batch size: DRAM bytes per launch scale with the algorithmic
    # bytes of the launch (same index, same budget), so report the measured ratio applied to this launch
    ratio = rec["dram_bytes"] / float(rec["algorithmic_bytes"])
    return ratio * alg_bytes, {"source": rec.get("source"), "dram_bytes_captured": rec["dram_bytes"],
                               "algorithmic_bytes_captured": rec["algorithmic_bytes"], "queries_captured": rec.get("nq"),
                               "traffic_over_algorithmic": ratio}


def b200_arm(args, rank, local_rank, world, quantized, config):
    import numpy as np
    import torch
    import __graft_entry__
    if not os.path.exists(__graft_entry__.LIB):
        __graft_entry__.build_cuda()
    from sptag_b200 import B200Index, capi

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a GPU: the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    dist = None
    if world > 1:
        import torch.distributed as dist
        import datetime
        dist.init_process_group("nccl", device_id=dev, timeout=datetime.timedelta(seconds=600))

    mode = args.mode if world > 1 else "single"
    do_main = mode in ("single", "auto", "replica")
    do_shard = mode in ("auto", "shard")
    line = None
    if do_main:
        line = main_leg(args, rank, local_rank, world, dev, dist, quantized, config, "replica" if world > 1 else "single")
    shard = None
    if do_shard:
        torch.cuda.empty_cache()
        shard = shard_leg(args, rank, local_rank, world, dev, dist, config)
    if rank == 0:
        if line is None:  # --mode shard: the shard figure is the line's value
            line = {"metric": "queries_per_second", "value": shard["value"], "unit": "queries/s", "n_gpus": args.gpus,
                    "steps": args.steps, "warmup": args.warmup, "ms_per_step": shard["ms_per_step"], "higher_is_better": True,
                    "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic",
                    "config": dict(config, parallelism="shard x%d" % world, n=shard["vectors_per_gpu"],
                                   workload=shard["workload"]),
                    "recall_at_10": None, "clocks": shard.pop("clocks", None), "e2e": shard["e2e"],
                    "gpu_launches": shard["gpu_launches"], "roofline": shard["roofline"], "cpu_baseline": None,
                    "parity_vs_reference": shard["parity_vs_reference"]}
        line["shard"] = shard
        if shard is not None and do_main:
            line["config"]["parallelism"] = ("replica x%d -> `value` (aggregate QPS, no collective); shard x%d -> key `shard` "
                                             "(config C5's form: NCCL all-gather + merge_topk_kernel)" % (world, world))
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()
    return 0


def main_leg(args, rank, local_rank, world, dev, dist, quantized, config, mode):
    """The C2-style leg: every rank holds the whole index and searches its own batch (world == 1: the single-GPU bench)."""
    import numpy as np
    import torch
    from sptag_b200 import B200Index, capi

    # ---- set-up (untimed): index folder, device-resident index, queries, ground truth ----
    if world > 1:
        if rank == 0:
            ensure_index(args, 0, dev)
        dist.barrier()
    folder = ensure_index(args, 0, dev)
    t0 = time.time()
    # the native loader streams the reference's files into HBM (sptag_b200_load); the numpy view of the folder is only
    # used by the untimed bookkeeping below (row size, ground truth)
    files = load_folder_arrays(folder)
    idx = B200Index.load(folder, device=local_rank)
    idx.set_param("MaxCheck", args.maxcheck)
    for kv in args.param:
        nm, v = kv.split("=", 1)
        idx.set_param(nm, v)
    log("index loaded into HBM in %.1fs (sptag_b200_load)" % (time.time() - t0))

    qseed = args.seed + 7 + rank
    d_q_f32 = gen_data(args, args.nq, qseed, dev)
    qdtype = torch.int8 if args.raw_type == "int8" else torch.float32
    d_q = d_q_f32.to(qdtype).contiguous()
    h_q = torch.empty((args.nq, args.dim), dtype=qdtype, pin_memory=True)
    h_q.copy_(d_q)
    d_ids = torch.empty((args.nq, args.k), dtype=torch.int32, device=dev)
    d_dists = torch.empty((args.nq, args.k), dtype=torch.float32, device=dev)
    d_stats = torch.zeros((args.nq, capi.STATS_PER_QUERY), dtype=torch.int32, device=dev)
    h_ids = torch.empty((args.nq, args.k), dtype=torch.int32, pin_memory=True)
    h_dists = torch.empty((args.nq, args.k), dtype=torch.float32, pin_memory=True)
    stream = torch.cuda.current_stream().cuda_stream

    def step_device(with_stats=False):
        idx.search_device(d_q.data_ptr(), args.nq, args.k, d_ids.data_ptr(), d_dists.data_ptr(),
                          d_stats.data_ptr() if with_stats else 0, stream)

    def step_e2e():
        # the call a user makes: host query buffer in, host results out (H2D + kernel + D2H, blocking)
        idx.search(h_q.numpy(), args.k, out_ids=h_ids.numpy(), out_dists=h_dists.numpy())

    def sync_all():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
            torch.cuda.synchronize()

    # one untimed pass with counters -> algorithmic bytes of one launch (SURVEY.md 8d)
    step_device(with_stats=True)
    torch.cuda.synchronize()
    st = d_stats.cpu().numpy().astype(np.int64)
    row_bytes = files.vectors.shape[1] * files.vectors.itemsize  # dim*4, or M code bytes when quantized
    alg_bytes = int((st[:, capi.ST_NDIST] * row_bytes + st[:, capi.ST_NEXPAND] * files.degree * 4
                     + st[:, capi.ST_NTREE] * (16 if args.algo == "kdt" else 12)).sum())
    res_ids = d_ids.cpu().numpy()
    res_d = d_dists.cpu().numpy()

    # recall@10 against exact search (untimed)
    from tools import gpu_index_builder as B
    if quantized:  # ground truth on the raw vectors (regenerated: the folder only holds codes)
        x_dev = gen_data(args, args.n, args.seed + 1000, dev)
    else:
        x_dev = torch.from_numpy(np.ascontiguousarray(files.vectors)).to(dev).float()   # int8 rows: exact truth on their float values
    truth = B.exact_topk(x_dev, d_q_f32, args.k, args.metric)
    del x_dev
    torch.cuda.empty_cache()
    recall = recall_at_k(res_ids, truth, args.k)
    log("recall@%d = %.4f, mean D_q = %.0f, E_q = %.0f, Tn_q = %.0f" % (
        args.k, recall, st[:, capi.ST_NDIST].mean(), st[:, capi.ST_NEXPAND].mean(), st[:, capi.ST_NTREE].mean()))

    # ---- timed region 1: inputs resident in HBM (value, roofline) ----
    sampler = ClockSampler(local_rank)
    if rank == 0 and not args.no_clocks:
        sampler.start()
        time.sleep(0.3)
    for _ in range(args.warmup):
        step_device()
    sync_all()
    launches0 = capi.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tm0 = time.time()
    ev0.record()
    for _ in range(args.steps):
        step_device()
    ev1.record()
    sync_all()
    tm1 = time.time()
    launches = capi.launch_count() - launches0
    if args.dump_outputs:
        last_ids, last_dists = d_ids.cpu().numpy(), d_dists.cpu().numpy()
    ms_total = ev0.elapsed_time(ev1)
    if world > 1:
        t = torch.tensor([ms_total], dtype=torch.float64, device=dev)
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        ms_total = float(t.item())
    ms_step = ms_total / args.steps
    queries_per_step = args.nq * world
    value = queries_per_step / (ms_step / 1000.0)

    # ---- optional: the same K steps with two batches in flight (alternating streams; the library gives each its own scratch) ----
    pipelined = None
    if args.in_flight == 2:
        s2 = torch.cuda.Stream(device=dev)
        d_ids2 = torch.empty_like(d_ids)
        d_dists2 = torch.empty_like(d_dists)

        def step_pipe(i):
            if i & 1:
                idx.search_device(d_q.data_ptr(), args.nq, args.k, d_ids2.data_ptr(), d_dists2.data_ptr(), 0, s2.cuda_stream)
            else:
                idx.search_device(d_q.data_ptr(), args.nq, args.k, d_ids.data_ptr(), d_dists.data_ptr(), 0, stream)

        for i in range(max(2, args.warmup)):
            step_pipe(i)
        sync_all()
        pe0, pe1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        s2.wait_stream(torch.cuda.current_stream())
        pe0.record()
        for i in range(args.steps):
            step_pipe(i)
        torch.cuda.current_stream().wait_stream(s2)
        pe1.record()
        sync_all()
        pms = pe0.elapsed_time(pe1)
        if world > 1:
            t = torch.tensor([pms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            pms = float(t.item())
        same = bool((d_ids2 == d_ids).all().item()) if args.steps >= 2 else None
        pipelined = {"value": queries_per_step / (pms / args.steps / 1000.0), "unit": "queries/s", "ms_per_step": pms / args.steps,
                     "batches_in_flight": 2, "results_identical_to_serial": same,
                     "note": "K steps, consecutive batches on alternating CUDA streams; each launch has its own scratch set"}

    # ---- timed region 2: end to end through the C-ABI with host buffers (pinned, then pageable) ----
    def time_e2e(fn):
        for _ in range(args.warmup):
            fn()
        sync_all()
        t0 = time.perf_counter()
        for _ in range(args.steps):
            fn()
        torch.cuda.synchronize()
        sec = time.perf_counter() - t0
        if world > 1:
            t = torch.tensor([sec], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            sec = float(t.item())
        return queries_per_step * args.steps / sec

    e2e_value = time_e2e(step_e2e)
    # the same call from ordinary (pageable) numpy buffers -- what a caller that never pins memory sees
    p_q = np.array(h_q.numpy(), copy=True)
    p_ids = np.empty((args.nq, args.k), np.int32)
    p_d = np.empty((args.nq, args.k), np.float32)
    e2e_pageable = time_e2e(lambda: idx.search(p_q, args.k, out_ids=p_ids, out_dists=p_d))
    clocks = None
    if rank == 0:
        sampler.stop()
        clocks = sampler.summary(tm0, tm1)

    if rank != 0:
        idx.close()
        return None
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, last_ids, last_dists)

    # ---- roofline of the dominant (only) kernel of a step ----
    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak = float(json.load(open(peaks_path))["hbm_gbs"])
        peak_src = "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    # kernel duration: the step on this stream is memset(4 B) + the search kernel; time the kernel alone
    # with the library's own CUDA events (recorded on the launching stream around the launch)
    kms = []
    for _ in range(5):
        step_device()  # rank 0 only from here on: no collectives
        kms.append(idx.last_kernel_ms())
    kernel_ms = float(np.mean(kms))
    achieved = alg_bytes / (kernel_ms / 1000.0) / 1e9
    kname = ("search_kernel<PQ,L2,BKT>" if quantized else "search_kernel<int8,L2,%s>" % args.algo.upper()
             if args.raw_type == "int8" else
             "search_kernel<%d,%s,%s>" % (args.dim if args.dim in (128, 768) else 0, args.metric, args.algo.upper()))
    wkey = "%s_%s_%dx%d_mc%d%s" % (args.algo, args.metric, args.n, args.dim, args.maxcheck,
                                    ("_%s%d" % (args.quantizer, args.pq_m)) if quantized else "")
    traffic, traffic_note = kept_traffic(wkey, alg_bytes)
    row_bytes_total = args.n * (args.pq_m if quantized else args.dim * (1 if args.raw_type == "int8" else 4))
    roofline = {"bound": "hbm" if row_bytes_total > 4 * L2_BYTES else "hbm (index partly or wholly L2-resident: see l2_note)",
                "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                "traffic": traffic, "traffic_note": traffic_note, "kernel": kname, "kernel_ms": kernel_ms,
                "kernel_ms_samples": [round(v, 3) for v in kms],
                "algorithmic_bytes_per_launch": alg_bytes, "peak_source": peak_src,
                "share_of_step": kernel_ms / ms_step}

    if row_bytes_total <= 4 * L2_BYTES:
        roofline["l2_note"] = ("the vector rows (%.0f MB) are not much larger than the 126 MB L2, so part of the algorithmic "
                               "bytes are served by L2 hits and never reach HBM: `achieved` / `frac` count algorithmic bytes "
                               "and can exceed the HBM peak here; the HBM roofline bounds the configurations whose rows are "
                               "several times the L2 (C2: 3.07 GB)" % (row_bytes_total / 1e6))
    if quantized:
        # The quantized kernel's HBM bytes are only the M code bytes per distance; what it really moves is the SDC table:
        # one 4-byte look-up per sub-vector, each a 32-byte L2 sector request unless lanes of the same instruction share a
        # sector.  Upper bound on the L2 -> SM traffic of one launch = look-ups x 32 B; the kept ncu capture gives the
        # sectors actually requested (l1tex__t_sectors_pipe_lsu_mem_global_op_ld).  Roof: the L2 slice throughput cap of
        # the microarchitecture notes (~6300 B/clk full chip, measured on B300; x the SM clock of this run).
        lookups = int(st[:, capi.ST_NDIST].sum()) * args.pq_m
        clk_mhz = (clocks or {}).get("sm_mhz") or 1965.0
        l2_peak = 6300.0 * clk_mhz * 1e6 / 1e9
        rec = None
        try:
            rec = json.load(open(os.path.join(ROOT, "profiles", "r02_ncu_traffic.json"))).get(wkey)
        except Exception:
            rec = None
        sect_ratio = (rec or {}).get("l1_global_ld_sectors_per_lookup")
        upper = lookups * 32.0
        roofline["l2_gather"] = {"bound": "l2 sector gather (SDC table)", "lookups_per_launch": lookups,
                                 "upper_bound_bytes": upper,
                                 "measured_sectors_per_lookup": sect_ratio,
                                 "achieved": (upper * (sect_ratio or 1.0)) / (kernel_ms / 1000.0) / 1e9, "unit": "GB/s",
                                 "peak": l2_peak, "peak_source": "B300_MICROARCH.md LTS cap 6300 B/clk x %.0f MHz (not measured on this box)" % clk_mhz,
                                 "frac": (upper * (sect_ratio or 1.0)) / (kernel_ms / 1000.0) / 1e9 / l2_peak}

    # ---- cpu baseline on a bounded sample (rank 0, N=1 only) + parity against the reference itself ----
    cpu_baseline = None
    parity = None
    if args.gpus == 1 and not args.no_cpu_baseline:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import reflib
        qn = h_q.numpy()
        threads = best_cpu_threads(folder, qn, args.k, args.maxcheck, each=quantized)
        probe, _, _ = cpu_search_leg(folder, qn, args.k, args.maxcheck, threads, min(args.nq, 512), each=quantized)
        sample = args.cpu_sample or int(max(512, min(args.nq, probe["value"] * 5.0)))
        cpu_baseline, cpu_ids, cpu_d = cpu_search_leg(folder, qn, args.k, args.maxcheck, threads, sample, repeats=3,
                                                      each=quantized)
        cpu_baseline.pop("seconds", None)
        cpu_baseline["host"] = host_info()
        cpu_baseline["threads_probed"] = sorted({os.cpu_count() or 1, max(1, (os.cpu_count() or 1) // 2)})
        same_ids = (cpu_ids == res_ids[:sample]).all(axis=1)
        same_bits = (cpu_d.view(np.int32) == res_d[:sample].view(np.int32)).all(axis=1)
        parity = {"queries_compared": sample, "identical_id_lists": int(same_ids.sum()),
                  "identical_distance_bits": int((same_ids & same_bits).sum())}
        # the reference's own WorkSpace counters (m_iNumberOfCheckedLeaves, NGQueue / SPTQueue sizes at exit), read
        # per query through the reference's work-space factory, against the kernel's counters
        if reflib.have_ref() and not quantized:
            nst = min(sample, 64)
            ridx = reflib.RefIndex.load(folder)
            ridx.set_param("MaxCheck", args.maxcheck)
            ridx.enable_stats()
            ok = 0
            for i in range(nst):
                _, _, rs = ridx.search_one_stats(qn[i], args.k)
                dev_row = st[i]
                ok += int(rs[0] == dev_row[capi.ST_CHECKED] and rs[2] == dev_row[capi.ST_NG_LEFT]
                          and rs[3] == dev_row[capi.ST_SPT_LEFT])
            parity["counter_queries"] = nst
            parity["identical_counters"] = ok
            parity["counters"] = "m_iNumberOfCheckedLeaves, NGQueue.size(), SPTQueue.size() at exit (WorkSpace.h:303-308)"

    line_config = dict(config)
    line_config["index_builder"] = ("reference (oracle/_ref VectorIndex::BuildIndex on the host cores)" if args.builder == "reference"
                                    else "tools/gpu_index_builder.py (set-up utility; same files go to both arms)")
    line = {"metric": "queries_per_second", "value": value, "unit": "queries/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True,
            "scaling": "weak", "vs_baseline": None, "dtype": "f32" if not quantized else "u8 codes, f32 SDC sums", "data": "synthetic",
            "config": line_config, "recall_at_10": recall, "clocks": clocks,
            "e2e": {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": args.nq * args.dim * h_q.element_size(),
                    "d2h_bytes_per_step": args.nq * args.k * 8, "host_buffers": "pinned",
                    "pageable_value": e2e_pageable},
            "gpu_launches": int(launches), "roofline": roofline, "cpu_baseline": cpu_baseline,
            "parity_vs_reference": parity}
    if pipelined is not None:
        line["pipelined"] = pipelined
    idx.close()
    return line


def shard_leg(args, rank, local_rank, world, dev, dist, config):
    """BASELINE config 5's form: vector-partition shards, one NCCL all-gather, merge on the GPU; parity against the
    reference searched shard by shard."""
    import copy
    import numpy as np
    import torch
    from sptag_b200 import B200Index, capi, sharded
    from tools import gpu_index_builder as B

    sargs = copy.copy(args)
    sargs.n = args.shard_n if args.mode == "auto" else args.n
    sargs.algo, sargs.quantizer, sargs.raw_type = "bkt", "none", "float"
    # shards of this size get the reference's own recipe for the initial graph (partition trees, 20 s) instead of the
    # 3-minute brute-force kNN: parity is about the same files on both sides, not about graph quality
    sargs.tpt_above = min(args.tpt_above, 1000000)
    files = build_in_memory(sargs, rank, dev)   # rank r builds and keeps shard r (no disk: 8 x 8 GB)
    id_offset = rank * sargs.n
    t0 = time.time()
    idx = B200Index.create(algo=capi.ALGO_BKT, value_type=files.value_type, metric=files.metric, vectors=files.vectors,
                           graph=files.graph, tree_starts=files.tree_starts, tree_nodes=files.nodes, device=local_rank,
                           id_offset=id_offset)
    idx.set_param("MaxCheck", args.maxcheck)
    for kv in args.param:
        nm, v = kv.split("=", 1)
        idx.set_param(nm, v)
    log("shard %d: %d x %d uploaded in %.1fs" % (rank, sargs.n, sargs.dim, time.time() - t0))

    d_q = gen_data(sargs, args.nq, args.seed + 7, dev).contiguous()   # the SAME batch on every rank
    h_q = torch.empty((args.nq, args.dim), dtype=torch.float32, pin_memory=True)
    h_q.copy_(d_q)
    d_ids = torch.empty((args.nq, args.k), dtype=torch.int32, device=dev)
    d_dists = torch.empty((args.nq, args.k), dtype=torch.float32, device=dev)
    d_stats = torch.zeros((args.nq, capi.STATS_PER_QUERY), dtype=torch.int32, device=dev)
    m_ids = torch.empty_like(d_ids)
    m_d = torch.empty_like(d_dists)
    stream = torch.cuda.current_stream().cuda_stream
    stats_on = [False]
    marks = []

    def local_search(q, k):
        idx.search_device(q.data_ptr(), args.nq, k, d_ids.data_ptr(), d_dists.data_ptr(),
                          d_stats.data_ptr() if stats_on[0] else 0, stream)
        return d_ids, d_dists

    def merge(g_ids, g_d, k):
        capi.merge_topk(local_rank, g_ids.data_ptr(), g_d.data_ptr(), world, args.nq, k, m_ids.data_ptr(), m_d.data_ptr(), stream)
        return m_ids, m_d

    def mark():
        if marks is not None and len(marks) < 4096:
            e = torch.cuda.Event(enable_timing=True)
            e.record()
            marks.append(e)

    ss = sharded.ShardedSearch(dist, local_search, merge, world, on_exchange_start=mark, on_exchange_end=mark)

    def sync_all():
        torch.cuda.synchronize()
        dist.barrier()
        torch.cuda.synchronize()

    stats_on[0] = True
    ss.search(d_q, args.k)
    stats_on[0] = False
    torch.cuda.synchronize()
    st = d_stats.cpu().numpy().astype(np.int64)
    alg_bytes = int((st[:, capi.ST_NDIST] * sargs.dim * 4 + st[:, capi.ST_NEXPAND] * files.degree * 4 + st[:, capi.ST_NTREE] * 12).sum())
    res_ids = m_ids.cpu().numpy()
    res_d = m_d.cpu().numpy()

    sampler = ClockSampler(local_rank)
    if rank == 0 and not args.no_clocks:
        sampler.start()
        time.sleep(0.3)
    for _ in range(args.warmup):
        ss.search(d_q, args.k)
    sync_all()
    del marks[:]
    launches0 = capi.launch_count()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    tm0 = time.time()
    ev0.record()
    for _ in range(args.steps):
        ss.search(d_q, args.k)
    ev1.record()
    sync_all()
    tm1 = time.time()
    launches = capi.launch_count() - launches0
    if rank == 0 and args.dump_outputs and args.mode == "shard":
        dump_outputs(args.dump_outputs, m_ids.cpu().numpy(), m_d.cpu().numpy())
    ms_total = ev0.elapsed_time(ev1)
    exch_ms = sum(marks[2 * i].elapsed_time(marks[2 * i + 1]) for i in range(len(marks) // 2)) / max(1, len(marks) // 2)
    t = torch.tensor([ms_total, exch_ms], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    ms_step = float(t[0].item()) / args.steps
    exch_ms = float(t[1].item())
    value = args.nq / (ms_step / 1000.0)

    # end to end: host queries in, merged host results out, every step
    h_ids = torch.empty((args.nq, args.k), dtype=torch.int32, pin_memory=True)
    h_d = torch.empty((args.nq, args.k), dtype=torch.float32, pin_memory=True)

    def step_e2e():
        d_q.copy_(h_q, non_blocking=True)
        ss.search(d_q, args.k)
        h_ids.copy_(m_ids, non_blocking=True)
        h_d.copy_(m_d, non_blocking=True)
        torch.cuda.synchronize()

    for _ in range(args.warmup):
        step_e2e()
    sync_all()
    t0 = time.perf_counter()
    for _ in range(args.steps):
        step_e2e()
    sec = time.perf_counter() - t0
    t = torch.tensor([sec], dtype=torch.float64, device=dev)
    dist.all_reduce(t, op=dist.ReduceOp.MAX)
    e2e_value = args.nq * args.steps / float(t.item())
    clocks = None
    if rank == 0:
        sampler.stop()
        clocks = sampler.summary(tm0, tm1)

    kms = []
    for _ in range(3):
        local_search(d_q, args.k)
        kms.append(idx.last_kernel_ms())
    kernel_ms = float(np.mean(kms))

    # ---- parity against the REFERENCE searched shard by shard (AggregatorService.cpp:215-412 analogue) ----
    parity = {"error": None}
    S = max(1, min(args.nq, args.shard_parity_sample))
    ref_ids = torch.full((S, args.k), -1, dtype=torch.int32, device=dev)
    ref_d = torch.zeros((S, args.k), dtype=torch.float32, device=dev)
    ref_sec = 0.0
    ref_ok = 1
    try:
        sys.path.insert(0, os.path.join(ROOT, "tests"))
        import reflib
        if not reflib.have_ref():
            raise RuntimeError("oracle/_ref is not built")
        ini = B.ini_text(sargs.metric, files.degree)
        ridx = reflib.RefIndex.load_memory(ini, files.vectors, files.graph, files.nodes, files.tree_starts)
        ridx.set_param("MaxCheck", args.maxcheck)
        threads = max(1, (os.cpu_count() or 1) // world)
        r_ids, r_d, ref_sec = ridx.search(h_q.numpy()[:S], args.k, threads=threads)
        r_ids = np.where(r_ids >= 0, r_ids + id_offset, r_ids).astype(np.int32)
        ref_ids.copy_(torch.from_numpy(r_ids))
        ref_d.copy_(torch.from_numpy(r_d))
        del ridx
    except Exception as e:  # parity must never take the timed numbers down with it
        ref_ok = 0
        parity["error"] = "rank %d: %s" % (rank, str(e)[:200])
    okt = torch.tensor([ref_ok], dtype=torch.int32, device=dev)
    dist.all_reduce(okt, op=dist.ReduceOp.MIN)
    g_ref_ids = torch.empty((world * S, args.k), dtype=torch.int32, device=dev)
    g_ref_d = torch.empty((world * S, args.k), dtype=torch.float32, device=dev)
    dist.all_gather_into_tensor(g_ref_ids, ref_ids)
    dist.all_gather_into_tensor(g_ref_d, ref_d)
    # the device-side per-shard lists of the same queries (before the merge), for a per-shard comparison as well
    ss.search(d_q, args.k)
    torch.cuda.synchronize()
    g_dev_ids, g_dev_d = ss.gathered()
    out = None
    if rank == 0:
        if int(okt.item()) == 1:
            gi = g_ref_ids.view(world, S, args.k).cpu().numpy()
            gd = g_ref_d.view(world, S, args.k).cpu().numpy()
            e_ids, e_d = sharded.merge_topk_host(gi, gd, args.k)     # host merge by (Dist, VID), QueryResultSet.h:17-26
            same_ids = (e_ids == res_ids[:S]).all(axis=1)
            same_bits = (e_d.view(np.int32) == res_d[:S].view(np.int32)).all(axis=1)
            di = g_dev_ids[:, :S].cpu().numpy()
            dd = g_dev_d[:, :S].cpu().numpy()
            per_shard = ((di == gi).all(axis=2) & (dd.view(np.int32) == gd.view(np.int32)).all(axis=2)).sum(axis=1)
            parity = {"queries_compared": S, "identical_id_lists": int(same_ids.sum()),
                      "identical_distance_bits": int((same_ids & same_bits).sum()),
                      "per_shard_identical_lists": [int(v) for v in per_shard],
                      "ids_from_other_shards": int((res_ids[:S] // sargs.n != 0).sum()),
                      "method": "each rank ran the unmodified reference (oracle/_ref, VectorIndex::LoadIndex from memory blobs + "
                                "SearchIndex(batch)) on ITS shard; the %d lists per query were merged on the host by (Dist, VID) "
                                "and compared with the device all-gather + merge_topk_kernel result" % world,
                      "reference_seconds_rank0": ref_sec}
        peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
        peak = float(json.load(open(peaks_path))["hbm_gbs"]) if os.path.exists(peaks_path) else 6650.0
        achieved = alg_bytes / (kernel_ms / 1000.0) / 1e9
        out = {"parallelism": "shard x%d" % world, "vectors_per_gpu": sargs.n, "corpus_vectors": sargs.n * world,
               "workload": "SPTAG-BKT, %d x %dx%d float32 %s shards, batch %d queries, k=%d, MaxCheck=%d" % (
                   world, sargs.n, sargs.dim, sargs.metric.lower(), args.nq, args.k, args.maxcheck),
               "value": value, "unit": "queries/s over the whole %d-vector corpus" % (sargs.n * world),
               "ms_per_step": ms_step, "search_kernel_ms": kernel_ms, "exchange_merge_ms": exch_ms,
               "exchange_bytes_per_rank": args.nq * args.k * 8,
               "limiter": "the per-shard search (%.1f ms); the exchange is 2 all-gathers of %d KB per rank + one merge kernel "
                          "(%.2f ms): launch/collective latency, not NVLink bandwidth" % (kernel_ms, args.nq * args.k * 4 // 1024, exch_ms),
               "e2e": {"value": e2e_value, "unit": "queries/s", "h2d_bytes_per_step": args.nq * args.dim * 4,
                       "d2h_bytes_per_step": args.nq * args.k * 8},
               "gpu_launches": int(launches), "collective": "NCCL all_gather_into_tensor x2 per step",
               "comm_nranks_seen": world,
               "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                            "traffic": None, "kernel": "search_kernel<%d,%s,BKT>" % (sargs.dim if sargs.dim in (128, 768) else 0, sargs.metric),
                            "kernel_ms": kernel_ms, "algorithmic_bytes_per_launch": alg_bytes, "scope": "rank 0's shard"},
               "parity_vs_reference": parity, "clocks": clocks}
    idx.close()
    return out


if __name__ == "__main__":
    sys.exit(main())
