#!/usr/bin/env python3
"""Benchmark of the `metagraph align` hot path on B200 (BASELINE.json metric: aligned reads/sec on
synthetic 150 bp reads).

Workloads (BENCH_CONFIG or --config):
  c2 (default, BASELINE.json configs[1]): 1 M synthetic 150 bp DNA reads per GPU (seed 42 + rank, 50 %
     reverse-complemented, error-free) against a k=31 BOSS graph of a 100 Mbp uniform random genome (seed 32,
     ~100 M nodes), exact-match seeder (--align-min-seed-length 31 --align-max-seed-length 31), CLI-default
     scoring. Weak scaling: every rank aligns its own 1 M reads.
  c3 (BASELINE.json configs[2], the north-star target): 10 M reads IN TOTAL with 5 % per-base errors (80 %
     substitutions, 10 % insertions, 10 % deletions) against the graph of a 1 Gbp genome (~1 B nodes), CLI-default
     seeder (MEM + sub-k seeds) with --align-min-exact-match 0. Strong scaling: 10 M / N reads per rank.
Both: seed complexity filter off (sdust is not vendored in the reference tree), index replicated per GPU (built
once on rank 0, BOSS arrays broadcast over NCCL), reads sharded, no collective on the data path.

One step = one pass of the hot path (query preparation + seeding + seed-and-extend) over the read batch of this
rank. `value` counts device time only (inputs resident in HBM; CUDA events on the launching stream around the
kernels, reported by the C-ABI in mgb_stats_t). `e2e` is the same metric through the reference-facing call
mgb_align_batch() with pinned HOST buffers: H2D of the reads, all kernels, D2H of the packed results and host
unpacking, and at N > 1 the gather of every rank's result set on rank 0 (export block -> NCCL send -> import),
all inside the timed region; rank 0 then reads the score of every alignment of the whole job.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402

K = 31
READ_LEN = 150
CPU_SUFFIX_INDEX = 12      # BOSS::index_suffix_ranges length of the CPU arm's graph (reference default)
CHUNK = 250_000            # c3 reads are generated in chunks so that a shard does not depend on the world size


def env_int(name, default):
    return int(os.environ.get(name, default))


def make_genome(G):
    rng = np.random.default_rng(32)
    return np.frombuffer(b"ACGT", dtype=np.uint8)[rng.integers(0, 4, G, dtype=np.uint8)]


def make_reads(genome, n, seed):
    """error-free reads, 50 % reverse-complemented; returns (uint8 buffer, uint64 offsets)"""
    rng = np.random.default_rng(seed)
    starts = rng.integers(0, len(genome) - READ_LEN, n)
    idx = starts[:, None] + np.arange(READ_LEN)[None, :]
    reads = genome[idx]
    comp = np.zeros(256, np.uint8)
    comp[list(b"ACGT")] = list(b"TGCA")
    rc = rng.random(n) < 0.5
    reads[rc] = comp[reads[rc]][:, ::-1]
    return np.ascontiguousarray(reads.reshape(-1)), np.arange(n + 1, dtype=np.uint64) * READ_LEN


def make_error_reads(genome, chunk_lo, chunk_hi, rate=0.05, chunk=CHUNK):
    """c3 reads of chunks [chunk_lo, chunk_hi): 150 bp windows, per output base `rate` errors split 80 / 10 / 10 into
    substitution (uniform replacement base) / insertion (a random base that consumes no genome) / deletion (one
    genome base skipped), then 50 % reverse-complemented. Chunk c is seeded with 4242 + c."""
    comp = np.zeros(256, np.uint8)
    comp[list(b"ACGT")] = list(b"TGCA")
    acgt = np.frombuffer(b"ACGT", dtype=np.uint8)
    parts = []
    for c in range(chunk_lo, chunk_hi):
        rng = np.random.default_rng(4242 + c)
        n = chunk
        starts = rng.integers(0, len(genome) - READ_LEN - 64, n)
        u = rng.random((n, READ_LEN))
        ins = u < rate * 0.1
        dele = (u >= rate * 0.1) & (u < rate * 0.2)
        sub = (u >= rate * 0.2) & (u < rate)
        # source offset of output base j: one per base that is not an insertion, plus the deletions up to j
        consumed = np.cumsum(~ins, axis=1, dtype=np.int16) - 1 + np.cumsum(dele, axis=1, dtype=np.int16)
        consumed = np.maximum(consumed, 0)
        reads = genome[starts[:, None] + consumed]
        rnd = acgt[rng.integers(0, 4, (n, READ_LEN), dtype=np.uint8)]
        repl = ins | sub
        reads[repl] = rnd[repl]
        rc = rng.random(n) < 0.5
        reads[rc] = comp[reads[rc]][:, ::-1]
        parts.append(np.ascontiguousarray(reads.reshape(-1)))
    buf = np.concatenate(parts) if parts else np.zeros(0, np.uint8)
    n_tot = (chunk_hi - chunk_lo) * chunk
    return buf, np.arange(n_tot + 1, dtype=np.uint64) * READ_LEN


class ClockSampler:
    """nvidia-smi clocks / throttle reasons sampled during the timed region (B200_PROFILING.md)."""

    def __init__(self, gpu_index=0):
        self.rows = []
        self.proc = None
        self.gpu_index = gpu_index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.gpu_index),
                 "--query-gpu=clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
                 "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
                 "clocks_event_reasons.sw_power_cap",
                 "--format=csv,noheader,nounits", "-lms", "100"],
                stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append(line.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=2)
        except Exception:
            pass
        sm, smax, reasons = [], [], set()
        for r in self.rows:
            f = [x.strip() for x in r.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); smax.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None,
                "sm_max_mhz": max(smax) if smax else None, "reasons": sorted(reasons), "samples": len(sm)}


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return json.load(open(p))["hbm_gbs"], "measured"
    return 6650.0, "fallback"


_ORACLE_CACHE = {}


def cpu_reference(boss, reads_buf, offsets, cfg, target_seconds, threads, n_max):
    """Times the CPU restatement of the reference algorithm (oracle/) on a bounded sample. The thread
    count is probed (all hardware threads, half, a quarter): on two-socket hosts the restatement, like
    any pointer-chasing code over one shared graph, peaks below the full thread count.
    Returns (reads/s, sample size, seconds, threads used)."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle_lib as O
    if "g" not in _ORACLE_CACHE:
        # the reference builds its graphs with a suffix-range index of length 12 (`metagraph build
        # --index-ranges 12`, cli/config/config.cpp:24-25; SURVEY 8d): the CPU arm runs with it
        _ORACLE_CACHE["g"] = O.OracleGraph(K, arrays=(boss.W, boss.last, boss.F), suffix_index=CPU_SUFFIX_INDEX)
    g = _ORACLE_CACHE["g"]
    def reads_of(a, b):
        return [bytes(reads_buf[int(offsets[i]):int(offsets[i + 1])]) for i in range(a, b)]
    if "threads" not in _ORACLE_CACHE:
        best = (0.0, threads)
        for th in sorted({max(1, threads // 4), max(1, threads // 2), threads}):
            probe = min(n_max, max(th * 200, 2000))
            rs = reads_of(0, probe)
            t = time.time(); g.align_tsv(cfg, rs, threads=th); dt = time.time() - t
            if probe / dt > best[0]:
                best = (probe / dt, th)
        _ORACLE_CACHE["threads"] = best[1]
        _ORACLE_CACHE["rate"] = best[0]
    th = _ORACLE_CACHE["threads"]
    n = int(min(n_max, max(2000, _ORACLE_CACHE["rate"] * target_seconds)))
    rs = reads_of(0, n)
    t = time.time(); g.align_tsv(cfg, rs, threads=th); dt = time.time() - t
    return n / dt, n, dt, th


def cpu_single_thread(reads_buf, offsets, cfg, n=1500):
    """single-thread rate of the same CPU arm (BASELINE.md asks for the 1-thread row); cpu_reference() first"""
    g = _ORACLE_CACHE["g"]
    n = min(n, len(offsets) - 1)
    rs = [bytes(reads_buf[int(offsets[i]):int(offsets[i + 1])]) for i in range(n)]
    t = time.time(); g.align_tsv(cfg, rs, threads=1); dt = time.time() - t
    return n / dt


def workload(name, world):
    """the benchmark workload `name` for `world` ranks"""
    from metagraph_b200.config import cli_defaults
    if name == "c2":
        G = env_int("BENCH_GENOME", 100_000_000)
        n_rank = env_int("BENCH_READS", 1_000_000)
        cfg = cli_defaults(K, min_seed_length=K, max_seed_length=K, result_nodes=env_int("BENCH_RESULT_NODES", 1),
                           no_exact_path_shortcut=bool(env_int("BENCH_NO_SHORTCUT", 0)))
        text = ("%d synthetic %d bp DNA reads/GPU (50%% rc, error-free) vs k=%d BOSS graph of a %d bp random "
                "genome, exact-match seeder, CLI-default scoring" % (n_rank, READ_LEN, K, G))
        return dict(name="c2 (BASELINE configs[1])", text=text, G=G, n_rank=n_rank, n_total=n_rank * world, cfg=cfg,
                    scaling="weak", seeder="exact (min=max seed length = k)", error_rate=0.0, chunk=0)
    G = env_int("BENCH_GENOME", 1_000_000_000)
    n_total = env_int("BENCH_READS", 10_000_000)
    chunk = min(CHUNK, max(1, n_total // (8 * 5)))        # 40 chunks at least: 1, 2, 4 and 8 ranks take whole chunks
    n_total = max(chunk * world, n_total // (chunk * world) * (chunk * world))
    cfg = cli_defaults(K, min_exact_match=0.0, result_nodes=env_int("BENCH_RESULT_NODES", 1),
                       no_exact_path_shortcut=bool(env_int("BENCH_NO_SHORTCUT", 0)))
    text = ("%d synthetic %d bp DNA reads in total (50%% rc, 5%% errors: 80/10/10 substitution/insertion/deletion) vs "
            "k=%d BOSS graph of a %d bp random genome, CLI-default seeder (MEM + sub-k seeds), min_exact_match 0, "
            "CLI-default scoring" % (n_total, READ_LEN, K, G))
    return dict(name="c3 (BASELINE configs[2])", text=text, G=G, n_rank=n_total // world, n_total=n_total, cfg=cfg,
                scaling="strong", seeder="CLI default: SuffixSeeder<UniMEMSeeder>, min_seed_length 19", error_rate=0.05,
                chunk=chunk)


def alignment_records(L, res, fields):
    """the alignments of a result set as a numpy structured array over the library's memory (no copy), restricted
    to `fields` of mgb_alignment_t; pointer fields read as uint64 addresses"""
    from metagraph_b200._lib import mgb_alignment_t
    types = dict(mgb_alignment_t._fields_)
    dt = np.dtype({"names": list(fields),
                   "formats": [np.uint64 if issubclass(types[f], ctypes._Pointer) else np.dtype(types[f]) for f in fields],
                   "offsets": [getattr(mgb_alignment_t, f).offset for f in fields],
                   "itemsize": ctypes.sizeof(mgb_alignment_t)})
    n_aln = int(L.mgb_results_num_alignments(res))
    if not n_aln:
        return np.zeros(0, dt)
    alns = L.mgb_results_alignments(res)
    raw = (ctypes.c_char * (n_aln * dt.itemsize)).from_address(ctypes.addressof(alns.contents))
    return np.frombuffer(raw, dtype=dt, count=n_aln)


OUTPUT_FIELDS = ("read_index", "orientation", "score", "offset", "query_begin", "query_len", "num_nodes",
                 "sequence_len", "num_cigar_ops")


def output_arrays(L, res, max_rows=1 << 20, n_detail=4096):
    """What a caller of mgb_align_batch receives, as float arrays for --dump-outputs: every scalar field of every
    alignment (of a seeded sample of `max_rows` alignments when there are more), and for a seeded sample of
    `n_detail` of those rows the CIGAR operations, the aligned sequence and the node path, flattened, each with an
    offsets array. Values are exact in the float type used (float32 below 2**24, float64 for node ids). Node paths
    are left out when the result set carries none (MGB_NODES_NONE), and no array is empty."""
    rec = alignment_records(L, res, OUTPUT_FIELDS + ("nodes", "sequence", "cigar"))
    rng = np.random.default_rng(0)
    rows = np.arange(len(rec)) if len(rec) <= max_rows else np.sort(rng.choice(len(rec), max_rows, replace=False))
    out = {"num_alignments": np.array([len(rec)], np.float64), "rows": rows.astype(np.float64)}
    for f in OUTPUT_FIELDS:
        out[f] = rec[f][rows].astype(np.float64 if f == "read_index" else np.float32)
    detail = rows[np.sort(rng.choice(len(rows), min(n_detail, len(rows)), replace=False))]
    cigar, seq, nodes = [], [], []
    for r in detail:
        a = rec[r]
        cigar.append(np.frombuffer(ctypes.string_at(int(a["cigar"]), 4 * int(a["num_cigar_ops"])), np.uint32))
        seq.append(np.frombuffer(ctypes.string_at(int(a["sequence"]), int(a["sequence_len"])), np.uint8))
        nodes.append(np.frombuffer(ctypes.string_at(int(a["nodes"]), 8 * int(a["num_nodes"])), np.uint64)
                     if a["nodes"] else np.zeros(0, np.uint64))
    def flat(parts, dtype):
        return np.concatenate(parts) if parts else np.zeros(0, dtype)
    ops = flat(cigar, np.uint32)   # packed (length << 3 | operation)
    out.update(detail_rows=detail.astype(np.float64), cigar_length=(ops >> 3).astype(np.float32),
               cigar_op=(ops & 7).astype(np.float32), sequence=flat(seq, np.uint8).astype(np.float32))
    variable = [("cigar", cigar), ("sequence", seq)]
    if any(len(p) for p in nodes):
        out["nodes"] = flat(nodes, np.uint64).astype(np.float64)
        variable.append(("nodes", nodes))
    for name, parts in variable:
        out[name + "_offsets"] = np.cumsum([0] + [len(p) for p in parts]).astype(np.float64)
    return {name: a for name, a in out.items() if a.size}


def rank_reads(wl, genome, rank, world):
    if wl["error_rate"] == 0.0:
        return make_reads(genome, wl["n_rank"], 42 + rank)
    per = wl["n_rank"] // wl["chunk"]
    return make_error_reads(genome, rank * per, (rank + 1) * per, wl["error_rate"], wl["chunk"])


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--config", default=os.environ.get("BENCH_CONFIG", "c2"), choices=["c2", "c3"])
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the alignments of the last timed step (rank 0's reads) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.dump_outputs and args.impl != "b200":
        ap.error("--dump-outputs writes the results of the b200 arm")

    rank = env_int("RANK", 0)
    world = env_int("WORLD_SIZE", 1)
    local_rank = env_int("LOCAL_RANK", 0)
    host_threads = os.cpu_count() or 1

    from metagraph_b200.aligner import B200Aligner, BOSSTable, DBGSuccinctIndex
    wl = workload(args.config, world)
    G, N, cfg = wl["G"], wl["n_rank"], wl["cfg"]
    config = {"workload": wl["text"], "name": wl["name"], "reads_per_gpu": N, "reads_total": wl["n_total"],
              "read_len": READ_LEN, "k": K, "genome_bp": G, "seeder": wl["seeder"],
              "result_nodes": "none (TSV consumer: cli/align.cpp:254-307 prints no node ids)" if cfg.result_nodes
                              else "u64 node path per alignment",
              "exact_path_shortcut": "off" if cfg.no_exact_path_shortcut else "on (reads whose k-mers all match: the "
                                     "extension is provably {L}= along them and is not run; same results, DESIGN.md)",
              "cpu_arm_suffix_index": CPU_SUFFIX_INDEX,
              "l2_policy": "inputs larger than L2 (index + node arrays + per-group arenas >> 126 MB)",
              "parallelism": "reads sharded x%d, index replicated" % world}

    # ---------------------------------------------------------------- reference arm (CPU) ----
    if args.impl == "reference":
        if rank != 0:
            return
        genome = make_genome(G)
        boss = BOSSTable.from_sequences(K, None, packed=(genome, np.array([0, G], dtype=np.uint64)),
                                        threads=min(host_threads, 32))   # torchrun pins OMP_NUM_THREADS=1
        if wl["error_rate"] == 0.0:
            buf, offsets = make_reads(genome, min(N, 400_000), 42)
        else:
            buf, offsets = make_error_reads(genome, 0, 1, wl["error_rate"], wl["chunk"])
        per_step = []
        sample_n = 0
        for s in range(args.warmup + args.steps):
            rate, n, dt, used_threads = cpu_reference(boss, buf, offsets, cfg, 8.0, host_threads, len(offsets) - 1)
            sample_n = n
            if s >= args.warmup:
                per_step.append((rate, dt))
        value = float(np.mean([r for r, _ in per_step]))
        line = {"impl": "reference", "metric": "aligned reads/sec (150 bp synthetic)", "value": value,
                "unit": "reads/s", "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
                "ms_per_step": float(np.mean([d for _, d in per_step]) * 1e3), "higher_is_better": True,
                "scaling": wl["scaling"], "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": config,
                "cpu_baseline": {"value": value, "unit": "reads/s", "cores": used_threads, "kind": "port",
                                 "single_thread": cpu_single_thread(buf, offsets, cfg),
                                 "sample": "%d reads of the same workload per step (CPU restatement of the "
                                           "reference algorithm, oracle/, graph with suffix-range index %d, best of "
                                           "%d/%d/%d threads = %d)"
                                           % (sample_n, CPU_SUFFIX_INDEX, max(1, host_threads // 4),
                                              max(1, host_threads // 2), host_threads, used_threads)},
                "e2e": {"value": value, "unit": "reads/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    # ---------------------------------------------------------------- B200 arm -----------------
    import torch
    import torch.distributed as dist
    if world > 1:
        torch.cuda.set_device(local_rank)
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    dev = torch.device("cuda", local_rank)
    num_sms = torch.cuda.get_device_properties(dev).multi_processor_count

    # index build on rank 0 (host, untimed), broadcast of the BOSS arrays over NCCL
    genome = make_genome(G)
    if rank == 0:
        t0 = time.time()
        boss = BOSSTable.from_sequences(K, None, packed=(genome, np.array([0, G], dtype=np.uint64)),
                                        threads=min(host_threads, 32))   # torchrun pins OMP_NUM_THREADS=1
        build_s = time.time() - t0
        meta = torch.tensor([len(boss.W)] + [int(x) for x in boss.F], dtype=torch.int64, device=dev)
    else:
        boss, build_s = None, 0.0
        meta = torch.zeros(6, dtype=torch.int64, device=dev)
    if world > 1:
        dist.broadcast(meta, 0)
        n1 = int(meta[0].item())
        Wt = torch.from_numpy(boss.W).to(dev) if rank == 0 else torch.empty(n1, dtype=torch.uint8, device=dev)
        Lt = torch.from_numpy(boss.last).to(dev) if rank == 0 else torch.empty(n1, dtype=torch.uint8, device=dev)
        dist.broadcast(Wt, 0)
        dist.broadcast(Lt, 0)
        if rank != 0:
            boss = BOSSTable(K, Wt.cpu().numpy(), Lt.cpu().numpy(), meta[1:6].cpu().numpy().astype(np.uint64))
        del Wt, Lt
    t0 = time.time()
    index = DBGSuccinctIndex(boss, device=local_rank)
    index_s = time.time() - t0
    aligner = B200Aligner(index, cfg)
    # torchrun pins OMP_NUM_THREADS=1: give this rank its share of the host cores for result unpacking
    aligner._L.mgb_set_host_threads(max(1, min(32, host_threads // max(world, 1))))

    buf_np, off_np = rank_reads(wl, genome, rank, world)
    del genome
    buf_pin = torch.empty(len(buf_np), dtype=torch.uint8, pin_memory=True)
    buf_pin.numpy()[:] = buf_np
    off_pin = torch.empty(len(off_np), dtype=torch.int64, pin_memory=True)
    off_pin.numpy()[:] = off_np.astype(np.int64)
    buf = buf_pin.numpy()
    offsets = off_pin.numpy().view(np.uint64)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()

    from metagraph_b200.sharding import ResultGather
    L = aligner._L
    gatherer = ResultGather(L, dev) if world > 1 else None
    gather_ms = []

    def score_sum(res):
        view = alignment_records(L, res, ("score",))
        return len(view), int(np.add.reduce(view["score"], dtype=np.int64))

    def step(gather, outputs=None):
        """one pass over this rank's reads; with `gather` every rank's result set goes to rank 0, which reads the
        score of every alignment of the whole job (checksum); otherwise each rank reads its own. `outputs` (a dict)
        receives output_arrays() of the result set."""
        res = aligner.align_batch_raw(buf, offsets)
        st = aligner.stats_of(res)
        if outputs is not None:
            outputs.update(output_arrays(L, res))
        if gather and gatherer is not None:
            tg = time.time()
            parts = gatherer.gather(res, rank * N)
            n_aln, chk = 0, 0
            if parts is not None:
                for _, h in parts:
                    a, c = score_sum(h)
                    n_aln += a; chk += c
                    L.mgb_results_free(h)
            gather_ms.append((time.time() - tg) * 1e3)
        else:
            n_aln, chk = score_sum(res)
        aligner.free_raw(res)
        return st, n_aln, chk

    # Region A -- `value`: the batch as ONE piece, so that the device timers around the kernels (CUDA events
    # on the launching stream, mgb_stats_t) do not overlap; inputs are in HBM when they start.
    # Region B -- `e2e`: the default call (a big batch is split into pieces on two streams so downloads and
    # unpacking overlap the kernels) plus, at N > 1, the gather of all result sets on rank 0; wall clock around
    # K whole steps from pinned host buffers.
    aligner.set_pipeline_pieces(1)
    for _ in range(args.warmup):
        step(False)
    sampler = ClockSampler(local_rank)
    barrier()
    if rank == 0:
        sampler.start()
    # the output copy of the last step is host work after its kernels: the device timers do not see it
    outputs = {} if args.dump_outputs and rank == 0 else None
    stats = [step(False, outputs if s == args.steps - 1 else None) for s in range(args.steps)]
    barrier()
    # the same region with the exact-path shortcut switched off (every extension runs): what the roofline / GCUPS
    # lines describe, and the device-timed rate without the shortcut
    stats_full = stats
    if not cfg.no_exact_path_shortcut:
        import dataclasses
        aligner_full = B200Aligner(index, dataclasses.replace(cfg, no_exact_path_shortcut=True))
        def step_full():
            res = aligner_full.align_batch_raw(buf, offsets)
            st = aligner_full.stats_of(res)
            n_aln, chk = score_sum(res)
            aligner_full.free_raw(res)
            return st, n_aln, chk
        step_full()
        barrier()
        stats_full = [step_full() for _ in range(args.steps)]
        barrier()
        assert [c for _, _, c in stats_full] == [c for _, _, c in stats], "the shortcut changed the results"
    aligner.set_pipeline_pieces(0)
    for _ in range(args.warmup):
        step(True)
    del gather_ms[:]
    barrier()
    t0 = time.time()
    stats_e2e = [step(True) for _ in range(args.steps)]
    barrier()
    wall = time.time() - t0
    clocks = sampler.stop() if rank == 0 else None

    dev_ms = sum(s["seed_kernel_ms"] + s["align_kernel_ms"] for s, _, _ in stats)
    # kernel times and DP counts of the full run (shortcut off) feed the roofline lines
    seed_ms = sum(s["seed_kernel_ms"] for s, _, _ in stats_full) / args.steps
    align_ms = sum(s["align_kernel_ms"] for s, _, _ in stats_full) / args.steps
    dev_ms_full = sum(s["seed_kernel_ms"] + s["align_kernel_ms"] for s, _, _ in stats_full)
    t = torch.tensor([dev_ms, wall * 1e3, float(np.mean(gather_ms)) if gather_ms else 0.0, dev_ms_full],
                     dtype=torch.float64, device=dev)
    tot = torch.tensor([sum(c for _, _, c in stats), sum(a for _, a, _ in stats)], dtype=torch.int64, device=dev)
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dist.all_reduce(tot, op=dist.ReduceOp.SUM)
    dev_ms_max, wall_ms_max, gather_ms_max, dev_ms_full_max = t.tolist()
    if rank == 0:
        # what rank 0 gathered in region B must be what the ranks computed in region A
        assert sum(c for _, _, c in stats_e2e) == int(tot[0].item()), "gathered results differ from the per-rank results"
        assert sum(a for _, a, _ in stats_e2e) == int(tot[1].item())

    if rank == 0:
        total_reads = N * world
        value = total_reads * args.steps / (dev_ms_max / 1e3)
        e2e = total_reads * args.steps / (wall_ms_max / 1e3)
        st = stats_full[-1][0]
        st_e2e = stats_e2e[-1][0]
        peak, peak_kind = measured_peaks()
        # dominant kernel and its algorithmic bytes per launch (DESIGN.md "Roofline")
        cols, cells = st["dp_columns"], st["dp_cells"]
        # seeding (SURVEY 8d): warm k-mer 96 B, cold k-mer 2 336 B. Error-free read: 2 x (1 cold + 119 warm); with e
        # error runs per read a strand restarts e times and keeps the k-mers no error touches (the survey's
        # 2 x [(1 + e) cold + hits warm] form)
        e_runs = wl["error_rate"] * READ_LEN
        hits = (READ_LEN - K + 1) * (1.0 - wl["error_rate"]) ** K
        seed_bytes_read = 2.0 * ((1.0 + e_runs) * 2336 + max(hits - 1.0 - e_runs, 0.0) * 96) if e_runs else 27520.0
        if align_ms >= seed_ms:
            kname, kms = "k_align", align_ms
            alg_bytes = cols * 128 + cells * 12
        else:
            kname, kms = "k_seed", seed_ms
            alg_bytes = N * seed_bytes_read
        achieved = alg_bytes / (kms / 1e3) / 1e9
        # DRAM traffic of the dominant kernel per launch: one ncu capture of this very workload and build
        # (profiles/r2_traffic.json, made by scripts/profile_bench.py), scaled per read; null otherwise
        traffic = None
        try:
            tr = json.load(open(os.path.join(ROOT, "profiles", "r2_traffic.json")))
            w = tr["workload"]
            if (w["read_len"], w["genome_bp"], w["k"], w["config"]) == (150, G, K, args.config):
                traffic = int((tr[kname]["dram_bytes_read"] + tr[kname]["dram_bytes_write"]) / w["reads"] * N)
        except (OSError, KeyError, ValueError):
            pass
        seed_alg = N * seed_bytes_read
        seed_gbs = seed_alg / (seed_ms / 1e3) / 1e9
        # int-pipe view of the extension (SURVEY 8d): 12 int32 ops per DP cell
        sm_clock = (clocks or {}).get("sm_mhz") or 1965.0
        gcups = cells / (align_ms / 1e3) / 1e9
        gcups_peak = num_sms * 128 * sm_clock * 1e6 / 12 / 1e9
        line = {
            "metric": "aligned reads/sec (150 bp synthetic)", "value": value, "unit": "reads/s",
            "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": dev_ms_max / args.steps, "higher_is_better": True, "scaling": wl["scaling"],
            "vs_baseline": None, "dtype": "int32", "data": "synthetic", "config": config,
            "clocks": clocks,
            "e2e": {"value": e2e, "unit": "reads/s", "h2d_bytes_per_step": int(st_e2e["h2d_bytes"]),
                    "d2h_bytes_per_step": int(st_e2e["d2h_bytes"]), "ms_per_step": wall_ms_max / args.steps,
                    "gather_ms_per_step": gather_ms_max if world > 1 else 0.0,
                    "gather": "every rank's result set exported, sent to rank 0 over NCCL and imported there, inside "
                              "the timed region" if world > 1 else "single rank: nothing to gather"},
            "gpu_launches": int(sum(s["kernel_launches"] for s, _, _ in stats + stats_e2e)),
            "roofline": {"bound": "hbm", "kernel": kname, "achieved": achieved, "peak": peak, "unit": "GB/s",
                         "frac": achieved / peak, "traffic": traffic, "peak_kind": peak_kind,
                         "algorithmic_bytes_per_launch": int(alg_bytes), "kernel_ms": kms},
            "kernels_ms_per_step": {"prepare+seed": seed_ms, "align": align_ms,
                                    "align_with_shortcut": sum(s["align_kernel_ms"] for s, _, _ in stats) / args.steps},
            "without_exact_path_shortcut": {"value": total_reads * args.steps / (dev_ms_full_max / 1e3), "unit": "reads/s",
                                            "ms_per_step": dev_ms_full_max / args.steps},
            # seeding against the HBM roofline (SURVEY 8d model of algorithmic bytes per read, both strands)
            "seeding": {"bound": "hbm", "kernel": "k_prepare+k_premap+k_seed(+k_subk)", "achieved": seed_gbs, "peak": peak,
                        "unit": "GB/s", "frac": seed_gbs / peak, "algorithmic_bytes_per_launch": int(seed_alg),
                        "algorithmic_bytes_per_read": seed_bytes_read},
            "extension": {"gcups": gcups, "gcups_int32_peak": gcups_peak, "frac": gcups / gcups_peak,
                          "dp_cells_per_step": int(cells), "dp_columns_per_step": int(cols), "sms": num_sms},
            "alignments_per_step": int(stats_e2e[-1][1]), "reads_retried_per_step": int(st["num_reads_retried"]),
            "index_build_s": build_s, "index_upload_s": index_s,
            "index_device_bytes": int(index.device_bytes),
        }
        if world == 1:
            # CPU baseline: oracle (port of the reference algorithm) on all host cores, bounded sample
            rate, n, dt, used_threads = cpu_reference(boss, buf_np, off_np, cfg, 10.0, host_threads, min(N, 400_000))
            line["cpu_baseline"] = {"value": rate, "unit": "reads/s", "cores": used_threads, "kind": "port",
                                    "single_thread": cpu_single_thread(buf_np, off_np, cfg),
                                    "sample": "first %d reads of the same workload, %.1f s wall, CPU restatement "
                                              "of the reference algorithm (oracle/), graph with suffix-range index "
                                              "%d, best of %d/%d/%d threads = %d"
                                              % (n, dt, CPU_SUFFIX_INDEX, max(1, host_threads // 4),
                                                 max(1, host_threads // 2), host_threads, used_threads)}
        print(json.dumps(line))
        if outputs is not None:
            os.makedirs(args.dump_outputs, exist_ok=True)
            for name, a in outputs.items():
                np.save(os.path.join(args.dump_outputs, name + ".npy"), a)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
