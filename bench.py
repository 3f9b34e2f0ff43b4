#!/usr/bin/env python
"""bench.py -- Mk-mers/s of the hot path (extract + count + index) on synthetic 150 bp reads, k=55.

One "step" = one pass of the hot path over one batch of synthetic reads:
    reads (2-bit packed)  ->  canonical (k+1)-mers  ->  XXH3 bucket partition  ->  per-bucket sort/unique/count
                           ->  boomphf-compatible MPHF over the distinct (k+1)-mers
i.e. what KMerDiskCounter::Count + KMerIndexBuilder::BuildIndex do in the reference
(kmer_index_builder.hpp:306-332,448-498). k-mers = N_reads x (L - K + 1) forward windows, K = k+1 = 56 (SURVEY 8d).

  value : whole-job throughput with the packed reads already resident in HBM when the timed region starts
  e2e   : same metric through the C ABI with HOST buffers: pinned-host -> device copy of the reads, the step, and the
          device -> host read of the result (bucket sizes + serialized KMerIndex) inside the timed region
  --impl reference : the UNMODIFIED reference (oracle/_ref/ref_probe bench mode) on the host cores, bounded sample

Timing: CUDA events on the stream the library runs on (it is handed torch's current stream), barrier + synchronize on
both sides, max over ranks. Inputs (>= 0.4 GB) and intermediates (tens of GB) are far larger than the 126 MB L2.
"""
import argparse
import json
import os
import subprocess
import sys
import tempfile
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

K_GRAPH = 55
K = K_GRAPH + 1
READ_LEN = 150
# --dump-outputs without --buckets: the bucket count decides which bucket every record lands in, so it must not follow the CPU count
# (10 x host threads) for two runs of the same command to be comparable output for output; 1280 = 10 x 128 threads
DUMP_BUCKETS = 1280


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--reads", type=int, default=int(os.environ.get("SGPU_BENCH_READS", 100_000_000)), help="reads per GPU")
    ap.add_argument("--buckets", type=int, default=0, help="0 = 10 x host threads, as the reference's graph path (construction.cpp:242); "
                                                            "with --dump-outputs, 0 = %d whatever the host" % DUMP_BUCKETS)
    ap.add_argument("--cpu-sample-reads", type=int, default=0, help="reads per reference-arm step; 0 = as many as fit the time budget (calibrated on a 1 M-read run)")
    ap.add_argument("--check-reads", type=int, default=2_000_000, help="N>1: reads per rank of the distributed-vs-single-GPU checksum check (0 = skip)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last timed step returned (bucket sizes, device checksums, a fixed seeded sample "
                         "of the counted records and of the serialized KMerIndex) as DIR/<name>.npy in float64/float32. The files depend "
                         "on --reads and --buckets only (and --gpus), not on the host's CPU count")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    return args


DUMP_BLOCKS, DUMP_BLOCK = 512, 1024            # records sampled by --dump-outputs: 512 blocks of 1024 consecutive records
DUMP_INDEX_HEAD, DUMP_INDEX_BLOCKS, DUMP_INDEX_BLOCK = 1 << 16, 256, 4096      # serialized KMerIndex bytes sampled


def _halves(a):
    """u64 values as their (low, high) 32-bit halves in float64, which holds them exactly"""
    import numpy as np
    a = np.asarray(a, np.uint64)
    return np.stack([a & np.uint64(0xFFFFFFFF), a >> np.uint64(32)], axis=-1).astype(np.float64)


def dump_outputs(out_dir, st, idx, suffix=""):
    """what a caller of the timed step receives -- the counted (k+1)-mer set (KMerDiskStorage) and its KMerIndex -- as .npy files of at
    most ~30 MB in all: the full bucket sizes and the device checksums over every record, and for a fixed seeded sample of record
    blocks the records, their multiplicities and their MPHF slots; the serialized index as its size and a seeded sample of its bytes"""
    import numpy as np
    os.makedirs(out_dir, exist_ok=True)
    rng = np.random.default_rng(12345)
    n = st.total_kmers()
    blk = min(DUMP_BLOCK, n)
    starts = np.unique((rng.random(DUMP_BLOCKS) * (n - blk + 1)).astype(np.int64)) if n else np.zeros(0, np.int64)
    keys = np.concatenate([st.kmers(int(s), blk) for s in starts]) if n else np.zeros((0, st.nw), np.uint64)
    counts = np.concatenate([st.counts(int(s), blk) for s in starts]) if n else np.zeros(0, np.uint32)
    ser = np.empty(idx.serialized_size(), np.uint8)
    idx.serialize_into(ser.ctypes.data, ser.size)
    pos = np.unique((rng.random(DUMP_INDEX_BLOCKS) * max(1, ser.size - DUMP_INDEX_BLOCK)).astype(np.int64))
    ser_sample = np.concatenate([ser[:DUMP_INDEX_HEAD]] + [ser[p:p + DUMP_INDEX_BLOCK] for p in pos])
    arrays = {
        "summary": np.array([n, ser.size, st.num_buckets(), st.k()], np.float64),
        "bucket_sizes": st.bucket_sizes().astype(np.float64),
        "kmer_checksums": _halves(st.checksum()),
        "kmers_sample": _halves(keys).reshape(len(keys), 2 * st.nw),
        "counts_sample": counts.astype(np.float64),
        "mphf_slots_sample": idx.seq_idx(keys).astype(np.float64) if len(keys) else np.zeros(0, np.float64),
        "kmer_index_bytes_sample": ser_sample.astype(np.float32),
    }
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + suffix + ".npy"), a)


def host_threads():
    try:
        return len(os.sched_getaffinity(0))
    except Exception:
        return os.cpu_count() or 1


# ---------------------------------------------------------------------------------------------------------------------
# synthetic reads (SURVEY 8d): uniform genome, uniform start, random strand, 1% substitutions; generated on the device
# ---------------------------------------------------------------------------------------------------------------------
def gen_reads_device(torch, n_reads, genome_len, seed, device):
    g = torch.Generator(device=device)
    g.manual_seed(seed)
    genome = torch.randint(0, 4, (genome_len,), dtype=torch.uint8, device=device, generator=g)
    nwr = (READ_LEN + 31) // 32
    words = torch.zeros(n_reads * nwr + 8, dtype=torch.int64, device=device)
    shifts = (torch.arange(32, device=device, dtype=torch.int64) * 2)
    ar = torch.arange(READ_LEN, device=device)
    chunk = 1_000_000
    for s in range(0, n_reads, chunk):
        c = min(chunk, n_reads - s)
        starts = torch.randint(0, genome_len - READ_LEN + 1, (c,), device=device, generator=g)
        reads = genome[starts[:, None] + ar[None, :]]
        strand = torch.rand(c, device=device, generator=g) < 0.5
        reads = torch.where(strand[:, None], (3 - reads).flip(1), reads)
        errs = torch.rand((c, READ_LEN), device=device, generator=g) < 0.01
        sub = torch.randint(1, 4, (c, READ_LEN), dtype=torch.uint8, device=device, generator=g)
        reads = torch.where(errs, (reads + sub) & 3, reads)
        padded = torch.zeros((c, nwr * 32), dtype=torch.int64, device=device)
        padded[:, :READ_LEN] = reads.to(torch.int64)
        w = (padded.view(c, nwr, 32) << shifts).sum(dim=2)
        words[s * nwr:(s + c) * nwr] = w.reshape(-1)
        del reads, padded, w, errs, sub, strand, starts
    offs = torch.arange(n_reads, device=device, dtype=torch.int64) * nwr
    lens = torch.full((n_reads,), READ_LEN, dtype=torch.int32, device=device)
    return words, offs, lens, nwr


def unpack_to_text(words_np, nwr, n, path):
    import numpy as np
    w = words_np[: n * nwr].reshape(n, nwr).astype(np.uint64)
    sh = (np.arange(32, dtype=np.uint64) * np.uint64(2))
    codes = ((w[:, :, None] >> sh[None, None, :]) & np.uint64(3)).astype(np.uint8).reshape(n, nwr * 32)[:, :READ_LEN]
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    txt = lut[codes]
    out = np.empty((n, READ_LEN + 1), dtype=np.uint8)
    out[:, :READ_LEN] = txt
    out[:, READ_LEN] = 10
    out.tofile(path)


class ClockSampler(threading.Thread):
    def __init__(self, gpu_index):
        super().__init__(daemon=True)
        self.gpu = gpu_index
        self.samples, self.reasons, self.maxclk = [], set(), None
        self.stop_ev = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        while not self.stop_ev.is_set():
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.gpu), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip().split(",")
                self.samples.append(float(out[0])); self.maxclk = float(out[1])
                for nm, v in zip(names, out[2:]):
                    if "Active" in v and "Not" not in v:
                        self.reasons.add(nm)
            except Exception:
                pass
            self.stop_ev.wait(0.2)

    def result(self):
        s = sorted(self.samples)
        return {"sm_mhz": s[len(s) // 2] if s else None, "sm_max_mhz": self.maxclk, "reasons": sorted(self.reasons), "samples": len(s)}


# ---------------------------------------------------------------------------------------------------------------------
# reference arm: the UNMODIFIED reference (oracle/_ref/ref_probe "bench": KMerDiskCounter::Count + KMerIndexBuilder::BuildIndex on
# in-memory read streams, all host threads, B = 10 x threads as construction.cpp:242) on a bounded prefix of the workload
# ---------------------------------------------------------------------------------------------------------------------
PROBE = os.path.join(ROOT, "oracle", "_ref", "ref_probe")
FULL_READS = 100_000_000


def _fs_of(path):
    """file-system type the reference's bucket files land on (BASELINE.md 3.3 asks for tmpfs vs disk)"""
    best, fstype = "", "unknown"
    try:
        for line in open("/proc/mounts"):
            f = line.split()
            if len(f) >= 3 and os.path.abspath(path).startswith(f[1]) and len(f[1]) > len(best):
                best, fstype = f[1], f[2]
    except Exception:
        pass
    return fstype


def _host_facts(workdir):
    ram = None
    try:
        import psutil
        ram = round(psutil.virtual_memory().total / 2**30)
    except Exception:
        pass
    return {"nproc": host_threads(), "ram_gib": ram, "workdir_fs": _fs_of(workdir)}


def _probe_bench(n, B, T, reps, d):
    """reps runs of the reference on the first n reads of the CPU sample generator; returns the per-run records"""
    rf = os.path.join(d, "reads_%d.txt" % n)
    if not os.path.exists(rf):
        _cpu_sample(n).tofile(rf)
    out = subprocess.run([PROBE, "bench", rf, str(K_GRAPH), str(B), str(T), os.path.join(d, "out_%d" % n), str(reps)], capture_output=True, text=True).stdout
    os.remove(rf)
    return [json.loads(l[6:]) for l in out.splitlines() if l.startswith("BENCH ")]


def _cpu_sample(n):
    """n reads of the workload's shape (150x coverage: genome of n bases, 1 % substitutions, random strand), as a text matrix"""
    import numpy as np
    from spades_b200.packing import synthetic_reads
    out = np.empty((n, READ_LEN + 1), dtype=np.uint8)
    lut = np.frombuffer(b"ACGT", dtype=np.uint8)
    step = 1_000_000
    codes = synthetic_reads(n, READ_LEN, max(READ_LEN + 1, n), 0.01, seed=42, as_codes=True) if n <= 4 * step else None
    if codes is not None:
        out[:, :READ_LEN] = lut[codes]
    else:                                      # large samples: piecewise (same genome, bounded temporaries)
        rng = np.random.default_rng(42)
        genome = rng.integers(0, 4, size=n, dtype=np.uint8)
        for s0 in range(0, n, step):
            c = min(step, n - s0)
            starts = rng.integers(0, n - READ_LEN + 1, size=c)
            r = genome[starts[:, None] + np.arange(READ_LEN)[None, :]]
            st = rng.random(c) < 0.5
            r[st] = (3 - r[st])[:, ::-1]
            e = rng.random(r.shape) < 0.01
            r[e] = (r[e] + rng.integers(1, 4, size=int(e.sum()), dtype=np.uint8)) & 3
            out[s0:s0 + c, :READ_LEN] = lut[r]
    out[:, READ_LEN] = 10
    return out


def run_reference(args, rank, world):
    if rank != 0:
        return
    T = host_threads()
    B = args.buckets or 10 * T
    if not os.path.exists(PROBE):
        print(json.dumps({"impl": "reference", "unavailable": "oracle/_ref/ref_probe was not built (needs /root/reference at build time)"}))
        return
    reps = args.warmup + args.steps
    with tempfile.TemporaryDirectory() as d:
        facts = _host_facts(d)
        # calibration on 1 M reads (also the first point of the size scaling), then the largest prefix whose `reps` runs fit ~4 minutes
        cal = _probe_bench(1_000_000, B, T, 2, d)[-1]
        cal_rate = cal["windows"] / cal["total_s"]
        n = args.cpu_sample_reads
        if n <= 0:
            per_rep_s = max(2.0, min(30.0, 240.0 / reps))
            n = int(cal_rate * per_rep_s / (READ_LEN - K + 1))
            ram_cap = int((facts["ram_gib"] or 64) * 2**30 * 0.25 / (READ_LEN + 1 + 2 * (READ_LEN - K + 1) * 16 * 0.6))    # text + spilled runs
            n = max(1_000_000, min(n, ram_cap, FULL_READS))
            n -= n % 100_000
        recs = _probe_bench(n, B, T, reps, d)
    timed = recs[args.warmup:]
    tot = sum(r["total_s"] for r in timed)
    windows = timed[0]["windows"]
    val = windows * len(timed) / tot / 1e6
    line = {"metric": "Mk-mers/s (extract+count+index) k=55, 150 bp reads", "value": val, "unit": "Mk-mers/s", "n_gpus": args.gpus,
            "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * tot / len(timed), "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u64", "data": "synthetic", "impl": "reference",
            "config": {"workload": "synthetic %d x 150 bp reads = the first %.1f %% of the 100 M-read bench workload's shape (150x coverage, 1%% substitutions), k=55 "
                                   "(K=56 canonical (k+1)-mers), %d buckets; the largest prefix whose %d runs fit the few-minute budget" % (n, 100.0 * n / FULL_READS, B, reps),
                       "k": K_GRAPH, "reads": n, "buckets": B, "sample_fraction": n / FULL_READS, "host": facts,
                       "size_scaling": [{"reads": 1_000_000, "Mk-mers/s": cal_rate / 1e6}, {"reads": n, "Mk-mers/s": val}]},
            "cpu_baseline": {"value": val, "unit": "Mk-mers/s", "cores": T, "kind": "reference",
                             "sample": "%d reads x 150 bp, in-memory read streams, count+index region of ref_probe (unmodified SPAdes KMerDiskCounter + KMerIndexBuilder), "
                                       "bucket files on %s" % (n, facts["workdir_fs"])},
            "e2e": {"value": val, "unit": "Mk-mers/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
    print(json.dumps(line))


def cpu_baseline(args):
    T = host_threads()
    B = args.buckets or 10 * T
    if os.path.exists(PROBE):
        with tempfile.TemporaryDirectory() as d:
            facts = _host_facts(d)
            r1 = _probe_bench(1_000_000, B, T, 2, d)[-1]
            rate1 = r1["windows"] / r1["total_s"]
            # second, larger point (~10 s of CPU work) so that the size dependence of the CPU path is visible
            n2 = int(min(10_000_000, max(2_000_000, rate1 * 10.0 / (READ_LEN - K + 1))))
            n2 -= n2 % 100_000
            r2 = _probe_bench(n2, B, T, 1, d)[-1]
            rate2 = r2["windows"] / r2["total_s"]
        return {"value": rate2 / 1e6, "unit": "Mk-mers/s", "cores": T, "kind": "reference",
                "sample": "%d reads x 150 bp (%.0f %% of the workload), unmodified SPAdes KMerDiskCounter::Count + KMerIndexBuilder::BuildIndex via oracle/_ref/ref_probe, "
                          "%d buckets, in-memory streams, bucket files on %s" % (n2, 100.0 * n2 / FULL_READS, B, facts["workdir_fs"]),
                "sample_fraction": n2 / FULL_READS, "host": facts,
                "size_scaling": [{"reads": 1_000_000, "Mk-mers/s": rate1 / 1e6}, {"reads": n2, "Mk-mers/s": rate2 / 1e6}]}
    # the plain-C oracle port (single thread)
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import oracle as O
    from spades_b200.packing import pack_fixed, synthetic_reads
    n = 100_000
    codes = synthetic_reads(n, READ_LEN, max(READ_LEN + 1, n), 0.01, seed=42, as_codes=True)
    words, offs, lens = pack_fixed(codes)
    t0 = time.time()
    ks = O.count(words, offs, lens, K, B, 0)
    O.Mphf(ks)
    dt = time.time() - t0
    return {"value": n * (READ_LEN - K + 1) / dt / 1e6, "unit": "Mk-mers/s", "cores": 1, "kind": "port", "sample": "%d reads x 150 bp, oracle/spades_oracle.c count+mphf" % n}


# ---------------------------------------------------------------------------------------------------------------------
def multi_gpu_check(torch, dist, ctx, dcounter, B, n_check, rank, world, dev):
    """N>1, before anything is timed: the distributed count of `world` shards against ONE GPU counting their union -- bucket sizes
    equal, and the order-independent device checksums of (records, multiplicities) add / xor up. Raises on a mismatch."""
    import numpy as np
    from spades_b200.kmer_index import DeBruijnReadKMerSplitter, KMerDiskCounter
    glen = max(READ_LEN + 1, n_check)
    w, o, l, nwr = gen_reads_device(torch, n_check, glen, 1000 + rank, dev)
    ctx.adopt_device_reads(w.data_ptr(), n_check * nwr, o.data_ptr(), l.data_ptr(), n_check)
    st = dcounter.Count(B)
    mine = st.checksum()
    bsz = torch.from_numpy(st.bucket_sizes().copy()).to(dev)
    st.free()
    dist.all_reduce(bsz, op=dist.ReduceOp.SUM)
    t = torch.tensor([mine[0], mine[1] - (1 << 64) if mine[1] >= (1 << 63) else mine[1], mine[3]], dtype=torch.int64, device=dev)   # sums wrap mod 2^64
    dist.all_reduce(t, op=dist.ReduceOp.SUM)
    xs = [None] * world
    dist.all_gather_object(xs, mine[2])
    ok, detail = True, None
    if rank == 0:
        x = 0
        for v in xs:
            x ^= v
        got = [int(t[0].item()), int(t[1].item()) & ((1 << 64) - 1), x, int(t[2].item()) & ((1 << 64) - 1)]
        parts = [gen_reads_device(torch, n_check, glen, 1000 + r, dev) for r in range(world)]
        uw = torch.cat([p_[0][: n_check * nwr] for p_ in parts] + [torch.zeros(8, dtype=torch.int64, device=dev)])
        uo = torch.cat([p_[1] + r * n_check * nwr for r, p_ in enumerate(parts)])
        ul = torch.cat([p_[2] for p_ in parts])
        del parts
        ctx.adopt_device_reads(uw.data_ptr(), world * n_check * nwr, uo.data_ptr(), ul.data_ptr(), world * n_check)
        ref = KMerDiskCounter(ctx, DeBruijnReadKMerSplitter(K)).Count(B)
        want = ref.checksum()
        want_bsz = ref.bucket_sizes()
        ref.free()
        torch.cuda.synchronize()
        ok = got == want and np.array_equal(want_bsz, bsz.cpu().numpy())
        detail = {"reads_per_rank": n_check, "distinct": want[0], "checksums_distributed": got, "checksums_single_gpu": want, "ok": ok}
        del uw, uo, ul
    flag = torch.tensor([1 if ok else 0], device=dev)
    dist.broadcast(flag, 0)
    del w, o, l
    torch.cuda.empty_cache()
    if int(flag.item()) != 1:
        raise RuntimeError("multi-GPU self check FAILED: distributed count != single-GPU count of the union: %s" % (detail,))
    return detail


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    import numpy as np
    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; this path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from spades_b200.kmer_index import Context, DeBruijnReadKMerSplitter, KMerDiskCounter, KMerIndexBuilder

    T = host_threads()
    B = args.buckets or (DUMP_BUCKETS if args.dump_outputs else 10 * T)
    n_reads = args.reads
    genome_len = max(READ_LEN + 1, n_reads)          # 150x coverage like config 3 (100 M reads over 100 Mbp)
    words, offs, lens, nwr = gen_reads_device(torch, n_reads, genome_len, 42 + rank, dev)
    torch.cuda.synchronize()
    torch.cuda.empty_cache()                         # the generator's temporaries go back to the driver before the library reserves its arena
    stream = torch.cuda.current_stream()
    ctx = Context(local_rank, stream=stream.cuda_stream)
    nwords = n_reads * nwr

    dcounter = None
    check = None
    if world > 1:
        from spades_b200.distributed import DistributedKMerCounter
        dcounter = DistributedKMerCounter(ctx, K)
        if args.check_reads > 0:
            check = multi_gpu_check(torch, dist, ctx, dcounter, B, min(args.check_reads, n_reads), rank, world, dev)

    def count(ctx_):
        # N>1: buckets are owned by ranks; one pull kernel per rank does the exchange + merge over NVLink peer memory
        if world > 1:
            return dcounter.Count(B)
        return KMerDiskCounter(ctx_, DeBruijnReadKMerSplitter(K)).Count(B)

    def step_resident():
        ctx.adopt_device_reads(words.data_ptr(), nwords, offs.data_ptr(), lens.data_ptr(), n_reads)
        st = count(ctx)
        idx = KMerIndexBuilder(ctx).BuildIndex(st)
        return st, idx

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- value: reads resident in HBM
    for _ in range(args.warmup):
        st, idx = step_resident(); idx.free(); st.free()
    phases = {k: 0.0 for k in ("extract_count_ms", "extract_scatter_ms", "exchange_ms", "refine_ms", "local_sort_ms", "compact_ms", "mphf_ms")}
    l0 = ctx.times()["launches"]
    sampler = ClockSampler(local_rank); sampler.start()
    barrier()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    distinct = instances = passes = 0
    last = None
    for i in range(args.steps):
        st, idx = step_resident()
        t = ctx.times()
        for kname in phases:
            phases[kname] += t[kname]
        distinct, instances, passes = st.total_kmers(), t["instances"], t["passes"]
        if args.dump_outputs and i == args.steps - 1:
            last = (st, idx)           # read back after the timed region
        else:
            idx.free(); st.free()
    e1.record(stream)
    barrier()
    ms = e0.elapsed_time(e1)
    sampler.stop_ev.set(); sampler.join()
    launches = ctx.times()["launches"] - l0
    peak = ctx.times()["peak_bytes"]
    if last is not None:
        dump_outputs(args.dump_outputs, *last, suffix="" if world == 1 else "_rank%d" % rank)
        last[1].free(); last[0].free()
    tms = torch.tensor([ms], device=dev)
    if world > 1:
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
    ms = float(tms.item())
    windows_per_step = n_reads * (READ_LEN - K + 1) * world
    value = windows_per_step * args.steps / (ms / 1e3) / 1e6

    # ---- e2e: host buffers in, host result out
    h_words = words[:nwords].cpu().pin_memory(); h_offs = offs.cpu().pin_memory(); h_lens = lens.cpu().pin_memory()
    d2h = 0
    h_index = None     # pinned host buffer the serialized KMerIndex lands in
    h_bsz = np.zeros(B, np.int64)

    def step_e2e():
        nonlocal d2h, h_index
        ctx.upload_reads(h_words.data_ptr(), nwords, h_offs.data_ptr(), h_lens.data_ptr(), n_reads)
        st = count(ctx)
        idx = KMerIndexBuilder(ctx).BuildIndex(st)
        need = idx.serialized_size()
        if h_index is None or h_index.numel() < need:
            h_index = torch.empty(int(need * 1.05) + 4096, dtype=torch.uint8).pin_memory()
        nser = idx.serialize_into(h_index.data_ptr(), h_index.numel())
        h_bsz[:] = st.bucket_sizes()
        d2h = nser + h_bsz.nbytes
        idx.free(); st.free()

    step_e2e()
    barrier()
    e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e2.record(stream)
    for _ in range(args.steps):
        step_e2e()
    e3.record(stream)
    barrier()
    ems = torch.tensor([e2.elapsed_time(e3)], device=dev)
    if world > 1:
        dist.all_reduce(ems, op=dist.ReduceOp.MAX)
    e2e_value = windows_per_step * args.steps / (float(ems.item()) / 1e3) / 1e6
    h2d = h_words.numel() * 8 + h_offs.numel() * 8 + h_lens.numel() * 4

    # ---- e2e_storage (N = 1): the same, plus what KMerDiskCounter::Count hands the reference's next stage -- every bucket's records
    # (the KMerDiskStorage contents, here 16 bytes x distinct) -- copied to pinned host memory. One warm-up step + the timed steps.
    e2e_storage = None
    if world == 1:
        try:
            import psutil
            need = int(distinct) * 16 + (1 << 20)
            if psutil.virtual_memory().available > need + (16 << 30):
                h_keys = torch.empty(need // 8, dtype=torch.int64, pin_memory=True)

                def step_storage():
                    ctx.upload_reads(h_words.data_ptr(), nwords, h_offs.data_ptr(), h_lens.data_ptr(), n_reads)
                    st = count(ctx)
                    idx = KMerIndexBuilder(ctx).BuildIndex(st)
                    nser = idx.serialize_into(h_index.data_ptr(), h_index.numel())
                    h_bsz[:] = st.bucket_sizes()
                    nk = st.total_kmers()
                    assert nk * 2 <= h_keys.numel()
                    st.download_keys_into(h_keys.data_ptr(), nk)
                    idx.free(); st.free()
                    return nser + h_bsz.nbytes + nk * 16
                step_storage()
                torch.cuda.synchronize()
                e4, e5 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                nst = args.steps
                e4.record(stream)
                for _ in range(nst):
                    d2h_s = step_storage()
                e5.record(stream)
                torch.cuda.synchronize()
                e2e_storage = {"value": windows_per_step * nst / (e4.elapsed_time(e5) / 1e3) / 1e6, "unit": "Mk-mers/s", "steps": nst,
                               "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h_s),
                               "what": "e2e + every bucket's sorted records (the KMerDiskStorage contents the reference's next stage reads) copied to pinned host memory"}
                del h_keys
            else:
                e2e_storage = {"skipped": "not enough free host memory to pin the k-mer set"}
        except Exception as ex:      # measurement extra: never fails the bench line
            e2e_storage = {"skipped": "%s: %s" % (type(ex).__name__, ex)}

    if rank == 0:
        W = 16
        steps = args.steps
        peaks = {}
        try:
            peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
        except Exception:
            pass
        peak_gbs, peak_src = (peaks["hbm_gbs"], "measured (MEASURED_PEAKS.json)") if "hbm_gbs" in peaks else (6650.0, "fallback (B200_PROFILING.md)")
        per_step = {k2: v / steps for k2, v in phases.items()}
        # algorithmic bytes per step of each kernel family (DESIGN.md 3): I = instances, D = distinct; SURVEY 8(d) counts the packed reads
        # ONCE for the partition kernel however many bucket-group passes re-read them
        I, D = instances, distinct
        alg = {
            "extract_scatter_ms": n_reads * nwr * 8 + I * W,                  # packed reads in, records out
            "extract_count_ms": n_reads * nwr * 8,                           # packed reads in
            "refine_ms": 2 * I * W,                                          # one read + one write of every record
            "local_sort_ms": I * W + D * (W + 4),                            # records in, distinct records + counts out
            "compact_ms": 2 * D * (W + 4),
            "exchange_ms": 2 * I * W,
        }
        dom = max(alg, key=lambda k2: per_step[k2])
        achieved = alg[dom] / (per_step[dom] / 1e3) / 1e9 if per_step[dom] > 0 else 0.0
        kernel_names = {"extract_scatter_ms": "levelA_scatter_roll_k (radix partition)", "extract_count_ms": "levelA_count_roll_k", "refine_ms": "refine_k (gather + MSD split)",
                        "local_sort_ms": "local_sort3_k", "compact_ms": "compact_k", "exchange_ms": "dist_pull_k (NVLink exchange+merge)"}
        launches_per_step = {"extract_scatter_ms": int(max(1, passes)), "refine_ms": None, "local_sort_ms": int(max(1, passes)), "compact_ms": int(max(1, passes)),
                             "extract_count_ms": 1, "exchange_ms": int(max(1, passes))}
        whole_alg = n_reads * nwr * 8 + 2 * I * W + 2 * D * W + D * (4 + 5.8 / 8)      # SURVEY 8(d): extract + count + index
        line = {
            "metric": "Mk-mers/s (extract+count+index) k=55, 150 bp reads", "value": value, "unit": "Mk-mers/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "u64",
            "data": "synthetic",
            "config": {"workload": "synthetic %d x 150 bp reads per GPU (uniform genome %d bp, 1%% substitutions, random strand), k=55: canonical (k+1)=56-mers, "
                                   "%d XXH3 buckets, sort/unique/count + boomphf MPHF (extract+count+index)" % (n_reads, genome_len, B),
                       "k": K_GRAPH, "reads_per_gpu": n_reads, "buckets": B, "distinct_kpomers": int(distinct), "instances": int(instances), "passes": int(passes),
                       "parallelism": ("1 GPU" if world == 1 else "%d GPUs: reads sharded, buckets owned by ranks, one pull kernel per rank exchanges + merges the partitions over NVLink peer memory" % world),
                       "l2": "inputs (%.1f GB) and intermediates larger than L2; no flush needed" % (nwords * 8 / 1e9), "peak_hbm_gb": peak / 1e9,
                       "multi_gpu_check": check},
            "clocks": sampler.result(), "gpu_launches": int(launches),
            "e2e": {"value": e2e_value, "unit": "Mk-mers/s", "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h),
                    "what": "pinned host reads -> sgpu_reads_upload -> sgpu_count -> sgpu_mphf_build -> sgpu_mphf_serialize + bucket sizes to host; sorted (k+1)-mers stay in HBM for the graph phases"},
            "e2e_storage": e2e_storage,
            "phases_ms_per_step": per_step,
            "roofline": {"bound": "hbm", "kernel": kernel_names[dom], "achieved": achieved, "peak": peak_gbs, "unit": "GB/s", "frac": achieved / peak_gbs,
                         "peak_source": peak_src,
                         # per-launch DRAM bytes (dram__bytes_read.sum + dram__bytes_write.sum) come from the committed ncu --set full capture of the
                         # SAME workload (profiles/, see NCU_TRAFFIC below); null when no capture of this kernel at this size exists
                         "traffic": (NCU_DRAM_PER_ALGORITHMIC_BYTE[dom][0] * alg[dom] / max(1, launches_per_step.get(dom) or 1)
                                     if dom in NCU_DRAM_PER_ALGORITHMIC_BYTE else None),
                         "traffic_source": NCU_DRAM_PER_ALGORITHMIC_BYTE[dom][1] if dom in NCU_DRAM_PER_ALGORITHMIC_BYTE else None,
                         "launches_per_step": launches_per_step.get(dom),
                         "algorithmic_bytes_per_step": int(alg[dom]),
                         "whole_step": {"algorithmic_bytes": int(whole_alg), "achieved": whole_alg / (ms / steps / 1e3) / 1e9, "frac": whole_alg / (ms / steps / 1e3) / 1e9 / peak_gbs},
                         "all": {kernel_names[k2]: (alg[k2] / (per_step[k2] / 1e3) / 1e9 if per_step[k2] > 0 else None) for k2 in alg}},
        }
        if not args.no_cpu_baseline:
            line["cpu_baseline"] = cpu_baseline(args)
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


# dram__bytes_read.sum + dram__bytes_write.sum of a kernel family per ALGORITHMIC byte, from the `ncu --set full` captures committed under
# profiles/ (ncu cannot profile the 100 M-read / 5-pass configuration itself: its kernel replay backs the 150 GB of device memory up to the
# host and returns no counters for the kernels that write the largest buffers; the captures are of the same kernels on smaller launches).
# roofline.traffic = this ratio x the algorithmic bytes of one launch of the timed run.
NCU_DRAM_PER_ALGORITHMIC_BYTE = {
    "local_sort_ms": (1.04, "profiles/r02g_ncu_full_100M_arena100_noids.csv: 11.3 GB read + 5.8 GB written for a launch of 0.70 G records"),
    "refine_ms": (0.80, "profiles/r02k_ncu_full_10M_warp_tiles.csv: 16.2 GB read + 8.1 GB written for 0.95 G records read twice and written once "
                        "(the second read of a piece is served by L2)"),
    "extract_count_ms": (7.0, "profiles/r02l_ncu_full_10M_levelA.csv: 0.65 GB read + 1.98 GB written (the 2-byte partition ids) for 0.375 GB of packed reads"),
}


if __name__ == "__main__":
    try:
        main()
    except BaseException as e:      # the failing rank's reason must be the LAST thing it prints (torchrun's summary hides earlier output)
        if isinstance(e, SystemExit) and e.code in (0, None):
            raise
        import traceback
        traceback.print_exc()
        msg = "bench.py rank %s FAILED: %s: %s" % (os.environ.get("RANK", "0"), type(e).__name__, e)
        sys.stdout.flush()
        print(msg, file=sys.stderr, flush=True)
        print(json.dumps({"error": msg}), flush=True)
        os._exit(1)
