#!/usr/bin/env python
"""bench.py — headline benchmark of the B200 LSM compaction / read engine (BASELINE.json metric:
compaction merged-GB/s + scan keys/s, next to the CPU path).

One "step" = one L0->L1 compaction of one hash partition (BASELINE.json configs[1]: 4 sorted runs x
2.5 M records, 16 B hashkey / 32 B sortkey / 256 B value, synthetic, fixed seed and `now`), with the
KeyWithTTLCompactionFilter fused.  Each rank (GPU) owns its own partition(s): weak scaling, no
collective on the data path (hash partitions are independent, SURVEY.md §8e).

  value    = whole-job merged GB/s, sum(user key + value bytes of all input records) / time, inputs already
             resident in HBM, timed with CUDA events on the engine's stream, max over ranks.
  e2e      = the same metric through the C ABI starting from HOST buffers: pipelined upload of the 4 runs
             (pinned host memory -> HBM, device index + Bloom build) + compaction + result struct back.
  roofline = the merge kernels (k_walk + k_emit, back to back on one stream): algorithmic bytes (B_in + B_out,
             key+value only) / their CUDA-event duration, against the measured HBM copy bandwidth in
             MEASURED_PEAKS.json; `traffic` is the DRAM byte count of an ncu capture of the same launch
             (profiles/traffic_r02.json), labelled with its source, or null.
  cpu_baseline = the oracle's block-level CPU compaction (heap merging iterator -> filter -> block builder,
             all host threads) on the SAME full workload (independent of the core count); its statistics are
             compared with the device's (`parity_checked`).  It is the oracle port, not RocksDB itself (RocksDB
             is neither in the reference tree nor in this image).  `--impl reference` times the same CPU path.
  reads    = get / prefix-scan legs on the resident partition (device and end-to-end numbers use the same
             statistic: the mean over the repetitions).
  sharded_reads = BASELINE.json configs[2]: a 256-partition table, partition p served by rank p % N, YCSB-C
             zipfian get + multi_get(hash_key) requests routed by crc64 like a client; per rank two multi-partition launches.
  sweep    = BASELINE.json configs[3] (N=1): manual-compact style L0..L4 merges with 30 % expired records at run
             sizes 8..256 MB, bottommost forced, roofline fraction per size.
  ycsb_a   = BASELINE.json configs[4] at small scale (N=1): 50/50 put+get through the rrdb surface.

--dump-outputs DIR writes, after the timed steps, what the last timed step returned (see dump_compaction, dump_reads) as
DIR/<name>.npy, so that two builds can be compared output for output; the inputs are seeded and identical from run to run.

Usage: python bench.py [--gpus N] [--steps K] [--warmup W] [--impl ours|reference] [--dump-outputs DIR]
"""
from __future__ import annotations

import argparse
import ctypes as C
import hashlib
import json
import os
import subprocess
import sys
import threading
import time
from concurrent.futures import ThreadPoolExecutor

import numpy as np

sys.dont_write_bytecode = True  # the benchmark leaves the source tree as it found it (it may be read-only)
ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))

NOW = 300_000_000
RUNS = 4
HK, SK, VAL = 16, 32, 256
STAT_FIELDS = ("in_records", "out_records", "in_bytes", "out_bytes", "dropped_shadowed", "dropped_tombstone", "dropped_expired",
               "dropped_user", "dropped_stale", "ttl_rewritten")


def load_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        with open(p) as f:
            j = json.load(f)
        return float(j["hbm_gbs"]), "measured (MEASURED_PEAKS.json, torch copy)"
    return 6650.0, "fallback (B200_PROFILING.md)"


def load_traffic():
    """DRAM bytes per launch from the committed ncu captures (tools/summarize_profiles.py writes the file)"""
    p = os.path.join(ROOT, "profiles", "traffic_r02.json")
    if os.path.exists(p):
        try:
            with open(p) as f:
                return json.load(f)
        except Exception:
            return {}
    return {}


def workload_config(records_per_run: int) -> dict:
    """the config both arms report (the driver compares them field by field)"""
    return {"workload": f"single-partition L0->L1 compaction per GPU: {RUNS} SSTs x {records_per_run} keys, "
                        f"{HK}B hashkey/{SK}B sortkey/{VAL}B value (BASELINE.json configs[1])",
            "filter": "KeyWithTTLCompactionFilter on", "bottommost": True}


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region."""

    def __init__(self, index: int):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop_flag = threading.Event()

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag.is_set():
            try:
                out = subprocess.run(["nvidia-smi", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-i",
                                      str(self.index)], capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            self.stop_flag.wait(0.2)

    def summary(self):
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = max([int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()] or [0])
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows for i in range(4) if len(r) > 2 + i and r[2 + i].startswith("Active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": mx or None, "reasons": reasons,
                "samples": len(sm)}


def gen_runs(records_per_run: int, seed: int):
    from incubator_pegasus_b200 import synth
    return synth.compaction_runs(k=RUNS, n_per_run=records_per_run, hk_len=HK, sk_len=SK, user_len=VAL, now=NOW,
                                 seed=seed)


def cpu_block_runs(runs):
    """block-encode the sample for the CPU path (setup, not timed)."""
    import oracle_py as orc
    return [orc.BlockRunCPU.from_run(orc.Run.from_records(r)) for r in runs]


def cpu_compaction(bruns, threads: int):
    """oracle block-level compaction on host cores; returns (merged GB/s, seconds, stats, merged block run)."""
    import oracle_py as orc
    fp = orc.filter_params(enabled=True)
    out, st, secs = orc.compact_blocks(bruns, True, fp, NOW, threads)
    return st.in_bytes / secs / 1e9, secs, st, out


# ---------------------------------------------------------------------------------------------------------------------
# --dump-outputs: float32 / float64 arrays, under 50 MB in all whatever the read batch sizes
# ---------------------------------------------------------------------------------------------------------------------
DUMP_RECORDS = 16384     # merged records sampled: 16384 x (50 B key + 268 B value) bytes as float32 is ~21 MB
DUMP_REQUESTS = 1 << 20  # per-request arrays of the read legs (every request at the default batch sizes)


def sample_index(n: int, cap: int, seed: int) -> np.ndarray:
    """0..n-1, or a fixed seeded sorted sample of cap of them"""
    if n <= cap:
        return np.arange(n)
    return np.sort(np.random.default_rng(seed).choice(n, size=cap, replace=False))


def padded_rows(buf: np.ndarray, off: np.ndarray, pick: np.ndarray) -> np.ndarray:
    """buf[off[i]:off[i + 1]] for i in pick as float32 rows, zero-padded to the longest (the lengths are dumped beside)"""
    start, length = off[pick].astype(np.int64), (off[pick + 1] - off[pick]).astype(np.int64)
    col = np.arange(int(length.max(initial=0)))
    inside = col < length[:, None]
    return np.where(inside, buf[np.where(inside, start[:, None] + col, 0)], 0).astype(np.float32)


def gather(buf: np.ndarray, start: np.ndarray, length: np.ndarray) -> np.ndarray:
    """buf[start[i]:start[i] + length[i]] for every i, concatenated"""
    start, length = start.astype(np.int64), length.astype(np.int64)
    end = np.cumsum(length)
    total = int(end[-1]) if end.size else 0
    return buf[np.repeat(start - end + length, length) + np.arange(total)]


def digest(*arrays) -> np.ndarray:
    """SHA-256 of the arrays' bytes, as 32 float32 values 0..255: equal iff the whole output is (not just the sample)"""
    h = hashlib.sha256()
    for a in arrays:
        h.update(np.ascontiguousarray(a).view(np.uint8))
    return np.frombuffer(h.digest(), np.uint8).astype(np.float32)


def write_arrays(out_dir: str, arrays: dict) -> None:
    os.makedirs(out_dir, exist_ok=True)
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


def dump_compaction(out_dir: str, stats, merged) -> None:
    """the compaction step's statistics (STAT_FIELDS, as the oracle reports them too), a seeded sample of the merged
    records (key and value bytes, lengths, sequence numbers, types) and a digest of the whole merged run"""
    pick = sample_index(merged.n, DUMP_RECORDS, seed=0)
    write_arrays(out_dir, {
        "compaction_stats": np.array([int(getattr(stats, f)) for f in STAT_FIELDS], np.float64),
        "compaction_sample_index": pick.astype(np.float64),
        "compaction_sample_keys": padded_rows(merged.keys, merged.key_off, pick),
        "compaction_sample_key_len": (merged.key_off[pick + 1] - merged.key_off[pick]).astype(np.float32),
        "compaction_sample_values": padded_rows(merged.vals, merged.val_off, pick),
        "compaction_sample_value_len": (merged.val_off[pick + 1] - merged.val_off[pick]).astype(np.float32),
        "compaction_sample_seq": merged.seq[pick].astype(np.float64),
        "compaction_sample_type": merged.type[pick].astype(np.float32),
        "compaction_digest": digest(merged.keys, merged.key_off, merged.vals, merged.val_off, merged.seq, merged.type),
    })


def dump_reads(out_dir: str, gres, garena: np.ndarray, sb) -> None:
    """the last get batch (status, expire_ts, expired flag, value length per key; digest of the values found) and the last
    prefix-scan batch (status and record count per request; digest of the records returned)"""
    g = np.ctypeslib.as_array(gres)
    found = g["status"] == 0
    gi = sample_index(g.shape[0], DUMP_REQUESTS, seed=1)
    s = np.ctypeslib.as_array(sb.results)
    si = sample_index(s.shape[0], DUMP_REQUESTS, seed=2)
    n_kv = int(sb.kbase[-1])
    kv = sb.kvs.reshape(-1, 5)[:n_kv]
    base = np.repeat(sb.abase[:-1], np.diff(sb.kbase)).astype(np.int64)
    write_arrays(out_dir, {
        "get_status": g["status"][gi].astype(np.float32),
        "get_expire_ts": g["expire_ts"][gi].astype(np.float64),
        "get_expired": g["expired"][gi].astype(np.float32),
        "get_value_len": g["value_len"][gi].astype(np.float32),
        "get_values_digest": digest(found, g["value_len"][found], gather(garena, g["value_off"][found], g["value_len"][found])),
        "scan_status": s["status"][si].astype(np.float32),
        "scan_n_kvs": s["n_kvs"][si].astype(np.float32),
        "scan_records_digest": digest(np.diff(sb.kbase), kv[:, [1, 3]], gather(sb.arena, base + kv[:, 0], kv[:, 1]),
                                      gather(sb.arena, base + kv[:, 2], kv[:, 3])),
    })


def zipf_ids(rng, n_items: int, n: int, theta: float = 0.99):
    """YCSB zipfian(theta) over n_items, scrambled."""
    w = 1.0 / np.power(np.arange(1, n_items + 1, dtype=np.float64), theta)
    cdf = np.cumsum(w)
    cdf /= cdf[-1]
    ranks = np.searchsorted(cdf, rng.random(n))
    perm = rng.permutation(n_items)
    return perm[np.minimum(ranks, n_items - 1)]


def read_workload(records_per_run: int, n_get: int, n_scan: int, seed: int):
    """keys of the read legs: zipfian hash keys of the synthetic data set; gets pick a random sort key."""
    from incubator_pegasus_b200 import synth
    rng = np.random.default_rng(seed + 77)
    per_run_hash = (int(records_per_run * 0.9) + 63) // 64  # own hash keys of runs 1.. (synth.compaction_runs)
    n_hash = (records_per_run + 63) // 64 + (RUNS - 1) * per_run_hash
    gh = zipf_ids(rng, n_hash, n_get).astype(np.uint64)
    gs = rng.integers(0, 64, n_get).astype(np.uint64)
    get_keys = synth.make_keys(gh, gs, HK, SK, seed)
    sh = zipf_ids(rng, n_hash, n_scan).astype(np.uint64)
    scan_keys = synth.make_keys(sh, np.zeros(n_scan, np.uint64), HK, SK, seed)[:, 2:2 + HK]
    return get_keys, scan_keys


def reference_arm(args, rank: int, world: int):
    """--impl reference: the CPU path (oracle port; RocksDB itself is not in the reference tree nor this image) on the same
    full workload, all host threads."""
    if rank != 0:
        return
    threads = os.cpu_count() or 1
    n = args.records_per_run
    bruns = cpu_block_runs(gen_runs(n, 1000))
    vals = []
    for i in range(args.warmup + args.steps):
        gbs, secs, st, out = cpu_compaction(bruns, threads)
        vals.append((gbs, secs))
        if args.dump_outputs and i == args.warmup + args.steps - 1:
            dump_compaction(args.dump_outputs, st, out.decode().records())
        del out
    in_bytes = int(st.in_bytes)
    timed = vals[args.warmup:]
    ms = 1e3 * sum(s for _, s in timed) / len(timed)
    v = in_bytes / (ms / 1e3) / 1e9
    line = {
        "impl": "reference", "metric": "compaction_merged_GBps", "value": v, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": ms, "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": workload_config(n),
        "cpu_baseline": {"value": v, "unit": "GB/s", "cores": threads, "kind": "port",
                         "what": "oracle-CPU block-level compaction (a restatement of the reference's RocksDB path, not RocksDB)",
                         "sample": f"{RUNS} x {n} records ({in_bytes / 1e9:.2f} GB merged) per step: the full workload"},
        "e2e": {"value": v, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE.json configs[2]: 256 partitions, YCSB-C zipfian get + multi_get(hash_key), partition p on rank p % N
# ---------------------------------------------------------------------------------------------------------------------
def sharded_read_leg(pgs, torch, dist, eng, rank, world, args, barrier, check_cpu):
    from incubator_pegasus_b200 import sharding
    t0 = time.time()
    table = sharding.Table(partition_count=args.partitions, n_hash=args.table_hashkeys, sortkeys_per_hash=64, hk_len=HK, sk_len=SK,
                           user_len=VAL, now=NOW)
    mine = sharding.partitions_of_rank(args.partitions, rank, world)
    parts, host_runs, n_rec, n_bytes = {}, {}, 0, 0
    for p in mine:
        runs = table.partition_runs(p)
        if not runs:
            continue
        part = eng.partition(app_id=2, pidx=p)
        brs = [pgs.build_run(r) for _, r in runs]
        part.upload_many(brs, levels=[lvl for lvl, _ in runs])
        parts[p] = part
        if check_cpu:
            host_runs[p] = brs
        n_rec += sum(r.n for _, r in runs)
        n_bytes += sum(int(b.data.shape[0]) for b in brs)
    gen_s = time.time() - t0
    gh, gs, sh = table.requests(args.n_get, args.n_scan)
    g_owner, s_owner = table.pidx[gh.astype(np.int64)], table.pidx[sh.astype(np.int64)]
    from incubator_pegasus_b200 import synth
    work = []  # (kind, partition, payload)
    my_gets = my_scans = 0
    pins = []

    def pinned_alloc(n, dt):  # request and answer buffers live in pinned memory, like a server's I/O buffers
        t = torch.empty(max(1, int(n)) * np.dtype(dt).itemsize, dtype=torch.uint8).pin_memory()
        pins.append(t)
        return t.numpy().view(dt)

    def pinned_copy(a):
        out = pinned_alloc(a.size, a.dtype)
        out[:] = a.reshape(-1)
        return out
    # gets: all of this rank's partitions in ONE launch (pgs_get_batch_multi: the shape a batching front end gives the engine)
    plist = sorted(parts)
    slot_of = {p: i for i, p in enumerate(plist)}
    sel = np.nonzero(np.isin(g_owner, plist))[0]
    if sel.size:
        keys = synth.make_keys(gh[sel], gs[sel], HK, SK, table.seed)
        flat = pinned_copy(np.ascontiguousarray(keys.reshape(-1)))
        off = pinned_copy(np.arange(sel.size + 1, dtype=np.uint32) * np.uint32(keys.shape[1]))
        kslot = pinned_copy(np.array([slot_of[int(p)] for p in g_owner[sel]], np.uint32))
        cap = int(sel.size) * (VAL + 16)
        res_buf = pinned_alloc(int(sel.size) * C.sizeof(pgs.GetResult), np.uint8)
        work.append(("get", -1, (flat, off, kslot, pinned_alloc(cap, np.uint8), (pgs.GetResult * int(sel.size)).from_buffer(res_buf),
                                 g_owner[sel].copy())))
        my_gets = int(sel.size)
    # prefix scans: likewise one launch over all of this rank's partitions (pgs_range_scan_many_multi)
    sel = np.nonzero(np.isin(s_owner, plist))[0]
    if sel.size:
        sslot = np.array([slot_of[int(p)] for p in s_owner[sel]], np.uint32)
        sb = pgs.ScanBatch(None, [table.hashkeys[int(h)].tobytes() for h in sh[sel]], 80, 24576, alloc=pinned_alloc,
                           parts=[parts[q] for q in plist], req_part=sslot)
        work.append(("scan", -1, (sb, s_owner[sel].copy())))
        my_scans = int(sel.size)
    lock = threading.Lock()
    tot = {"found": 0, "returned": 0, "kernel_ms": 0.0, "calls": 0}

    verify = [True]  # the first pass counts what was found (checked against the oracle); the timed passes only serve

    def serve(item):
        kind, p, payload = item
        if kind == "get":
            flat, off, kslot, arena, res, _owners = payload
            st, res, _, _ = pgs.get_batch_multi([parts[q] for q in plist], flat, off, kslot, NOW, arena, res)
            assert st == 0, st
            ms = eng.last_kernel_ms
            found = sum(1 for i in range(off.shape[0] - 1) if res[i].status == 0) if verify[0] else 0
            with lock:
                tot["found"] += found; tot["kernel_ms"] += ms; tot["calls"] += 1
        else:
            sb = payload[0]
            st = sb.run(NOW)
            assert st == 0, st
            ms = eng.last_kernel_ms
            with lock:
                tot["returned"] += int(sb.kbase[-1]); tot["kernel_ms"] += ms; tot["calls"] += 1

    pool = ThreadPoolExecutor(max_workers=args.read_threads)
    list(pool.map(serve, work))  # warm-up pass (also the answer that is checked below)
    first = dict(tot)
    verify[0] = False
    walls = []
    for _ in range(args.steps):
        tot.update(found=0, returned=0, kernel_ms=0.0, calls=0)
        barrier()
        w0 = time.perf_counter()
        list(pool.map(serve, work))
        barrier()
        walls.append(time.perf_counter() - w0)
    pool.shutdown()
    wall = sum(walls) / len(walls)
    t = torch.tensor([wall, float(my_gets), float(tot["returned"]), float(my_scans), float(n_rec), tot["kernel_ms"], float(tot["calls"])],
                     dtype=torch.float64, device="cuda")
    tmax = t.clone()
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        dist.all_reduce(tmax, op=dist.ReduceOp.MAX)
    wall_max = float(tmax[0])
    out = {
        "workload": f"{args.partitions} partitions x 3 runs (L2 full, L1 30 %, L0 10 % newer versions), {args.table_hashkeys} hash keys x 64 sort keys; "
                    f"YCSB-C zipfian(0.99) over hash keys: {args.n_get} get(hk,sk) + {args.n_scan} multi_get(hk, all sort keys), "
                    f"routed by crc64(hash_key) % {args.partitions}; partition p on rank p % N; per rank the gets of all its partitions go through "
                    f"one pgs_get_batch_multi launch and the prefix scans through one pgs_range_scan_many_multi launch, the two calls on separate host threads",
        "scaling": "strong", "collective": "none on the data path (partitions are independent)",
        "partitions_per_rank": len(parts), "records_resident": int(t[4]),
        "get_keys_per_s": float(t[1]) / wall_max, "scan_keys_per_s": float(t[2]) / wall_max,
        "requests_per_s": (float(t[1]) + float(t[3])) / wall_max, "ms_per_pass": wall_max * 1e3,
        "statistic": "mean over repetitions of the host wall clock around the pass (barrier + synchronize both sides), max over ranks",
        "e2e": True, "kernel_ms_sum_all_ranks": float(t[5]), "calls_per_pass_all_ranks": int(t[6]),
        "load_imbalance": float(tmax[1]) * world / max(1.0, float(t[1])),
        "load_imbalance_note": "largest rank's share of the gets / the mean: zipfian keys are not spread evenly over partitions",
        "table_build_s": round(gen_s, 1),
    }
    if check_cpu:  # N=1: the oracle answers the same requests on the same block runs
        import oracle_py as orc
        threads = os.cpu_count() or 1
        c_found = c_ret = 0
        c_secs = 0.0
        for kind, p, payload in work:  # gets: the oracle answers them partition by partition
            if kind != "get":
                continue
            flat, off, _kslot, _arena, _res, owners = payload
            klen = int(off[1] - off[0])
            for q in plist:
                selq = np.nonzero(owners == q)[0]
                if not selq.size:
                    continue
                bruns = [orc.BlockRunCPU.from_blocks(b) for b in reversed(host_runs[q])]  # newest first
                sub = np.ascontiguousarray(flat.reshape(-1, klen)[selq].reshape(-1))
                f, _vb, secs = orc.get_many(bruns, sub, np.arange(selq.size + 1, dtype=np.uint32) * np.uint32(klen), NOW, threads)
                c_found += f
                c_secs += secs
        for kind, p, payload in work:
            if kind == "get":
                continue
            sb, owners = payload
            for q in plist:  # scans: likewise partition by partition
                selq = np.nonzero(owners == q)[0]
                if not selq.size:
                    continue
                bruns = [orc.BlockRunCPU.from_blocks(b) for b in reversed(host_runs[q])]  # newest first
                hks = np.frombuffer(b"".join(bytes(sb.reqs[int(i)].start.data[2:2 + HK]) for i in selq), np.uint8)
                cnt, _nb, secs = orc.prefix_scan_many(bruns, hks, np.arange(selq.size + 1, dtype=np.uint32) * np.uint32(HK), NOW, threads)
                c_ret += cnt
                c_secs += secs
        out["parity_checked"] = bool(c_found == first["found"] and c_ret == first["returned"])
        out["cpu_baseline"] = {"requests_per_s": (my_gets + my_scans) / c_secs, "cores": threads, "kind": "port",
                               "what": "oracle-CPU lookups on the same block runs (not RocksDB)",
                               "sample": f"the same {my_gets} gets + {my_scans} prefix scans, {c_secs:.2f} s"}
        if not out["parity_checked"]:
            raise SystemExit(f"bench.py: sharded reads disagree with the oracle: found {first['found']} vs {c_found}, returned {first['returned']} vs {c_ret}")
    for part in parts.values():
        part.close()
    return out


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE.json configs[3]: manual compaction sweep, 30 % expired, run sizes 8..256 MB, bottommost forced
# ---------------------------------------------------------------------------------------------------------------------
def sweep_leg(pgs, eng, args, peak):
    from incubator_pegasus_b200 import synth
    out = []
    rec_bytes = 2 + HK + SK + 12 + VAL
    for mb in args.sweep_mb:
        n = max(1000, (mb << 20) // rec_bytes)
        rng = np.random.default_rng(900 + mb)
        runs = synth.compaction_runs(k=5, n_per_run=n, hk_len=HK, sk_len=SK, user_len=VAL, now=NOW, seed=2000 + mb)
        for r in runs:  # 30 % of the records already expired (synth's own mix has 10 %)
            nv = r.val_off.shape[0] - 1
            has = (r.val_off[1:] - r.val_off[:-1]) >= 4
            pick = np.nonzero(has & (rng.random(nv) < 0.30))[0]
            ets = (NOW - rng.integers(1, 86401, pick.size)).astype(">u4").view(np.uint8).reshape(-1, 4)
            for j in range(4):
                r.vals[(r.val_off[pick] + j).astype(np.int64)] = ets[:, j]
        part = eng.partition(app_id=3, pidx=mb)
        ids = part.upload_many([pgs.build_run(r) for r in runs], levels=[4, 3, 2, 1, 0])
        ms = []
        for i in range(2 + args.steps):
            res = part.compact(ids, out_level=4, bottommost=1, now=NOW, enabled=True, flags=3)
            if i >= 2:
                ms.append(res.merge_kernel_ms)
        k_ms = sum(ms) / len(ms)
        algo = int(res.in_bytes + res.out_bytes)
        out.append({"run_mb": mb, "runs": 5, "records": int(res.in_records), "survivors": int(res.out_records),
                    "dropped_expired": int(res.dropped_expired), "merge_kernel_ms": k_ms, "device_ms": float(res.device_ms),
                    "merged_GBps": res.in_bytes / (k_ms / 1e3) / 1e9,
                    "roofline_frac": algo / (k_ms / 1e3) / 1e9 / peak})
        part.close()
    return {"workload": "manual_compact sweep: 5 runs (L0..L4) of equal size, 30 % of the values expired, TTL filter on, bottommost forced "
                        f"(BASELINE.json configs[3]); merge kernels timed with CUDA events, mean of {args.steps} after 2 warm-ups",
            "sizes": out}


# ---------------------------------------------------------------------------------------------------------------------
# BASELINE.json configs[4] at small scale: YCSB-A, 50/50 put + get through the rrdb surface (one key per call)
# ---------------------------------------------------------------------------------------------------------------------
def ycsb_a_leg(pgs, eng, args):
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    from rrdb_harness import Backend
    be = Backend("gpu", eng, app_id=5, pidx=0, opts={"memtable_bytes": 4 << 20})
    rng = np.random.default_rng(5)
    n_keys, n_ops = args.ycsb_keys, args.ycsb_ops
    val = bytes(rng.integers(0, 256, 100, dtype=np.uint8))
    for i in range(n_keys):  # load phase
        be.put(b"user%08d" % i, b"f0", val, now=NOW)
    be.flush(NOW)
    ids = zipf_ids(rng, n_keys, n_ops)
    is_put = rng.random(n_ops) < 0.5
    hits = 0
    t0 = time.perf_counter()
    for i in range(n_ops):
        hk = b"user%08d" % int(ids[i])
        if is_put[i]:
            be.put(hk, b"f0", val, now=NOW)
        else:
            hits += be.get(hk, b"f0", now=NOW)["error"] == 0
    secs = time.perf_counter() - t0
    be.close()
    return {"workload": f"YCSB-A shaped: {n_keys} keys loaded, {n_ops} ops 50/50 put+get, zipfian(0.99), one key per rrdb call "
                        "(pgs_rrdb_put / pgs_rrdb_get: memtable in place + HBM runs), driven from Python through ctypes",
            "ops_per_s": n_ops / secs, "get_hit_frac": hits / max(1, int((~is_put).sum())), "seconds": secs,
            "note": "single-key calls are launch-latency bound; the batched read legs above are the throughput path"}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--records-per-run", type=int, default=2_500_000)
    ap.add_argument("--skip-cpu", action="store_true")
    ap.add_argument("--skip-e2e", action="store_true")
    ap.add_argument("--skip-reads", action="store_true")
    ap.add_argument("--skip-sharded", action="store_true")
    ap.add_argument("--skip-sweep", action="store_true")
    ap.add_argument("--skip-ycsb", action="store_true")
    ap.add_argument("--n-get", type=int, default=262144)
    ap.add_argument("--n-scan", type=int, default=16384)
    ap.add_argument("--partitions", type=int, default=256)
    ap.add_argument("--table-hashkeys", type=int, default=65536)
    ap.add_argument("--read-threads", type=int, default=8)
    ap.add_argument("--sweep-mb", type=int, nargs="*", default=[8, 16, 32, 64, 128, 256])
    ap.add_argument("--ycsb-keys", type=int, default=20000)
    ap.add_argument("--ycsb-ops", type=int, default=20000)
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned as DIR/<name>.npy (rank 0)")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be at least 1 and --warmup at least 0")

    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))

    if args.impl == "reference":
        reference_arm(args, rank, world)
        return

    import torch
    import torch.distributed as dist
    import incubator_pegasus_b200 as pgs

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the engine has no CPU path)")
    torch.cuda.set_device(local_rank)
    nccl = None
    if world > 1:
        os.environ.setdefault("MASTER_ADDR", "127.0.0.1")
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
        probe = torch.ones(1, device="cuda")
        dist.all_reduce(probe)  # the only collectives of this program: barriers and reductions of the timings
        nccl = {"backend": "nccl", "nranks": int(probe.item()), "used_for": "barriers + timing reductions only; the data path has no collective"}

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    # ---- inputs: this rank's partition ---------------------------------------------------------
    t0 = time.time()
    runs = gen_runs(args.records_per_run, 1000 + rank)
    host_runs = [pgs.build_run(r) for r in runs]  # flush side: records -> data blocks (host)
    in_bytes = sum(int(r.keys.shape[0] + r.vals.shape[0]) for r in runs)
    n_records = sum(r.n for r in runs)
    gen_s = time.time() - t0
    # pinned host copies of the block bytes for the end-to-end leg
    pinned, pinned_tensors = [], []
    for hr in host_runs:
        t = torch.empty(hr.data.shape[0], dtype=torch.uint8).pin_memory()
        t.numpy()[:] = hr.data
        pinned.append(pgs.BlockRun(t.numpy(), hr.blk_off, hr.blk_size))
        pinned_tensors.append(t)
    h2d_bytes = sum(int(p.data.shape[0]) for p in pinned)

    eng = pgs.Engine(device=local_rank)
    part = eng.partition(app_id=1, pidx=rank)
    ids = part.upload_many(pinned)
    stream = torch.cuda.ExternalStream(eng.stream, device=torch.device("cuda", local_rank))
    KEEP = 1 | 2  # PGS_COMPACT_KEEP_INPUTS | PGS_COMPACT_DISCARD_OUTPUT: repeat the same job

    def step(flags=KEEP):
        return part.compact(ids, out_level=1, bottommost=1, now=NOW, enabled=True, flags=flags)

    for _ in range(args.warmup):
        res = step()
    sampler = ClockSampler(local_rank)
    sampler.start()
    barrier()
    launches0 = eng.launches
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    merge_ms, plan_ms, walk_ms, emit_ms = [], [], [], []
    w0 = time.perf_counter()
    with torch.cuda.stream(stream):
        ev0.record(stream)
        for i in range(args.steps):
            # --dump-outputs: the last step installs its merged run so that it can be read back; the device work is the same
            res = step(1 if args.dump_outputs and i == args.steps - 1 else KEEP)
            merge_ms.append(res.merge_kernel_ms)
            plan_ms.append(res.device_ms - res.merge_kernel_ms)
            walk_ms.append(res.walk_ms)
            emit_ms.append(res.emit_ms)
        ev1.record(stream)
    barrier()
    wall_ms = (time.perf_counter() - w0) * 1e3
    sampler.stop_flag.set()
    dev_ms = ev0.elapsed_time(ev1)
    launches = eng.launches - launches0
    t = torch.tensor([dev_ms], dtype=torch.float64, device="cuda")
    if world > 1:
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
    max_ms = float(t.item())
    ms_per_step = max_ms / args.steps
    value = world * in_bytes / (ms_per_step / 1e3) / 1e9
    if args.dump_outputs:
        if rank == 0:
            dump_compaction(args.dump_outputs, res, pgs.decode_blocks(part.download(res.new_run_id)))
        part.drop(res.new_run_id)  # the read legs below see the same 4 runs as without the dump

    # ---- end to end through the C ABI from host buffers ------------------------------------------
    e2e = None
    if not args.skip_e2e:
        part2 = eng.partition(app_id=1, pidx=rank + 1000)
        split = {"upload": 0.0, "compact": 0.0, "drop": 0.0}

        def e2e_step():
            t0 = time.perf_counter()
            rid = part2.upload_many(pinned)                    # pipelined H2D of the runs + device index / Bloom build
            t1 = time.perf_counter()
            r = part2.compact(rid, out_level=1, bottommost=1, now=NOW, enabled=True)  # result struct comes back
            t2 = time.perf_counter()
            if r.new_run_id:
                part2.drop(r.new_run_id)
            t3 = time.perf_counter()
            split["upload"] += (t1 - t0) * 1e3; split["compact"] += (t2 - t1) * 1e3; split["drop"] += (t3 - t2) * 1e3
            return r

        e2e_step()
        barrier()
        split.update(upload=0.0, compact=0.0, drop=0.0)
        e0 = time.perf_counter()
        n_e2e = args.steps
        for _ in range(n_e2e):
            e2e_step()
        barrier()
        e_ms = (time.perf_counter() - e0) * 1e3 / n_e2e
        te = torch.tensor([e_ms], dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(te, op=dist.ReduceOp.MAX)
        # what the host link of this box delivers for a plain pinned -> device copy (context for the number above)
        probe = torch.empty(min(1 << 30, int(pinned_tensors[0].numel())), dtype=torch.uint8, device="cuda")
        src = pinned_tensors[0][: probe.numel()]
        probe.copy_(src, non_blocking=True)
        torch.cuda.synchronize()
        p0, p1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        p0.record()
        probe.copy_(src, non_blocking=True)
        p1.record()
        torch.cuda.synchronize()
        h2d_probe = probe.numel() / (p0.elapsed_time(p1) / 1e3) / 1e9
        del probe
        e2e = {"value": world * in_bytes / (float(te.item()) / 1e3) / 1e9, "unit": "GB/s",
               "h2d_bytes_per_step": h2d_bytes, "d2h_bytes_per_step": 128, "ms_per_step": float(te.item()),
               "timed": "host wall clock around upload_many(4 runs)+compact, barrier+synchronize both sides",
               "h2d_link_probe_GBps": round(h2d_probe, 1),
               "link_bound_ms": round(h2d_bytes / h2d_probe / 1e6, 2),
               "host_ms_per_step": {k: round(v / n_e2e, 2) for k, v in split.items()}}
        part2.close()

    # ---- read path on the same partition (4 overlapping runs resident): YCSB-C shaped, zipfian hash keys ----------
    reads = None
    traffic = load_traffic()
    peak, peak_src = load_peaks()
    if not args.skip_reads:
        pins = []

        def pinned_alloc(n, dt):  # host buffers of the read legs live in pinned memory, like a server's I/O buffers
            t = torch.empty(int(n) * np.dtype(dt).itemsize, dtype=torch.uint8).pin_memory()
            pins.append(t)
            return t.numpy().view(dt)

        gk, sk = read_workload(args.records_per_run, args.n_get, args.n_scan, 1000 + rank)
        gkeys = pinned_alloc(gk.size, np.uint8)
        gkeys[:] = gk.reshape(-1)
        goff = pinned_alloc(args.n_get + 1, np.uint32)
        goff[:] = np.arange(args.n_get + 1, dtype=np.uint32) * np.uint32(gk.shape[1])
        hashkeys = [bytes(r) for r in sk]
        garena_cap = args.n_get * (VAL + 8)
        garena_buf = pinned_alloc(garena_cap, np.uint8)
        gres_buf = (pgs.GetResult * args.n_get)()
        # gets
        part.get_batch(gkeys, goff, NOW, arena_cap=garena_cap, arena=garena_buf, results=gres_buf)
        g_ms, g_wall, found, probes = [], [], 0, 0
        for _ in range(args.steps):
            barrier()
            t0 = time.perf_counter()
            st, gres, garena, gused = part.get_batch(gkeys, goff, NOW, arena_cap=garena_cap, arena=garena_buf, results=gres_buf)
            g_wall.append((time.perf_counter() - t0) * 1e3)
            g_ms.append(eng.last_kernel_ms)
            probes = eng.last_blocks_probed
            skipped = eng.last_runs_skipped
        found = sum(1 for i in range(args.n_get) if gres[i].status == 0)
        # prefix scans = multi_get(hash_key, all sort keys)
        sb = part.prefix_scan_batch(hashkeys, max_records=80, arena_stride=24576, alloc=pinned_alloc)  # request structs marshalled once
        assert sb.run(NOW) == 0
        s_ms, s_wall = [], []
        for _ in range(args.steps):
            barrier()
            t0 = time.perf_counter()
            st = sb.run(NOW)  # host request structs in, packed records out (host buffers)
            s_wall.append((time.perf_counter() - t0) * 1e3)
            s_ms.append(eng.last_kernel_ms)
            assert st == 0, st
        sres, abase, kbase = sb.results, sb.abase, sb.kbase
        if args.dump_outputs and rank == 0:
            dump_reads(args.dump_outputs, gres, garena, sb)
        returned = int(kbase[-1])
        iterated = int(sum(sres[i].iter_count for i in range(args.n_scan)))
        scan_bytes = int(abase[-1])
        mean = lambda xs: sum(xs) / len(xs)
        gm, sm, gw, sw = mean(g_ms), mean(s_ms), mean(g_wall), mean(s_wall)
        nb_log = 18
        get_algo = probes * (4096 + nb_log * 58) + args.n_get * (2 + HK + SK) + int(gused)
        scan_algo = returned * 2 * (2 + HK + SK + 12 + VAL) + (iterated - returned) * (2 + HK + SK + 12 + VAL)
        vals = torch.tensor([args.n_get / (gm / 1e3), args.n_get / (gw / 1e3), returned / (sm / 1e3), returned / (sw / 1e3)],
                            dtype=torch.float64, device="cuda")
        if world > 1:
            dist.all_reduce(vals, op=dist.ReduceOp.SUM)  # partitions are independent: whole-job keys/s = sum over ranks

        def roof(kernel, algo, ms):
            tr = traffic.get(kernel)
            r = {"bound": "hbm", "kernel": kernel, "achieved": algo / (ms / 1e3) / 1e9, "peak": peak, "unit": "GB/s",
                 "frac": algo / (ms / 1e3) / 1e9 / peak, "algorithmic_bytes_per_launch": algo,
                 "formula": "SURVEY.md §8(d): blocks probed x (4 KB block + index path) + keys + values returned" if kernel == "k_get"
                            else "SURVEY.md §8(d): records iterated x record bytes + records returned x record bytes"}
            if tr:  # DRAM bytes of the same launch shape under ncu (time from this run's CUDA events)
                r["traffic"] = tr["dram_bytes_per_launch"]
                r["traffic_source"] = tr.get("source")
                r["dram_frac"] = tr["dram_bytes_per_launch"] / (ms / 1e3) / 1e9 / peak
            else:
                r["traffic"] = None
            return r

        reads = {
            "statistic": "mean over the repetitions, for the device (kernel CUDA events) and the e2e (host wall clock) numbers alike",
            "get": {"metric": "get_keys_per_s", "value": float(vals[0]), "e2e": float(vals[1]), "unit": "keys/s", "batch": args.n_get,
                    "kernel_ms": gm, "e2e_ms": gw, "found_frac": found / args.n_get, "blocks_probed_per_key": probes / args.n_get,
                    "bloom_runs_skipped_per_key": skipped / args.n_get,
                    "roofline": roof("k_get", get_algo, gm)},
            "scan": {"metric": "scan_keys_per_s", "value": float(vals[2]), "e2e": float(vals[3]), "unit": "keys/s", "requests": args.n_scan,
                     "returned_per_launch": returned, "iterated_per_launch": iterated, "kernel_ms": sm, "e2e_ms": sw, "d2h_bytes": scan_bytes,
                     "roofline": roof("k_scan_fwd", scan_algo, sm)},
            "workload": "YCSB-C shaped: zipfian(0.99) hash keys over the 4 resident overlapping runs; get(hk,sk) and multi_get(hk, all sort keys)",
        }
        if rank == 0 and world == 1 and not args.skip_cpu:
            import oracle_py as orc
            threads = os.cpu_count() or 1
            bruns = [orc.BlockRunCPU.from_blocks(hr) for hr in reversed(host_runs)]  # newest first
            ng, tot_s, tot_n = args.n_get, 0.0, 0
            while tot_s < 2.0 and tot_n < 200 * ng:  # repeat the batch until the sample is a couple of seconds of wall time
                f, vb, secs = orc.get_many(bruns, gkeys, goff, NOW, threads)
                tot_s += secs
                tot_n += ng
            reads["get"]["cpu_baseline"] = {"value": tot_n / tot_s, "unit": "keys/s", "cores": threads, "kind": "port",
                                            "sample": f"{tot_n} gets ({ng}-key batch repeated) over the same 4 block runs, {tot_s:.2f} s"}
            reads["get"]["parity_checked"] = bool(f == found)
            nsc = args.n_scan
            hk_flat = np.ascontiguousarray(sk[:nsc].reshape(-1))
            hk_off = (np.arange(nsc + 1, dtype=np.uint32) * np.uint32(HK))
            tot_s, tot_n, tot_q = 0.0, 0, 0
            while tot_s < 2.0 and tot_q < 200 * nsc:
                cnt, nb_, secs = orc.prefix_scan_many(bruns, hk_flat, hk_off, NOW, threads)
                tot_s += secs
                tot_n += cnt
                tot_q += nsc
            reads["scan"]["cpu_baseline"] = {"value": tot_n / tot_s, "unit": "keys/s", "cores": threads, "kind": "port",
                                             "sample": f"{tot_q} prefix scans ({tot_n} records) over the same 4 block runs, {tot_s:.2f} s"}
            reads["scan"]["parity_checked"] = bool(cnt == returned)
            del bruns
            if not (reads["get"]["parity_checked"] and reads["scan"]["parity_checked"]):
                raise SystemExit(f"bench.py: read legs disagree with the oracle: gets found {found} vs {f}, scan records {returned} vs {cnt}")

    # ---- roofline of the merge kernels --------------------------------------------------------------
    k_ms = sum(merge_ms) / len(merge_ms)
    algo_bytes = int(res.in_bytes + res.out_bytes)
    achieved = algo_bytes / (k_ms / 1e3) / 1e9
    tr_w, tr_e = traffic.get("k_walk"), traffic.get("k_emit")
    roofline = {"bound": "hbm", "kernel": "k_walk+k_emit", "achieved": achieved, "peak": peak, "unit": "GB/s",
                "frac": achieved / peak, "peak_source": peak_src, "algorithmic_bytes_per_launch": algo_bytes, "kernel_ms": k_ms,
                "kernels_ms": {"k_walk": sum(walk_ms) / len(walk_ms), "k_emit": sum(emit_ms) / len(emit_ms),
                               "plan (k_plan+k_seg_bounds+k_seg_layout)": sum(plan_ms) / len(plan_ms)},
                "traffic": (tr_w["dram_bytes_per_launch"] + tr_e["dram_bytes_per_launch"]) if tr_w and tr_e else None,
                "traffic_source": tr_w.get("source") if tr_w and tr_e else None}

    # ---- CPU baseline on the same full workload + parity of the statistics (rank 0, N=1 only) -----------
    cpu, parity = None, None
    if rank == 0 and world == 1 and not args.skip_cpu:
        threads = os.cpu_count() or 1
        gbs, secs, st = cpu_compaction(cpu_block_runs(runs), threads)[:3]
        cpu = {"value": gbs, "unit": "GB/s", "cores": threads, "kind": "port",
               "what": "oracle-CPU block-level compaction (a restatement of the reference's RocksDB path, not RocksDB)",
               "sample": f"{RUNS} runs x {args.records_per_run} records ({st.in_bytes / 1e9:.2f} GB merged): the full workload, {secs:.2f} s"}
        diff = {f: (int(getattr(res, f)), int(getattr(st, f))) for f in STAT_FIELDS if int(getattr(res, f)) != int(getattr(st, f))}
        parity = not diff
        if diff:
            raise SystemExit(f"bench.py: compaction statistics differ from the oracle at bench size: {diff}")

    sharded = None
    if not args.skip_sharded:
        sharded = sharded_read_leg(pgs, torch, dist, eng, rank, world, args, barrier, check_cpu=(rank == 0 and world == 1 and not args.skip_cpu))
    sweep = ycsb = None
    if world == 1 and not args.skip_sweep:
        sweep = sweep_leg(pgs, eng, args, peak)
    if world == 1 and not args.skip_ycsb:
        ycsb = ycsb_a_leg(pgs, eng, args)

    if rank == 0:
        cfg = workload_config(args.records_per_run)
        cfg.update({"records_per_step_per_gpu": n_records, "merged_bytes_per_step_per_gpu": in_bytes,
                    "survivors": int(res.out_records), "segments": int(res.n_tiles),
                    "l2": "inputs (2.9 GB of blocks) larger than the 126 MB L2", "input_gen_s": round(gen_s, 1)})
        line = {
            "metric": "compaction_merged_GBps", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": cfg,
            "roofline": roofline, "cpu_baseline": cpu, "parity_checked": parity, "e2e": e2e, "reads": reads,
            "sharded_reads": sharded, "sweep": sweep, "ycsb_a": ycsb, "nccl": nccl, "gpu_launches": int(launches),
            "clocks": sampler.summary(), "wall_ms_per_step": wall_ms / args.steps,
        }
        print(json.dumps(line), flush=True)
    part.close()
    eng.close()
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
