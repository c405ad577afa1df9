#!/usr/bin/env python
"""bench.py -- extract GB/s (uncompressed) of the PNA data-chunk hot path on B200, vs the host-CPU path.

Workload of the headline line (BASELINE.json configs[1], weak-scaled): each GPU extracts one shard of `--entries` x 4 MiB
files, zstd level 3 + AES-256-CTR, layout FHED,fSIZ,PHSF,FDAT(16),FDAT(C),FEND.  A "step" = one pass of the whole hot path
over the shard: CRC-32 check of every chunk, AES-256-CTR decrypt, zstd decode.

  value         kernel-only: archive already resident in HBM, CUDA events on the library's stream, max over ranks
  e2e           the same through the C++ host layer over the C ABI with HOST buffers: pinned archive -> H2D -> kernels -> D2H
                pinned outputs; e2e.pcie = the step's own transfers (same buffers, same bytes) copied by ALL ranks at the same
                time, each direction alone and both at once -- the box's concurrent transfer floor for this N
  roofline      dominant stage, algorithmic bytes / event time vs the measured HBM copy peak
  cpu_baseline  the oracle (reference dataflow restated on libzstd / OpenSSL / zlib, chunk CRC by the PCLMULQDQ folding method
                crc32fast uses) on the host cores, with single-core per-stage rates beside it
  create        BASELINE config 4's shape on the same shard (GPU zstd + AES-256-CTR + FDAT CRC-32)
  configs       (N = 1 only) the five BASELINE.json configurations at their stated sizes: cfg1, cfg3, cfg4_zstd, cfg4_deflate, cfg5

`--impl reference` times the CPU path alone (the reference is Rust; there is no cargo in this image, so the oracle port runs).
Inputs are synthetic (corpus.py), produced outside every timed region by the oracle's encoders, i.e. the same libzstd
level-3 streaming frames / zlib level-6 streams the reference writes.

`--dump-outputs DIR` writes what the last timed step of the extract and create paths returned to a caller (rank 0), so that
two builds can be compared output for output on the same seeded inputs:
  extract_files_sample, create_streams_sample   float32 bytes: all of them up to DUMP_SAMPLE_BYTES, beyond that windows at
                                                 seeded places, listed as rows [entry, offset, length] in *_sample_where
  extract_files_crc32, create_streams_crc32     float64 CRC-32 of every whole decoded file / created stream
  extract_files_length, create_streams_length   float64 bytes of every decoded file / created stream
  extract_chunk_crc32, create_chunk_crc32       float64 chunk CRCs the kernels computed (every chunk of the archive / FDAT)
"""
from __future__ import annotations

import argparse
import ctypes as C
import importlib
import json
import os
import statistics
import subprocess
import sys
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "oracle"))
import benchlib  # noqa: E402
import corpus  # noqa: E402

FILE_SIZE = benchlib.FILE_SIZE
PASSWORD = b"bench-password"
SALT = b"pna-bench-salt16"     # fixed, so that the PHSF chunks, and with them the archive bytes, repeat from run to run
KEY = bytes(range(32))
DUMP_SAMPLE_BYTES = 4 << 20    # per sampled output; both paths' dumps stay under 40 MB at 1024 entries
DUMP_WINDOW = 4096


def sample_bytes(blobs, seed: int):
    """Bytes of `blobs` (uint8 arrays): all of them when they total at most DUMP_SAMPLE_BYTES, else windows of up to
    DUMP_WINDOW bytes at places drawn from `seed`.  Returns (bytes as float32, rows [blob, offset, length] as float64)."""
    lens = np.array([b.size for b in blobs], dtype=np.int64)
    if lens.sum() <= DUMP_SAMPLE_BYTES:
        where = np.stack([np.arange(len(blobs)), np.zeros(len(blobs), dtype=np.int64), lens], axis=1)
    else:
        rng = np.random.default_rng(seed)
        k = DUMP_SAMPLE_BYTES // DUMP_WINDOW
        blob = np.sort(rng.integers(0, len(blobs), k))
        n = np.minimum(lens[blob], DUMP_WINDOW)
        off = (rng.random(k) * (lens[blob] - n + 1)).astype(np.int64)
        where = np.stack([blob, off, n], axis=1)
    data = np.concatenate([blobs[b][o:o + n] for b, o, n in where] + [np.zeros(0, dtype=np.uint8)])
    return data.astype(np.float32), where.astype(np.float64)


def dump_outputs(d: str, path: str, what: str, blobs, chunk_crcs, seed: int):
    """`path`'s outputs as DIR/<path>_<what>_{sample,sample_where,crc32,length}.npy and DIR/<path>_chunk_crc32.npy"""
    os.makedirs(d, exist_ok=True)
    data, where = sample_bytes(blobs, seed)
    arrays = {f"{what}_sample": data, f"{what}_sample_where": where,
              f"{what}_crc32": np.array([zlib.crc32(b) for b in blobs], dtype=np.float64),
              f"{what}_length": np.array([b.size for b in blobs], dtype=np.float64),
              "chunk_crc32": np.asarray(chunk_crcs, dtype=np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(d, f"{path}_{name}.npy"), a)


def make_shard(rank: int, entries: int, threads: int, world: int = 1):
    """Plain files + oracle-encoded streams (zstd 3 + AES-256-CTR) of this rank's shard.  Not timed.  (Kept for tools/.)"""
    shard = importlib.import_module("portable-network-archive_b200.shard")
    idx = shard.rank_entries([FILE_SIZE] * (entries * world), rank, world)
    files = benchlib.gen_files(idx, threads)
    plain, offs = benchlib.pack(files)
    streams, s_offs, _ = benchlib.oracle_encode(plain, offs, 2, 3, 1, 1, KEY, threads, seed=1234 + rank)
    return files, [streams[s_offs[i]:s_offs[i + 1]].tobytes() for i in range(entries)], KEY


def build_archive(streams, sizes, phsf: str, into=None):
    """PNA container bytes around per-entry streams (list of bytes).  (Kept for tools/.)"""
    buf, s_offs = benchlib.pack(streams)
    return benchlib.frame_archive(buf, s_offs, sizes, bytes([0, 0, 0, 2, 1, 1]), phsf, 16, "corpus/%07d.bin", into or (lambda n: np.empty(n, dtype=np.uint8)), 1)


class ClockSampler:
    QUERY = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.active,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, gpu_index: int):
        self.p = None
        try:
            self.p = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.QUERY}", "--format=csv,noheader,nounits", "-lms", "100",
                                       "-i", str(gpu_index)], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.p = None

    def stop(self):
        if not self.p:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.p.terminate()
        try:
            out = self.p.communicate(timeout=5)[0]
        except Exception:
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 9:
                continue
            try:
                sm.append(float(f[1]))
                mx.append(float(f[2]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[5:9]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def cpu_box():
    model = ""
    try:
        for line in open("/proc/cpuinfo"):
            if line.startswith("model name"):
                model = line.split(":", 1)[1].strip()
                break
    except OSError:
        pass
    return {"model": model, "logical_cpus": os.cpu_count()}


def reference_arm(args, ncpu):
    """The reference's own CPU implementation of the path (oracle port) on all host threads: extract dataflow, bounded sample."""
    E = args.entries
    sample = min(E, 256)
    files = benchlib.gen_files(range(sample), ncpu)
    sizes = [len(f) for f in files]
    U = sum(sizes)
    plain, offs = benchlib.pack(files)
    streams, s_offs, _ = benchlib.oracle_encode(plain, offs, 2, 3, 1, 1, KEY, ncpu, seed=1234)
    for _ in range(max(args.warmup, 1)):
        benchlib.oracle_decode_time(streams, s_offs, sizes, 2, 1, 1, KEY, ncpu, crc_impl=2)
    tot = 0.0
    for _ in range(args.steps):   # buffer set-up is outside the timed region (inputs / outputs resident in RAM)
        dt, out, o_offs = benchlib.oracle_decode_time(streams, s_offs, sizes, 2, 1, 1, KEY, ncpu, crc_impl=2)
        tot += dt
    assert out[o_offs[0]:o_offs[1]].tobytes() == files[0]
    dtz, _, _ = benchlib.oracle_decode_time(streams, s_offs, sizes, 2, 1, 1, KEY, ncpu, crc_impl=1, passes=2)
    dth, _, _ = benchlib.oracle_decode_time(streams, s_offs, sizes, 2, 1, 1, KEY, max(1, ncpu // 2), crc_impl=2, passes=2)
    v = U * args.steps / tot / 1e9
    return v, tot / args.steps, {
        "value": v, "unit": "GB/s", "cores": ncpu, "kind": "port",
        "sample": f"{sample} x 4 MiB entries per step (oracle: libzstd + OpenSSL AES-NI + PCLMULQDQ folding chunk CRC as crc32fast; "
                  f"1 iterating/CRC thread + {ncpu} workers, reference extract dataflow)",
        "with_zlib_table_crc_GBps": U / dtz / 1e9, "with_half_the_workers_GBps": U / dth / 1e9,
        "single_core": benchlib.single_core_rates(files[0] * 8, KEY), "box": cpu_box()}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--entries", type=int, default=1024, help="4 MiB files per GPU (cfg2: 8192 over 8 GPUs)")
    ap.add_argument("--e2e-steps", type=int, default=7)
    ap.add_argument("--workers", type=int, default=0, help="host worker threads of the end-to-end path (0: 4, or the rank's cores if fewer)")
    ap.add_argument("--group-mib", type=int, default=128, help="compressed MiB per pipelined entry group (end-to-end path)")
    ap.add_argument("--create-workers", type=int, default=4)
    ap.add_argument("--create-group-mib", type=int, default=256)
    ap.add_argument("--create", type=int, default=1, help="also measure the create path (GPU zstd + AES-CTR + CRC) on the same files")
    ap.add_argument("--configs", type=int, default=1, help="at N = 1: also run BASELINE.json configs 1, 3, 4, 5 at their stated sizes")
    ap.add_argument("--config-scale", type=float, default=1.0, help="shrink the configs (development runs); 1.0 = stated sizes")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the outputs of the last timed extract and create steps to DIR/*.npy (see the module docstring)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    cpus = benchlib.cpu_affinity_for_rank(local_rank, world) or list(range(os.cpu_count() or 1))
    threads = max(1, len(cpus))
    E = args.entries
    workers = args.workers or max(2, min(4, threads))
    cfg = {"workload": f"cfg2 shard: extract {E} x 4 MiB files per GPU, zstd level 3 + AES-256-CTR, chunk CRC-32 check "
                       f"(32 GiB / 8 GPUs at the full config)", "entries_per_gpu": E, "file_bytes": FILE_SIZE,
           "codec": "zstd-3", "cipher": "aes-256-ctr", "parallelism": f"entry-sharded x{world}, no collective",
           "l2": "inputs (C+U per step ~5.7 GiB) far exceed the 126 MB L2; no flush needed"}

    if args.impl == "reference":
        if rank != 0:
            return
        ncpu = os.cpu_count() or 1
        os.sched_setaffinity(0, range(ncpu)) if hasattr(os, "sched_setaffinity") else None
        v, s_per_step, cb = reference_arm(args, ncpu)
        line = {"impl": "reference", "metric": "extract_uncompressed_GBps", "value": v, "unit": "GB/s", "n_gpus": args.gpus,
                "steps": args.steps, "warmup": args.warmup, "ms_per_step": s_per_step * 1e3, "higher_is_better": True,
                "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": cfg, "cpu_baseline": cb,
                "e2e": {"value": v, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch
    import torch.distributed as dist
    torch.cuda.set_device(local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    pna = importlib.import_module("portable-network-archive_b200")
    host = importlib.import_module("portable-network-archive_b200._host")
    ctx = pna.Context(local_rank)

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    def sum_over_ranks(x: float) -> float:
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.SUM)
        return float(t.item())

    # ---- inputs (not timed).  The global corpus has world x entries files; the rank's share comes from the same LPT partition by
    # entry that the extract path uses (portable-network-archive_b200/shard.py) -- no collective, every rank derives it alone.
    run_configs = bool(args.configs) and world == 1
    shard = importlib.import_module("portable-network-archive_b200.shard")
    idx = shard.rank_entries([FILE_SIZE] * (E * world), rank, world)
    n_cfg4 = int(4096 * args.config_scale) if run_configs else 0
    have = set(idx)
    extra = [i for i in range(max(n_cfg4, 0)) if i not in have] if run_configs else []
    all_files = benchlib.gen_files(list(idx) + extra[:max(0, n_cfg4 - len(idx))], threads)
    files = all_files[:E]
    sizes = [len(f) for f in files]
    U = sum(sizes)
    plain_np, p_offs = benchlib.pack(files)
    streams_np, s_offs, _ = benchlib.oracle_encode(plain_np, p_offs, 2, 3, 1, 1, KEY, threads, seed=1234 + rank)
    Cbytes = int(s_offs[-1])
    opts = pna.WriteOptions(compression=2, encryption=1, cipher_mode=1, password=PASSWORD, kdf_params={"i": 1000}, salt=SALT)
    # the shard's streams were encrypted with KEY; record it as the options' derived key (the KDF is host work, once per archive)
    archive_buf = benchlib.frame_archive(streams_np, s_offs, sizes, bytes([0, 0, 0, 2, 1, 1]), opts.phsf, 16, "corpus/%07d.bin", ctx.pinned, threads)
    arch_bytes = int(archive_buf.size)
    ro = pna.ReadOptions.with_password(PASSWORD)
    ro._keys[opts.phsf] = KEY

    archive = pna.Archive.read_header(archive_buf, ctx, verify=False)   # index pass (host); CRC runs inside the plan
    plan, ents = archive.extract_plan(ro)
    assert len(ents) == E
    stream = torch.cuda.ExternalStream(ctx.stream)
    # ---- kernel-only: W warm-ups, K timed steps, CUDA events on the library's stream
    for _ in range(max(args.warmup, 1)):
        plan.run()
    torch.cuda.synchronize()
    l0 = ctx.launch_count
    sampler = ClockSampler(local_rank) if rank == 0 else None
    barrier()
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    ev0.record(stream)
    for _ in range(args.steps):
        plan.run()
    ev1.record(stream)
    barrier()
    ms_total = ev0.elapsed_time(ev1)
    launches = ctx.launch_count - l0
    clocks = sampler.stop() if sampler else None
    ms_step = max_over_ranks(ms_total / args.steps)
    counts = plan.counts()
    stage_ms = plan.stage_ms()                     # last timed step, CUDA events between stages on the same stream
    # parity spot-check of what was just timed
    outs, st, _ = plan.fetch(sizes)
    crcs, broken = plan.crc_results()
    assert st == [0] * E and broken == 0, "decode failed"
    for k in range(0, E, max(1, E // 16)):
        assert outs[k].tobytes() == files[k], "GPU output differs from the source file"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, "extract", "files", outs, crcs, seed=1)
    del outs
    plan.close()

    # ---- end to end through the reference-facing host API (C++ pna::Archive over the C ABI) with HOST buffers:
    # index pass over the pinned archive bytes, then entry groups pipelined over `workers` threads x 2 contexts (H2D + chunk CRC
    # check + decrypt + decode + D2H into pinned output), everything inside the timed region
    out_pinned = ctx.pinned(U + 16 * E + 64)
    e2e_times = []
    for it in range(args.e2e_steps + 1):
        barrier()
        t0 = time.perf_counter()
        ha = host.HostArchive(archive_buf)
        ha.set_key(opts.phsf, KEY)
        _, offs, stv = ha.extract_files(out=out_pinned, device=local_rank, workers=workers, group_bytes=args.group_mib << 20, verify=True)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        ha.close()
        if it > 0:
            e2e_times.append(dt)
    if e2e_times:
        assert stv == [0] * E
        for k in range(0, E, max(1, E // 16)):
            assert out_pinned[int(offs[k]):int(offs[k]) + sizes[k]].tobytes() == files[k], "e2e output differs from the source file"
    e2e_s = max_over_ranks(statistics.median(e2e_times)) if e2e_times else float('nan')
    # PCIe yardstick: the step's OWN transfers (the pinned archive up, U bytes down into the pinned output buffer) copied by EVERY
    # rank at the same time -- each direction alone, then both at once, which is what the pipelined path does.  The slowest rank's
    # both-at-once time is the concurrent transfer floor of the step at this N; everything above it is pipeline fill and host work.
    pcie = None
    if e2e_times:
        best = None
        for _ in range(2):
            barrier()
            pr = ctx.transfer_probe(archive_buf, out_pinned[:U])
            barrier()
            best = pr if best is None or pr["both_ms"] < best["both_ms"] else best
        floor_ms = max_over_ranks(best["both_ms"])
        h_ms, d_ms = max_over_ranks(best["h2d_ms"]), max_over_ranks(best["d2h_ms"])
        pcie = {"ranks_concurrent": world, "h2d_alone_GBps_aggregate": world * archive_buf.size / h_ms / 1e6,
                "d2h_alone_GBps_aggregate": world * U / d_ms / 1e6,
                "both_at_once_ms": floor_ms, "both_at_once_GBps_aggregate": world * (archive_buf.size + U) / floor_ms / 1e6,
                "rank0": {k: round(v, 3) for k, v in best.items()},
                "transfer_floor_ms": floor_ms, "e2e_over_floor": e2e_s * 1e3 / floor_ms,
                "how": "pna_cuda_transfer_probe: the step's pinned buffers and byte counts, all ranks after a barrier, CUDA events, max over ranks"}

    # ---- create path (BASELINE config 4 shape: GPU zstd encode + AES-256-CTR + FDAT CRC-32) on the same files
    create = None
    if args.create:
        import pna_oracle as O
        rng = np.random.Generator(np.random.PCG64(99 + rank))
        plain_pinned = ctx.pinned(U)
        plain_pinned[:] = plain_np[:U]
        views = [plain_pinned[int(p_offs[i]):int(p_offs[i + 1])] for i in range(E)]
        enc_ents = [{"plain": v, "compression": 2, "level": 3, "encryption": 1, "cipher_mode": 1, "key": KEY, "iv": rng.bytes(16),
                     "max_chunk_size": 0} for v in views]
        eplan = ctx.encode_plan(enc_ents)
        for _ in range(max(args.warmup, 1)):
            eplan.run()
        torch.cuda.synchronize()
        l1 = ctx.launch_count
        barrier()
        c0, c1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        c0.record(stream)
        for _ in range(args.steps):
            eplan.run()
        c1.record(stream)
        barrier()
        c_ms = max_over_ranks(c0.elapsed_time(c1) / args.steps)
        c_launches = ctx.launch_count - l1
        c_stage = eplan.stage_ms()
        outp = ctx.pinned(sum(eplan.bounds))
        streams_gpu, crcs_gpu, cst = eplan.fetch(into=outp)
        assert cst == [0] * E
        c_gpu = sum(int(s.size) for s in streams_gpu)
        for k in range(0, E, max(1, E // 8)):   # the reference pipeline must read what we wrote, CRCs must match
            s = streams_gpu[k].tobytes()
            assert O.decode_stream(s, 2, 1, 1, KEY, None) == files[k], "GPU-created stream is not reference-readable"
            assert int(crcs_gpu[k][0]) == O.chunk_crc(b"FDAT", s[16:])
        if args.dump_outputs and rank == 0:
            dump_outputs(args.dump_outputs, "create", "streams", streams_gpu, np.concatenate(crcs_gpu + [np.zeros(0, np.uint32)]), seed=2)
        eplan.close()
        ce2e = []
        names = [f"corpus/{i:07d}.bin" for i in range(E)]
        arch_out = ctx.pinned(int(U * 1.02) + (64 << 20))
        ivs = rng.bytes(16 * E)
        for it in range(args.e2e_steps + 1):
            barrier()
            t0 = time.perf_counter()
            blob = host.create_archive(list(zip(names, views)), compression=2, level=3, encryption=1, cipher_mode=1, key=KEY, phsf=opts.phsf,
                                       ivs=ivs, max_chunk_size=0, device=local_rank, workers=args.create_workers,
                                       group_bytes=args.create_group_mib << 20, out=arch_out)
            torch.cuda.synchronize()
            dt = time.perf_counter() - t0
            if it > 0:
                ce2e.append(dt)
        if ce2e:   # the created archive must extract bit-exactly with ours (all) and with the reference reader (oracle; small runs)
            hb = host.HostArchive(blob)
            hb.set_key(opts.phsf, KEY)
            o2, of2, st2 = hb.extract_files(device=local_rank, workers=workers)
            assert st2 == [0] * E
            for k in range(0, E, max(1, E // 16)):
                assert o2[int(of2[k]):int(of2[k]) + sizes[k]].tobytes() == files[k]
            if E <= 64:
                assert [d for _, d in O.extract_all(blob.tobytes(), PASSWORD, _keys={opts.phsf: KEY})] == files
            del o2
            hb.close()
        ce2e_s = max_over_ranks(statistics.median(ce2e)) if ce2e else float("nan")
        create = {"metric": "create_uncompressed_GBps", "value": world * U / (c_ms * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": c_ms,
                  "e2e": {"value": world * U / ce2e_s / 1e9, "unit": "GB/s", "h2d_bytes_per_step": int(U) * world, "d2h_bytes_per_step": int(c_gpu) * world,
                          "ms_per_step": ce2e_s * 1e3},
                  "codec": "gpu zstd + aes-256-ctr + crc32", "stage_ms": c_stage,
                  "gpu_launches": c_launches, "ratio": U / c_gpu, "c_gpu_over_c_ref": c_gpu / Cbytes,
                  "checked": "sampled streams decoded by the oracle (libzstd + OpenSSL) == source files; FDAT CRCs == zlib crc32"}
        for b in (outp, plain_pinned, arch_out):
            ctx.pinned_free(b)
        del outp, plain_pinned, arch_out, views, enc_ents, streams_gpu

    # ---- CPU baseline on this box's cores (rank 0, N=1 only): bounded sample of the same workload
    cpu = None
    cpu_create = None
    if rank == 0 and world == 1:
        ncpu = threads
        sample = min(E, 256)
        so = s_offs[:sample + 1]
        benchlib.oracle_decode_time(streams_np, so, sizes[:sample], 2, 1, 1, KEY, ncpu, crc_impl=2)
        dt, _, _ = benchlib.oracle_decode_time(streams_np, so, sizes[:sample], 2, 1, 1, KEY, ncpu, crc_impl=2, passes=3)
        dtz, _, _ = benchlib.oracle_decode_time(streams_np, so, sizes[:sample], 2, 1, 1, KEY, ncpu, crc_impl=1, passes=2)
        dth, _, _ = benchlib.oracle_decode_time(streams_np, so, sizes[:sample], 2, 1, 1, KEY, max(1, ncpu // 2), crc_impl=2, passes=2)
        Us = sum(sizes[:sample])
        if args.create:
            _, _, dtc = benchlib.oracle_encode(plain_np, p_offs[:sample + 1], 2, 3, 1, 1, KEY, ncpu)
            cpu_create = {"value": Us / dtc / 1e9, "unit": "GB/s", "cores": ncpu, "kind": "port",
                          "sample": f"{sample} x 4 MiB entries, oracle encode (libzstd level 3 streaming + OpenSSL AES-256-CTR), {ncpu} threads"}
        cpu = {"value": Us / dt / 1e9, "unit": "GB/s", "cores": ncpu, "kind": "port",
               "sample": f"{sample} x 4 MiB entries x3 passes (oracle: libzstd + OpenSSL AES-NI + PCLMULQDQ folding chunk CRC as crc32fast; "
                         f"1 iterating/CRC thread + {ncpu} worker threads, reference extract dataflow)",
               "with_zlib_table_crc_GBps": Us / dtz / 1e9, "with_half_the_workers_GBps": Us / dth / 1e9,
               "single_core": benchlib.single_core_rates(files[0] * 8, KEY), "box": cpu_box()}

    # ---- BASELINE.json configs 1, 3, 4, 5 at their stated sizes (N = 1 only; each with value, e2e, cpu_baseline, parity check)
    configs = None
    if run_configs and rank == 0:
        del archive
        ctx.pinned_free(archive_buf)
        ctx.pinned_free(out_pinned)
        del archive_buf, out_pinned
        import benchcfg
        configs = benchcfg.run_all(pna, host, ctx, all_files, threads, args.config_scale, workers)

    if world > 1:
        barrier()
        dist.destroy_process_group()
    if rank != 0:
        return
    peaks = {}
    try:
        peaks = json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))
    except Exception:
        pass
    peak = float(peaks.get("hbm_gbs", 6650.0))
    # per-stage algorithmic bytes (DESIGN.md): seq = bitstreams in (<= C) + 8 B records out; lz = records + literals in, U out
    alg = {"crc": Cbytes, "cipher": 2 * Cbytes, "zstd_scan": 0, "zstd_seq": Cbytes + 8 * counts["sequences"],
           "zstd_lit": Cbytes + counts["literal_bytes"], "zstd_prefix": 0,
           "zstd_lz": 8 * counts["sequences"] + counts["literal_bytes"] + U, "inflate": 0, "store": 0}
    dom = max(stage_ms, key=lambda k: stage_ms[k])
    step_alg = Cbytes + U                           # fully fused accounting: ciphertext read once, plaintext written once
    dom_ms = stage_ms[dom]
    roof = {"bound": "hbm", "kernel": dom, "achieved": alg[dom] / (dom_ms * 1e-3) / 1e9 if dom_ms > 0 else None, "peak": peak,
            "unit": "GB/s", "peak_source": "measured (MEASURED_PEAKS.json hbm_gbs)" if peaks else "fallback 6650",
            "traffic": None, "stage_ms": stage_ms, "stage_share": {k: v / sum(stage_ms.values()) for k, v in stage_ms.items()},
            "stage_frac_of_peak": {k: (alg[k] / (v * 1e-3) / 1e9 / peak if v > 0.01 and alg.get(k) else None) for k, v in stage_ms.items()},
            "step_algorithmic_GBps": step_alg / (ms_step * 1e-3) / 1e9, "step_frac": step_alg / (ms_step * 1e-3) / 1e9 / peak}
    roof["frac"] = roof["achieved"] / peak if roof["achieved"] else None
    roof["algorithmic_bytes"] = alg[dom]
    try:   # DRAM bytes of the dominant kernel per launch from the committed ncu --set full capture of this same configuration
        tr = None
        for name in ("r2_traffic.json", "r1_traffic.json"):
            pth = os.path.join(ROOT, "profiles", name)
            if os.path.exists(pth):
                tr = (name, json.load(open(pth)))
                break
        k = tr[1]["kernels"].get(dom + "_kernel") if tr else None
        if k and E == 1024:
            roof["traffic"] = k["dram_read_bytes"] + k["dram_write_bytes"]
            roof["traffic_source"] = f"profiles/{tr[0]} (ncu --set full, one launch, same --entries)"
    except Exception:
        pass
    value = world * U / (ms_step * 1e-3) / 1e9
    line = {"metric": "extract_uncompressed_GBps", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
            "dtype": "u8", "data": "synthetic", "config": dict(cfg, compressed_bytes_per_gpu=Cbytes, plain_bytes_per_gpu=U,
                                                             ratio=U / Cbytes, host_cpus_per_rank=threads, e2e_workers=workers),
            "clocks": clocks, "gpu_launches": launches,
            "e2e": {"value": world * U / e2e_s / 1e9, "unit": "GB/s", "h2d_bytes_per_step": arch_bytes * world,
                    "d2h_bytes_per_step": int(U) * world, "ms_per_step": e2e_s * 1e3, "ms_all_steps_rank0": [round(t * 1e3, 2) for t in e2e_times], "pcie": pcie,
                    "path": f"pna::Archive::read_header_from_slice + extract_files (C++ host layer, {workers} worker threads x 2 contexts, {args.group_mib} MiB entry groups software-pipelined create->run->fetch): index pass, H2D, chunk CRC check, decrypt, decode, D2H to pinned buffers; host clock"},
            "roofline": roof}
    if cpu:
        line["cpu_baseline"] = cpu
    if create:
        if cpu_create:
            create["cpu_baseline"] = cpu_create
        line["create"] = create
    if configs:
        line["configs"] = configs
    print(json.dumps(line))


if __name__ == "__main__":
    main()
