#!/usr/bin/env python
"""bench.py -- BASELINE.json metric: Inflate GB/s (uncompressed) on 1 GiB synthetic DEFLATE @1/2/4/8 GPU vs the CPU path.

  python bench.py --gpus N --steps K --warmup W [--config 2|3|4|5] [--impl reference] [--dump-outputs DIR]

Default = BASELINE config 2 (SURVEY.md 8d): 16 384 gzip members x 64 KiB of synthetic wiki-like text, one dynamic-Huffman
block per member, ~394 MiB compressed -> 1 GiB, per GPU.  One JSON line on rank 0:

  value      device-resident (compressed members already in HBM -> decoded bytes in HBM; b200z_inflate_batch_device),
             CUDA events on the launching stream, max over ranks.
             N > 1 (one process per GPU, members dealt to the ranks, weak scaling: every rank owns its own 1 GiB): the
             timed step is decode PLUS the reassembly north_star names -- the ranks' shards all-gathered over NVLink so that
             every GPU holds the whole stream in order.  The stream is cut into chunks (chunk-major: chunk c of the stream =
             the ranks' c-th shares side by side), so the all-gather of chunk c runs behind the decode of chunk c+1.
             `decode_only` carries the same step without the collective, `strong` the metric's fixed-size variant (1 GiB in
             total: every rank decodes 1/N of it, then the gather), `per_rank` what every rank measured by itself.
  e2e        the same metric through the reference-facing call GZipDecoderWeb.decodeBytes == b200z_gzip_decode(host in,
             host out): pinned host buffers, H2D + framing walk + kernels + D2H inside the timed region.
  roofline   HBM bound; algorithmic bytes = C + U per pass (compressed read once + output written once).
  cpu_baseline / --impl reference
             the C oracle (a restatement of the pure-Dart Inflate; the reference itself is Dart and no Dart SDK exists here
             or on the GPU box -- profiles/r2_dart_probe.txt) on the host cores: a pool of pinned threads made once, a
             bounded sample, best of 5.
  configs    (N = 1 only, --no-side-configs skips) the other BASELINE configs at their full sizes, each with value, e2e,
             roofline, cpu_baseline and a parity check: 3 Deflate level 6 on 256 MiB, 4 BZip2Decoder on 512 MiB of 900 kB
             blocks, 5 ZipDecoder on a 1024-member 4 GiB zip.  --config K makes K the line's own metric (4 and 5 shard over
             the ranks of a torchrun job).
  --dump-outputs DIR
             (config 2) after the timed steps, what the last step handed its caller, as float .npy files in DIR
             (dump_outputs): two builds run with the same arguments decode the same input and can be compared file by file.
"""
from __future__ import annotations

import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

UNIT = 65536
N_UNITS = int(os.environ.get("B200Z_BENCH_UNITS", 16384))
CACHE = os.environ.get("B200Z_CACHE", "/tmp/b200z_cache")
WORKLOAD2 = "gzip-multimember-64KiB-dynamic (BASELINE config 2)"


def config2_dict():
    """The `config` object of BOTH arms (the driver compares them key by key)."""
    return {"workload": WORKLOAD2, "units_per_gpu": N_UNITS, "unit_bytes": UNIT, "uncompressed_bytes_per_gpu": N_UNITS * UNIT,
            "sharding": "members dealt to the ranks (chunk-major), one all-gather of every chunk behind the next chunk's decode",
            "l2": "inputs larger than L2 (394 MiB in + 1 GiB out per pass vs 126 MB L2)"}


def peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        try:
            return float(json.load(open(p))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
        except Exception:
            pass
    return 6650.0, "fallback (B200_PROFILING.md)"


DUMP_UNITS = 128  # 128 units x 64 KiB of decoded bytes as float32: 32 MiB, so that a whole dump stays under 64 MB
DUMP_SEED = 0xB200


def dump_outputs(out_dir: str, full: np.ndarray, status: np.ndarray, out_len: np.ndarray, in_used: np.ndarray):
    """--dump-outputs: the arrays one step of b200z_inflate_batch_device returns, as .npy files in out_dir.
      status, out_len, in_used        float32 [units of this rank]; every value is below 2**24, so float32 holds it exactly
      decoded_sample                  float32 [DUMP_UNITS, UNIT]: the decoded bytes of whole 64 KiB units of the stream
                                      (N > 1: of the gathered stream), a fixed, seeded sample -- all of it would take 4 GiB
      decoded_sample_units            float64 [DUMP_UNITS]: which units of the stream those are (ascending)"""
    os.makedirs(out_dir, exist_ok=True)
    n_total = full.size // UNIT
    units = np.sort(np.random.default_rng(DUMP_SEED).choice(n_total, size=min(DUMP_UNITS, n_total), replace=False))
    arrays = {"status": status.astype(np.float32), "out_len": out_len.astype(np.float32), "in_used": in_used.astype(np.float32),
              "decoded_sample": full.reshape(n_total, UNIT)[units].astype(np.float32),
              "decoded_sample_units": units.astype(np.float64)}
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, name + ".npy"), a)


class ClockSampler:
    """nvidia-smi clocks + throttle reasons DURING the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index: int):
        self.index = index
        self.proc = None
        self.lines = []

    def start(self):
        q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
             "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
             "clocks_event_reasons.sw_power_cap")
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}",
                                          "--format=csv,noheader,nounits", "-lms", "25"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            self.t = threading.Thread(target=self._read, daemon=True)
            self.t.start()
        except Exception:
            self.proc = None

    def _read(self):
        for ln in self.proc.stdout:
            self.lines.append(ln.strip())

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        try:
            self.proc.wait(timeout=5)
        except Exception:
            self.proc.kill()
        sm, mx, reasons = [], [], set()
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        for ln in self.lines:
            f = [x.strip() for x in ln.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0]))
                mx.append(float(f[1]))
            except ValueError:
                continue
            for nm, v in zip(names, f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(nm)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


# ---------------------------------------------------------------------------------------------
# the CPU side: the oracle on a pool of pinned threads (oracle/bench_threads.c)
# ---------------------------------------------------------------------------------------------
class OrcJob(C.Structure):
    _fields_ = [("kind", C.c_int), ("arg", C.c_int), ("inp", C.c_void_p), ("in_len", C.c_size_t), ("out_len", C.c_size_t),
                ("status", C.c_int)]


JOB_GZIP, JOB_INFLATE, JOB_DEFLATE, JOB_BZ2_DECODE, JOB_BZ2_ENCODE = 0, 1, 2, 3, 4
_ORC = None


def load_oracle():
    global _ORC
    if _ORC is None:
        subprocess.run(["make", "-s", "-C", os.path.join(ROOT, "oracle")], check=False)
        _ORC = C.CDLL(os.path.join(ROOT, "oracle", "liboracle.so"))
        _ORC.orc_bench_jobs.restype = C.c_double
        _ORC.orc_set_runaway_limit(C.c_int64(1 << 40))
    return _ORC


def oracle_jobs(jobs, threads: int, repeats: int):
    """jobs = [(kind, arg, address, length)] -> (best seconds, [seconds of every repeat], bytes produced, statuses)."""
    L = load_oracle()
    arr = (OrcJob * len(jobs))()
    for j, (kind, arg, addr, ln) in zip(arr, jobs):
        j.kind, j.arg, j.inp, j.in_len = kind, arg, addr, ln
    times = (C.c_double * repeats)()
    best = L.orc_bench_jobs(arr, len(jobs), threads, repeats, times)
    return best, list(times), sum(j.out_len for j in arr), [j.status for j in arr]


def oracle_deflate_bytes(data: bytes, level: int) -> bytes:
    """(parity check of the side configs only)"""
    L = load_oracle()
    out, n, crc = C.POINTER(C.c_uint8)(), C.c_size_t(), C.c_uint32()
    st = L.orc_deflate_bytes(data, C.c_size_t(len(data)), level, 15, C.byref(out), C.byref(n), C.byref(crc))
    r = C.string_at(out, n.value)
    L.orc_free(out)
    assert st == 0
    return r


def gzip_member_jobs(blob: np.ndarray, member_off, n_units: int, threads: int):
    """One job per range of whole members (the reference decodes a range with one member loop); 4 ranges per thread."""
    n_units = min(n_units, len(member_off) - 1)
    per = max(1, n_units // max(1, threads * 4))
    jobs = []
    for a in range(0, n_units, per):
        b = min(a + per, n_units)
        lo, hi = int(member_off[a]), int(member_off[b])
        jobs.append((JOB_GZIP, 0, blob.ctypes.data + lo, hi - lo))
    return jobs, n_units


def cpu_baseline_config2(blob, moff, cores):
    blob = np.ascontiguousarray(blob)
    jobs, sample = gzip_member_jobs(blob, moff, min(len(moff) - 1, 128 * cores), cores)
    best, times, total, st = oracle_jobs(jobs, cores, 5)
    assert all(s == 0 for s in st) and total == sample * UNIT, (set(st), total)
    return {"value": total / best / 1e9, "unit": "GB/s", "cores": cores, "kind": "port",
            "sample": f"first {sample} members ({total >> 20} MiB out), best of 5 passes ({best:.3f} s; all: "
                      f"{[round(t, 3) for t in times]}), C oracle restating the pure-Dart GZipDecoderWeb/Inflate (no Dart SDK "
                      "on the box), a pool of pinned threads made once, member ranges dealt to them"}


def gpu_local_cpus(local_rank: int):
    """CPUs on the NUMA node the GPU's PCIe link hangs off (/sys/bus/pci/devices/<bdf>/local_cpulist), restricted to the
    CPUs this process may use; None when the box does not say.  One process per GPU bound to its GPU's node is how the
    end-to-end path is meant to be deployed: the pinned staging buffers are then allocated on the memory the DMA reaches
    without crossing the socket link."""
    try:
        import torch
        p = torch.cuda.get_device_properties(local_rank)
        bdf = "%04x:%02x:%02x.0" % (p.pci_domain_id, p.pci_bus_id, p.pci_device_id)
        txt = open(f"/sys/bus/pci/devices/{bdf}/local_cpulist").read().strip()
        cpus = set()
        for part in txt.split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus.update(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        cpus &= os.sched_getaffinity(0)
        return cpus or None
    except Exception:
        return None


# ---------------------------------------------------------------------------------------------
# --impl reference
# ---------------------------------------------------------------------------------------------
def run_reference(args, rank, world):
    """The reference's CPU implementation of the path on this box's host cores.  The reference is pure Dart and cannot run
    here (no Dart SDK, no network): the arm times the C oracle, a restatement of the same algorithm (kind "port"), with all
    host threads -- a pinned pool, a bounded sample of the arm's own workload per step."""
    if rank != 0:
        return
    from archive_b200 import synth
    cores = os.cpu_count() or 1
    if args.config != 2:
        return run_reference_side(args, cores)
    sample_units = int(os.environ.get("B200Z_REF_UNITS", min(N_UNITS, 256 * max(1, cores // 2))))
    w = synth.gzip_workload(sample_units, UNIT, stream0=0, cache_dir=CACHE)
    blob = np.ascontiguousarray(w["blob"])
    jobs, sample_units = gzip_member_jobs(blob, w["member_off"], sample_units, cores)
    if args.warmup > 0:
        oracle_jobs(jobs, cores, 1)
    best, times, total, st = oracle_jobs(jobs, cores, args.steps + 1)  # (the pool's first pass is its warm-up)
    assert all(s == 0 for s in st)
    steps = times[1:]
    t = sum(steps)
    val = total * len(steps) / t / 1e9
    line = {
        "impl": "reference", "metric": "inflate_uncompressed_GBps", "value": val, "unit": "GB/s", "n_gpus": args.gpus,
        "steps": args.steps, "warmup": args.warmup, "ms_per_step": 1e3 * t / len(steps), "higher_is_better": True,
        "scaling": "weak", "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": config2_dict(),
        "cpu_baseline": {"value": val, "unit": "GB/s", "cores": cores, "kind": "port",
                         "sample": f"{sample_units} members ({total >> 20} MiB out) per step, best step "
                                   f"{total / min(steps) / 1e9:.2f} GB/s, C oracle restating the pure-Dart GZipDecoderWeb/"
                                   "Inflate, a pool of pinned threads, member ranges dealt to them"},
        "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
    }
    print(json.dumps(line), flush=True)


# ---------------------------------------------------------------------------------------------
# the other BASELINE configs (side results of the default line; --config K makes one the line itself)
# ---------------------------------------------------------------------------------------------
def _timed_calls(fn, reps):
    ts = []
    for _ in range(reps):
        t0 = time.perf_counter()
        fn()
        ts.append(time.perf_counter() - t0)
    return ts


def side_config3(L, cores, reps=3):
    """Deflate level 6 on 256 MiB of the synthetic text through b200z_deflate_raw (host in, host out, pinned): the only
    entry point the encoder has, so value == e2e.  Parity: the first 32 MiB compressed alone are byte-identical to the
    oracle's Deflate(level: 6) of the same bytes; the full output inflates back to the input (CRC-32)."""
    from archive_b200 import _ffi, synth
    n = int(os.environ.get("B200Z_C3_MIB", 256)) << 20
    text = synth.text(n, stream=100)
    h_in = L.b200z_host_alloc(n)
    C.memmove(h_in, text.ctypes.data, n)
    cap = L.b200z_deflate_bound(n)
    h_out = L.b200z_host_alloc(cap)
    out_len, crc = C.c_size_t(0), C.c_uint32(0)

    def call(k=n):
        rc = L.b200z_deflate_raw(h_in, k, 6, 15, h_out, cap, C.byref(out_len), C.byref(crc))
        assert rc == 0, _ffi.last_error()

    call()
    ts = _timed_calls(call, reps)
    z = C.string_at(h_out, out_len.value)
    c_bytes = out_len.value
    ok_round = zlib.crc32(zlib.decompress(z, -15)) == zlib.crc32(text.tobytes()) == crc.value
    k = min(n, int(os.environ.get("B200Z_C3_ORACLE_MIB", 32)) << 20)
    call(k)
    mine = C.string_at(h_out, out_len.value)
    sample = np.ascontiguousarray(text[:k])
    best, times, total, st = oracle_jobs([(JOB_DEFLATE, 6, sample.ctypes.data, k)], 1, 1)
    identical = oracle_deflate_bytes(sample.tobytes(), 6) == mine
    L.b200z_host_free(h_in)
    L.b200z_host_free(h_out)
    dt = min(ts)
    peak, src = peaks()
    return {"workload": f"Deflate level 6, {n >> 20} MiB synthetic text, one stream (BASELINE config 3)",
            "metric": "deflate6_input_GBps", "value": n / dt / 1e9, "unit": "GB/s", "ms_per_step": dt * 1e3,
            "e2e": {"value": n / dt / 1e9, "unit": "GB/s", "h2d_bytes_per_step": n, "d2h_bytes_per_step": c_bytes,
                    "call": "b200z_deflate_raw(host in, host out) == Deflate(bytes, level: 6).getBytes(), pinned buffers"},
            "roofline": {"bound": "hbm", "achieved": (n + c_bytes) / dt / 1e9, "peak": peak, "unit": "GB/s",
                         "frac": (n + c_bytes) / dt / 1e9 / peak, "traffic": None, "peak_source": src,
                         "note": "algorithmic bytes U + C over the whole call (copies included: the encoder has no "
                                 "device-resident entry point)"},
            "cpu_baseline": {"value": k / best / 1e9, "unit": "GB/s", "cores": 1, "kind": "port",
                             "sample": f"first {k >> 20} MiB, {best:.2f} s, C oracle restating Deflate (one stream is one "
                                       "serial parse in the reference)"},
            "parity": {"identical_to_oracle": bool(identical), "sample": f"first {k >> 20} MiB compressed alone",
                       "full_output_inflates_to_input": bool(ok_round), "ratio": round(n / c_bytes, 3)}}


def make_bz2_stream(L, text: np.ndarray):
    from archive_b200 import _ffi
    m = text.size
    cap = L.b200z_bzip2_bound(m)
    zbuf = np.empty(cap, dtype=np.uint8)
    zl = C.c_size_t(0)
    rc = L.b200z_bzip2_encode(text.ctypes.data, m, zbuf.ctypes.data, cap, C.byref(zl))
    assert rc == 0, _ffi.last_error()
    return zbuf[:zl.value].copy()


def side_config4(L, cores, world=1, rank=0, dist=None, reps=3):
    """BZip2Decoder(verify) on 512 MiB of text in 900 kB blocks (one BZh9 stream, written by the device encoder whose bytes
    the tests pin to the oracle's).  N = 1: b200z_bzip2_decode host -> host.  N > 1: blocks sharded over the ranks
    (shard.bzip2_decode_sharded: per-block reports exchanged, decoded bytes stay on the rank that produced them)."""
    from archive_b200 import _ffi, shard, synth
    m = int(os.environ.get("B200Z_C4_MIB", 512)) << 20
    text = synth.text(m, stream=200)
    z = make_bz2_stream(L, text)
    h_z = L.b200z_host_alloc(z.size)
    C.memmove(h_z, z.ctypes.data, z.size)
    if world == 1:
        src_crc = zlib.crc32(text.tobytes())
        h_o = L.b200z_host_alloc(m + 1024)
        ol = C.c_size_t(0)

        def call():
            rc = L.b200z_bzip2_decode(h_z, z.size, 1, h_o, m + 1024, C.byref(ol))
            assert rc == 0, _ffi.last_error()

        call()
        ts = _timed_calls(call, reps)
        ok = ol.value == m and zlib.crc32(C.string_at(h_o, m)) == src_crc
        L.b200z_host_free(h_o)
        dt = min(ts)
    else:
        import torch
        gloo = dist.new_group(backend="gloo")
        ocap = m // world + (64 << 20)
        h_o = L.b200z_host_alloc(ocap)
        zv = (C.c_uint8 * z.size).from_address(h_z)
        ts, r = [], None
        for i in range(reps + 1):
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            r = shard.bzip2_decode_sharded(zv, verify=True, group=gloo, out_buf=(h_o, ocap))
            torch.cuda.synchronize()
            dist.barrier()
            ts.append(time.perf_counter() - t0)
        ok = r["kind"] == "ok" and r["total"] == m
        for off, v in r["pieces"]:
            ok = ok and zlib.crc32(v) == zlib.crc32(text[off:off + len(v)].tobytes())
        t = torch.tensor([min(ts[1:]), 0.0 if ok else 1.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt, ok = float(t[0]), float(t[1]) == 0.0
        L.b200z_host_free(h_o)
    L.b200z_host_free(h_z)
    peak, src = peaks()
    res = {"workload": f"BZip2Decoder(verify), {m >> 20} MiB of text in 900 kB blocks, one BZh9 stream (BASELINE config 4)",
           "metric": "bzip2_decode_uncompressed_GBps", "value": m / dt / 1e9, "unit": "GB/s", "ms_per_step": dt * 1e3, "n_gpus": world,
           "scaling": "strong",
           "e2e": {"value": m / dt / 1e9, "unit": "GB/s", "h2d_bytes_per_step": int(z.size) * world, "d2h_bytes_per_step": m,
                   "call": "b200z_bzip2_decode(host in, host out)" if world == 1 else
                           "b200z_bzip2_decode_shard per rank (every rank scans the stream, decodes its blocks)"},
           "roofline": {"bound": "hbm", "achieved": (m + int(z.size)) / dt / 1e9, "peak": peak, "unit": "GB/s",
                        "frac": (m + int(z.size)) / dt / 1e9 / peak, "traffic": None, "peak_source": src,
                        "note": "algorithmic bytes C + U over the whole call (host copies included)"},
           "parity": {"output_equals_source": bool(ok), "blocks": (m + 899980) // 899981}}
    if rank == 0:
        k = int(os.environ.get("B200Z_C4_ORACLE_MIB", 24)) << 20
        zs = make_bz2_stream(L, np.ascontiguousarray(text[:k]))
        best, times, total, st = oracle_jobs([(JOB_BZ2_DECODE, 1, zs.ctypes.data, zs.size)], 1, 1)
        res["cpu_baseline"] = {"value": total / best / 1e9, "unit": "GB/s", "cores": 1, "kind": "port",
                               "sample": f"a {k >> 20} MiB stream of the same text, {best:.2f} s, C oracle restating "
                                         "BZip2Decoder (one stream is one serial loop in the reference)"}
        res["parity"]["oracle_decodes_sample_to_source_size"] = bool(st[0] == 0 and total == k)
    return res


def _zip_member_job(a):
    """One member of the synthetic zip, made where it is compressed (nothing but the compressed bytes crosses a pipe)."""
    i, size, stream = a
    from archive_b200 import synth
    b = synth.text(size, stream=stream + i).tobytes()
    return synth.deflate_raw_flushed(b, 65536), zlib.crc32(b)


def make_zip(n_members: int, size: int, stream: int = 7000):
    from concurrent.futures import ProcessPoolExecutor
    from archive_b200 import synth
    with ProcessPoolExecutor(max_workers=min(96, os.cpu_count() or 1)) as ex:
        parts = list(ex.map(_zip_member_job, [(i, size, stream) for i in range(n_members)], chunksize=2))
    data = synth.zip_from_deflated([(f"member{i:04d}.txt", z, crc, size) for i, (z, crc) in enumerate(parts)])
    return data, [crc for _, crc in parts]


def side_config5(L, cores, world=1, rank=0, dist=None, reps=3):
    """ZipDecoder end to end on a 1024-member x 4 MiB synthetic .zip (method 8, a full-flush point every 64 KiB -- still one
    valid DEFLATE stream per member): b200z_zip_list + ONE b200z_zip_extract call, host in, host out.  N > 1: the members are
    packed onto the ranks (shard.pack_members), every rank extracts its share."""
    from archive_b200 import _ffi, shard
    n = int(os.environ.get("B200Z_C5_MEMBERS", 1024))
    size = int(os.environ.get("B200Z_C5_MEMBER_MIB", 4)) << 20
    data, crcs = make_zip(n, size)
    zl = len(data)
    h_in = L.b200z_host_alloc(zl)
    C.memmove(h_in, data, zl)
    cnt = C.c_size_t(0)
    ents = (_ffi.ZipEntry * n)()
    assert L.b200z_zip_list(h_in, zl, ents, n, C.byref(cnt)) == 0 and cnt.value == n
    mine = list(range(n)) if world == 1 else shard.pack_members([ents[i].comp_size for i in range(n)], world)[rank]
    k = len(mine)
    sub = (_ffi.ZipEntry * k)(*[ents[i] for i in mine])
    tot = k * size
    h_out = L.b200z_host_alloc(max(tot, 1))
    off = (C.c_uint64 * k)(*[j * size for j in range(k)])
    room = (C.c_uint64 * k)(*[size] * k)
    ol, st = (C.c_uint64 * k)(), (C.c_int32 * k)()

    def call():
        rc = L.b200z_zip_extract(h_in, zl, sub, k, h_out, tot, off, room, ol, st, 0)
        assert rc == 0, _ffi.last_error()

    if world > 1:
        import torch
        ts = []
        for i in range(reps + 1):
            dist.barrier()
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            call()
            torch.cuda.synchronize()
            dist.barrier()
            ts.append(time.perf_counter() - t0)
        ts = ts[1:]
    else:
        call()
        ts = _timed_calls(call, reps)
    out = np.ctypeslib.as_array((C.c_uint8 * tot).from_address(h_out))
    ok = all(s == 0 for s in st) and all(o == size for o in ol)
    ok = ok and all(zlib.crc32(out[j * size:(j + 1) * size].tobytes()) == crcs[mine[j]] for j in range(0, k, 7))
    dt = min(ts)
    if world > 1:
        import torch
        t = torch.tensor([dt, 0.0 if ok else 1.0], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        dt, ok = float(t[0]), float(t[1]) == 0.0
    U = n * size
    peak, src = peaks()
    res = {"workload": f"ZipDecoder on a {n}-member x {size >> 20} MiB synthetic .zip, method 8, full-flush points every 64 KiB "
                       "(BASELINE config 5)",
           "metric": "zip_extract_uncompressed_GBps", "value": U / dt / 1e9, "unit": "GB/s", "ms_per_step": dt * 1e3, "n_gpus": world,
           "scaling": "strong",
           "e2e": {"value": U / dt / 1e9, "unit": "GB/s", "h2d_bytes_per_step": zl * world, "d2h_bytes_per_step": U,
                   "call": "b200z_zip_extract(host zip, host out): every member of the rank's share in one call"},
           "roofline": {"bound": "hbm", "achieved": (U + zl) / dt / 1e9, "peak": peak, "unit": "GB/s", "frac": (U + zl) / dt / 1e9 / peak,
                        "traffic": None, "peak_source": src, "note": "algorithmic bytes C + U over the whole call (host copies included)"},
           "parity": {"members_ok_crc32": bool(ok), "checked": "status / size of every member, CRC-32 of every 7th against the generator's"}}
    if rank == 0:
        ks = min(n, 4 * cores)
        arr = np.frombuffer(data, dtype=np.uint8)
        jobs = [(JOB_INFLATE, 0, arr.ctypes.data + ents[i].data_off, ents[i].comp_size) for i in range(ks)]
        best, times, total, sts = oracle_jobs(jobs, cores, 3)
        res["cpu_baseline"] = {"value": total / best / 1e9, "unit": "GB/s", "cores": cores, "kind": "port",
                               "sample": f"{ks} members ({total >> 20} MiB out), best of 2 passes ({best:.2f} s), C oracle "
                                         "restating Inflate, one member per job on a pool of pinned threads"}
        res["parity"]["oracle_inflates_sample_members"] = bool(all(s == 0 for s in sts) and total == ks * size)
    L.b200z_host_free(h_in)
    L.b200z_host_free(h_out)
    return res


def run_reference_side(args, cores):
    """--impl reference --config 3|4|5: the oracle on a bounded sample of that config's workload."""
    from archive_b200 import synth
    cfg = args.config
    if cfg == 3:
        k = 16 << 20
        text = np.ascontiguousarray(synth.text(k, stream=100))
        jobs, threads, metric, per = [(JOB_DEFLATE, 6, text.ctypes.data, k)], 1, "deflate6_input_GBps", k
        wl = "Deflate level 6 (BASELINE config 3), 16 MiB sample of the 256 MiB text, one stream"
    elif cfg == 4:
        import bz2
        k = 16 << 20
        text = synth.text(k, stream=200).tobytes()
        z = np.frombuffer(bz2.compress(text, 9), dtype=np.uint8).copy()
        jobs, threads, metric, per = [(JOB_BZ2_DECODE, 1, z.ctypes.data, z.size)], 1, "bzip2_decode_uncompressed_GBps", k
        wl = "BZip2Decoder(verify) (BASELINE config 4), a 16 MiB stream of the same text"
    else:
        ks, size = 2 * cores, 4 << 20
        text = synth.text(ks * size, stream=700)
        zs = [np.frombuffer(synth.deflate_raw_flushed(text[i * size:(i + 1) * size].tobytes(), 65536), dtype=np.uint8).copy()
              for i in range(ks)]
        jobs = [(JOB_INFLATE, 0, z.ctypes.data, z.size) for z in zs]
        threads, metric, per = cores, "zip_extract_uncompressed_GBps", ks * size
        wl = f"ZipDecoder members (BASELINE config 5), {ks} members x 4 MiB"
    best, times, total, st = oracle_jobs(jobs, threads, args.steps + 1)
    steps = times[1:]
    val = per * len(steps) / sum(steps) / 1e9
    print(json.dumps({"impl": "reference", "metric": metric, "value": val, "unit": "GB/s", "n_gpus": args.gpus, "steps": args.steps,
                      "warmup": args.warmup, "ms_per_step": 1e3 * sum(steps) / len(steps), "higher_is_better": True, "scaling": "strong",
                      "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": {"workload": wl},
                      "cpu_baseline": {"value": val, "unit": "GB/s", "cores": threads, "kind": "port", "sample": wl},
                      "e2e": {"value": val, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}), flush=True)


# ---------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200z")
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5])
    ap.add_argument("--no-e2e", action="store_true")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-side-configs", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write what the last timed step computed to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and (args.impl == "reference" or args.config != 2):
        ap.error("--dump-outputs dumps the config 2 decode of the GPU arm")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    if args.impl == "reference":
        run_reference(args, rank, world)
        return
    args.warmup = max(args.warmup, 3)

    import torch
    import torch.distributed as dist
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- the product path has no CPU fallback")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        # the collective's kernel has to get onto the SMs BESIDE the decode of the next chunk (whose persistent CTAs would
        # otherwise take every SM the moment the previous chunk drains): NCCL's stream gets the higher priority
        opts = None
        try:
            opts = dist.ProcessGroupNCCL.Options(is_high_priority_stream=True)
        except Exception:
            pass
        dist.init_process_group("nccl", device_id=dev, pg_options=opts)

    from archive_b200 import _ffi, synth
    L = _ffi.ensure_init(local_rank)
    cores = os.cpu_count() or 1

    if args.config != 2:
        fn = {3: side_config3, 4: side_config4, 5: side_config5}[args.config]
        sampler = ClockSampler(local_rank)
        if rank == 0:
            sampler.start()
        launches0 = L.b200z_launch_count()
        ranks = () if args.config == 3 else (world, rank, dist if world > 1 else None)
        res = fn(L, cores, *ranks, reps=args.steps)
        launches = L.b200z_launch_count() - launches0
        clocks = sampler.stop() if rank == 0 else None
        if rank == 0:
            line = {"metric": res.pop("metric"), "value": res.pop("value"), "unit": res.pop("unit"), "n_gpus": world, "steps": args.steps,
                    "warmup": 1, "ms_per_step": res.pop("ms_per_step"), "higher_is_better": True, "scaling": res.pop("scaling", "strong"),
                    "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": {"workload": res.pop("workload")},
                    "gpu_launches": int(launches), "clocks": clocks}
            line.update(res)
            print(json.dumps(line), flush=True)
        if world > 1:
            dist.destroy_process_group()
        return

    # ---------------- workload: every rank owns its own re-drawn 1 GiB (weak scaling) ----------------
    t_gen = time.time()
    stream0 = int(os.environ.get("B200Z_BENCH_STREAM0", rank * 4096))  # (every rank its own re-drawn text)
    w = synth.gzip_workload(N_UNITS, UNIT, stream0=stream0, cache_dir=CACHE)
    blob, moff = w["blob"], w["member_off"]
    n = N_UNITS
    hdr = 18  # synth.gzip_member with the BC hint: 10 + 2 + 6
    in_off = (moff[:-1] + hdr).astype(np.uint64)
    in_len = (moff[1:] - moff[:-1] - hdr).astype(np.uint32)  # member payload incl. the 8-byte trailer
    C_bytes, U_bytes = int(len(blob)), n * UNIT
    gen_s = time.time() - t_gen
    # the stream every GPU ends up holding, chunk-major: chunk c = the ranks' c-th shares side by side
    NCH = 4 if world > 1 else 1
    upc = n // NCH                       # units per rank per chunk
    cb = upc * UNIT                      # bytes per rank per chunk
    unit_idx = np.arange(n)
    out_off = ((unit_idx // upc) * (world * cb) + rank * cb + (unit_idx % upc) * UNIT).astype(np.uint64)
    out_cap = np.full(n, UNIT, dtype=np.uint32)

    d_in = torch.empty(C_bytes + 64, dtype=torch.uint8, device=dev)
    d_in[:C_bytes].copy_(torch.from_numpy(blob.copy()))
    d_full = torch.empty(world * U_bytes, dtype=torch.uint8, device=dev)
    d_in_off = torch.from_numpy(in_off.view(np.int64)).to(dev)
    d_in_len = torch.from_numpy(in_len.view(np.int32)).to(dev)
    d_out_off = torch.from_numpy(out_off.view(np.int64)).to(dev)
    d_out_cap = torch.from_numpy(out_cap.view(np.int32)).to(dev)
    d_out_len = torch.zeros(n, dtype=torch.int32, device=dev)
    d_status = torch.full((n,), -99, dtype=torch.int32, device=dev)
    d_used = torch.zeros(n, dtype=torch.int32, device=dev)
    # (the workspace mirrors the output layout the batch addresses: a chunk's units sit inside world * cb bytes)
    ws_bytes = L.b200z_inflate_workspace_bytes(upc, C_bytes, world * cb)
    d_ws = torch.empty(ws_bytes, dtype=torch.uint8, device=dev)
    stream = torch.cuda.Stream(device=dev)  # a real (non-NULL) stream: the library launches on it, the events time it
    torch.cuda.set_stream(stream)
    chunk_out_off = torch.from_numpy((out_off - (unit_idx // upc).astype(np.uint64) * np.uint64(world * cb)).view(np.int64)).to(dev)

    def decode_chunk(c, units=upc):
        a = c * upc
        rc = L.b200z_inflate_batch_device(d_in.data_ptr(), d_in_off.data_ptr() + 8 * a, d_in_len.data_ptr() + 4 * a,
                                          d_full.data_ptr() + c * world * cb, chunk_out_off.data_ptr() + 8 * a,
                                          d_out_cap.data_ptr() + 4 * a, d_out_len.data_ptr() + 4 * a, d_status.data_ptr() + 4 * a,
                                          d_used.data_ptr() + 4 * a, units, d_ws.data_ptr(), ws_bytes, stream.cuda_stream)
        if rc:
            raise RuntimeError(_ffi.last_error())

    def step_decode_only():
        for c in range(NCH):
            decode_chunk(c)

    def step():  # decode + reassembly: the all-gather of chunk c runs behind the decode of chunk c + 1
        if world == 1:
            return step_decode_only()
        works = []
        for c in range(NCH):
            decode_chunk(c)
            full_c = d_full[c * world * cb:(c + 1) * world * cb]
            works.append(dist.all_gather_into_tensor(full_c, full_c[rank * cb:(rank + 1) * cb], async_op=True))
        for wk in works:
            wk.wait()

    spr = n // world // NCH if world > 1 else 0  # strong scaling: units per rank per chunk of a 1 GiB stream

    def step_strong():  # 1 GiB in total: every rank decodes 1/N of it, chunk by chunk, and the shards are gathered
        works = []
        sb = spr * UNIT
        for c in range(NCH):
            decode_chunk(c, spr)  # (the first spr units of the rank's c-th share: they land at rank * cb of chunk c)
            full_c = d_full[c * world * cb:(c + 1) * world * cb]
            for r in range(world):  # shards of spr units sit cb apart: one broadcast per shard == an all-gather of strided pieces
                works.append(dist.broadcast(full_c[r * cb:r * cb + sb], src=r, async_op=True))
        for wk in works:
            wk.wait()

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def timed(fn, steps, warmup):
        for _ in range(warmup):
            fn()
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            fn()
        e1.record()
        barrier()
        ms_own = e0.elapsed_time(e1)
        ms = ms_own
        if world > 1:
            t = torch.tensor([ms], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            ms = float(t.item())
        return ms, ms_own

    # ---------------- device-resident timing ----------------
    sampler = ClockSampler(local_rank)
    sampler.start()
    L.b200z_profile_enable(0)
    launches0 = L.b200z_launch_count()
    ms_total, ms_own = timed(step, args.steps, args.warmup)
    launches = (L.b200z_launch_count() - launches0) * args.steps // (args.steps + args.warmup)  # timed steps only
    ms_step = ms_total / args.steps
    value = world * U_bytes / (ms_step * 1e-3) / 1e9
    my_clocks = sampler.stop()

    # correctness gate on what the timed region produced: status, lengths, and CRC-32 against the trailers
    st = d_status.cpu().numpy()
    ol = d_out_len.cpu().numpy()
    us = d_used.cpu().numpy()
    assert (st == 0).all(), f"unit status {np.unique(st)}"
    assert (ol == UNIT).all()
    assert (us.astype(np.int64) + 8 == in_len.astype(np.int64)).all()
    check_idx = np.linspace(0, n - 1, 512).astype(int)
    host_full = d_full.cpu().numpy()
    for i in check_idx:
        m_end = int(moff[i + 1])
        crc = int.from_bytes(blob[m_end - 8:m_end - 4].tobytes(), "little")
        o = int(out_off[i])
        assert zlib.crc32(host_full[o:o + UNIT].tobytes()) == crc, f"unit {i} CRC mismatch"
    gathered_ok = None
    if world > 1:  # the gathered stream: every rank's share of every chunk is what that rank decoded (CRC of a sample, exchanged)
        def piece(r, c):
            return host_full[c * world * cb + r * cb:c * world * cb + r * cb + 4 * UNIT].tobytes()
        mine = torch.tensor([zlib.crc32(piece(rank, c)) for c in range(NCH)], dtype=torch.int64, device=dev)
        allc = [torch.zeros_like(mine) for _ in range(world)]
        dist.all_gather(allc, mine)
        gathered_ok = all(zlib.crc32(piece(r, c)) == int(allc[r][c]) for r in range(world) for c in range(NCH))
        assert gathered_ok, "the gathered stream differs from what its owners decoded"
    if args.dump_outputs and rank == 0:
        dump_outputs(args.dump_outputs, host_full, st, ol, us)
    del host_full

    # per-kernel breakdown (separate pass so event records do not sit inside the headline region)
    L.b200z_profile_enable(1)
    for _ in range(args.steps):
        step_decode_only()
    torch.cuda.synchronize()
    fms, dms, ems, nb = C.c_double(), C.c_double(), C.c_double(), C.c_uint64()
    L.b200z_profile_read(C.byref(fms), C.byref(dms), C.byref(ems), C.byref(nb))
    L.b200z_profile_enable(0)
    k_fast, k_dec, k_exp = (v.value / args.steps for v in (fms, dms, ems))

    # the other inflate kernel on the same step (the library reads B200Z_FAST at every launch)
    was = os.environ.get("B200Z_FAST")
    other = "0" if (was or "1") != "0" else "1"
    os.environ["B200Z_FAST"] = other
    try:
        ms_a, _ = timed(step_decode_only, args.steps, args.warmup)
        alt = {"kernel": "k_inflate_fast, one CTA per unit in shared memory (B200Z_FAST=1)" if other == "1"
               else "k_inflate_decode + k_inflate_expand (B200Z_FAST=0)",
               "value": world * U_bytes / (ms_a / args.steps * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": ms_a / args.steps,
               "all_units_ok": bool((d_status.cpu().numpy() == 0).all()),
               "dram_bytes_per_pass": 1431698328 if other == "1" else 6980970000,
               "note": "decode only, same buffers; DRAM bytes from profiles/ (ncu)"}
    finally:
        if was is None:
            del os.environ["B200Z_FAST"]
        else:
            os.environ["B200Z_FAST"] = was

    decode_only = strong = per_rank = None
    if world > 1:
        ms_d, ms_d_own = timed(step_decode_only, args.steps, args.warmup)
        decode_only = {"value": world * U_bytes / (ms_d / args.steps * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": ms_d / args.steps}
        ms_s, _ = timed(step_strong, args.steps, args.warmup)
        strong = {"value": (world * NCH * spr * UNIT) / (ms_s / args.steps * 1e-3) / 1e9, "unit": "GB/s", "ms_per_step": ms_s / args.steps,
                  "scaling": "strong", "total_bytes": world * NCH * spr * UNIT, "units_per_rank": NCH * spr,
                  "note": "the metric's fixed size: 1 GiB in total, every rank decodes 1/N of it and the shards are gathered "
                          "(one broadcast per shard) so that every GPU holds the GiB"}
        mine = {"rank": rank, "ms_per_step": ms_own / args.steps, "decode_only_ms_per_step": ms_d_own / args.steps,
                "k_inflate_fast_ms": k_fast, "k_inflate_decode_ms": k_dec, "k_inflate_expand_ms": k_exp,
                "sm_mhz": my_clocks.get("sm_mhz"), "reasons": my_clocks.get("reasons"), "compressed_bytes": C_bytes}
        per_rank = [None] * world
        dist.all_gather_object(per_rank, mine)

    # ---------------- end to end through the reference-facing call, host buffers ----------------
    e2e = None
    if not args.no_e2e:
        all_cpus = os.sched_getaffinity(0)
        near = gpu_local_cpus(local_rank)
        if near and near != all_cpus:
            os.sched_setaffinity(0, near)  # for the staging buffers' placement and the calling thread; undone below
        h_in = torch.empty(C_bytes, dtype=torch.uint8).pin_memory()
        h_in.numpy()[:] = blob
        h_out = torch.empty(U_bytes, dtype=torch.uint8).pin_memory()
        out_len = C.c_size_t(0)

        def e2e_step():
            rc = L.b200z_gzip_decode(h_in.data_ptr(), C_bytes, 0, h_out.data_ptr(), U_bytes, C.byref(out_len))
            if rc:
                raise RuntimeError(_ffi.last_error())

        for _ in range(2):
            e2e_step()
        barrier()
        t0 = time.perf_counter()
        k = max(3, min(args.steps, 10))
        for _ in range(k):
            e2e_step()
        torch.cuda.synchronize()
        dt = (time.perf_counter() - t0) / k
        if world > 1:
            t = torch.tensor([dt], dtype=torch.float64, device=dev)
            dist.all_reduce(t, op=dist.ReduceOp.MAX)
            dt = float(t.item())
        assert out_len.value == U_bytes
        ho = h_out.numpy()
        for i in check_idx[::16]:
            m_end = int(moff[i + 1])
            crc = int.from_bytes(blob[m_end - 8:m_end - 4].tobytes(), "little")
            assert zlib.crc32(ho[i * UNIT:(i + 1) * UNIT].tobytes()) == crc
        e2e = {"value": world * U_bytes / dt / 1e9, "unit": "GB/s", "h2d_bytes_per_step": C_bytes,
               "d2h_bytes_per_step": U_bytes, "ms_per_step": dt * 1e3,
               "call": "b200z_gzip_decode(host in, host out) == GZipDecoderWeb.decodeBytes, pinned host buffers",
               "cpu_binding": ("%d CPUs of the GPU's NUMA node" % len(near)) if near and near != all_cpus else "none"}
        if near and near != all_cpus:
            os.sched_setaffinity(0, all_cpus)
        del h_in, h_out

    # ---------------- CPU baseline beside it (rank 0, every N; bounded sample) ----------------
    cpu = None
    if rank == 0 and not args.no_cpu_baseline:
        cpu = cpu_baseline_config2(blob, moff, cores)

    # ---------------- the other configs (N = 1) ----------------
    configs = None
    if rank == 0 and world == 1 and not args.no_side_configs:
        del d_in, d_full, d_ws
        torch.cuda.empty_cache()
        configs = {}
        for k_, fn in (("3", side_config3), ("4", side_config4), ("5", side_config5)):
            try:
                t0 = time.time()
                configs[k_] = fn(L, cores)
                configs[k_]["wall_s"] = round(time.time() - t0, 1)
            except Exception as ex:  # a side config must not take the headline down with it
                configs[k_] = {"error": repr(ex)[:300]}

    if rank == 0:
        peak, peak_src = peaks()
        kernel_s = (k_fast + k_dec + k_exp) * 1e-3
        achieved = (C_bytes + U_bytes) / kernel_s / 1e9
        traffic = None
        tp = os.path.join(ROOT, "profiles", "traffic.json")
        if os.path.exists(tp):
            try:
                traffic = json.load(open(tp)).get("dram_bytes_per_pass")
            except Exception:
                traffic = None
        cfg = config2_dict()
        line = {
            "metric": "inflate_uncompressed_GBps", "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_step, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "u8", "data": "synthetic", "config": cfg,
            "workload_facts": {"compressed_bytes_per_gpu": C_bytes, "chunks": NCH, "generate_s": round(gen_s, 1), "text_stream0": stream0,
                               "B200Z_FAST": os.environ.get("B200Z_FAST", "1 (default)"),
                               "B200Z_FAST_SPARE_SMS": os.environ.get("B200Z_FAST_SPARE_SMS", "0 (default)")},
            "e2e": e2e, "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic, "peak_source": peak_src,
                         "algorithmic_bytes_per_pass": C_bytes + U_bytes,
                         "kernels": {"k_inflate_fast_ms": k_fast, "k_inflate_decode_ms": k_dec, "k_inflate_expand_ms": k_exp},
                         "note": "one pass = k_inflate_fast (clean units, all in shared memory) + the exact pair k_inflate_decode / "
                                 "k_inflate_expand over what it leaves (nothing on this workload); achieved = (C+U) / their "
                                 "CUDA-event time; traffic = ncu DRAM bytes of k_inflate_fast per pass (profiles/traffic.json)"},
            "cpu_baseline": cpu, "clocks": my_clocks, "alt_kernel": alt,
        }
        if world > 1:
            line["collective"] = {"what": "all_gather_into_tensor of every chunk (NCCL over NVLink), in place, behind the next "
                                          "chunk's decode", "bytes_received_per_rank_per_step": (world - 1) * U_bytes,
                                  "gathered_stream_checked": gathered_ok}
            line["decode_only"] = decode_only
            line["strong"] = strong
            line["per_rank"] = per_rank
        if configs is not None:
            line["configs"] = configs
        print(json.dumps(line), flush=True)
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
