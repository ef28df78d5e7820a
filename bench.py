#!/usr/bin/env python3
"""bench.py -- zstd block-encode throughput (input GB/s) on N B200s, BASELINE.json's metric.

A step = one pass of the hot path over one batch per GPU:
  --level 1 (default)  16384 synthetic-text chunks of 64 KiB = 1 GiB per GPU, SpeedFastest (BASELINE config 2)
  --level 2            8192 chunks of 128 KiB = 1 GiB per GPU, SpeedDefault (BASELINE config 5: 8 GiB over 8 GPUs)
`value` is timed with CUDA events around K launches with inputs resident in HBM (inputs are 8x larger than L2, so no
cache flush is needed); `e2e` goes through the host-buffer C-ABI call with pinned host input/output (H2D + encode +
D2H inside the timed region) on the same number of chunks.  Multi-GPU: one process per GPU, bound to the GPU's NUMA
node, each with its own 1 GiB (weak scaling), no collective on the data path; time = max over ranks.
`--impl reference` (and `cpu_baseline` of the default arm) time the CPU oracle -- the C restatement of the reference's
Go encoder; the Go toolchain is absent -- on all host cores over ONE un-looped pass of rank 0's 1 GiB: the same bytes
the GPU arm encodes.
"""
import argparse
import ctypes
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.dont_write_bytecode = True    # runs from the built tree, which may be read-only: nothing is written into it
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tests"))

LEVELS = {1: {"chunk": 65536, "nchunks": 16384, "name": "SpeedFastest"},
          2: {"chunk": 131072, "nchunks": 8192, "name": "SpeedDefault"},
          3: {"chunk": 131072, "nchunks": 8192, "name": "SpeedBetterCompression"}}
DATA_SEED = 1000


def metric_name(level):
    return "zstd %s encode GB/s (input)" % LEVELS[level]["name"]


def hbm_peak():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        return float(json.load(open(p))["hbm_gbs"]), "measured"
    return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    def __init__(self, index):
        super().__init__(daemon=True)
        self.index = index
        self.rows = []
        self.stop = False

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), f"--query-gpu={q}", "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([x.strip() for x in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        import statistics
        sm = [float(r[0]) for r in self.rows if r and r[0].replace(".", "").isdigit()]
        mx = [float(r[1]) for r in self.rows if len(r) > 1 and r[1].replace(".", "").isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = [names[k] for k in range(4) if any(len(r) > 2 + k and r[2 + k].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": statistics.median(sm) if sm else None, "sm_max_mhz": max(mx) if mx else None, "reasons": reasons,
                "samples": len(self.rows)}


def host_cores():
    """Host cores this process may really use: CPU affinity capped by the cgroup CPU quota."""
    n = len(os.sched_getaffinity(0)) if hasattr(os, "sched_getaffinity") else (os.cpu_count() or 1)
    try:
        q, per = open("/sys/fs/cgroup/cpu.max").read().split()
        if q != "max":
            n = max(1, min(n, int(float(q) / float(per) + 0.999)))
    except Exception:
        pass
    return n


def cpu_reference_rate(blob, chunk, level, threads, seconds=0.0):
    """Oracle (C restatement of zstd.Encoder.EncodeAll at `level`) on `threads` host threads, one pooled encoder per
    thread (zstd/encoder.go:90-99), one EncodeAll per chunk.  blob: uint8 array of whole chunks; every thread encodes
    its contiguous share once (seconds = 0: a single un-looped pass) or repeatedly until `seconds` have passed.
    Returns (GB/s, wall seconds, ratio)."""
    import helpers as H
    L = H.oracle()
    from concurrent.futures import ThreadPoolExecutor
    c = ctypes
    cap = L.orc_zstd_max_encoded_size(chunk, level, 1) + 64
    L.orc_zstd_cctx_new.restype = c.c_void_p
    L.orc_zstd_cctx_free.argtypes = [c.c_void_p]
    L.orc_zstd_bench_chunks.restype = c.c_int64
    L.orc_zstd_bench_chunks.argtypes = [c.c_void_p, c.c_void_p, c.c_size_t, c.c_size_t, c.c_int, c.c_int, c.c_void_p,
                                        c.c_size_t, c.c_double, c.c_void_p]
    nchunks = blob.size // chunk
    threads = max(1, min(threads, nchunks))
    bufs = [c.create_string_buffer(cap) for _ in range(threads)]
    ctxs = [L.orc_zstd_cctx_new() for _ in range(threads)]
    per = nchunks // threads
    done = (c.c_uint64 * threads)()

    def work(t):
        lo = t * per
        cnt = per if t < threads - 1 else nchunks - lo
        r = L.orc_zstd_bench_chunks(ctxs[t], blob.ctypes.data + lo * chunk, chunk, cnt, level, 1, bufs[t], cap,
                                    float(seconds), c.byref(done, 8 * t))  # ctypes releases the GIL
        assert r > 0
        return r
    t0 = time.perf_counter()
    with ThreadPoolExecutor(threads) as ex:
        outs = list(ex.map(work, range(threads)))
    dt = time.perf_counter() - t0
    for x in ctxs:
        L.orc_zstd_cctx_free(x)
    nbytes = sum(int(d) for d in done)
    return nbytes / dt / 1e9, dt, sum(outs) / (nchunks * chunk)


def make_data(nbytes, device, seed):
    """The workload bytes: deterministic for (device type, seed).  Both arms call this with the same arguments on
    rank 0, so the CPU arm encodes exactly the bytes the GPU arm does."""
    import helpers as H
    return H.synth_text_torch(nbytes, device, seed=seed)


DUMP_BYTES = 64 << 20
DUMP_SEED = 7


def dump_outputs(path, dst, sizes, suffix=""):
    """Writes what the timed encode returned in its last step, so that two builds can be compared output for output:
    sizes.npy (every frame's size, float64), frames.npy (the frame bytes of a fixed, seeded sample of chunks, one row of
    `slot` float32 values per chunk, zero past the frame's end) and frame_index.npy (the sampled chunks), 64 MB at most."""
    import torch
    os.makedirs(path, exist_ok=True)
    n, slot = dst.shape
    k = max(0, min(n, 64, (DUMP_BYTES - 16 * n) // (4 * slot)))
    idx = np.sort(np.random.Generator(np.random.PCG64(DUMP_SEED)).choice(n, size=k, replace=False))
    rows = dst[torch.from_numpy(idx).to(dst.device)].cpu().numpy()
    rows[np.arange(slot)[None, :] >= sizes[idx][:, None]] = 0
    np.save(os.path.join(path, "sizes%s.npy" % suffix), sizes.astype(np.float64))
    np.save(os.path.join(path, "frame_index%s.npy" % suffix), idx.astype(np.float64))
    np.save(os.path.join(path, "frames%s.npy" % suffix), rows.astype(np.float32))


def pci_bus_id(index):
    try:
        out = subprocess.run(["nvidia-smi", "-i", str(index), "--query-gpu=pci.bus_id", "--format=csv,noheader"],
                             capture_output=True, text=True, timeout=10).stdout.strip()
        return out or None
    except Exception:
        return None


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--level", type=int, default=1, choices=[1, 2, 3])
    ap.add_argument("--nchunks", type=int, default=0, help="chunks per GPU (default: 1 GiB worth)")
    ap.add_argument("--e2e-chunks", type=int, default=0, help="chunks per e2e step (default: all)")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--no-secondary", action="store_true", help="skip the decode / S2 / huff0 / chunk-API side measurements")
    ap.add_argument("--dump-outputs", metavar="DIR", help="write a seeded sample of the last timed step's frames and all "
                                                          "frame sizes to DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs dumps the GPU encoder's outputs; --impl reference keeps none")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    warm = max(args.warmup, 3)
    level = args.level
    CHUNK = LEVELS[level]["chunk"]
    n = args.nchunks or LEVELS[level]["nchunks"]
    METRIC = metric_name(level)
    config = {"workload": "zstd %s (level %d), %d x %d KiB independent chunks of synthetic enwik-like text per GPU, "
                          "one frame per chunk, CRC on" % (LEVELS[level]["name"], level, n, CHUNK >> 10),
              "chunk_bytes": CHUNK, "chunks_per_gpu": n, "l2": "inputs (1 GiB/GPU) larger than L2, no flush needed",
              "parallelism": "chunks sharded over %d GPU(s), no collective" % world}

    import helpers as H
    import torch

    if args.impl == "reference":
        if rank != 0:
            return
        nthreads = host_cores()
        dev = torch.device("cuda", local_rank) if torch.cuda.is_available() else torch.device("cpu")
        blob = make_data(n * CHUNK, dev, DATA_SEED).cpu().numpy()
        steps = max(1, args.steps)
        for _ in range(min(args.warmup, 1)):
            cpu_reference_rate(blob[: 256 * CHUNK], CHUNK, level, nthreads)
        rates = [cpu_reference_rate(blob, CHUNK, level, nthreads) for _ in range(steps)]
        gbs = sum(r[0] * r[1] for r in rates) / sum(r[1] for r in rates)
        line = {"metric": METRIC, "value": gbs, "unit": "GB/s", "n_gpus": args.gpus, "steps": steps, "warmup": args.warmup,
                "ms_per_step": 1e3 * sum(r[1] for r in rates) / steps, "higher_is_better": True, "scaling": "weak",
                "vs_baseline": None, "dtype": "u8", "data": "synthetic", "impl": "reference", "config": config,
                "cpu_baseline": {"value": gbs, "unit": "GB/s", "cores": nthreads, "kind": "port",
                                 "sample": "one un-looped pass per step over the %d chunks (%.2f GiB) the GPU arm's rank 0 "
                                           "encodes (same generator, same seed); oracle C restatement of the Go encoder (Go "
                                           "toolchain absent), one EncodeAll per chunk on a pooled encoder, %d threads"
                                           % (n, n * CHUNK / 2**30, nthreads),
                                 "ratio": rates[-1][2]},
                "e2e": {"value": gbs, "unit": "GB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}
        print(json.dumps(line))
        return

    import torch.distributed as dist
    assert torch.cuda.is_available(), "bench.py needs a GPU (no CPU fallback)"
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    # host placement before any pinned allocation: this rank's CPUs and host buffers on the GPU's NUMA node
    from compress_b200 import shard
    numa = None
    orig_affinity = os.sched_getaffinity(0) if hasattr(os, "sched_getaffinity") else None
    bdf = pci_bus_id(local_rank)
    if bdf:
        numa = shard.bind_to_gpu_numa(bdf)
    nthreads = host_cores()
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from compress_b200 import zstd
    enc = zstd.Encoder(level=level, device=local_rank, max_chunks=1184)  # host-path batch: 8 x 64 KiB chunks per SM
    src = make_data(n * CHUNK, dev, DATA_SEED + rank)
    dst = torch.empty((n, enc.slot), dtype=torch.uint8, device=dev)
    outs = torch.empty((n,), dtype=torch.int64, device=dev)

    def barrier():
        torch.cuda.synchronize()
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    for _ in range(warm):
        enc.encode_device(src, dst=dst, out_sizes=outs)
    barrier()
    sampler = ClockSampler(local_rank)
    sampler.start()
    launches0 = enc.launches
    enc.profile(True)
    ev = [torch.cuda.Event(enable_timing=True) for _ in range(args.steps + 1)]
    ev[0].record()
    for k in range(args.steps):
        enc.encode_device(src, dst=dst, out_sizes=outs)
        ev[k + 1].record()
    barrier()
    step_ms = [ev[k].elapsed_time(ev[k + 1]) for k in range(args.steps)]
    total_ms = ev[0].elapsed_time(ev[args.steps])
    kernel_launches = enc.launches - launches0
    kms, kcalls = enc.profile_read()
    enc.profile(False)
    outs_h = outs.cpu().numpy()
    assert (outs_h > 0).all(), "encode error"
    if args.dump_outputs:
        dump_outputs(args.dump_outputs, dst, outs_h, "" if world == 1 else "_rank%d" % rank)
    out_bytes = int(outs_h.sum())
    in_bytes = n * CHUNK
    peak, peak_kind = hbm_peak()
    side = {}

    if not args.no_secondary:
        # ---- decode of the frames just produced (SURVEY 8d "decode GB/s (output bytes)"), device-resident
        dec = zstd.Decoder(device=local_rank)
        dsz = outs.to(torch.int32)
        dout = torch.empty((n, CHUNK), dtype=torch.uint8, device=dev)
        dres = torch.empty((n,), dtype=torch.int64, device=dev)
        for _ in range(2):
            dec.decode_device(dst, dsz, src_stride=enc.slot, dst=dout, dst_cap=CHUNK, out_sizes=dres)
        torch.cuda.synchronize()
        d0, d1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        d0.record()
        for _ in range(3):
            dec.decode_device(dst, dsz, src_stride=enc.slot, dst=dout, dst_cap=CHUNK, out_sizes=dres)
        d1.record()
        torch.cuda.synchronize()
        dec_ms = d0.elapsed_time(d1) / 3
        assert bool((dres == CHUNK).all()) and torch.equal(dout.view(-1), src), "decode mismatch"
        dec.profile(True)                      # per-kernel times: the stages run one after the other in this mode
        for _ in range(2):
            dec.decode_device(dst, dsz, src_stride=enc.slot, dst=dout, dst_cap=CHUNK, out_sizes=dres)
        dk = {k: v / 2 for k, v in dec.profile_read().items()}
        dec.profile(False)
        side["decode"] = {"value": in_bytes / (dec_ms / 1e3) / 1e9, "unit": "GB/s (output bytes, this rank)", "ms": dec_ms,
                          "roofline_frac": (in_bytes + out_bytes) / (dec_ms / 1e3) / 1e9 / peak,
                          "kernel_ms": dk,
                          "note": "staged decode (scan, literals beside sequences, execute, xxh64, one-warp decoder for marked "
                                  "inputs) of the frames produced above; verified equal to the input"}
        del dout
        dec.close()

    if not args.no_secondary:
        # ---- frame mode (SURVEY 8f-1): the same bytes as 1 MiB inputs, ONE multi-block frame each (EncodeAll of a large
        # input, zstd/encoder.go:796-830); blocks see the history before them
        fs = 1 << 20
        nf = in_bytes // fs
        foffs, flens = [i * fs for i in range(nf)], [fs] * nf
        fdst = torch.empty(nf * (fs + 4096), dtype=torch.uint8, device=dev)
        for _ in range(2):
            _, foff, fsz = enc.encode_frames_device(src, foffs, flens, dst=fdst)
        torch.cuda.synchronize()
        f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        f0.record()
        for _ in range(3):
            _, foff, fsz = enc.encode_frames_device(src, foffs, flens, dst=fdst)
        f1.record()
        torch.cuda.synchronize()
        fms = f0.elapsed_time(f1) / 3
        fz, fo = fsz.cpu().numpy(), foff.cpu().numpy().astype(np.int64)
        assert (fz > 0).all(), "frame mode error"
        import helpers as _H
        probe = bytes(fdst[int(fo[nf // 2]): int(fo[nf // 2]) + int(fz[nf // 2])].cpu().numpy())
        assert _H.libzstd_decode(probe, fs) == bytes(src[(nf // 2) * fs:(nf // 2 + 1) * fs].cpu().numpy()), "frame mode decode mismatch"
        side["frame_mode"] = {"value": nf * fs / (fms / 1e3) / 1e9, "unit": "GB/s (input, this rank)", "ms": fms, "frames": nf,
                              "frame_bytes": fs, "ratio": float(fz.sum()) / (nf * fs),
                              "note": "one multi-block frame per 1 MiB input (b2c_zstd_encode_frames_device); one frame checked "
                                      "with libzstd"}
        del fdst

    if not args.no_secondary and level == 1:
        # ---- BASELINE config 3: S2 / Snappy block encode + decode of the same chunks, device-resident
        from compress_b200 import s2 as s2mod
        from compress_b200 import _lib as _lib_mod
        s2c = s2mod.Codec(device=local_rank)
        s2res = {}
        s2dst = torch.empty((n, s2mod.SLOT), dtype=torch.uint8, device=dev)
        s2sz = torch.empty((n,), dtype=torch.int64, device=dev)
        dout = torch.empty((n, CHUNK), dtype=torch.uint8, device=dev)
        dres = torch.empty((n,), dtype=torch.int64, device=dev)
        for name, snappy, better in (("s2", False, False), ("snappy", True, False), ("s2_better", False, True),
                                     ("snappy_better", True, True)):
            for _ in range(2):
                s2c.encode_device(src, snappy=snappy, better=better, dst=s2dst, out_sizes=s2sz)
            torch.cuda.synchronize()
            a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            a0.record()
            for _ in range(3):
                s2c.encode_device(src, snappy=snappy, better=better, dst=s2dst, out_sizes=s2sz)
            a1.record()
            torch.cuda.synchronize()
            ems = a0.elapsed_time(a1) / 3
            s2out = int(s2sz.sum())
            s2i = s2sz.to(torch.int32)
            for _ in range(2):
                s2c.decode_device(s2dst, s2i, src_stride=s2mod.SLOT, dst=dout, dst_cap=CHUNK, out_sizes=dres)
            torch.cuda.synchronize()
            a0.record()
            for _ in range(3):
                s2c.decode_device(s2dst, s2i, src_stride=s2mod.SLOT, dst=dout, dst_cap=CHUNK, out_sizes=dres)
            a1.record()
            torch.cuda.synchronize()
            dms = a0.elapsed_time(a1) / 3
            assert bool((dres == CHUNK).all()) and torch.equal(dout.view(-1), src), "s2 decode mismatch"
            s2res[name] = {"encode_gbs": in_bytes / (ems / 1e3) / 1e9, "encode_ms": ems, "ratio": s2out / in_bytes,
                           "decode_gbs": in_bytes / (dms / 1e3) / 1e9, "decode_ms": dms,
                           "encode_roofline_frac": (in_bytes + s2out) / (ems / 1e3) / 1e9 / peak}
        del dout, s2dst
        # the framing format around the same blocks (s2.Writer.EncodeBuffer): identifier + one checksummed chunk per block
        sdst = torch.empty(int(_lib_mod.lib.b2c_s2_stream_bound(in_bytes, CHUNK)) + 16, dtype=torch.uint8, device=dev)
        for _ in range(2):
            _, stot, serr = s2c.encode_stream_device(src, dst=sdst)
        torch.cuda.synchronize()
        a0.record()
        for _ in range(3):
            _, stot, serr = s2c.encode_stream_device(src, dst=sdst)
        a1.record()
        torch.cuda.synchronize()
        sms = a0.elapsed_time(a1) / 3
        assert int(serr.item()) == 0
        s2res["stream"] = {"encode_gbs": in_bytes / (sms / 1e3) / 1e9, "encode_ms": sms, "ratio": int(stot.cpu().numpy()[0]) / in_bytes,
                           "note": "b2c_s2_encode_stream_device: blocks + CRC32-C + placement into one S2 stream"}
        del sdst
        side["s2"] = s2res

        # ---- BASELINE config 4: standalone huff0 Compress4X / Decompress4X, 262143-byte blocks of the same text
        from compress_b200 import huff0 as hufmod
        hc = hufmod.Codec(device=local_rank)
        hb, hstride = 262143, 262144
        hn = in_bytes // hstride
        hsz = torch.full((hn,), hb, dtype=torch.int32, device=dev)
        hdst = torch.empty((hn, hstride), dtype=torch.uint8, device=dev)
        hout = torch.empty((hn,), dtype=torch.int64, device=dev)
        for _ in range(2):
            hc.compress_device(src, hstride, hsz, True, dst=hdst, out_sizes=hout)
        torch.cuda.synchronize()
        a0, a1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        a0.record()
        for _ in range(3):
            hc.compress_device(src, hstride, hsz, True, dst=hdst, out_sizes=hout)
        a1.record()
        torch.cuda.synchronize()
        hc_ms = a0.elapsed_time(a1) / 3
        assert int(hout.min()) > 0
        hcsz = hout.to(torch.int32)
        hdec = torch.empty((hn, hstride), dtype=torch.uint8, device=dev)
        hres = torch.empty((hn,), dtype=torch.int64, device=dev)
        for _ in range(2):
            hc.decompress_device(hdst.view(-1), hstride, hcsz, hsz, hstride, True, dst=hdec, out_sizes=hres)
        torch.cuda.synchronize()
        a0.record()
        for _ in range(3):
            hc.decompress_device(hdst.view(-1), hstride, hcsz, hsz, hstride, True, dst=hdec, out_sizes=hres)
        a1.record()
        torch.cuda.synchronize()
        hd_ms = a0.elapsed_time(a1) / 3
        assert bool((hres == hb).all()) and torch.equal(hdec[:, :hb], src.view(hn, hstride)[:, :hb]), "huff0 mismatch"
        side["huff0"] = {"blocks": hn, "block_bytes": hb, "compress4x_gbs": hn * hb / (hc_ms / 1e3) / 1e9, "compress_ms": hc_ms,
                         "ratio": float(hout.sum()) / (hn * hb), "decompress4x_gbs": hn * hb / (hd_ms / 1e3) / 1e9,
                         "decompress_ms": hd_ms}
        del hdec, hdst

    # ---- end to end through the host-buffer C-ABI call (pinned host in/out), all chunks of the workload
    ne = min(args.e2e_chunks or n, n)
    host_in = src[: ne * CHUNK].cpu().pin_memory()
    host_out = torch.empty(ne * CHUNK + ne * 32 + 64, dtype=torch.uint8, pin_memory=True)
    for _ in range(2):
        enc.encode_packed(host_in, dst=host_out)
    barrier()
    t0 = time.perf_counter()
    e2e_steps = max(2, min(args.steps, 5))
    for _ in range(e2e_steps):
        _, e_total, _, _ = enc.encode_packed(host_in, dst=host_out)
    torch.cuda.synchronize()
    e2e_s = (time.perf_counter() - t0) / e2e_steps
    # the same bytes moved with no kernel in between (H2D and D2H on two streams): the ceiling of this call on this host
    s_in, s_out = torch.cuda.Stream(device=dev), torch.cuda.Stream(device=dev)
    dtmp = torch.empty(ne * CHUNK, dtype=torch.uint8, device=dev)
    dpk = torch.empty(int(e_total), dtype=torch.uint8, device=dev)
    barrier()
    t0 = time.perf_counter()
    for _ in range(e2e_steps):
        with torch.cuda.stream(s_in):
            dtmp.copy_(host_in, non_blocking=True)
        with torch.cuda.stream(s_out):
            host_out[: int(e_total)].copy_(dpk, non_blocking=True)
    torch.cuda.synchronize()
    copy_s = (time.perf_counter() - t0) / e2e_steps
    del dtmp, dpk
    sampler.stop = True
    sampler.join(timeout=2)

    if not args.no_secondary and level == 1 and world == 1:
        # ---- the other host-buffer entry points a cgo shim calls: per-chunk pointer tables, one synchronous call each.
        # Timed around the C call only (argument arrays are built before): what the shim pays.
        from compress_b200._lib import lib
        from compress_b200 import s2 as s2mod
        m = 2048
        hin = host_in.numpy()
        cap = int(lib.b2c_zstd_bound(CHUNK, 1)) + 16
        outb = np.empty((m, cap), dtype=np.uint8)
        srcs = (ctypes.c_void_p * m)(*[hin.ctypes.data + i * CHUNK for i in range(m)])
        ssz = (ctypes.c_size_t * m)(*([CHUNK] * m))
        dsts = (ctypes.c_void_p * m)(*[outb.ctypes.data + i * cap for i in range(m)])
        dcap = (ctypes.c_size_t * m)(*([cap] * m))
        res = (ctypes.c_int64 * m)()

        def timed(fn, *a):
            fn(*a)
            t0 = time.perf_counter()
            rc = fn(*a)
            dt = time.perf_counter() - t0
            assert rc == 0
            return dt
        tc = timed(lib.b2c_zstd_encode_chunks, enc._ctx, 1, 3, srcs, ssz, dsts, dcap, res, m)
        fsz = [int(r) for r in res]
        assert min(fsz) > 0
        dec = zstd.Decoder(device=local_rank)
        back = np.empty((m, CHUNK), dtype=np.uint8)
        fs = (ctypes.c_size_t * m)(*fsz)
        bdst = (ctypes.c_void_p * m)(*[back.ctypes.data + i * CHUNK for i in range(m)])
        bcap = (ctypes.c_size_t * m)(*([CHUNK] * m))
        res2 = (ctypes.c_int64 * m)()
        td = timed(lib.b2c_zstd_decode_chunks, dec._ctx, dsts, fs, bdst, bcap, res2, m)
        assert all(int(r) == CHUNK for r in res2) and bytes(back.reshape(-1)[: m * CHUNK]) == bytes(hin[: m * CHUNK])
        dec.close()
        s2c = s2mod.Codec(device=local_rank)
        ts = timed(lib.b2c_s2_encode_chunks, s2c._ctx, 1, 0, srcs, ssz, dsts, dcap, res, m)
        s2c.close()
        side["e2e_chunk_apis"] = {"chunks": m, "note": "one synchronous C-ABI call over 2048 separately addressed 64 KiB chunks in pageable "
                                                      "host memory (pointer tables), wall clock around the call",
                                  "b2c_zstd_encode_chunks_gbs": m * CHUNK / tc / 1e9, "b2c_zstd_decode_chunks_gbs": m * CHUNK / td / 1e9,
                                  "b2c_s2_encode_chunks_gbs": m * CHUNK / ts / 1e9}

    # max over ranks
    total_ms_max, e2e_s_max, copy_s_max = shard.max_over_ranks([total_ms, e2e_s, copy_s], device=dev)
    value = world * in_bytes * args.steps / (total_ms_max / 1e3) / 1e9
    e2e_val = world * ne * CHUNK / e2e_s_max / 1e9
    # dominant kernel of the pipeline, from the CUDA events recorded around every kernel of the timed steps
    per_step = {k: v / args.steps for k, v in kms.items()}
    dom = max(per_step, key=per_step.get)
    dom_s = per_step[dom] / 1e3
    achieved = (in_bytes + out_bytes) / dom_s / 1e9
    step_s = (sum(step_ms) / len(step_ms)) / 1e3
    traffic, traffic_src = None, None
    tj = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tj):
        try:
            tjd = json.load(open(tj))
            traffic = tjd.get("%s@L%d" % (dom, level))
            traffic_src = "profiles/traffic.json (ncu dram__bytes of a separate capture of the same command; not measured in this run)"
        except Exception:
            traffic = None
    if rank == 0:
        line = {"metric": METRIC, "value": value, "unit": "GB/s", "n_gpus": world, "steps": args.steps, "warmup": warm,
                "ms_per_step": total_ms_max / args.steps, "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
                "dtype": "u8", "data": "synthetic", "config": config, "ratio": out_bytes / in_bytes,
                "hbm_input_fraction": (value / world) / peak,
                "gpu_launches": int(kernel_launches),
                "clocks": sampler.summary(),
                "numa_node": numa,
                "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                             "traffic": traffic, "traffic_source": traffic_src, "peak_kind": peak_kind, "kernel": dom,
                             "algorithmic_bytes_per_launch": (in_bytes + out_bytes) / max(1, kcalls // max(1, args.steps)),
                             "kernel_ms_per_step": per_step, "pipeline_launches_per_step": kcalls // max(args.steps, 1),
                             "pipeline_frac": (in_bytes + out_bytes) / step_s / 1e9 / peak},
                "e2e": {"value": e2e_val, "unit": "GB/s", "h2d_bytes_per_step": ne * CHUNK, "d2h_bytes_per_step": int(e_total),
                        "api": "b2c_zstd_encode_packed (pinned host in/out; H2D, kernels and D2H on three streams, two slots)",
                        "chunks_per_step": ne,
                        "copy_only_gbs": world * ne * CHUNK / copy_s_max / 1e9,
                        "copy_only_note": "same H2D + D2H bytes on two streams with no kernels: the host-side ceiling of this call"}}
        line.update(side)
        if not args.no_cpu_baseline:
            if orig_affinity is not None:
                os.sched_setaffinity(0, orig_affinity)     # the CPU arm may use every core the process was given
            nthreads = host_cores()
            blob = src.cpu().numpy()          # rank 0's bytes: what `--impl reference` generates too
            gbs, dt, ratio = cpu_reference_rate(blob, CHUNK, level, nthreads)
            g1, d1, _ = cpu_reference_rate(blob[: 512 * CHUNK], CHUNK, level, 1)
            line["cpu_baseline"] = {"value": gbs, "unit": "GB/s", "cores": nthreads, "kind": "port",
                                    "sample": "one un-looped pass over the %d chunks (%.2f GiB) rank 0 encoded on the GPU, %.1f s on "
                                              "%d threads (oracle C restatement of the Go encoder, one EncodeAll per chunk, pooled "
                                              "encoders); 1 thread on the first 512 chunks: %.3f GB/s" % (n, in_bytes / 2**30, dt, nthreads, g1),
                                    "ratio": ratio}
        print(json.dumps(line))
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
