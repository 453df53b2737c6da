#!/usr/bin/env python
"""bench.py -- headline benchmark of the B200 rANS hot path (BASELINE.json metric).

Step      = one bit-exact round trip of the hot path over one batch: encode the
            batch (rb200_encode: encode kernel + directory scan + compaction), then
            decode it (rb200_decode: one kernel), device-resident, through the C-ABI.
Workload  = BASELINE.json configs[1]: 1 GiB i.i.d. uniform bytes, one static
            256-symbol model (scale_bits 12), word coder, 32-way interleaved chunks.
            Per-GPU work is fixed (weak scaling): every rank round-trips its own shard.
value     = symbols round-tripped per second over all ranks (Gsymbols/s, 1 symbol = 1 byte)
e2e       = the same round trip through the host-pointer C-ABI calls (pinned host
            buffers, H2D/D2H inside the timed region).
roofline  = the decode kernel (the north-star kernel) against measured HBM copy bandwidth;
            the encode call is reported beside it.
--impl reference times the reference's own CPU coders (oracle/_ref, built from the
reference sources) on all host cores on a bounded sample of the same workload.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

METRIC = "Gsymbols/s decode+encode (bit-exact round-trip)"
UNIT = "Gsymbols/s"
HEADLINE = "uniform_1GiB_word32"
WORKLOADS = {
    # name: coder, scale_bits, generator, BASELINE.json config it stands for
    "uniform_1GiB_word32": ("word", 12, "uniform", "configs[1]: 1 GiB uniform bytes, static model, 32-way decode"),
    "zipf1.1_1GiB_alias32": ("alias", 16, "zipf", "configs[2]: 1 GiB Zipf(1.1), alias-method lookup"),
    "text_1GiB_word32": ("word", 12, "text", "configs[3]: one 1 GiB shard of the 8 GiB text-like stream (book1 byte histogram)"),
    "blocks_64KiB_word32": ("blocks", 12, "blocks", "configs[4]: this GPU's 8192 of the 64 Ki blocks of 64 KiB, one model per block"),
    "uniform_1GiB_rans64": ("rans64", 14, "uniform", "the reference's CPU-baseline coder (rans64.h) on the GPU"),
}
DECODE_KERNEL = {"word": "word_decode_tma_kernel", "alias": "alias_decode_persist_kernel", "blocks": "block_decode_kernel",
                 "rans64": "rans64_decode_kernel"}
BLOCK_SIZE = 65536


def parse_args():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=10)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--workload", default=HEADLINE, choices=sorted(WORKLOADS))
    ap.add_argument("--configs", default="auto", choices=["auto", "all", "none"],
                    help="also measure the other BASELINE configs (reduced steps) into the line's `configs` object; "
                         "auto = yes when --workload is the headline one")
    ap.add_argument("--config-steps", type=int, default=3)
    ap.add_argument("--size", type=int, default=1 << 30, help="symbols per GPU")
    ap.add_argument("--chunk", type=int, default=int(os.environ.get("RB200_CHUNK", 8192)), help="symbols per 32-way chunk stream")
    ap.add_argument("--e2e-steps", type=int, default=5)
    ap.add_argument("--cpu-sample", type=int, default=256 << 20, help="bytes of the workload the in-line CPU baseline is timed on")
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last step returned (compressed blob, chunk directory, "
                         "decoded symbols; seeded samples of the large ones) as DIR/<name>.npy")
    return ap.parse_args()


# ------------------------------------------------------------------ synthetic data

def text_probs():
    """Order-0 distribution of the reference's test file book1 (82 symbols, 4.527 bit/symbol; SURVEY 8(d) C4),
    from the committed fixture tests/golden/book1_hist.json (made by tests/golden/make_book1_hist.py)."""
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "tests", "golden", "book1_hist.json")) as f:
        counts = np.asarray(json.load(f)["counts"], dtype=np.float64)
    return counts / counts.sum()


def synth_torch(kind, n, seed, device):
    """Seeded synthetic symbols generated on the device (so 1 GiB need not cross PCIe)."""
    import torch
    g = torch.Generator(device=device)
    g.manual_seed(0x5EED0000 + seed)
    if kind == "uniform":
        return torch.randint(0, 256, (n,), dtype=torch.uint8, device=device, generator=g)
    if kind == "blocks":
        # every 64 KiB block has its own distribution: Zipf ranks pushed through a per-block permutation
        nb = n // BLOCK_SIZE
        p = 1.0 / torch.arange(1, 257, dtype=torch.float64) ** 1.3
        cdf = torch.cumsum(p / p.sum(), 0).to(device=device, dtype=torch.float32)
        out = torch.empty(n, dtype=torch.uint8, device=device)
        perms = torch.argsort(torch.rand(nb, 256, device=device, generator=g), dim=1).to(torch.uint8)
        step_blocks = 1024
        for b0 in range(0, nb, step_blocks):
            b1 = min(nb, b0 + step_blocks)
            u = torch.rand((b1 - b0) * BLOCK_SIZE, device=device, generator=g)
            ranks = torch.searchsorted(cdf, u).clamp_(max=255).view(b1 - b0, BLOCK_SIZE)
            out[b0 * BLOCK_SIZE:b1 * BLOCK_SIZE] = torch.gather(perms[b0:b1], 1, ranks).reshape(-1)
        return out
    if kind == "zipf":
        p = 1.0 / torch.arange(1, 257, dtype=torch.float64) ** 1.1
    elif kind == "text":
        p = torch.from_numpy(text_probs())
    else:
        raise ValueError(kind)
    cdf = torch.cumsum(p / p.sum(), 0).to(device=device, dtype=torch.float32)
    out = torch.empty(n, dtype=torch.uint8, device=device)
    step = 1 << 26
    for lo in range(0, n, step):
        m = min(step, n - lo)
        u = torch.rand(m, device=device, generator=g)
        out[lo:lo + m] = torch.searchsorted(cdf, u).clamp_(max=255).to(torch.uint8)
    return out


def synth_numpy(kind, n, seed):
    rng = np.random.default_rng(0x5EED0000 + seed)
    if kind == "uniform":
        return rng.integers(0, 256, n, dtype=np.uint8)
    if kind == "zipf":
        p = 1.0 / np.arange(1, 257) ** 1.1
    else:
        p = text_probs()
    cdf = np.cumsum(p / p.sum())
    out = np.empty(n, np.uint8)
    step = 1 << 24
    for lo in range(0, n, step):
        m = min(step, n - lo)
        out[lo:lo + m] = np.minimum(np.searchsorted(cdf, rng.random(m)), 255).astype(np.uint8)
    return out


# ------------------------------------------------------------------ clocks

class ClockSampler:
    Q = ("clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")

    def __init__(self, index):
        self.proc = None
        try:
            self.proc = subprocess.Popen(["nvidia-smi", "-i", str(index), f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "20"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
        except Exception:
            self.proc = None

    def stop(self):
        if not self.proc:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        time.sleep(0.15)
        self.proc.terminate()
        try:
            out, _ = self.proc.communicate(timeout=5)
        except Exception:
            self.proc.kill()
            out = ""
        sm, mx, reasons = [], [], set()
        for line in out.strip().splitlines():
            f = [x.strip() for x in line.split(",")]
            if len(f) < 7:
                continue
            try:
                sm.append(float(f[0])); mx.append(float(f[1]))
            except ValueError:
                continue
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), f[3:7]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": float(np.median(sm)) if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "samples": len(sm), "reasons": sorted(reasons)}


def ncu_traffic(workload, chunk, kernel):
    """dram__bytes_read.sum + dram__bytes_write.sum per launch of `kernel` on `workload`, from the committed
    `ncu --set full` captures (profiles/ncu_traffic.json, regenerated by tools/ncu_traffic.py), or None when no capture
    of this build's kernel exists for the workload / chunk size."""
    try:
        with open(os.path.join(ROOT, "profiles", "ncu_traffic.json")) as f:
            t = json.load(f)
        w = t["workloads"][workload]
        if w["chunk_syms"] == chunk:
            return w["dram_bytes_per_launch"].get(kernel)
    except Exception:
        pass
    return None


def measured_peak():
    try:
        with open(os.path.join(ROOT, "MEASURED_PEAKS.json")) as f:
            return float(json.load(f)["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs, burst copy)"
    except Exception:
        return 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------ reference arm / cpu baseline

_CPU_SAMPLES = {}


def _cpu_sample(kind, nbytes):
    """The CPU arm's input (generated once per process: 1 GiB of numpy random draws takes seconds)."""
    key = (kind, nbytes)
    if key not in _CPU_SAMPLES:
        _CPU_SAMPLES.clear()
        _CPU_SAMPLES[key] = synth_numpy(kind, nbytes, seed=1)
    return _CPU_SAMPLES[key]


def cpu_reference_run(kind, coder, scale_bits, nbytes, runs, threads, single_thread=True):
    """Time the reference's own CPU coders (oracle/_ref) on `nbytes` of the workload."""
    import oracle
    data = _cpu_sample(kind, nbytes)
    if oracle.Reference.available():
        ref = oracle.Reference()
        which = "alias" if coder == "alias" else "simd"
        r = ref.cpu_baseline(which, data, threads, runs=runs, scale_bits=scale_bits if coder == "alias" else None)
        r64 = ref.cpu_baseline("rans64", data, threads, runs=max(1, runs - 1), scale_bits=14)
        if not (r["ok"] and r64["ok"]):
            raise RuntimeError("reference CPU round trip failed")
        kind_s = "reference"
        paths = {
            ("main_alias.cpp 2-way alias" if coder == "alias" else "main_simd.cpp 8-way scalar enc + SSE4.1 dec"): r,
            "main64.cpp rans64 2-way": r64,
        }
    else:   # the C port (oracle/rans_oracle.c), single thread
        orc = oracle.Oracle()
        cid = oracle.CODER_ALIAS if coder == "alias" else oracle.CODER_WORD
        freqs, cum = orc.model(data, scale_bits)
        nl = 2 if coder == "alias" else 8
        t0 = time.perf_counter()
        stream = orc.encode(cid, data, freqs, cum, nl, scale_bits)
        t1 = time.perf_counter()
        dec, _ = orc.decode(cid, stream, data.size, freqs, cum, nl, scale_bits)
        t2 = time.perf_counter()
        assert np.array_equal(dec, data)
        kind_s, threads = "port", 1
        paths = {"oracle/rans_oracle.c port": {"enc_s": t1 - t0, "dec_s": t2 - t1, "bytes": stream.size, "ok": True}}
    best_name, best = min(paths.items(), key=lambda kv: kv[1]["enc_s"] + kv[1]["dec_s"])
    rt = nbytes / (best["enc_s"] + best["dec_s"]) / 1e9
    detail = {k: {"encode_gsym_s": round(nbytes / v["enc_s"] / 1e9, 4), "decode_gsym_s": round(nbytes / v["dec_s"] / 1e9, 4),
                  "compressed_bytes": v["bytes"]} for k, v in paths.items()}
    if kind_s == "reference" and threads > 1 and single_thread:      # SURVEY 8(d): single-thread figures beside the all-core ones
        small = data[:min(nbytes, 32 << 20)]
        st = {("main_alias.cpp 2-way alias" if coder == "alias" else "main_simd.cpp 8-way scalar enc + SSE4.1 dec"):
              ref.cpu_baseline("alias" if coder == "alias" else "simd", small, 1, runs=2, scale_bits=scale_bits if coder == "alias" else None),
              "main64.cpp rans64 2-way": ref.cpu_baseline("rans64", small, 1, runs=2, scale_bits=14)}
        for k, v in st.items():
            detail[k]["single_thread_encode_gsym_s"] = round(small.size / v["enc_s"] / 1e9, 4)
            detail[k]["single_thread_decode_gsym_s"] = round(small.size / v["dec_s"] / 1e9, 4)
    return {"value": rt, "unit": UNIT, "cores": threads, "kind": kind_s,
            "sample": f"{nbytes >> 20} MiB of the {kind} workload, one contiguous slice per thread, best of {runs}; "
                      f"round trip = encode + decode; fastest path: {best_name}",
            "paths": detail}


def run_reference(args, rank, world):
    """--impl reference: the reference's own CPU coders (oracle/_ref, or the C port where the reference could not be
    built) on the SAME workload and size as our arm, all host threads; every step is one full round trip."""
    if rank != 0:
        return
    coder, sb, kind, _ = WORKLOADS[args.workload]
    if coder == "blocks":
        coder, kind = "word", "zipf"        # the reference has no per-block driver: one model over the same bytes
    threads = os.cpu_count() or 1
    n = args.size
    t0 = time.perf_counter()
    for _ in range(args.warmup):
        cpu_reference_run(kind, coder, sb, n, runs=1, threads=threads, single_thread=False)
    vals, base = [], None
    for _ in range(args.steps):
        base = cpu_reference_run(kind, coder, sb, n, runs=1, threads=threads, single_thread=False)
        vals.append(base["value"])
    ms = [1e3 * n / (v * 1e9) for v in vals]
    v = n / (float(np.mean(ms)) * 1e-3) / 1e9
    base["value"] = v
    base["sample"] = f"the whole workload ({n >> 20} MiB), one contiguous slice per thread, {args.steps} timed round trips"
    print(json.dumps({
        "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
        "warmup": args.warmup, "ms_per_step": float(np.mean(ms)), "higher_is_better": True, "scaling": "weak",
        "vs_baseline": None, "dtype": "u32", "data": "synthetic",
        "config": {"workload": args.workload, "symbols_per_gpu": n, "symbols_per_step": n,
                   "note": "CPU, host cores only; the box's cores are shared by all ranks, so the value does not grow with --gpus"},
        "cpu_baseline": base,
        "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
        "gpu_launches": 0, "wall_s": round(time.perf_counter() - t0, 2),
    }))


# ------------------------------------------------------------------ our arm

class Rig:
    """What one rank needs to measure workloads: device, stream, context, process group."""

    def __init__(self, rank, local_rank, world):
        import torch
        import ryg_rans_b200 as rb
        if not torch.cuda.is_available():
            raise SystemExit("bench.py: no CUDA device visible; the rANS hot path has no CPU fallback")
        self.torch, self.rb = torch, rb
        self.rank, self.local_rank, self.world = rank, local_rank, world
        torch.cuda.set_device(local_rank)
        self.dev = torch.device("cuda", local_rank)
        self.dist = None
        if world > 1:
            import torch.distributed as dist
            dist.init_process_group("nccl", device_id=self.dev)
            self.dist = dist
        self.ctx = rb.Context(local_rank, torch.cuda.current_stream().cuda_stream)

    def barrier(self):
        if self.dist:
            self.dist.barrier()
        self.torch.cuda.synchronize()

    def max_over_ranks(self, values):
        t = self.torch.tensor(values, dtype=self.torch.float64, device=self.dev)
        if self.dist:
            self.dist.all_reduce(t, op=self.dist.ReduceOp.MAX)
        return t.tolist()


DUMP_BYTES = 16_000_000        # per written array; at most four arrays, so a dump stays within 64 MB


def dump_outputs(dump_dir, outputs):
    """Write each device array as <dump_dir>/<name>.npy: float64 when its values could exceed float32's 24-bit exact
    range (the directory's byte offsets), float32 otherwise.  An array with more elements than fit DUMP_BYTES is
    reduced to the elements at distinct sorted positions drawn from a generator seeded with 0, so two runs with the
    same arguments write the same positions."""
    import torch
    os.makedirs(dump_dir, exist_ok=True)
    for name, t in outputs.items():
        t = t.reshape(-1)
        dtype = np.float64 if t.dtype == torch.int64 else np.float32
        keep = DUMP_BYTES // np.dtype(dtype).itemsize
        if t.numel() > keep:
            idx = np.sort(np.random.default_rng(0).choice(t.numel(), keep, replace=False))
            t = t[torch.from_numpy(idx).to(t.device)]
        np.save(os.path.join(dump_dir, name + ".npy"), t.cpu().numpy().astype(dtype))


def measure(rig, workload, n, chunk, steps, warmup, e2e_steps, headline, dump_dir=None):
    """One workload on every rank: bit-exact check, K timed round trips (device-resident, CUDA events on the
    context's stream, max over ranks), the host-buffer e2e number, and -- for the headline -- the blob gather.
    With `dump_dir`, rank 0 writes the outputs of the last timed step there (dump_outputs)."""
    torch, rb, ctx, dev, world = rig.torch, rig.rb, rig.ctx, rig.dev, rig.world
    coder_name, sb, kind, stands_for = WORKLOADS[workload]
    coder = {"word": rb.CODER_WORD, "alias": rb.CODER_ALIAS, "rans64": rb.CODER_RANS64, "blocks": rb.CODER_WORD}[coder_name]
    blocks = coder_name == "blocks"
    if blocks:
        if BLOCK_SIZE % chunk:
            raise SystemExit("--chunk must divide the 64 KiB block size")
        n = max(BLOCK_SIZE, (n // BLOCK_SIZE) * BLOCK_SIZE)
        if n == 1 << 30:
            n = 8192 * BLOCK_SIZE                      # 64 Ki blocks over 8 GPUs = 8192 blocks (512 MiB) per GPU
    data = synth_torch(kind, n, seed=rig.rank, device=dev)
    n_chunks = ctx.chunk_count(n, chunk)
    cap = ctx.encode_bound(n, chunk)
    blob = torch.empty(cap, dtype=torch.uint8, device=dev)
    offsets = torch.zeros(n_chunks + 1, dtype=torch.int64, device=dev)
    out = torch.empty(n, dtype=torch.uint8, device=dev)
    model_bytes, model, n_blocks, bfreqs = 0, None, 0, None
    if blocks:
        n_blocks = n // BLOCK_SIZE
        bfreqs = torch.zeros(n_blocks * 256, dtype=torch.int16, device=dev)
        model_bytes = 512 * n_blocks                  # the per-block frequency tables travel with the blob (SURVEY 8d)

        def enc():                                    # per-block models are part of encoding a block: one fused launch
            ctx.blocks_model_encode_device(data.data_ptr(), n_blocks, BLOCK_SIZE, bfreqs.data_ptr(), chunk, blob.data_ptr(), cap,
                                           offsets.data_ptr())

        def dec(blob_size):
            ctx.blocks_decode_device(blob.data_ptr(), blob_size, offsets.data_ptr(), bfreqs.data_ptr(), n_blocks, BLOCK_SIZE, chunk,
                                     out.data_ptr())
    else:
        # rb200_model_from_data: histogram on the GPU, the reference's normalize_freqs on the host, tables uploaded
        model = rb.Model.from_data(ctx, coder, sb, device_ptr=data.data_ptr(), n=n)

        def enc():
            ctx.encode_device(model, data.data_ptr(), n, chunk, blob.data_ptr(), cap, offsets.data_ptr())

        def dec(blob_size):
            ctx.decode_device(model, blob.data_ptr(), blob_size, offsets.data_ptr(), chunk, out.data_ptr(), n)

    # warm-up + bit-exact verification (outside the timed region)
    enc()
    ctx.sync()
    blob_size = int(offsets[-1].item())
    for _ in range(max(warmup, 3)):
        enc()
        dec(blob_size)
    ctx.sync()
    if not torch.equal(out, data):
        raise SystemExit(f"bench.py: {workload}: round trip is NOT bit-exact")
    out.zero_()

    launches0 = ctx.launches
    ev = [[torch.cuda.Event(enable_timing=True) for _ in range(3)] for _ in range(steps)]
    sampler = ClockSampler(rig.local_rank) if (rig.rank == 0 and headline) else None
    rig.barrier()
    t_start = torch.cuda.Event(enable_timing=True)
    t_end = torch.cuda.Event(enable_timing=True)
    t_start.record()
    for k in range(steps):
        ev[k][0].record()
        enc()
        ev[k][1].record()
        dec(blob_size)
        ev[k][2].record()
    t_end.record()
    torch.cuda.synchronize()
    rig.barrier()
    clocks = sampler.stop() if sampler else None
    launches = ctx.launches - launches0
    ctx.sync()
    if not torch.equal(out, data):
        raise SystemExit(f"bench.py: {workload}: timed round trip is NOT bit-exact")
    if dump_dir and rig.rank == 0:
        outputs = {"blob": blob[:blob_size], "offsets": offsets, "decoded": out}
        if blocks:
            outputs["block_freqs"] = bfreqs
        dump_outputs(dump_dir, outputs)
    total_ms, enc_ms, dec_ms = rig.max_over_ranks([t_start.elapsed_time(t_end),
                                                   float(np.mean([e[0].elapsed_time(e[1]) for e in ev])),
                                                   float(np.mean([e[1].elapsed_time(e[2]) for e in ev]))])

    # ---- the one exchange step (SURVEY 8e): compressed blobs + directories to rank 0 over NCCL, through the C-ABI
    gather = None
    if rig.dist and headline:
        gather = measure_gather(rig, blob, blob_size, offsets, n_chunks, enc, steps)

    # ---- e2e: host pointers through the C-ABI, copies inside the timed region
    e2e = None
    if e2e_steps > 0:
        e2e = measure_e2e(rig, workload, data, n, chunk, cap, n_chunks, model, coder, sb, n_blocks, e2e_steps)

    peak, peak_src = measured_peak()
    algo_bytes = n + blob_size + model_bytes         # SURVEY 8(d): (1 + c) bytes per symbol (+ 512 B per block model)
    dec_gbs = algo_bytes / (dec_ms * 1e-3) / 1e9
    enc_gbs = algo_bytes / (enc_ms * 1e-3) / 1e9
    per_step = launches // max(steps, 1)               # launches of one encode call + one decode call
    dk = DECODE_KERNEL[coder_name]
    res = {
        "stands_for": stands_for,
        "value": world * n * steps / (total_ms * 1e-3) / 1e9, "unit": UNIT, "steps": steps, "ms_per_step": total_ms / steps,
        "bit_exact": True, "symbols_per_gpu": n, "chunk_syms": chunk, "coder": coder_name, "scale_bits": sb,
        "compressed_bytes_per_symbol": blob_size / n,
        "decode_ms": dec_ms, "encode_ms": enc_ms,
        "decode_gsym_s": world * n / (dec_ms * 1e-3) / 1e9, "encode_gsym_s": world * n / (enc_ms * 1e-3) / 1e9,
        "roofline": {"kernel": dk, "bound": "hbm", "achieved": dec_gbs, "peak": peak, "unit": "GB/s", "frac": dec_gbs / peak,
                     "traffic": ncu_traffic(workload, chunk, dk) if n == (8192 * BLOCK_SIZE if blocks else 1 << 30) else None,
                     "algorithmic_bytes_per_launch": algo_bytes, "peak_source": peak_src},
        "roofline_encode_call": {"launches_per_call": per_step - 1, "bound": "hbm", "achieved": enc_gbs, "peak": peak,
                                 "unit": "GB/s", "frac": enc_gbs / peak, "algorithmic_bytes_per_call": algo_bytes,
                                 "traffic": ncu_traffic(workload, chunk, "encode_call")
                                 if n == (8192 * BLOCK_SIZE if blocks else 1 << 30) else None},
        "gpu_launches": launches, "e2e": e2e,
    }
    if clocks is not None:
        res["clocks"] = clocks
    if gather is not None:
        res.update(gather)
    del data, blob, offsets, out, bfreqs
    if model is not None:
        model.close()
    torch.cuda.empty_cache()
    return res


def measure_gather(rig, blob, blob_size, offsets, n_chunks, enc, steps):
    """The only communication of the path: every rank's blob + directory to rank 0 (rb200_gather_blobs: ncclAllGather
    of the sizes, then grouped ncclSend / ncclRecv).  Reports the gather alone and an encode+gather step."""
    torch, dev = rig.torch, rig.dev
    from ryg_rans_b200.shard import NcclGather
    g = NcclGather(rig.ctx, rig.rank, rig.world, rig.dist)
    total = g.total_bytes(blob_size, n_chunks)             # rank 0 learns the sizes once (all ranks take part)
    gblob = torch.empty(max(total[0], 16), dtype=torch.uint8, device=dev) if rig.rank == 0 else None
    gdir = torch.empty(total[1] + 1, dtype=torch.int64, device=dev) if rig.rank == 0 else None

    def gather():
        g.gather(blob.data_ptr(), blob_size, offsets.data_ptr(), n_chunks,
                 gblob.data_ptr() if gblob is not None else 0, gblob.numel() if gblob is not None else 0,
                 gdir.data_ptr() if gdir is not None else 0)
    gather()                                               # warm-up: NCCL channel set-up
    rig.barrier()
    e0, e1, e2 = (torch.cuda.Event(enable_timing=True) for _ in range(3))
    e0.record()
    gather()
    e1.record()
    for _ in range(steps):                                 # encode + gather back to back: what a sharded encoder pays
        enc()
        gather()
    e2.record()
    torch.cuda.synchronize()
    rig.barrier()
    gather_ms, both_ms = rig.max_over_ranks([e0.elapsed_time(e1), e1.elapsed_time(e2) / steps])
    if rig.rank == 0:
        assert gblob.numel() % 16 == 0 and int(gdir[-1].item()) == total[0], "gathered container is inconsistent"
    g.close()
    return {"nccl_blob_gather_ms": gather_ms, "encode_plus_gather_ms": both_ms,
            "gather_note": "rb200_gather_blobs over the NCCL communicator: rank 0 NVLink ingress is the limit "
                           "(world-1 blobs into one GPU)"}


def measure_e2e(rig, workload, data, n, chunk, cap, n_chunks, model, coder, sb, n_blocks, e2e_steps):
    """The same round trip through the host-pointer C-ABI calls: pinned host buffers, H2D/D2H inside the timed region,
    wall clock, max over ranks.  `with_model` adds rb200_model_from_data (histogram + normalisation + table upload)."""
    import ctypes as C
    torch, rb, ctx = rig.torch, rig.rb, rig.ctx
    lib = ctx.lib
    blocks = model is None
    # first-touch the pinned buffers on the GPU's own NUMA node (what `numactl --cpunodebind` would do for a caller)
    numa_node, saved_affinity = bind_to_gpu_numa_node(rig.local_rank)
    h_in = torch.empty(n, dtype=torch.uint8).pin_memory()
    h_in.copy_(data)
    h_blob = torch.empty(cap, dtype=torch.uint8).pin_memory()
    h_out = torch.empty(n, dtype=torch.uint8).pin_memory()
    h_off = np.zeros(n_chunks + 1, np.uint64)
    h_freqs = torch.empty(max(n_blocks, 1) * 256, dtype=torch.int16).pin_memory()
    size = C.c_size_t(0)

    def step(with_model):
        if blocks:
            lib.check(lib.dll.rb200_blocks_model_encode(ctx.h, h_in.data_ptr(), n_blocks, BLOCK_SIZE, h_freqs.data_ptr(), chunk,
                                                        h_blob.data_ptr(), cap, h_off.ctypes.data, C.byref(size), rb.MEM_HOST), ctx.h)
            lib.check(lib.dll.rb200_blocks_decode(ctx.h, h_blob.data_ptr(), size.value, h_off.ctypes.data, h_freqs.data_ptr(),
                                                  n_blocks, BLOCK_SIZE, chunk, h_out.data_ptr(), rb.MEM_HOST), ctx.h)
            return
        m = rb.Model.from_data(ctx, coder, sb, device_ptr=None, data=h_in.numpy()) if with_model else model
        lib.check(lib.dll.rb200_encode(ctx.h, m.h, h_in.data_ptr(), n, chunk, h_blob.data_ptr(), cap, h_off.ctypes.data,
                                       C.byref(size), rb.MEM_HOST), ctx.h)
        lib.check(lib.dll.rb200_decode(ctx.h, m.h, h_blob.data_ptr(), size.value, h_off.ctypes.data, chunk,
                                       h_out.data_ptr(), n, rb.MEM_HOST), ctx.h)
        if with_model:
            m.close()

    def timed(with_model):
        step(with_model)     # warm-up (allocates staging)
        rig.barrier()
        t0 = time.perf_counter()
        for _ in range(e2e_steps):
            step(with_model)
        torch.cuda.synchronize()
        dt = time.perf_counter() - t0
        if not torch.equal(h_out, h_in):
            raise SystemExit(f"bench.py: {workload}: e2e round trip is NOT bit-exact")
        return rig.max_over_ranks([dt])[0]

    dt = timed(False)
    dt_model = None if blocks else timed(True)
    if saved_affinity is not None:
        os.sched_setaffinity(0, saved_affinity)
    moved = int(n + size.value + 8 * (n_chunks + 1) + (512 * n_blocks if blocks else 0))
    res = {"value": rig.world * n * e2e_steps / dt / 1e9, "unit": UNIT, "host_numa_node": numa_node,
           "h2d_bytes_per_step": moved, "d2h_bytes_per_step": moved, "steps": e2e_steps,
           "pcie_gbs_per_direction_per_rank": moved * e2e_steps / dt / 1e9,
           "note": ("rb200_blocks_model_encode + rb200_blocks_decode" if blocks else "rb200_encode + rb200_decode")
                   + " with RB200_MEM_HOST on pinned buffers, wall clock",
           "bound": "PCIe: each call streams its input in and its output back concurrently; with both directions busy the "
                    "slower one gets 43-47 GB/s on this box (tools/pcie_probe.py, profiles/r1_pcie_copies.log)"}
    if dt_model is not None:
        res["with_model"] = {"value": rig.world * n * e2e_steps / dt_model / 1e9, "unit": UNIT,
                             "note": "the same plus rb200_model_from_data (one more pass of the input over PCIe for the histogram, "
                                     "normalize_freqs on the host, table upload) in every step"}
    return res


def run_ours(args, rank, local_rank, world):
    rig = Rig(rank, local_rank, world)
    head = measure(rig, args.workload, args.size, args.chunk, args.steps, args.warmup, args.e2e_steps, headline=True,
                   dump_dir=args.dump_outputs)
    configs = {}
    want = args.configs == "all" or (args.configs == "auto" and args.workload == HEADLINE and args.size == 1 << 30)
    if want:
        for name in WORKLOADS:
            if name == args.workload:
                continue
            configs[name] = measure(rig, name, args.size, args.chunk, args.config_steps, 3, min(args.e2e_steps, 2), headline=False)
    if rank != 0:
        if rig.dist:
            rig.dist.barrier()
            rig.dist.destroy_process_group()
        return
    coder_name = WORKLOADS[args.workload][0]
    per_step = head["gpu_launches"] // max(args.steps, 1)
    line = {
        "metric": METRIC, "value": head["value"], "unit": UNIT, "n_gpus": world, "steps": args.steps, "warmup": max(args.warmup, 3),
        "ms_per_step": head["ms_per_step"], "higher_is_better": True, "scaling": "weak", "vs_baseline": None,
        "dtype": "u32", "data": "synthetic",
        "config": {"workload": args.workload, "stands_for": head["stands_for"], "symbols_per_gpu": head["symbols_per_gpu"],
                   "chunk_syms": args.chunk, "lanes": 32, "coder": coder_name, "scale_bits": head["scale_bits"],
                   "compressed_bytes_per_symbol": head["compressed_bytes_per_symbol"],
                   "l2": "inputs (1 GiB symbols + ~1 GiB blob) exceed the 126 MB L2; no flush needed",
                   "step": "encode call (%d launch%s) + decode call (1 launch), device-resident, through the C-ABI"
                           % (per_step - 1, "" if per_step == 2 else "es")},
    }
    for k in ("decode_gsym_s", "encode_gsym_s", "decode_ms", "encode_ms", "roofline", "roofline_encode_call", "gpu_launches",
              "clocks", "e2e", "nccl_blob_gather_ms", "encode_plus_gather_ms", "gather_note"):
        if k in head:
            line[k] = head[k]
    if "encode_plus_gather_ms" in head:        # a second SCALE-visible number: the round trip with the gather in it
        n = head["symbols_per_gpu"]
        line["value_with_gather"] = world * n / ((head["encode_plus_gather_ms"] + head["decode_ms"]) * 1e-3) / 1e9
    if configs:
        line["configs"] = configs
    if world == 1 and not args.no_cpu_baseline:
        _, sb, kind, _ = WORKLOADS[args.workload]
        try:
            line["cpu_baseline"] = cpu_reference_run("zipf" if coder_name == "blocks" else kind,
                                                     "word" if coder_name == "blocks" else coder_name, sb,
                                                     min(args.cpu_sample, head["symbols_per_gpu"]), runs=2, threads=os.cpu_count() or 1)
        except Exception as e:  # the baseline must not take the GPU number down with it
            line["cpu_baseline"] = {"error": repr(e)}
    print(json.dumps(line), flush=True)
    if rig.dist:
        rig.dist.barrier()
        rig.dist.destroy_process_group()


def bind_to_gpu_numa_node(dev_index):
    """Restrict this process to the CPUs of the NUMA node GPU `dev_index` hangs off.  Returns (node, previous
    affinity) or (None, None) when the topology cannot be read; the caller restores the affinity."""
    try:
        import torch
        props = torch.cuda.get_device_properties(dev_index)
        if hasattr(props, "pci_bus_id"):
            bdf = "%04x:%02x:%02x.0" % (props.pci_domain_id, props.pci_bus_id, props.pci_device_id)
        else:
            bdf = subprocess.run(["nvidia-smi", "--query-gpu=pci.bus_id", "--format=csv,noheader", "-i", str(dev_index)],
                                 capture_output=True, text=True, timeout=20).stdout.strip().lower()[-12:]
        path = "/sys/bus/pci/devices/%s/numa_node" % bdf
        node = int(open(path).read())
        if node < 0:
            return None, None
        cpus = set()
        for part in open("/sys/devices/system/node/node%d/cpulist" % node).read().strip().split(","):
            if "-" in part:
                a, b = part.split("-")
                cpus |= set(range(int(a), int(b) + 1))
            elif part:
                cpus.add(int(part))
        saved = os.sched_getaffinity(0)
        cpus &= saved
        if not cpus:
            return None, None
        os.sched_setaffinity(0, cpus)
        return node, saved
    except Exception:  # noqa: BLE001 -- topology files are optional
        return None, None


def main():
    args = parse_args()
    rank = int(os.environ.get("RANK", 0))
    local_rank = int(os.environ.get("LOCAL_RANK", 0))
    world = int(os.environ.get("WORLD_SIZE", 1))
    if args.impl == "reference":
        run_reference(args, rank, world)
    else:
        run_ours(args, rank, local_rank, world)


if __name__ == "__main__":
    main()
