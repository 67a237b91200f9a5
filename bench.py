#!/usr/bin/env python
"""bench.py — throughput of the Predict()/Perceive() hot path on B200 (BASELINE.json metric).

    python bench.py [--gpus N] [--steps K] [--warmup W] [--streams S] [--step-bytes B] [--dump-outputs DIR]
    python bench.py --impl reference ...           # the reference's own CPU implementation on the box's host cores

Workload = BASELINE.json configs[1]: synthetic enwik8-shaped ASCII text (tools/gen_synth.py, seed 0xE9E80001),
coded by the COMPLETE predictor: every model group (54 small models, PPMD, LSTM, FXCM, PAQ8, the 47 gated mixers, SSE)
is device resident; the only input is the byte stream, the only output the probability of every bit. A "step" advances
every stream by --step-bytes bytes (8x as many coded bits). One stream = one reference Predictor = one file.

`value`     input MB/s, streams' bytes already in HBM when the timed region starts. Default --streams 1: the single-file
            figure every BASELINE config is about (latency bound: one bit depends on the previous one).
`aggregate` the same with as many independent files per GPU as fit HBM (labelled; not the headline).
`e2e`       `value`'s workload through cmixb200_code_batch with pinned HOST buffers: H2D of the step's bytes and D2H of
            its probabilities inside the timed region.
`roofline`  the gated-mixer kernel (SURVEY §8d): 450 000 algorithmic B per coded bit / its CUDA-event duration on its own
            stream, against MEASURED_PEAKS.json; `kernels` lists every bulk kernel's measured time per coded bit so that
            the share of each (and the pole) is visible.
`bpc`       cross entropy of the coded prefix from the device's probabilities, next to the reference's on the same bytes.
--dump-outputs DIR writes what the last timed step returned (see dump_outputs) so that two builds can be compared output for
output: the inputs depend only on the arguments.
Multi-GPU (torchrun): independent files per rank, no data-path collective (weak scaling); time = max over ranks.
"""
import argparse
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

os.environ.setdefault("CUDA_DEVICE_MAX_CONNECTIONS", "32")   # before the CUDA context: one work queue per library stream
os.environ.setdefault("CMIXB200_PPMD_MB", "1024")            # PPMD arenas: the library's default is the reference's 14 000 MB heap per stream;
                                                             # the bench files are 20 KB, 1 GB is ample and lets the aggregate figure fit more streams

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.join(ROOT, "tools"))

# algorithmic bytes per coded bit (DESIGN.md §4) and ncu's DRAM bytes per coded bit of one launch (profiles/)
ALGO_BYTES_PER_BIT = {
    "mix_kernel_v3": 450_000,       # SURVEY.md §8(d): 55 172 fp32 weights read + written, + input vectors
    "paq8_kernel": 212_000,         # 28 selected int16 weight sets x 1552 read + written (174 KB) + ~273 live contexts x (64 B bucket line r/w + StateMap cells)
    "fxcm_kernel": 34_000,          # 10 selected weight rows x 512 int16 read + written (20 KB) + ~100 live contexts x 140 B
}
NCU_DRAM_BYTES_PER_BIT = {
    "mix_kernel_v3": 34_786,        # profiles/r01_ncu_full_metrics.csv: (63.16 MB + 8.09 MB) / 2048 bits
    "paq8_kernel": 22_483,          # profiles/r02_ncu_producers.txt: (22.28 MB + 0.74 MB) / 1024 bits (weight sets stay in shared memory)
    "fxcm_kernel": 4_100,           # profiles/r02_ncu_producers.txt
}
KERNELS = ["mix_kernel_v3", "small_kernel", "lstm_kernel", "ppmd_kernel", "fxcm_kernel", "paq8_kernel"]
SEED = 0xE9E80001


def measured_hbm_peak():
    try:
        return float(json.load(open(os.path.join(ROOT, "MEASURED_PEAKS.json")))["hbm_gbs"]), "measured"
    except Exception:
        return 6650.0, "fallback"


class ClockSampler(threading.Thread):
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md)."""

    def __init__(self, index):
        super().__init__(daemon=True)
        self.rows, self.stop_flag, self.index = [], False, index

    def run(self):
        q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
             "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap")
        while not self.stop_flag:
            try:
                out = subprocess.run(["nvidia-smi", "-i", str(self.index), "--query-gpu=" + q, "--format=csv,noheader,nounits"],
                                     capture_output=True, text=True, timeout=5).stdout.strip()
                if out:
                    self.rows.append([c.strip() for c in out.split(",")])
            except Exception:
                pass
            time.sleep(0.2)

    def summary(self):
        if not self.rows:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["unavailable"]}
        sm = sorted(float(r[0]) for r in self.rows)
        reasons = [name for i, name in enumerate(["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"])
                   if any(r[2 + i].lower().startswith("active") for r in self.rows)]
        return {"sm_mhz": sm[len(sm) // 2], "sm_max_mhz": float(self.rows[0][1]), "reasons": reasons}


def bench_text(n_bytes, stream_id=0):
    from gen_synth import synth_text
    return np.frombuffer(synth_text(n_bytes, SEED + stream_id), dtype=np.uint8).copy()


def bench_stream(n_file, stream_id=0):
    """What the predictor sees for an n_file-byte input under `cmix -n`: runner.cpp's stream, i.e. NoPreprocess's 5-byte block
    header (type DEFAULT, big-endian length; preprocessor.cpp:591-600, one segment) followed by the file."""
    head = np.frombuffer(bytes([0]) + int(n_file).to_bytes(4, "big"), dtype=np.uint8)
    return np.concatenate([head, bench_text(n_file, stream_id)])


N_E2E = 10
N_AGG = 3
DUMP_LIMIT = 64 << 20


def dump_outputs(directory, arrays, limit=DUMP_LIMIT):
    """Write every array as directory/<name>.npy (float32 or float64). Past `limit` bytes in all, each array is replaced by the
    same fixed, seeded sample of its flattened elements (sorted positions), sized so that the files stay within the limit."""
    os.makedirs(directory, exist_ok=True)
    total = sum(a.nbytes for a in arrays.values())
    for name, a in arrays.items():
        assert a.dtype in (np.float32, np.float64), name
        if total > limit:
            keep = a.size * limit // total
            a = a.reshape(-1)[np.sort(np.random.default_rng(0).choice(a.size, keep, replace=False))]
        np.save(os.path.join(directory, name + ".npy"), a)


def file_bytes(B, W, K):
    """Length of the synthetic file of one stream: every step of the run consumes fresh bytes of it. The vocabulary (the LSTM's
    symbol set, runner.cpp:196-203) is taken over the whole file, in both arms."""
    return B * (W + K + 1 + N_E2E + N_AGG) - 5      # + the 5-byte block header = a whole number of steps


def reference_run(binary, n_file, n_bytes, step_bytes):
    """One process of the reference (oracle/ref_driver.cpp `time` mode, pinned to core 0) coding the first n_bytes of the
    n_file-byte bench text of stream 0."""
    import tempfile
    with tempfile.TemporaryDirectory() as tmp:
        src = os.path.join(tmp, "in.txt")
        open(src, "wb").write(bench_text(n_file).tobytes())
        cmd = [binary, "time", "n", src, str(n_bytes), "-", str(step_bytes)]
        if subprocess.run(["which", "taskset"], capture_output=True).returncode == 0:
            cmd = ["taskset", "-c", "0"] + cmd
        out = subprocess.run(cmd, capture_output=True, text=True, timeout=3000)
        return json.loads([l for l in out.stdout.splitlines() if l.startswith("{")][-1])


def cpu_baseline(n_file, sample_bytes):
    """The unmodified reference on one host core (it has no threads): the project-flag build (-Ofast, makefile:4; -march=x86-64-v3
    so that the binary built in the CPU container runs here) is the timed baseline, the strict-FP build (the parity oracle) is
    reported next to it. Whole predictor, constructor excluded, `cmix -n` equivalent on the first sample_bytes of the bench text."""
    ref = os.path.join(ROOT, "oracle", "_ref")
    fast, strict = os.path.join(ref, "oracle_dump_fast"), os.path.join(ref, "oracle_dump")
    if not os.path.exists(strict):
        return {"value": None, "unit": "MB/s", "cores": 1, "kind": "unavailable", "sample": "oracle/_ref not built (make -C oracle ref)"}
    r_strict = reference_run(strict, n_file, sample_bytes, 0)
    r_fast = reference_run(fast, n_file, sample_bytes, 0) if os.path.exists(fast) else None
    r = r_fast or r_strict
    return {"value": r["bytes"] / r["code_s"] / 1e6, "unit": "MB/s", "cores": 1, "kind": "reference", "host_cores": os.cpu_count(),
            "build": "-Ofast -march=x86-64-v3 (project flags)" if r_fast else "-O2 strict FP",
            "sample": "first %d bytes of the same stream as stream 0 (block header + file, same vocabulary), whole predictor, one stream, taskset -c 0, constructor (%.1f s) excluded" % (r["bytes"], r["ctor_s"]),
            "strict_value": r_strict["bytes"] / r_strict["code_s"] / 1e6, "bpc_reference": r_strict["bpc"], "bpc_reference_fast_build": r_fast["bpc"] if r_fast else None}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=5)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--streams", type=int, default=int(os.environ.get("CMIXB200_BENCH_STREAMS", "1")), help="independent files per GPU for `value`")
    ap.add_argument("--aggregate-streams", type=int, default=int(os.environ.get("CMIXB200_BENCH_AGG", "7")), help="files per GPU for the aggregate figure (0 = skip)")
    ap.add_argument("--step-bytes", type=int, default=1024)
    ap.add_argument("--cpu-sample-bytes", type=int, default=4096)
    ap.add_argument("--dump-outputs", metavar="DIR", help="write the probabilities the last timed step returned to DIR/p.npy "
                    "(float32, one row of step-bytes x 8 per stream; with several ranks DIR/p_rank<r>.npy)")
    args = ap.parse_args()
    if args.steps < 1:
        ap.error("--steps must be at least 1")
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    S, B, K, W = args.streams, args.step_bytes, args.steps, args.warmup
    config = {"workload": "configs[1]: synthetic enwik8-shaped ASCII text (seed 0xE9E80001), `cmix -n` equivalent; complete predictor, every model "
                          "group device resident (small models, PPMD, LSTM, FXCM, PAQ8, 47 mixers, SSE); no replayed inputs",
              "streams_per_gpu": S, "step_bytes_per_stream": B, "ppmd_arena_mb": int(os.environ["CMIXB200_PPMD_MB"]),
              "parallelism": "independent files sharded over %d rank(s), no data-path collective" % max(world, args.gpus),
              "l2": "inputs larger than L2: every coded byte walks ~22 GB of per-stream HBM tables (hashed buckets of ~330 contexts, 40 mixer weight sets)"}

    if args.impl == "reference":
        if rank != 0:
            return 0
        ref = os.path.join(ROOT, "oracle", "_ref")
        binary = os.path.join(ref, "oracle_dump_fast") if os.path.exists(os.path.join(ref, "oracle_dump_fast")) else os.path.join(ref, "oracle_dump")
        sample = max(256, min(B, 1024))                 # bounded sample per step: the reference needs ~2-5 ms per byte
        r = reference_run(binary, file_bytes(B, W, K), sample * (W + K), sample)
        steps = r["step_s"][W:W + K]
        v = sample * len(steps) / sum(steps) / 1e6
        cb = {"value": v, "unit": "MB/s", "cores": 1, "kind": "reference", "host_cores": os.cpu_count(),
              "build": "-Ofast -march=x86-64-v3 (project flags)" if binary.endswith("_fast") else "-O2 strict FP",
              "sample": "%d steps of %d bytes of the bench text after %d warm-up steps, one process (constructor %.1f s excluded), one stream, taskset -c 0"
                        % (len(steps), sample, W, r["ctor_s"])}
        config["streams_per_gpu"] = 1
        print(json.dumps({"impl": "reference", "metric": "input_MB_per_s", "value": v, "unit": "MB/s", "n_gpus": args.gpus, "steps": K, "warmup": W,
                          "ms_per_step": sum(steps) / len(steps) * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32",
                          "data": "synthetic", "config": config, "cpu_baseline": cb, "bpc": r["bpc"],
                          "e2e": {"value": v, "unit": "MB/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return 0

    import torch
    import cmix_b200
    from cmix_b200.capi import code_batch, code_batch_device
    from cmix_b200.sharding import stream_block, reduce_timing
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device - the B200 path has no CPU fallback")
    dist = None
    if world > 1:
        if os.environ.get("NCCL_DEBUG", "VERSION").upper() == "VERSION":
            os.environ["NCCL_DEBUG"] = "WARN"               # keep NCCL's version banner off stdout: rank 0 prints ONE JSON line
        import torch.distributed as dist_mod
        dist = dist_mod
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank))
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    n_e2e = N_E2E
    total_steps = (file_bytes(B, W, K) + 5) // B
    S_total = max(S, args.aggregate_streams)
    free0 = torch.cuda.mem_get_info(dev)[0]
    streams = []
    for s in stream_block(S_total * world, world, rank):
        if len(streams) >= S_total:
            break
        text = bench_stream(file_bytes(B, W, K), stream_id=s)
        vocab = np.ones(256, dtype=np.uint8)
        if text.size >= 10000:                               # runner.cpp:14,197: short streams keep the full symbol set
            vocab[:] = 0
            vocab[np.unique(text)] = 1
        P = cmix_b200.Predictor(vocab, device=local_rank)
        streams.append(dict(P=P, text=text, pos=0, d_bytes=torch.from_numpy(text).to(dev), d_out=torch.empty(B * total_steps * 8, dtype=torch.float32, device=dev)))
        if len(streams) == 1:   # every stream owns ~22 GB of model tables: run as many as fit (the same number on every rank)
            per_stream = free0 - torch.cuda.mem_get_info(dev)[0] + (256 << 20)
            fit = max(1, int(0.94 * free0 // per_stream))
            if dist:
                t_fit = torch.tensor([fit], device=dev, dtype=torch.int64)
                dist.all_reduce(t_fit, op=dist.ReduceOp.MIN)
                fit = int(t_fit.item())
            S_total = min(S_total, fit)
            S = min(S, fit)
            config["hbm_per_stream_gb"] = round(per_stream / 1e9, 2)
    config["streams_per_gpu"] = S
    torch.cuda.synchronize()

    def run(group, n_steps, timed_kernels=False):
        """n_steps further steps of every stream in `group` (each continues at its own cursor);
        returns (seconds max over ranks, bytes over all ranks, launches, kernel ms dict)."""
        preds = [st["P"] for st in group]
        if timed_kernels:
            for p in preds:
                p.time_mix_kernel(True)
        launches0 = sum(p.kernel_launches for p in preds)
        torch.cuda.synchronize()
        if dist:
            dist.barrier()
        ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        ev0.record()
        t0 = time.perf_counter()
        for _ in range(n_steps):
            code_batch_device(preds, [st["d_bytes"][st["pos"]:st["pos"] + B] for st in group], B, None, None,
                              [st["d_out"][st["pos"] * 8:(st["pos"] + B) * 8] for st in group])
            for st in group:
                st["pos"] += B
        ev1.record()
        torch.cuda.synchronize()
        dt = max(time.perf_counter() - t0, ev0.elapsed_time(ev1) / 1e3)
        nbytes = len(group) * B * n_steps
        if dist:
            dt, nbytes = reduce_timing(dist, dev, dt, nbytes)
            dist.barrier()
        kms = {}
        if timed_kernels:
            for w, name in enumerate(KERNELS):
                ms = n = 0
                for p in preds:
                    a, b = p.kernel_ms(w)
                    ms += a
                    n += b
                kms[name] = (ms, n)
            for p in preds:
                p.time_mix_kernel(False)
        return dt, nbytes, sum(p.kernel_launches for p in preds) - launches0, kms

    head = streams[:S]
    run(head, W)                                          # warm-up (untimed)
    sampler = ClockSampler(local_rank)
    sampler.start()
    dt, total_bytes, launches, kms = run(head, K, timed_kernels=True)
    sampler.stop_flag = True
    sampler.join(timeout=2)
    value = total_bytes / dt / 1e6
    if args.dump_outputs:
        last = torch.stack([st["d_out"][(st["pos"] - B) * 8:st["pos"] * 8] for st in head]).cpu().numpy()
        dump_outputs(args.dump_outputs, {"p" if world == 1 else "p_rank%d" % rank: last}, DUMP_LIMIT // world)

    # ---- end to end through the C-ABI with pinned HOST buffers: the same streams continue ----
    preds = [st["P"] for st in head]
    lo = (W + K) * B
    h_bytes = [torch.from_numpy(st["text"][lo:lo + (n_e2e + 1) * B].copy()).pin_memory() for st in head]
    h_out = [torch.empty((n_e2e + 1) * B * 8, dtype=torch.float32).pin_memory() for _ in head]
    code_batch(preds, h_bytes, B, None, None, h_out)         # one untimed step sizes the staging buffers
    torch.cuda.synchronize()
    if dist:
        dist.barrier()
    t0 = time.perf_counter()
    for j in range(1, n_e2e + 1):
        code_batch(preds, [t[j * B:] for t in h_bytes], B, None, None, [t[j * B * 8:] for t in h_out])
    torch.cuda.synchronize()
    dt_e2e = time.perf_counter() - t0
    if dist:
        tt = torch.tensor([dt_e2e], device=dev, dtype=torch.float64)
        dist.all_reduce(tt, op=dist.ReduceOp.MAX)
        dt_e2e = float(tt.item())
    e2e_value = S * n_e2e * B * world / dt_e2e / 1e6
    if not all(bool(torch.isfinite(o).all()) and float(o.min()) >= 0.0 and float(o.max()) <= 1.0 for o in h_out):
        raise SystemExit("bench.py: end-to-end probabilities out of range")

    # ---- aggregate: as many independent files per GPU as fit HBM (labelled, not the headline) ----
    aggregate = None
    for st in head:
        st["pos"] += (n_e2e + 1) * B                         # the end-to-end steps consumed these bytes
    if S_total > S:
        n_agg = N_AGG
        run(streams[S:], 1)                                  # the extra streams' first step is their warm-up
        dt_a, bytes_a, _, _ = run(streams, n_agg)
        aggregate = {"value": bytes_a / dt_a / 1e6, "unit": "MB/s", "streams_per_gpu": len(streams), "steps": n_agg,
                     "note": "independent files advanced together in one launch set; each is an untouched single-stream predictor (the reference runs one per process)"}

    # ---- the decoder's order on one stream (not part of `value`) ----
    lock = None
    if rank == 0:
        P0 = head[0]["P"]
        bits = np.unpackbits(head[0]["text"][:16])
        for b in bits[:16]:
            P0.Predict(); P0.Perceive(int(b))
        t0 = time.perf_counter()
        for b in bits[16:]:
            P0.Predict(); P0.Perceive(int(b))
        P0.Predict()
        lock = {"us_per_bit": (time.perf_counter() - t0) / (bits.size - 16) * 1e6, "bits": int(bits.size - 16), "note": "cmixb200_predict/perceive through ctypes, every model resident, host clock"}

    if rank == 0:
        peak, peak_kind = measured_hbm_peak()
        n_bits = S * B * K * 8
        per_bit = {k: (v[0] * 1e3 / n_bits if n_bits else None) for k, v in kms.items()}      # us per coded bit (kernels overlap on their own streams)
        pole = max(per_bit, key=lambda k: per_bit[k] or 0) if per_bit else None
        roof = {}
        for kname in ("paq8_kernel", "fxcm_kernel", "mix_kernel_v3"):
            ms, n = kms.get(kname, (0.0, 0))
            if ms <= 0 or n == 0:
                continue
            bits_per_launch = n_bits / n
            ach = ALGO_BYTES_PER_BIT[kname] * bits_per_launch / (ms / n / 1e3) / 1e9
            roof[kname] = {"achieved": ach, "frac": ach / peak, "launches": n, "ms_total": ms, "bits_per_launch": bits_per_launch,
                           "algorithmic_bytes_per_bit": ALGO_BYTES_PER_BIT[kname], "traffic": NCU_DRAM_BYTES_PER_BIT[kname] * bits_per_launch}
        dom = pole if pole in roof else "mix_kernel_v3"
        p_dev = head[0]["d_out"][W * B * 8:(W + K) * B * 8].cpu().numpy().astype(np.float64)
        bits_coded = np.unpackbits(head[0]["text"][W * B:(W + K) * B])
        out = {
            "metric": "input_MB_per_s", "value": value, "unit": "MB/s", "n_gpus": world if world > 1 else args.gpus, "steps": K, "warmup": W,
            "ms_per_step": dt / K * 1e3, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "f32", "data": "synthetic", "config": config,
            "clocks": sampler.summary(),
            "e2e": {"value": e2e_value, "unit": "MB/s", "h2d_bytes_per_step": S * B, "d2h_bytes_per_step": S * B * 8 * 4, "steps": n_e2e,
                    "note": "cmixb200_code_batch with pinned host buffers: the step's bytes go up and its probabilities come back inside the timed region (bytes per rank per step)"},
            "gpu_launches": int(launches),
            "roofline": {"bound": "hbm", "kernel": dom, "achieved": roof[dom]["achieved"], "peak": peak, "unit": "GB/s", "frac": roof[dom]["frac"],
                         "traffic": roof[dom]["traffic"], "traffic_unit": "B per launch",
                         "traffic_source": "ncu --set full DRAM read+write of one launch per coded bit (profiles/r02_ncu_producers.txt, r01_ncu_full_metrics.csv) x bits per launch",
                         "peak_source": "MEASURED_PEAKS.json (%s)" % peak_kind, "per_kernel": roof,
                         "note": "the dominant kernel is the one the stream waits for (longest CUDA-event time per coded bit). Every kernel of this path is LATENCY bound, "
                                 "not bandwidth bound: bit t+1 cannot start before bit t is perceived, the integer models walk dependent hash-bucket chains and every "
                                 "fp32 dot product is one serial FADD chain (bit-exact parity), so the HBM fraction is small by construction"},
            "kernels": {"us_per_coded_bit": per_bit, "pole": pole, "note": "CUDA events on each kernel's own stream; the kernels of a sub-chunk overlap, the stream advances at the pole's pace"},
            "single_stream": {"MB_per_s": value / max(S * world, 1), "hours_per_100MB": 100.0 / max(value / max(S * world, 1), 1e-12) / 3600.0},
            "aggregate": aggregate,
            "bits_per_s": total_bytes * 8 / dt,
            "bpc": float(-np.log2(np.where(bits_coded == 1, p_dev, 1 - p_dev).clip(1.0 / 65536, 1)).sum() / max(bits_coded.size // 8, 1)),
            "bpc_note": "timed region of stream 0 (bytes %d..%d of the bench text); cpu_baseline.bpc_reference is the reference on its first cpu-sample bytes" % (W * B, (W + K) * B),
            "lockstep": lock,
        }
        if world == 1:
            try:
                out["cpu_baseline"] = cpu_baseline(file_bytes(B, W, K), args.cpu_sample_bytes)
                n = min(args.cpu_sample_bytes, (W + K) * B)
                # the device's cross entropy on the same prefix the CPU sample covers
                p0 = head[0]["d_out"][:n * 8].cpu().numpy().astype(np.float64)
                b0 = np.unpackbits(head[0]["text"][:n])
                out["bpc_on_cpu_sample"] = float(-np.log2(np.where(b0 == 1, p0, 1 - p0).clip(1.0 / 65536, 1)).sum() / n)
                out["bpc_sample_bytes"] = n
            except Exception as e:  # the baseline is reported, never required for the GPU number
                out["cpu_baseline"] = {"value": None, "unit": "MB/s", "cores": 1, "kind": "unavailable", "sample": repr(e)}
        if world > 1:
            print(json.dumps(out))
    for st in streams:
        st["P"].close()
    # ---- the decompress direction on the device (SURVEY §8f rank 1; not part of `value`): one file, 512 bytes ----
    if rank == 0 and world == 1:
        try:
            nd = 512
            src = bench_stream(file_bytes(B, W, K))
            vocab = np.ones(256, dtype=np.uint8)
            if src.size >= 10000:
                vocab[:] = 0
                vocab[np.unique(src)] = 1
            enc = cmix_b200.Predictor(vocab, device=local_rank)
            enc.coder_begin(2 * nd + 64)
            enc.code_bytes(src[:nd])
            archive = enc.coder_finish()
            enc.close()
            dec = cmix_b200.Predictor(vocab, device=local_rank)
            torch.cuda.synchronize()
            t0 = time.perf_counter()
            back = dec.decode_bytes(archive, nd)
            dt_dec = time.perf_counter() - t0
            dec.close()
            out["device_decode"] = {"us_per_bit": dt_dec / (nd * 8) * 1e6, "bytes": nd, "round_trip_ok": bool(back.tobytes() == src[:nd].tobytes()),
                                    "note": "cmixb200_decode_bytes: predict kernels, arithmetic-decoder step and perceive kernels queued per bit, the bit never visits the host"}
        except Exception as e:
            out["device_decode"] = {"error": repr(e)}
        print(json.dumps(out))
    if dist:
        dist.destroy_process_group()
    return 0


if __name__ == "__main__":
    sys.exit(main())
