#!/usr/bin/env python
"""bench.py -- face-tokens/sec of the MeshAnything-350M hot path on B200 (BASELINE.json metric).

One "step" = one full pass of the hot path over one batch of synthetic inputs: generate()
of `--faces`*9+2 tokens for `--batch` shapes per GPU (default: BASELINE.json configs[1] = batch 1,
800-face cap, greedy).  Weak scaling: every rank runs the same per-GPU batch on its own shapes;
the only collective is the weight broadcast at init.

    python bench.py [--gpus N] [--steps K] [--warmup W] [--config {2,3,4,5}] [--batch B] [--faces F] [--sampling]
    python bench.py --impl reference ...      # the CPU oracle on the host cores (bounded sample)
    python bench.py ... --dump-outputs DIR    # also write the last timed step's output as DIR/faces.npy

--config selects a BASELINE.json configuration (index + 1): 2 = batch 1, 800 faces, greedy (default, the one the metric
is quoted on); 3 = batch 64, 800 faces, top-k/top-p sampling; 4 = the same per GPU, meant for --gpus 8 (512 shapes);
5 = batch 32 per GPU, 1600 faces (256 shapes on 8 GPUs), sampling.  The default run also appends an `extra` block:
bounded decode-step measurements of configs 3 and 5 (200 steps at three context lengths each, KV cache zero-filled and
the sequence state moved there with ma_decode_slots_seek), each with its own roofline.
"""
from __future__ import annotations

import argparse
import json
import os
import subprocess
import sys
import threading
import time

ROOT = os.path.dirname(os.path.abspath(__file__))
if ROOT not in sys.path:
    sys.path.insert(0, ROOT)

import torch  # noqa: E402

METRIC = "face-tokens/sec (350M, 800-face cap)"
UNIT = "tokens/s"
KV_BYTES_PER_POS = 98304          # 24 layers x K,V x 1024 x fp16  (SURVEY.md 8d)


def measured_peaks():
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        return float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json)"
    return 6650.0, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks + throttle reasons sampled DURING the timed region (B200_PROFILING.md)."""
    Q = ("index,clocks.sm,clocks.max.sm,power.draw,clocks_event_reasons.hw_slowdown,"
         "clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,"
         "clocks_event_reasons.sw_power_cap")

    def __init__(self, index: int):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--query-gpu={self.Q}", "--format=csv,noheader,nounits",
                                          "-lms", "200", "-i", str(self.index)], stdout=subprocess.PIPE, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([c.strip() for c in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        sm = sorted(int(r[1]) for r in self.rows if len(r) >= 8 and r[1].isdigit())
        mx = [int(r[2]) for r in self.rows if len(r) >= 8 and r[2].isdigit()]
        reasons = set()
        for r in self.rows:
            if len(r) >= 8:
                for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[4:8]):
                    if v.lower().startswith("active"):
                        reasons.add(name)
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": sorted(reasons), "samples": len(sm)}


def synthetic_prefix(batch: int, first: int) -> torch.Tensor:
    """Stand-in for processed_point_feature while the encoder leg is timed separately: fp32 [B,257,1024],
    shape i seeded with 1000+i (SURVEY.md 8d)."""
    rows = []
    for i in range(batch):
        g = torch.Generator().manual_seed(1000 + first + i)
        rows.append(torch.randn(257, 1024, generator=g) * 0.7)
    return torch.stack(rows)


_ORACLE_THREADS = None   # OpenMP team size picked once per process by the calibration below


def _usable_cpus() -> int:
    """Logical CPUs this process may actually run on: affinity mask and cgroup CPU quota, not os.cpu_count()."""
    n = os.cpu_count() or 1
    try:
        n = min(n, len(os.sched_getaffinity(0)))
    except (AttributeError, OSError):
        pass
    for path in ("/sys/fs/cgroup/cpu.max", "/sys/fs/cgroup/cpu/cpu.cfs_quota_us"):
        try:
            txt = open(path).read().split()
            if path.endswith("cpu.max"):
                if txt[0] != "max":
                    n = min(n, max(1, int(int(txt[0]) / int(txt[1]) + 0.5)))
            else:
                q = int(txt[0])
                period = int(open("/sys/fs/cgroup/cpu/cpu.cfs_period_us").read())
                if q > 0:
                    n = min(n, max(1, int(q / period + 0.5)))
        except (OSError, ValueError, IndexError):
            pass
    return n


def cpu_oracle_tokens_per_s(sd, n_layers: int, seconds: float = 12.0):
    """The oracle (CPU restatement of the reference decoder) on the host cores: prefill + as many greedy
    decode steps as fit in ~`seconds`, with the OpenMP team size that is fastest on this host (one thread per logical
    CPU can be several times slower than fewer threads when the container may not use all of them: every candidate runs
    a few decode steps first and the best is kept).  Reported baseline only."""
    global _ORACLE_THREADS
    from oracle import decoder as orc
    from oracle.decoder import OracleDecoder, greedy_pick
    ncpu = os.cpu_count() or 1
    oracle = OracleDecoder(sd, n_layers, 257 + 4096)
    prefix = synthetic_prefix(1, 0)[0]
    if _ORACLE_THREADS is not None:
        orc.set_threads(_ORACLE_THREADS)
    t0 = time.time()
    logits = oracle.prefill(prefix)
    t_prefill = time.time() - t0
    tok = greedy_pick(logits)
    n = 0
    tried = {}
    if _ORACLE_THREADS is None:
        cands = sorted({c for c in (ncpu, _usable_cpus(), 96, 64, 48, 32, 24, 16, 8, 4) if 1 <= c <= ncpu}, reverse=True)
        for c in cands:
            orc.set_threads(c)
            tc = time.time()
            k = 0
            while k < 4 or (time.time() - tc < 0.4 and k < 24):   # at least 4 steps, at most ~0.4 s per candidate
                logits = oracle.step(tok, n + 1)
                tok = greedy_pick(logits)
                n += 1
                k += 1
            tried[c] = k / (time.time() - tc)
        _ORACLE_THREADS = max(tried, key=tried.get)
        orc.set_threads(_ORACLE_THREADS)
    n0, t1 = n, time.time()
    while time.time() - t1 < seconds and n < 4000:
        logits = oracle.step(tok, n + 1)
        tok = greedy_pick(logits)
        n += 1
    dt = time.time() - t1
    cal = (" (team sizes tried, tokens/s: " + ", ".join(f"{c}: {v:.1f}" for c, v in tried.items()) + ")") if tried else ""
    return {"value": (n - n0) / dt, "unit": UNIT, "cores": _ORACLE_THREADS, "kind": "port",
            "sample": f"oracle/decoder_oracle.c: 257-token prefill ({t_prefill:.2f}s, not counted) + {n - n0} greedy "
                      f"decode steps at context {257 + n0}..{257 + n} in {dt:.1f}s, batch 1, {n_layers} layers, "
                      f"OpenMP on {_ORACLE_THREADS} of {ncpu} logical CPUs{cal}"}


def batched_decode_steps(arena, n_layers, B, F, sampling, contexts, steps=200, warm=20):
    """Bounded measurement of the batched decode step (BASELINE configs 3-5) at chosen context lengths: the KV cache is
    zero-filled, every slot is moved to the context with ma_decode_slots_seek and `steps` steps are timed with CUDA
    events (device time, CUDA graphs as in ma_decode_generate).  Returns per-context step time, face-tokens/s and the
    achieved fraction of the HBM roofline (weights once per step + KV of B sequences)."""
    import ctypes as C
    from meshanything_b200 import capi
    from meshanything_b200.config import DEC
    L = capi.lib()
    dev = arena.device
    max_new = DEC.max_new_tokens(F)
    tmax = 257 + max_new
    peak, peak_src = measured_peaks()
    kv_bytes = L.ma_kv_cache_bytes(n_layers, B, tmax)
    kv = torch.zeros(kv_bytes, dtype=torch.uint8, device=dev)
    ws = torch.empty(L.ma_decoder_workspace_bytes(B, tmax), dtype=torch.uint8, device=dev)
    ids = torch.full((B, max_new), 2, dtype=torch.int32, device=dev)
    samp = capi.Sampling(int(sampling), 50, 0.95, 0)
    st = capi.stream_ptr()
    capi.check(L.ma_decode_slots_init(B, tmax, 2, capi.ptr(ws), st), "slots_init")
    wbytes = arena.weight_bytes_per_step()
    rows = []
    for ctx in contexts:
        ctx = min(ctx, tmax - steps - warm - 4)

        def run(n, c):
            capi.check(L.ma_decode_slots_step(C.byref(arena.c), B, tmax, max_new, n, c + 1, C.byref(samp), -1, 2,
                                              capi.ptr(kv), capi.ptr(ws), capi.ptr(ids), 0, st), "slots_step")
        capi.check(L.ma_decode_slots_seek(B, tmax, ctx, ctx - 256, 5, capi.ptr(ws), st), "slots_seek")
        run(warm, ctx)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        run(steps, ctx + warm)
        e1.record()
        torch.cuda.synchronize()
        ms = e0.elapsed_time(e1) / steps
        mid = ctx + warm + steps // 2
        alg = wbytes + B * KV_BYTES_PER_POS * (mid + 1)
        rows.append({"context": mid, "ms_per_step": ms, "tokens_per_s": B / (ms / 1e3), "algorithmic_bytes": alg,
                     "achieved_GBps": alg / (ms / 1e3) / 1e9, "frac": alg / (ms / 1e3) / 1e9 / peak})
    del kv, ws
    torch.cuda.empty_cache()
    # harmonic mean over the three contexts ~ a full generate (steps are spread evenly over the contexts)
    tps = len(rows) / sum(1.0 / r["tokens_per_s"] for r in rows)
    return {"batch_per_gpu": B, "faces": F, "sampling": bool(sampling), "kv_cache_GB": kv_bytes / 1e9,
            "steps_timed_per_context": steps, "contexts": rows, "tokens_per_s_over_contexts": tps,
            "peak_GBps": peak, "peak_source": peak_src,
            "kernels": "gemm_ws_kernel (tcgen05, swap-AB, K slices in a cluster) + attention_stream_kernel + sample_kernel in one CUDA graph per step"
                       if sampling else "gemm_canon_kernel + attention_stream_kernel + sample_kernel in one CUDA graph per step",
            "note": "decode steps only (no encoder / prefill / detokenizer); KV zero-filled, state set by ma_decode_slots_seek"}


DUMP_LIMIT_BYTES = 64 << 20


def dump_faces(out_dir: str, faces: torch.Tensor) -> None:
    """Writes what MeshAnything.forward returned in the last timed step -- face coordinates [B, F, 3, 3], NaN where no
    face was generated -- as out_dir/faces.npy in float32, so that two builds can be compared output for output.
    Above DUMP_LIMIT_BYTES a fixed sample of whole shapes (seed 0, ascending shape index) is written instead."""
    import numpy as np
    a = faces.detach().float().cpu()
    if a.numel() * 4 > DUMP_LIMIT_BYTES:
        keep = max(1, DUMP_LIMIT_BYTES // (a[0].numel() * 4))
        rows = torch.randperm(a.shape[0], generator=torch.Generator().manual_seed(0))[:keep].sort().values
        a = a[rows]
    os.makedirs(out_dir, exist_ok=True)
    np.save(os.path.join(out_dir, "faces.npy"), a.numpy())


CONFIGS = {2: dict(batch=1, faces=800, sampling=False), 3: dict(batch=64, faces=800, sampling=True),
           4: dict(batch=64, faces=800, sampling=True), 5: dict(batch=32, faces=1600, sampling=True)}


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=3)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--config", type=int, default=2, choices=[2, 3, 4, 5], help="BASELINE.json configs[config-1]")
    ap.add_argument("--batch", type=int, default=None, help="shapes per GPU (overrides --config)")
    ap.add_argument("--faces", type=int, default=None)
    ap.add_argument("--no-extra", action="store_true", help="skip the bounded config-3/5 decode-step block")
    ap.add_argument("--lean", action="store_true",
                    help="only the contract's two timed regions (value, e2e): no separate stage / short-context runs; the "
                         "roofline then uses the whole step's time (for the long multi-GPU configurations)")
    ap.add_argument("--layers", type=int, default=24)
    ap.add_argument("--sampling", action="store_true")
    ap.add_argument("--flags", type=int, default=0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="write the output of the last timed step (rank 0's shapes) as DIR/faces.npy")
    args = ap.parse_args()
    if args.steps < 1 or args.warmup < 0:
        ap.error("--steps must be >= 1 and --warmup >= 0")
    if args.dump_outputs and args.impl != "ours":
        ap.error("--dump-outputs writes the GPU path's outputs (--impl ours)")
    cfg = CONFIGS[args.config]
    if args.batch is None:
        args.batch = cfg["batch"]
    if args.faces is None:
        args.faces = cfg["faces"]
    args.sampling = args.sampling or cfg["sampling"]

    from meshanything_b200 import parallel
    from meshanything_b200.checkpoint import decoder_specs, make_state_dict
    from meshanything_b200.config import DEC

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    F, B, NL = args.faces, args.batch, args.layers
    max_new = DEC.max_new_tokens(F)
    face_tokens_per_seq = 9 * F
    workload = f"BASELINE configs[{args.config - 1}]: 350M ({NL} layers), batch={B}/GPU, {F}-face cap ({max_new} new tokens), " + (
        "top-k 50 / top-p 0.95 sampling" if args.sampling else "greedy decode")

    specs = decoder_specs(NL)

    # ------------------------------------------------------------------ reference arm (CPU oracle)
    if args.impl == "reference":
        if rank != 0:
            return
        sd = make_state_dict(specs, 0)
        vals = []
        base = None
        for _ in range(max(1, args.warmup > 0) + args.steps):
            base = cpu_oracle_tokens_per_s(sd, NL, seconds=8.0)
            vals.append(base["value"])
        vals = vals[-args.steps:]
        v = sum(vals) / len(vals)
        base["value"] = v
        print(json.dumps({
            "impl": "reference", "metric": METRIC, "value": v, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": 1000.0 / v, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16 weights/activations, f32 accumulate", "data": "synthetic",
            "config": {"workload": workload, "note": "bounded sample of the same workload on the host cores"},
            "cpu_baseline": base,
            "e2e": {"value": v, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}}))
        return

    # ------------------------------------------------------------------ our arm
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device (the product path has no CPU fallback)")
    # stdout must carry exactly ONE JSON line: libraries that print to fd 1 (NCCL's version banner) go to stderr
    sys.stdout.flush()
    saved_stdout = os.dup(1)
    os.dup2(2, 1)
    rank, world, local = parallel.init_from_env()
    dev = torch.device("cuda", local)
    torch.cuda.set_device(dev)
    from meshanything_b200 import capi
    from meshanything_b200.decoder import Generator

    import argparse as _ap
    from meshanything_b200.checkpoint import all_specs
    from meshanything_b200.inputs import synthetic_pc_normal
    from MeshAnything.models.meshanything import MeshAnything
    full_specs = all_specs(NL)
    sd_host = make_state_dict(full_specs, 0) if rank == 0 else None
    bstats = {}
    sd = parallel.broadcast_state_dict(sd_host, full_specs, dev, stats=bstats)  # ONE NCCL broadcast; no collective in the step
    del sd_host
    margs = _ap.Namespace(llm="facebook/opt-350m", codebook_size=8192, codebook_dim=1024, n_max_triangles=F, seed=0)
    model = MeshAnything(margs)
    if NL != 24:
        model.expected_keys = lambda: list(full_specs.keys())
    model.load_state_dict(sd, strict=True, device=dev)
    arena = model._dec
    del sd
    torch.cuda.empty_cache()
    tmax = 257 + max_new
    gen = model._generator(B)
    flags = args.flags | capi.GEN_NO_EARLY_EXIT
    pc_host = synthetic_pc_normal(B, first=rank * B).pin_memory()     # fp16 [B,4096,6]
    pc_dev = pc_host.to(dev)
    _, prefix_dev = model.point_encoder.encode_with_prefix(pc_dev)
    prefix_dev = prefix_dev.clone()

    def one_step_resident():                                          # the whole hot path, inputs resident in HBM
        return model(pc_dev, sampling=args.sampling)

    def one_step_e2e():                                               # public API, host buffers in and out
        return model(pc_host, sampling=args.sampling).to("cpu")

    def barrier():
        if world > 1:
            torch.distributed.barrier()
        torch.cuda.synchronize()

    def timed(fn, k):
        barrier()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(k):
            out = fn()
        e1.record()
        barrier()
        ms = e0.elapsed_time(e1)
        if world > 1:
            t = torch.tensor([ms], device=dev)
            torch.distributed.all_reduce(t, op=torch.distributed.ReduceOp.MAX)
            ms = float(t.item())
        return ms, out

    for _ in range(args.warmup):
        one_step_resident()
    launches0 = capi.lib().ma_launch_count()
    sampler = ClockSampler(local)
    sampler.start()
    try:
        ms, out = timed(one_step_resident, args.steps)
    finally:
        clocks = sampler.stop()   # never leave the nvidia-smi sampler running
    launches = capi.lib().ma_launch_count() - launches0
    if args.dump_outputs and rank == 0:
        dump_faces(args.dump_outputs, out)
    ms_e2e, out_e2e = timed(one_step_e2e, args.steps)
    e2e_remeasured = None
    if ms_e2e > 1.5 * ms:   # the e2e pass only adds ~50 KB of copies: a large gap is a disturbed measurement, not the path
        e2e_remeasured = ms_e2e
        ms_e2e, out_e2e = timed(one_step_e2e, args.steps)
    mega_err = gen.mega_error() if (B == 1 and not args.sampling) else 0
    # stage split of one pass (encoder / decode loop / detokenizer), device timed
    if args.lean:
        ms_enc, ms_gen, gen_out = 0.0, ms, (model.last_ids,)
    else:
        ms_enc, _ = timed(lambda: model.point_encoder.encode_with_prefix(pc_dev), args.steps)
        ms_gen, gen_out = timed(lambda: gen.generate(prefix_dev, max_new, do_sample=args.sampling, seed=0, flags=flags),
                                args.steps)
    ms_all = ms

    ids = gen_out[0]
    ms = ms_gen   # the roofline below is about the decode loop
    n_tokens = world * B * face_tokens_per_seq * args.steps
    value = n_tokens / (ms_all / 1000.0)
    e2e_value = n_tokens / (ms_e2e / 1000.0)

    # ---- roofline of the decode step (the HBM-bound part): algorithmic bytes per token-step / time per step
    peak, peak_src = measured_peaks()
    wbytes = arena.weight_bytes_per_step()
    n_dec = max_new - 1                                           # decode steps per generate (step 0 is the prefill)
    kv_read = sum(KV_BYTES_PER_POS * (257 + i) for i in range(1, max_new)) * B
    kv_write = KV_BYTES_PER_POS * n_dec * B
    alg_bytes_per_gen = wbytes * n_dec + kv_read + kv_write
    # short-context GEMV-dominated slice: (T(300 tokens) - T(100 tokens)) / 200 steps
    def short(nn):
        g2 = Generator(arena, B, tmax)
        for _ in range(2):
            g2.generate(prefix_dev, nn, flags=flags)
        t, _ = timed(lambda: g2.generate(prefix_dev, nn, flags=flags), 3)
        return t / 3
    n_lo, n_hi = (100, 300) if max_new >= 300 else (max(2, max_new // 4), max_new)
    if args.lean:
        t100 = n_lo * ms / args.steps / max_new
        t300 = n_hi * ms / args.steps / max_new
    else:
        t100, t300 = short(n_lo), short(n_hi)
    us_step_short = (t300 - t100) / float(n_hi - n_lo) * 1000.0
    short_bytes = wbytes + KV_BYTES_PER_POS * B * (257 + (n_lo + n_hi) // 2 + 1)
    t_prefill_ms = t100 - (n_lo - 1) * us_step_short / 1000.0
    dec_ms = ms / args.steps - max(0.0, t_prefill_ms)             # decode-loop part of one generate
    achieved = alg_bytes_per_gen / (dec_ms / 1000.0) / 1e9
    traffic = None   # DRAM bytes per decode token from the committed ncu --set full capture of the same kernel
    for tag in ("r02", "r01"):     # the newest committed `ncu --set full` capture of the persistent kernel
        tpath = os.path.join(ROOT, "profiles", f"traffic_{tag}.json")
        if B == 1 and not args.sampling and os.path.exists(tpath):
            traffic = json.load(open(tpath))["traffic_bytes_per_token"]
            break
    roofline = {
        "bound": "hbm",
        "kernel": ("decode_mega_kernel (persistent: all 121 phases of a token, 512 tokens per launch)"
                   if (B == 1 and not args.sampling and not (flags & capi.GEN_NO_MEGA)) else
                   "decode step = 97 fast_gemv_kernel + 24 attention_kernel launches (one CUDA graph)" if B == 1 else
                   "decode step: gemm_ws_kernel (tcgen05 swap-AB, K slices in a cluster) + attention_stream_kernel + sample_kernel, one CUDA graph"
                   if args.sampling else "decode step (gemm_canon + attention kernels, one CUDA graph)"),
        "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak, "peak_source": peak_src,
        "traffic": traffic,
        "algorithmic_bytes_per_launch": alg_bytes_per_gen / n_dec,
        "launch": "one decode step (one token of every sequence); bytes = fp16 weights %d + KV read/write averaged over the run" % wbytes,
        "us_per_step_avg": dec_ms * 1000.0 / n_dec,
        "short_context": {"us_per_step": us_step_short, "bytes_per_step": short_bytes,
                          "achieved": short_bytes / us_step_short / 1e3, "frac": short_bytes / us_step_short / 1e3 / peak,
                          "note": "steps at context ~%d..%d (GEMV-dominated): (T(%d)-T(%d))/%d" % (257 + n_lo, 257 + n_hi, n_hi, n_lo, n_hi - n_lo)},
        "prefill_ms": t_prefill_ms,
        "lean": bool(args.lean),
    }

    extra = None
    if rank == 0 and world == 1 and args.config == 2 and B == 1 and NL == 24 and not args.no_extra:
        del gen
        model._gens.clear()
        torch.cuda.empty_cache()
        try:
            extra = {"config3_batch64_F800_sampling": batched_decode_steps(arena, NL, 64, 800, True, [450, 3850, 7300]),
                     "config5_batch32_F1600_sampling": batched_decode_steps(arena, NL, 32, 1600, True, [450, 7300, 14400])}
        except Exception as e:  # noqa: BLE001  (an extra must never cost the headline line)
            extra = {"error": str(e)[:300]}
    if rank == 0:
        cpu = None
        if not args.no_cpu_baseline and world == 1:
            cpu = cpu_oracle_tokens_per_s(make_state_dict(specs, 0), NL)
        line = {
            "metric": METRIC, "value": value, "unit": UNIT, "n_gpus": world, "steps": args.steps,
            "warmup": args.warmup, "ms_per_step": ms_all / args.steps, "higher_is_better": True, "scaling": "weak",
            "vs_baseline": None, "dtype": "f16 weights/activations, f32 accumulate", "data": "synthetic",
            "config": {"workload": workload, "global_batch": B * world, "parallelism": f"dp{world} (batch sharded, "
                       "weights broadcast once over NCCL)",
                       "weight_broadcast": {"bytes": bstats.get("bytes"), "ms": bstats.get("ms"),
                                            "note": "one collective at init, outside the timed region; Linear parameters as fp16"},
                       "inputs": "pc_normal fp16 [B,4096,6] resident in HBM; one step = encoder + generate + detokenize",
                       "stage_ms": {"encoder": ms_enc / args.steps, "generate": ms_gen / args.steps,
                                    "detokenize_and_rest": max(0.0, (ms_all - ms_enc - ms_gen) / args.steps)},   # separate runs: noise can exceed it
                       "l2": "inputs larger than L2: 623.5 MB of weights + KV streamed per token (L2 = 126 MB)",
                       "checkpoint": "synthetic seed 0 (random weights: no early EOS, every sequence runs the cap)"},
            "roofline": roofline, "cpu_baseline": cpu,
            "e2e": {"value": e2e_value, "unit": UNIT, "h2d_bytes_per_step": int(pc_host.numel() * 2),
                    "d2h_bytes_per_step": int(out_e2e.numel() * 4),
                    "api": "MeshAnything.models.meshanything.MeshAnything.forward(pc_normal on the host) -> .cpu()",
                    "first_attempt_ms_discarded": e2e_remeasured},
            "gpu_launches": int(launches), "clocks": clocks, "extra": extra,
            "check": {"first_ids": ids[0, :8].cpu().tolist(), "persistent_kernel_poll_timeouts": int(mega_err)},
        }
        sys.stdout.flush()
        os.dup2(saved_stdout, 1)
        print(json.dumps(line), flush=True)
        os.dup2(2, 1)
    if world > 1:
        torch.distributed.destroy_process_group()


if __name__ == "__main__":
    main()
