#!/usr/bin/env python
"""bench.py -- Llama-3-8B AWQ-INT4 batch-1 decode on B200 (BASELINE.json configs[1] at N = 1, configs[4] = tensor-parallel decode at
N > 1), the reference's own CPU path beside it.

    python bench.py --gpus N --steps K --warmup W            # this repo's CUDA path (one rank per GPU under torchrun)
    python bench.py --impl reference --gpus N --steps K --warmup W   # the reference's own AVX CPU path (rank 0 only)
    python bench.py ... --dump-outputs DIR   # also write what the last timed step returned as DIR/*.npy (same inputs every run)

A "step" is one decode token of the synthetic Llama-3-8B (random AWQ-INT4 weights in the reference's QM_CUDA layout, random-filled
fp16 KV cache).  The K timed steps are spread evenly over context lengths 1 -> max_ctx, so ms_per_step estimates the mean cost per
token of a 1 -> 4096 generation.  `value` = tokens/s with token ids already in HBM (tce_llama_decode); `e2e` = the same through the host
entry point (tce_llama_decode_host): token id/position copied from pinned host memory and the fp32 logits row + greedy token copied
back, every step, inside the timed region.  N > 1 defaults to tensor-parallel decode of ONE sequence (column/row sharded linears,
two all-reduces per layer over NVLink peer memory inside the persistent kernel); `tp_parity_rel_err` compares its logits with a
single-GPU run of the same weights before timing.  One JSON line on stdout (rank 0).  See DESIGN.md "Measurement".
"""
from __future__ import annotations

import argparse
import os as _os

_os.environ["NCCL_DEBUG"] = _os.environ.get("TCE_NCCL_DEBUG", "WARN")  # a pod-wide NCCL_DEBUG=VERSION prints to stdout
_os.environ.setdefault("NCCL_DEBUG_FILE", "/dev/stderr")  # NCCL's version / debug lines must not land on stdout next to the JSON line

import json
import os
import sys
import threading
import time
from pathlib import Path

ROOT = Path(__file__).resolve().parent
sys.path.insert(0, str(ROOT))

METRIC = "llama3_8b_awq_int4_batch1_decode_tokens_per_s"
UNIT = "tok/s"


def load_traffic():
    """dram__bytes_read + dram__bytes_write of one decode_persistent_kernel launch from this round's `ncu --set full` capture
    (profiles/roofline_traffic.json, written by tools/ncu_launch_summary.py); None if absent."""
    p = ROOT / "profiles" / "roofline_traffic.json"
    try:
        d = json.loads(p.read_text())
        return d.get("dram_bytes_per_launch"), d.get("source")
    except Exception:
        return None, None


def workload_config(geom, args, world: int, tp: bool) -> dict:
    """The `config` object both arms report (identical keys and values): names the workload, no model-architecture keys."""
    return {
        "workload": (f"{geom.name} AWQ-INT4 g128 batch-1 decode, timed steps spread over ctx 1->{args.max_ctx}" if args.ctx < 0
                     else f"{geom.name} AWQ-INT4 g128 batch-1 decode at ctx {args.ctx}"),
        "sequences": 1 if (world == 1 or tp) else world,
        "max_ctx": args.max_ctx,
        "parallelism": (f"tp{world}: one sequence, column/row sharded linears, 2 all-reduces per layer over NVLink peer memory" if tp else
                        (f"{world} independent sequences, one per GPU (no collective)" if world > 1 else "single GPU")),
    }


def env_rank():
    return int(os.environ.get("RANK", "0")), int(os.environ.get("LOCAL_RANK", "0")), int(os.environ.get("WORLD_SIZE", "1"))


# ------------------------------------------------------------------------------------------------------------------
# clocks: sample NVML during the timed region (B200_PROFILING.md timing hygiene)
# ------------------------------------------------------------------------------------------------------------------
class ClockSampler:
    REASONS = {0x1: "gpu_idle", 0x2: "applications_clocks_setting", 0x4: "sw_power_cap", 0x8: "hw_slowdown", 0x10: "sync_boost",
               0x20: "sw_thermal_slowdown", 0x40: "hw_thermal_slowdown", 0x80: "hw_power_brake_slowdown", 0x100: "display_clock_setting"}

    def __init__(self, index: int):
        self.samples, self.reasons, self.max_mhz = [], set(), None
        self._stop = threading.Event()
        self._thr = None
        try:
            import pynvml

            pynvml.nvmlInit()
            self.nv = pynvml
            self.h = pynvml.nvmlDeviceGetHandleByIndex(index)
            self.max_mhz = pynvml.nvmlDeviceGetMaxClockInfo(self.h, pynvml.NVML_CLOCK_SM)
        except Exception:
            self.nv = None

    def _run(self):
        while not self._stop.is_set():
            try:
                self.samples.append(self.nv.nvmlDeviceGetClockInfo(self.h, self.nv.NVML_CLOCK_SM))
                r = self.nv.nvmlDeviceGetCurrentClocksEventReasons(self.h) if hasattr(self.nv, "nvmlDeviceGetCurrentClocksEventReasons") \
                    else self.nv.nvmlDeviceGetCurrentClocksThrottleReasons(self.h)
                for bit, name in self.REASONS.items():
                    if r & bit and name != "gpu_idle":
                        self.reasons.add(name)
            except Exception:
                pass
            self._stop.wait(0.02)

    def __enter__(self):
        if self.nv:
            self._thr = threading.Thread(target=self._run, daemon=True)
            self._thr.start()
        return self

    def __exit__(self, *a):
        self._stop.set()
        if self._thr:
            self._thr.join()

    def summary(self):
        s = sorted(self.samples)
        return {"sm_mhz": (s[len(s) // 2] if s else None), "sm_max_mhz": self.max_mhz, "reasons": sorted(self.reasons), "samples": len(s)}


def load_peaks():
    p = ROOT / "MEASURED_PEAKS.json"
    if p.exists():
        d = json.loads(p.read_text())
        return d, float(d["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    return {}, 6650.0, "fallback (B200_PROFILING.md 6.65 TB/s)"


# ------------------------------------------------------------------------------------------------------------------
# reference arm / cpu_baseline: the reference's AVX W4A8 path (oracle/_ref/libtce_ref_avx.so) on the host cores
# ------------------------------------------------------------------------------------------------------------------
class CpuReferenceDecode:
    """The linears of one decode token driven through the reference's own CPU kernel (Linear_FP_int4::forward's
    mat_mul_accelerator_int8_int4_fast_no_offset, QM_x86 g32 format, oracle/ref_shim.cc fills matmul_params like
    llm/src/ops/linear.cc:171-236) with all host threads.  `token()` runs EVERY linear of a token once -- num_layers x (q k v o gate up
    down) + lm_head -- cycling over `distinct` separately allocated layers so that the weights do not stay cache resident.  Attention
    and norms are NOT part of the timed value, which therefore flatters the reference: reference_attention_cost() below measures what its
    attention module adds per token on the same host and the lines report it next to the value."""

    def __init__(self, geom, distinct: int = 4, threads: int = 0, with_lm_head: bool = True):
        import numpy as np

        from oracle import capi

        self.np, self.capi, self.geom = np, capi, geom
        # the reference's worker pool is a function-local static sized by the FIRST call of the process (kernels/avx/matmul_avx_int8_int4.cc:340), so
        # the thread count is fixed here, before any call; `threads` = 0: every host thread
        self.cores = threads if threads > 0 else (os.cpu_count() or 1)
        if capi.ref_available("avx"):
            self.kind, self.X = "reference", capi.ref("avx")
        else:
            self.kind, self.X, self.cores = "port", None, 1
        hd, E, F = geom.head_dim, geom.embed_dim, geom.hidden_dim
        shapes = [(geom.num_heads * hd, E), (geom.num_kv_heads * hd, E), (geom.num_kv_heads * hd, E), (E, geom.num_heads * hd), (F, E), (F, E), (E, F)]
        rng = np.random.default_rng(0)
        self.distinct = max(1, min(distinct, geom.num_layers))
        self.layers = [[(self._make(oc, ic, rng), oc, ic) for oc, ic in shapes] for _ in range(self.distinct)]
        self.lm = (self._make(geom.vocab_size if with_lm_head else 128, E, rng), geom.vocab_size if with_lm_head else 128, E)
        if with_lm_head:
            self.token()  # warm-up (also creates the reference's static thread pool with `cores` threads)

    def _make(self, oc, ic, rng):
        np, capi = self.np, self.capi
        B = capi.aligned_empty((oc, ic // 2), np.uint8)
        B[:] = rng.integers(0, 256, (oc, ic // 2), dtype=np.uint8)
        S = capi.aligned_empty((oc, ic // 32), np.float32)
        S[:] = (rng.random((oc, ic // 32), dtype=np.float32) + 0.5) * 0.004
        A = capi.aligned_empty((1, ic), np.float32)
        A[:] = rng.standard_normal((1, ic), dtype=np.float32)
        Cc = capi.aligned_empty((1, oc), np.float32)
        xi8 = capi.aligned_empty((ic,), np.int8)
        xs = capi.aligned_empty((ic // 32,), np.float32)
        return A, B, S, Cc, xi8, xs

    def _run(self, t, oc, ic):
        A, B, S, Cc, xi8, xs = t
        if self.X is not None:
            self.X.ref_w4a8_avx(A.ctypes.data, B.ctypes.data, S.ctypes.data, Cc.ctypes.data, xi8.ctypes.data, xs.ctypes.data, 1, ic, oc, self.cores)
        else:  # oracle port of the naive path (scalar, 1 core): only when oracle/_ref could not be built
            self.capi.naive_mat_mul_int4(self.np.asarray(A), self.np.asarray(B), self.np.asarray(S), 8.0, 32)

    def token(self) -> float:
        t0 = time.perf_counter()
        for l in range(self.geom.num_layers):
            for t, oc, ic in self.layers[l % self.distinct]:
                self._run(t, oc, ic)
        self._run(*self.lm)
        return time.perf_counter() - t0

    def ops(self):
        """the linears of one token in execution order: (tensors, oc, ic, weight bytes)"""
        seq = []
        for l in range(self.geom.num_layers):
            for t, oc, ic in self.layers[l % self.distinct]:
                seq.append((t, oc, ic, oc * ic // 2))
        seq.append((*self.lm, self.lm[1] * self.lm[2] // 2))
        return seq

    def slice_runner(self, slices: int):
        """Bounded samples: a step = the next 1/`slices` of a token's linears (by weight bytes, in execution order, continuing where the previous
        step stopped), so that `slices` consecutive steps are exactly one full token.  Returns step() -> (seconds, fraction of a token done)."""
        seq = self.ops()
        total = float(sum(o[3] for o in seq))
        state = {"i": 0}

        def step():
            done, t0 = 0.0, time.perf_counter()
            while True:
                t, oc, ic, nbytes = seq[state["i"] % len(seq)]
                self._run(t, oc, ic)
                state["i"] += 1
                done += nbytes
                if done >= total / slices - 1e-9:
                    break
            return time.perf_counter() - t0, done / total

        return step

    def describe(self, n):
        g = self.geom
        return (f"{n} full tokens: every linear of a {g.name} decode step ({g.num_layers} layers x 7 + lm_head) through the reference's W4A8 AVX kernel "
                f"(g32 CPU format), {self.distinct} distinct layers' weights cycled; attention/norms not included (see excluded_attention)")


def reference_attention_cost(geom, cores: int, ctx: int = 512, steps: int = 8):
    """What the linears-only CPU number leaves out, measured instead of assumed: one layer of the reference's OWN Int4llamaAttention module (CPU build
    compiled in place, oracle/_ref/libtce_ref_llama.so: q/k/v/o linears, RoPE, KV concat, the GQA `repeat` copies, BMM_F32T, softmax --
    llm/src/nn_modules/non_cuda/Int4llamaAttention.cc:288-442) at this model's widths, timed per single-token call after a prompt of 1 and of `ctx`
    tokens with NUM_THREAD = `cores`.  The difference is the attention core at that context; x num_layers = its cost per token.  Bounded: a few seconds."""
    import shutil
    import tempfile

    import numpy as np

    from oracle import capi

    if not (capi.REF_DIR / "libtce_ref_llama.so").exists():
        return {"unavailable": "oracle/_ref/libtce_ref_llama.so not built"}
    hd, E, H, KVH = geom.head_dim, geom.embed_dim, geom.num_heads, geom.num_kv_heads
    rng = np.random.default_rng(3)
    W = {name: (rng.standard_normal((rows, E)) * 0.02).astype(np.float32) for name, rows in (("q_proj", H * hd), ("k_proj", KVH * hd), ("v_proj", KVH * hd), ("o_proj", E))}
    max_sq = ctx + steps + 8
    cosb, sinb = capi.rope_tables(max_sq, hd, geom.rope_theta)
    root = tempfile.mkdtemp(prefix="tce_ref_attn_")
    try:
        capi.write_llama_attention_params(root, W, cosb, sinb, np.float32(1.0 / np.sqrt(hd)))
        per_step = {}
        for past in (1, ctx):
            hidden = rng.standard_normal((past + steps, E)).astype(np.float32)
            *_, secs = capi.ref_int4_llama_attention(root, hidden, E, H, KVH, past, steps, max_sq, num_thread=cores, timing=True)
            per_step[past] = secs / steps
    finally:
        shutil.rmtree(root, ignore_errors=True)
    core = max(0.0, per_step[ctx] - per_step[1])
    return {"module": "Int4llamaAttention::forward (reference CPU build), one layer, single-token calls", "cores": cores, "ctx": ctx,
            "ms_per_layer_at_ctx_1": per_step[1] * 1e3, f"ms_per_layer_at_ctx_{ctx}": per_step[ctx] * 1e3,
            "attention_core_ms_per_token": core * 1e3 * geom.num_layers,
            "note": f"the timed value covers the linears only; at ctx {ctx} the reference's attention core (everything in the module besides its four linears) adds this "
                    f"many ms per token ({geom.num_layers} layers), growing about linearly with the context"}


def pick_reference_threads(model: str) -> int:
    """NUM_THREAD is the reference user's choice (llm/application/chat.cc:123,156).  Its static pthread pool does not scale to every thread of a
    128-thread host (measured: 128 threads are ~8x slower than 8 on the linears of a token), so the arm uses the best of a few counts, each probed
    in its own process (the pool size is fixed by a process's first call) on one layer's seven linears."""
    import subprocess

    cores = os.cpu_count() or 1
    best, best_t = cores, float("inf")
    for c in sorted({x for x in (4, 8, 16, 32, 64, cores) if x <= cores}):
        try:
            r = subprocess.run([sys.executable, str(Path(__file__).resolve()), "--probe-threads", str(c), "--model", model], capture_output=True, text=True,
                               timeout=180)
            t = float(r.stdout.strip().splitlines()[-1])
        except Exception:
            continue
        if t < best_t:
            best, best_t = c, t
    return best


def probe_threads(args):
    from tinychatengine_b200.llama import GEOMETRIES

    ref = CpuReferenceDecode(GEOMETRIES[args.model], distinct=1, threads=args.probe_threads, with_lm_head=False)
    ts = []
    for _ in range(4):
        t0 = time.perf_counter()
        for t, oc, ic in ref.layers[0]:
            ref._run(t, oc, ic)
        ts.append(time.perf_counter() - t0)
    print(sorted(ts)[1])


def cpu_baseline(geom, budget_s: float):
    ref = CpuReferenceDecode(geom, threads=pick_reference_threads(geom.name))
    times = []
    t0 = time.perf_counter()
    while not times or (time.perf_counter() - t0 < budget_s and len(times) < 16):
        times.append(ref.token())
    med = sorted(times)[len(times) // 2]
    out = {"value": 1.0 / med, "unit": UNIT, "cores": ref.cores, "kind": ref.kind, "sample": ref.describe(len(times))}
    try:
        out["excluded_attention"] = reference_attention_cost(geom, ref.cores)
    except Exception as ex:
        out["excluded_attention"] = {"error": repr(ex)}
    return out


def cpu_baseline_w8a8(budget_s: float = 6.0):
    """configs[2] beside the GPU number: the six linears of one Int8OPTDecoderLayer-shaped layer at the Llama-2-7B widths, M = 1, through the
    reference's own AVX int8 kernels (oracle/_ref/libtce_ref_avx.so: mat_mul_accelerator_int8_fast_32unroll_over_column for q/k/v/fc1,
    ..._bfp32_ofp32_over_column for out_proj/fc2 -- the methods W8A8B8O8Linear / W8A8BFP32OFP32Linear call at m == 1, kernels/avx/matmul_avx_int8.cc),
    NUM_THREAD = the fastest of a few (these kernels create their threads per call); the BMMs / softmax / LayerNormQ of the layer are not included."""
    import numpy as np

    from oracle import capi

    if not capi.ref_available("avx"):
        return {"unavailable": "oracle/_ref/libtce_ref_avx.so not built"}
    E, F = 4096, 11008
    rng = np.random.default_rng(1)
    mats = []  # (variant, A, B, bias8, biasf, q_min): weights of 3 distinct layers are cycled so that they do not stay cache resident
    for _ in range(3):
        layer = []
        for variant, n, k, q_min in ((1, E, E, -128), (1, E, E, -128), (1, E, E, -128), (5, E, E, -128), (1, F, E, 0), (5, E, F, -128)):
            B = capi.aligned_empty((n, k), np.int8)
            B[:] = rng.integers(-127, 128, (n, k), dtype=np.int8)
            A = capi.aligned_empty((1, k), np.int8)
            A[:] = rng.integers(-127, 128, (1, k), dtype=np.int8)
            b8 = rng.integers(-127, 128, (n,), dtype=np.int8) if variant == 1 else None
            bf = rng.standard_normal(n).astype(np.float32) if variant == 5 else None
            layer.append((variant, A, B, b8, bf, q_min))
        mats.append(layer)
    wbytes = 4 * E * E + 2 * E * F

    def one_layer(layer, threads):
        t0 = time.perf_counter()
        for variant, A, B, b8, bf, q_min in layer:
            capi.ref_int8_matmul(variant, A, B, b8, bf, 0.00050354, 0.0213013, q_min, 127, kind="avx", num_thread=threads)
        return time.perf_counter() - t0

    cores = os.cpu_count() or 1
    cands = [c for c in (4, 8, 16, 32) if c <= cores] or [1]  # the over_column kernels need N % (8 * threads) == 0: 4096 and 11008 allow up to 32
    best, best_t = cands[0], float("inf")
    for c in cands:
        one_layer(mats[0], c)
        t = min(one_layer(mats[i % 3], c) for i in range(1, 4))
        if t < best_t:
            best, best_t = c, t
    times, t0, i = [], time.perf_counter(), 0
    while not times or (time.perf_counter() - t0 < budget_s and len(times) < 64):
        times.append(one_layer(mats[i % 3], best))
        i += 1
    med = sorted(times)[len(times) // 2]
    return {"ms_per_layer_linears": med * 1e3, "weight_GB_per_s": wbytes / med / 1e9, "tok_s_at_32_layers": 1.0 / (32 * med), "cores": best, "kind": "reference",
            "sample": f"{len(times)} passes over the six linears of one layer (M = 1; q/k/v/o 4096x4096, fc1 11008x4096 ReLU, fc2 4096x11008), 3 layers' weights cycled; "
                      "the reference's AVX int8 kernels; attention BMMs / softmax / LayerNormQ not included"}


def cpu_baseline_prefill(cores: int, model: str = "llama2-13b", m: int = 128):
    """configs[3] beside the GPU number, as SURVEY.md 8(d) asks: the reference's AVX W4A8 path on a REDUCED prompt -- the seven linears of one layer of the
    13B model at M = 128 rows (2048 rows of all 40 layers would take minutes) -- timed once after a warm-up and scaled to tokens/s of the full model
    (x num_layers; attention / norms / lm_head not included), labelled as such.  `cores`: the pool size this process already fixed (see CpuReferenceDecode)."""
    import numpy as np

    from oracle import capi
    from tinychatengine_b200.llama import GEOMETRIES

    if not capi.ref_available("avx"):
        return {"unavailable": "oracle/_ref/libtce_ref_avx.so not built"}
    g = GEOMETRIES[model]
    hd, E, F = g.head_dim, g.embed_dim, g.hidden_dim
    shapes = [(g.num_heads * hd, E), (g.num_kv_heads * hd, E), (g.num_kv_heads * hd, E), (E, g.num_heads * hd), (F, E), (F, E), (E, F)]
    rng = np.random.default_rng(2)
    X = capi.ref("avx")
    ops = []
    for oc, ic in shapes:
        B = capi.aligned_empty((oc, ic // 2), np.uint8)
        B[:] = rng.integers(0, 256, (oc, ic // 2), dtype=np.uint8)
        S = capi.aligned_empty((oc, ic // 32), np.float32)
        S[:] = (rng.random((oc, ic // 32), dtype=np.float32) + 0.5) * 0.004
        A = capi.aligned_empty((m, ic), np.float32)
        A[:] = rng.standard_normal((m, ic), dtype=np.float32)
        ops.append((A, B, S, capi.aligned_empty((m, oc), np.float32), capi.aligned_empty((m * ic,), np.int8), capi.aligned_empty((m * ic // 32,), np.float32), oc, ic))

    def layer():
        t0 = time.perf_counter()
        for A, B, S, Cc, xi8, xs, oc, ic in ops:
            X.ref_w4a8_avx(A.ctypes.data, B.ctypes.data, S.ctypes.data, Cc.ctypes.data, xi8.ctypes.data, xs.ctypes.data, m, ic, oc, cores)
        return time.perf_counter() - t0

    layer()
    t = min(layer(), layer())
    flops = 2.0 * m * sum(oc * ic for *_, oc, ic in ops)
    return {"model": model, "rows": m, "s_per_layer_linears": t, "linear_tflops": flops / t / 1e12, "tok_per_s_scaled": m / (t * g.num_layers), "cores": cores,
            "kind": "reference",
            "sample": f"one layer's seven linears at M = {m} through the reference's W4A8 AVX kernel (g32 CPU format), best of 2 after a warm-up; "
                      f"tok/s scaled by {g.num_layers} layers (attention, norms, lm_head not included): an estimate, not a measurement of a {2048}-token prompt"}


def run_reference(args):
    rank, _, world = env_rank()
    if rank != 0:
        return
    from tinychatengine_b200.llama import GEOMETRIES

    geom = GEOMETRIES[args.model]
    ref = CpuReferenceDecode(geom, threads=pick_reference_threads(geom.name))
    # a step is a bounded sample of the token: K steps + W warm-up steps must end within a few minutes whatever K is.  One full token costs t_tok on
    # this host (measured by the constructor's warm-up token and one more here); a step covers 1/slices of a token's linears, continuing in execution
    # order, so every linear is timed in proportion and `slices` steps are exactly one token.
    t_tok = ref.token()
    budget_s = 150.0
    slices = max(1, int(-(-(args.steps + args.warmup) * t_tok // budget_s)))
    step = ref.slice_runner(slices)
    for _ in range(args.warmup):
        step()
    t0 = time.perf_counter()
    samples = [step() for _ in range(args.steps)]
    wall = time.perf_counter() - t0
    times = [t for t, _ in samples]
    tok_s = sum(f for _, f in samples) / sum(times)
    tp = args.gpus > 1 and args.parallel == "tp"
    line = {"impl": "reference", "metric": METRIC, "value": tok_s, "unit": UNIT, "n_gpus": args.gpus, "steps": args.steps, "warmup": args.warmup,
            "ms_per_step": 1e3 * sum(times) / args.steps, "ms_per_token": 1e3 / tok_s, "higher_is_better": True, "scaling": "strong" if tp else "weak", "vs_baseline": None,
            "dtype": "w4a8 (int8 act x int4 weight, fp32 acc)", "data": "synthetic",
            "config": workload_config(geom, args, args.gpus, tp),  # the same workload as our arm; the reference has no GPU path here: rank 0's host cores
            "reference_path": f"the reference's AVX W4A8 kernels (oracle/_ref, compiled in place) with NUM_THREAD = {ref.cores} (the fastest of 4..{os.cpu_count()} probed on this host); "
                              f"each step = 1/{slices} of a token's linears in execution order ({slices} steps = one full token)",
            "cpu_baseline": {"value": tok_s, "unit": UNIT, "cores": ref.cores, "kind": ref.kind,
                             "sample": f"{args.steps} steps of 1/{slices} token each = {sum(f for _, f in samples):.2f} tokens; " + ref.describe(0).split(": ", 1)[1]},
            "e2e": {"value": tok_s, "unit": UNIT, "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0}, "gpu_launches": 0, "wall_s": wall}
    try:  # what the value leaves out, measured on this host (never allowed to hide the line)
        line["excluded_attention"] = reference_attention_cost(geom, ref.cores)
        core_ms = line["excluded_attention"].get("attention_core_ms_per_token")
        if core_ms is not None:
            line["excluded_attention"]["tok_s_with_attention_at_that_ctx"] = 1e3 / (1e3 / tok_s + core_ms)
    except Exception as ex:
        line["excluded_attention"] = {"error": repr(ex)}
    print(json.dumps(line), flush=True)


# ------------------------------------------------------------------------------------------------------------------
# secondary configs measured in the same run (BASELINE.json configs[2], configs[3]) and the reference's CUDA kernel on this GPU
# ------------------------------------------------------------------------------------------------------------------
def gpu_reference_gemv(model, geom, dev):
    """The reference's own gemv_kernel_g128 (kernels/cuda/gemv_cuda.cu, compiled unchanged for sm_100a into oracle/_ref) over every
    GEMV of one decode step on the model's real weights: the GPU-side baseline SURVEY.md 8(d) config 2 names."""
    import torch

    from oracle import capi

    if not capi.ref_available("cuda"):
        return None
    L = capi.ref_cuda()
    hd = geom.head_dim
    xs = {ic: torch.randn((1, ic), device=dev).to(torch.float16) for ic in (geom.embed_dim, geom.num_heads * hd, geom.hidden_dim)}
    ys = {}

    def run_all():
        for l in range(geom.num_layers):
            T = model.layer_tensors(l)
            for name in ("q", "k", "v", "o", "gate", "up", "down"):
                w, z, s = T[name]
                oc, ic = w.shape[0], w.shape[1] * 8
                y = ys.setdefault(oc, torch.empty((1, oc), dtype=torch.float16, device=dev))
                L.ref_cuda_gemv(xs[ic].data_ptr(), w.data_ptr(), z.data_ptr(), s.data_ptr(), y.data_ptr(), 1, ic, oc)
        w, z, s = model.tensors[-1]
        oc, ic = w.shape[0], w.shape[1] * 8
        y = ys.setdefault(oc, torch.empty((1, oc), dtype=torch.float16, device=dev))
        L.ref_cuda_gemv(xs[ic].data_ptr(), w.data_ptr(), z.data_ptr(), s.data_ptr(), y.data_ptr(), 1, ic, oc)

    ds = torch.cuda.default_stream(dev)  # the reference launches on the legacy default stream
    torch.cuda.synchronize(dev)
    with torch.cuda.stream(ds):
        run_all()
        torch.cuda.synchronize(dev)
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        reps = 3
        e0.record(ds)
        for _ in range(reps):
            run_all()
        e1.record(ds)
        torch.cuda.synchronize(dev)
    ms = e0.elapsed_time(e1) / reps
    return {"kernel": "reference gemv_kernel_g128 (kernels/cuda/gemv_cuda.cu:140-194) built for sm_100a, all GEMVs of one step, eager launches",
            "ms_per_token_gemvs_only": ms, "tok_s_gemvs_only": 1e3 / ms}


def run_extras(ctx, dev, stream, peaks):
    """configs[3] (Llama-2-13B 2048-token prefill) and configs[2] (Llama-2-7B-shaped W8A8 decoder layer) on this GPU, CUDA events."""
    out = {}
    try:
        from tools.prefill_bench import prefill_once

        out["prefill_13b_2048"] = prefill_once(ctx, dev, stream, "llama2-13b", 2048, peaks)
    except Exception as ex:  # a secondary number must never hide the headline
        out["prefill_13b_2048"] = {"error": repr(ex)}
    try:
        from tools.w8a8_layer_bench import w8a8_layer

        out["w8a8_7b"] = w8a8_layer(ctx, dev, stream, peaks)
    except Exception as ex:
        out["w8a8_7b"] = {"error": repr(ex)}
    return out


# ------------------------------------------------------------------------------------------------------------------
# our arm
# ------------------------------------------------------------------------------------------------------------------
def dump_outputs(out_dir, arrays, rank: int, world: int):
    """--dump-outputs: one DIR/<name>.npy per array (float32 / float64); with N > 1 every rank writes its own, suffixed _rank<r>."""
    import numpy as np

    os.makedirs(out_dir, exist_ok=True)
    suffix = "" if world == 1 else f"_rank{rank}"
    for name, a in arrays.items():
        np.save(os.path.join(out_dir, f"{name}{suffix}.npy"), a)


def run_ours(args):
    import numpy as np
    import torch
    import torch.distributed as dist

    rank, local_rank, world = env_rank()
    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device -- tinychatengine_b200 has no CPU fallback (use --impl reference for the CPU arm)")
    torch.cuda.set_device(local_rank)
    dev = torch.device("cuda", local_rank)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)
    from tinychatengine_b200 import llama as LL
    from tinychatengine_b200.runtime import Context

    geom = LL.GEOMETRIES[args.model]
    stream = torch.cuda.Stream(dev)
    tp = world > 1 and args.parallel == "tp"
    extra = {}
    outs = {} if args.dump_outputs else None
    with torch.cuda.stream(stream):
        ctx = Context(local_rank, stream)
        K, W = args.steps, args.warmup
        gen = torch.Generator(device="cpu")
        gen.manual_seed(99)
        toks = torch.randint(0, geom.vocab_size, (K + W,), generator=gen).tolist()
        # timed positions spread over 1 -> max_ctx (ctx length = pos); warm-up at mid context
        pos_list = [args.max_ctx // 2] * W + [min(args.max_ctx - 1, int(round(i * (args.max_ctx - 1) / max(1, K - 1)))) for i in range(K)]
        if args.ctx >= 0:
            pos_list = [args.ctx] * (W + K)

        def barrier():
            if world > 1:
                dist.barrier()
            torch.cuda.synchronize(dev)

        def fill_cache(m, g):
            # random-filled KV cache so every context length is "already generated"; seeded so that every run decodes the same inputs
            gen = torch.Generator(device=dev)
            gen.manual_seed(4321)
            for l in range(g.num_layers):
                m.kv_cache(l, 0).normal_(0, 0.5, generator=gen)
                m.kv_cache(l, 1).normal_(0, 0.5, generator=gen)

        def timed(m, vocab_local, outs=None):
            """(device-resident ms, host entry point ms, clocks) over the K timed steps of model m; `outs` (a dict) receives what the last
            step of each entry point returned: the device logits of tce_llama_decode, the host logits and greedy token of tce_llama_decode_host"""
            tokpos_all = torch.tensor(list(zip(toks, pos_list)), dtype=torch.int32, device=dev)
            tokpos = torch.zeros(2, dtype=torch.int32, device=dev)
            logits_pinned = torch.empty(vocab_local, dtype=torch.float32).pin_memory()
            for i in range(W):
                tokpos.copy_(tokpos_all[i])
                m.decode(tokpos)
            barrier()
            e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            with ClockSampler(local_rank) as clk:
                e0.record(stream)
                for i in range(W, W + K):
                    tokpos.copy_(tokpos_all[i])
                    m.decode(tokpos)
                e1.record(stream)
                barrier()
            ms_dev = e0.elapsed_time(e1)
            if outs is not None:
                outs["logits"] = m.logits().cpu().numpy()
            for i in range(W):
                m.decode_host(toks[i], pos_list[i], logits_pinned)
            barrier()
            e2, e3 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
            e2.record(stream)
            for i in range(W, W + K):
                nxt = m.decode_host(toks[i], pos_list[i], logits_pinned)
            e3.record(stream)
            barrier()
            if outs is not None:
                outs["e2e_logits"] = logits_pinned.numpy().copy()
                outs["e2e_next_token"] = np.array([nxt], dtype=np.float64)
            return ms_dev, e2.elapsed_time(e3), clk.summary()

        if tp:
            # tensor-parallel decode of ONE sequence: every rank generates the same full weights (same seed) and keeps its 1/N shard
            if geom.num_kv_heads % world or geom.num_heads % world or (geom.hidden_dim // world) % 128:
                raise SystemExit(f"{geom.name}: does not split over {world} ranks on head / 128-channel group boundaries")
            Wfull = LL.make_random_weights(geom, dev, seed=1234)
            Wl, gl = LL.shard_weights(Wfull, geom, rank, world)
            model = LL.LlamaModel(ctx, gl, max_ctx=args.max_ctx, weights=Wl, tp_rank=rank, tp_size=world)
            model.tp_connect()
            # ---- parity: 4 steps against a single-GPU run of the same weights (rank 0), before any timing ----
            ptoks, ppos = [11, 4242, 77777, 5], [0, 1, 2, 3]
            lg_local = torch.empty(gl.vocab_size, dtype=torch.float32)
            full_logits = []
            for tkn, ps in zip(ptoks, ppos):
                model.decode_host(tkn, ps, lg_local)
                shards = [torch.empty(gl.vocab_size, dtype=torch.float32, device=dev) for _ in range(world)]
                dist.all_gather(shards, lg_local.to(dev))
                full_logits.append(torch.cat(shards).cpu())
            single = LL.LlamaModel(ctx, geom, max_ctx=args.max_ctx, weights=Wfull) if (rank == 0 or args.replicas_too) else None
            parity = None
            if rank == 0:
                lg = torch.empty(geom.vocab_size, dtype=torch.float32)
                parity = 0.0
                for (tkn, ps), got in zip(zip(ptoks, ppos), full_logits):
                    single.decode_host(tkn, ps, lg)
                    parity = max(parity, float((got - lg).abs().max() / lg.abs().max()))
                extra["tp_parity_rel_err"] = parity
                extra["tp_parity_note"] = "max |logits_tp - logits_1gpu| / max |logits_1gpu| over 4 decode steps of the same weights (rank 0 runs the single-GPU model)"
            fill_cache(model, gl)
            ms_dev, ms_e2e, clocks = timed(model, gl.vocab_size, outs)
            if args.replicas_too:
                fill_cache(single, geom)
                r_dev, _, _ = timed(single, geom.vocab_size)
                rt = torch.tensor([r_dev], dtype=torch.float64, device=dev)
                dist.all_reduce(rt, op=dist.ReduceOp.MAX)
                extra["replicas_tok_s"] = world * K / (rt.item() * 1e-3)
            if single is not None:
                single.close()
            vocab_local = gl.vocab_size
        else:
            gl = geom
            model = LL.LlamaModel(ctx, geom, max_ctx=args.max_ctx, seed=1234 + rank)
            fill_cache(model, geom)
            ms_dev, ms_e2e, clocks = timed(model, geom.vocab_size, outs)
            vocab_local = geom.vocab_size
        kernels_per_step = model.kernels_per_step
        if outs is not None:
            dump_outputs(args.dump_outputs, outs, rank, world)
        if rank == 0 and world == 1 and not args.no_extras:
            peaks, _, _ = load_peaks()
            try:
                extra["gpu_reference"] = gpu_reference_gemv(model, geom, dev)
            except Exception as ex:
                extra["gpu_reference"] = {"error": repr(ex)}
        model.close()
        if rank == 0 and world == 1 and not args.no_extras:
            extra.update(run_extras(ctx, dev, stream, peaks))
        if world > 1 and not args.no_extras:
            # configs[3] at N GPUs.  The prompt pass is tensor-bound and a 2048-token prompt of the 13B model fits one GPU, so it scales as N
            # independent prompts (data parallel, no collective on the data path): aggregate = N x FLOPs / the slowest rank's time.
            pre, pre_err = None, None
            try:
                from tools.prefill_bench import prefill_once

                pre = prefill_once(ctx, dev, stream, "llama2-13b", 2048, load_peaks()[0])
            except Exception as ex:  # a secondary number must never hide the headline
                pre_err = repr(ex)
            pre_ms = torch.tensor([pre["ms"] if pre else float("inf")], dtype=torch.float64, device=dev)
            dist.all_reduce(pre_ms, op=dist.ReduceOp.MAX)  # every rank reaches this line, whatever happened above
            if rank == 0:
                slowest = pre_ms.item()
                if pre is not None and slowest != float("inf"):
                    scale = pre["ms"] / slowest
                    extra["prefill_13b_2048"] = {
                        "model": pre["model"], "n": pre["n"], "prompts": world, "parallelism": f"{world} independent prompts, one per GPU (no collective)",
                        "ms": slowest, "tok_per_s": world * pre["tok_per_s"] * scale, "linear_tflops": world * pre["linear_tflops"] * scale,
                        "linear_plus_attn_tflops": world * pre["linear_plus_attn_tflops"] * scale, "rank0_ms": pre["ms"],
                        "note": "aggregate over all GPUs, timed as the slowest rank (max over ranks of the best-of-3 CUDA-event time)"}
                else:
                    extra["prefill_13b_2048"] = {"error": pre_err or "a rank failed"}

    times = torch.tensor([ms_dev, ms_e2e], dtype=torch.float64, device=dev)
    if world > 1:
        dist.all_reduce(times, op=dist.ReduceOp.MAX)
    ms_dev, ms_e2e = times.tolist()
    if rank == 0:
        _, peak, peak_src = load_peaks()
        wbytes = LL.weight_bytes_per_token(geom)
        mean_ctx = sum(pos_list[W:]) / K
        kvbytes = LL.kv_bytes_per_token(geom, int(mean_ctx))
        seqs = 1 if (tp or world == 1) else world
        tok_s = seqs * K / (ms_dev * 1e-3)
        e2e_tok_s = seqs * K / (ms_e2e * 1e-3)
        per_gpu_bytes = (wbytes + kvbytes) / (world if tp else 1)
        achieved = per_gpu_bytes / (ms_dev / K * 1e-3) / 1e9
        traffic, traffic_src = load_traffic()
        persistent = kernels_per_step == 1
        line = {
            "metric": METRIC, "value": tok_s, "unit": UNIT, "n_gpus": world, "steps": K, "warmup": W, "ms_per_step": ms_dev / K,
            "higher_is_better": True, "scaling": "strong" if tp else "weak", "vs_baseline": None,
            "dtype": "w4a16 (int4 weights; activations fp16 -> 32-bit block fixed point = four int8 digit planes; int32 accumulate, fp32 scale)",
            "data": "synthetic",
            "config": workload_config(geom, args, world, tp),
            "mean_ctx": mean_ctx,
            "l2": "inputs larger than L2: 3.9 GB of weights stream per step vs 126 MB L2",
            "clocks": clocks,
            "e2e": {"value": e2e_tok_s, "unit": UNIT, "h2d_bytes_per_step": 12, "d2h_bytes_per_step": vocab_local * 4 + 4},
            "gpu_launches": K * kernels_per_step,
            "roofline": {"bound": "hbm",
                         "kernel": ("decode_persistent_kernel (1 launch per step: every weight, scale/zero and KV byte of the token streams through its TMA ring)"
                                    if persistent else f"{kernels_per_step} kernels per step (kernel-per-op graph path)"),
                         "achieved": achieved, "peak": peak, "unit": "GB/s", "frac": achieved / peak,
                         "traffic": traffic if (persistent and world == 1) else None, "traffic_source": traffic_src if (persistent and world == 1) else None,
                         "peak_source": peak_src,
                         "algorithmic_bytes_per_launch": per_gpu_bytes / (1 if persistent else kernels_per_step),
                         "avg_launch_us": ms_dev / K * 1e3 / kernels_per_step,
                         "note": "per GPU; algorithmic bytes = packed weights + fp16 scales + 4-bit zeros (SURVEY.md 8d: 3.899 GB) + KV rows at the mean context"
                                 + (", divided by the tensor-parallel degree" if tp else "")},
        }
        # tensor-parallel parity / replica keys stay at the top level; the other workloads of BASELINE.json measured in the same run
        # (prefill_13b_2048, w8a8_7b, gpu_reference) go under "extra"
        top = {k: v for k, v in extra.items() if k.startswith("tp_") or k.startswith("replicas")}
        line.update(top)
        rest = {k: v for k, v in extra.items() if k not in top}
        if rest:
            line["extra"] = rest
        if world == 1 and not args.no_cpu_baseline:
            try:
                line["cpu_baseline"] = cpu_baseline(geom, args.cpu_budget)
            except Exception as ex:  # the baseline must never hide the GPU number
                line["cpu_baseline"] = {"error": repr(ex)}
            # the reference's CPU path timed beside the two secondary configs as well (bounded samples; SURVEY.md 8d)
            if "extra" in line:
                for key, fn in (("w8a8_7b", lambda: cpu_baseline_w8a8(min(6.0, args.cpu_budget))),
                                ("prefill_13b_2048", lambda: cpu_baseline_prefill(int(line["cpu_baseline"].get("cores", 8))))):
                    if isinstance(line["extra"].get(key), dict):
                        try:
                            line["extra"][key]["cpu_baseline"] = fn()
                        except Exception as ex:
                            line["extra"][key]["cpu_baseline"] = {"error": repr(ex)}
        print(json.dumps(line), flush=True)
    ctx.close()
    if world > 1:
        dist.barrier()
        dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=None, help="timed steps (default: 128; 8 with --impl reference)")
    ap.add_argument("--warmup", type=int, default=8)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--model", default="llama3-8b")
    ap.add_argument("--max-ctx", type=int, default=4096)
    ap.add_argument("--ctx", type=int, default=-1, help="fixed context length for every step (default: sweep 1 -> max_ctx)")
    ap.add_argument("--cpu-budget", type=float, default=12.0)
    ap.add_argument("--no-cpu-baseline", action="store_true")
    ap.add_argument("--probe-threads", type=int, default=0, help=argparse.SUPPRESS)  # internal: time one layer's linears on the reference with N threads
    ap.add_argument("--no-extras", action="store_true", help="skip gpu_reference / prefill_13b_2048 / w8a8_7b (the last two: N = 1 only)")
    # N > 1 default = tensor-parallel decode of ONE sequence (BASELINE config 5, strong scaling); "replicas" = one independent batch-1
    # sequence per GPU (no data-path collective, weak scaling), also reported as `replicas_tok_s` beside the tensor-parallel value
    ap.add_argument("--parallel", default="tp", choices=["tp", "replicas"])
    ap.add_argument("--no-replicas", dest="replicas_too", action="store_false", help="N>1 tp: skip the secondary replicas measurement")
    ap.add_argument("--dump-outputs", metavar="DIR", default=None,
                    help="after the timed steps, write what the last one returned (logits, greedy token) as DIR/<name>.npy")
    args = ap.parse_args()
    if args.steps is not None and args.steps < 1:
        ap.error("--steps must be at least 1")
    if args.dump_outputs and args.impl == "reference":
        ap.error("--dump-outputs writes the outputs of this project's decode step; the reference arm times bare linears")
    if args.warmup < 3:
        args.warmup = 3
    if args.probe_threads:
        probe_threads(args)
        return
    if args.impl == "reference":
        if args.steps is None:
            args.steps = 8  # a full token costs seconds on the host: keep the default invocation within minutes
        run_reference(args)
    else:
        if args.steps is None:
            args.steps = 128
        run_ours(args)


if __name__ == "__main__":
    main()
