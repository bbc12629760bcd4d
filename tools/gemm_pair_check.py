#!/usr/bin/env python
"""Check + time the W4A16 large-M GEMM (tce_w4a16_gemm: int4 -> fp16 expansion + CTA-pair tcgen05 GEMM) against a torch fp32 reference
of the dequantised weights: a few ragged shapes for correctness, the Llama-2-13B prefill shapes for speed.
    python tools/gemm_pair_check.py
"""
import json
import sys
from pathlib import Path

import torch

sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from tinychatengine_b200.runtime import Context, random_w4  # noqa: E402


def dequant(w, z, s, ic):
    oc = w.shape[0]
    wi = w.to(torch.int64) & 0xFFFFFFFF
    q = torch.stack([(wi >> (4 * i)) & 0xF for i in range(8)], dim=2).reshape(oc, ic).float()
    zi = z.to(torch.int64) & 0xFFFFFFFF
    zn = torch.stack([(zi >> (4 * i)) & 0xF for i in range(8)], dim=2).reshape(oc, -1)[:, : ic // 128].float()
    sc = s[:, : ic // 128].float()
    return ((q.reshape(oc, ic // 128, 128) - zn[:, :, None]) * sc[:, :, None]).reshape(oc, ic)


def main():
    dev = torch.device("cuda", 0)
    ctx = Context(0)
    ok = True
    for (m, oc, ic) in [(16, 256, 128), (128, 512, 1024), (200, 1000, 1152), (333, 4096, 4096), (17, 44, 256), (130, 300, 11008), (2048, 5120, 5120)]:
        w, z, s = random_w4(oc, ic, dev, 7 + m, random_zeros=True)
        x = torch.randn((m, ic), device=dev).to(torch.float16)
        y = ctx.w4a16_gemv(x, w, z, s, gemm=True).float()
        ref = x.float() @ dequant(w, z, s, ic).t()
        err = float((y - ref).abs().max() / ref.abs().max())
        good = err < 2e-3
        ok &= good
        print(json.dumps({"check": [m, oc, ic], "rel_err": err, "ok": good}), flush=True)
    if not ok:
        raise SystemExit(1)
    M = 2048
    for name, (oc, ic) in {"13B qkv 15360x5120": (15360, 5120), "13B o 5120x5120": (5120, 5120), "13B gate_up 27648x5120": (27648, 5120),
                           "13B down 5120x13824": (5120, 13824)}.items():
        w, z, s = random_w4(oc, ic, dev, 5, random_zeros=True)
        x = torch.randn((M, ic), device=dev).to(torch.float16)
        y = torch.empty((M, oc), dtype=torch.float16, device=dev)
        for _ in range(3):
            ctx.w4a16_gemv(x, w, z, s, out=y, gemm=True)
        torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(10):
            ctx.w4a16_gemv(x, w, z, s, out=y, gemm=True)
        e1.record()
        torch.cuda.synchronize()
        t = e0.elapsed_time(e1) / 10 * 1e-3
        print(json.dumps({"shape": name, "M": M, "ms": round(t * 1e3, 4), "tflops": round(2.0 * M * oc * ic / t / 1e12, 1)}), flush=True)


if __name__ == "__main__":
    main()
