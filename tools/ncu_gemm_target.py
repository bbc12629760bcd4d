"""Target for `ncu -k regex:gemm_pair`: four W4A16 GEMM calls at the Llama-2-13B q|k|v prefill shape (M = 2048, 15360 x 5120) through tce_w4a16_gemm
(int4 -> fp16 expansion + the CTA-pair GEMM).  See profiles/README.md (prefill section)."""
import sys, torch
from pathlib import Path
sys.path.insert(0, str(Path(__file__).resolve().parents[1]))
from tinychatengine_b200.runtime import Context, random_w4
dev = torch.device("cuda", 0)
ctx = Context(0)
oc, ic, M = 15360, 5120, 2048
w, z, s = random_w4(oc, ic, dev, 5, random_zeros=True)
x = torch.randn((M, ic), device=dev).to(torch.float16)
y = torch.empty((M, oc), dtype=torch.float16, device=dev)
for _ in range(4):
    ctx.w4a16_gemv(x, w, z, s, out=y, gemm=True)
torch.cuda.synchronize()
