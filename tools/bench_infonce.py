"""Kernel-only timing of the fused InfoNCE tensor-core kernel at the headline shape (CUDA events;
the pre-pass is done once outside the timed loop).  Usage: bench_infonce.py [B] [reps]"""
import json, os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from rangeclip_b200 import _lib, ops
B = int(sys.argv[1]) if len(sys.argv) > 1 else 64
reps = int(sys.argv[2]) if len(sys.argv) > 2 else 10
dev = torch.device("cuda:0")
D, K = 512, 256
H = int(os.environ.get("BENCH_H", 256)); W = int(os.environ.get("BENCH_W", 256))
HW = H * W
g = torch.Generator(device=dev).manual_seed(0)
x = torch.empty(B, D, HW, device=dev, dtype=torch.bfloat16)
for b in range(B):
    x[b] = torch.randn(D, HW, device=dev, generator=g).to(torch.bfloat16)
t = torch.nn.functional.normalize(torch.randn(K, D, device=dev, generator=g), dim=1)
y = torch.randint(0, K, (B * HW,), device=dev, generator=g, dtype=torch.int32)
w = torch.ones(B * HW, device=dev)
tb, ttb = ops.text_to_bf16(t)
L = _lib.lib(); st = torch.cuda.current_stream().cuda_stream
ws_bytes = int(L.rc_infonce_workspace_bytes(B, D, HW, K, _lib.RC_BF16))
ws = torch.empty(ws_bytes, device=dev, dtype=torch.uint8)
acc = torch.zeros(4, device=dev, dtype=torch.float64)
acc[3] = B * HW
lse = torch.empty(B * HW, device=dev)
dx = torch.empty_like(x)
_lib.check(L.rc_infonce_prepass(x.data_ptr(), _lib.RC_BF16, B, D, HW, ws.data_ptr(), ws_bytes, st), "prepass")
def run(bwd=True):
    _lib.check(L.rc_infonce_bf16(x.data_ptr(), _lib.RC_BF16, B, D, HW, tb.data_ptr(), ttb.data_ptr(), K, y.data_ptr(), w.data_ptr(),
                                 1 / 0.07, lse.data_ptr(), acc[0:].data_ptr(), acc[1:].data_ptr(), acc[3:].data_ptr(), None,
                                 dx.data_ptr() if bwd else None, None, acc[2:].data_ptr() if bwd else None, ws.data_ptr(), ws_bytes,
                                 1, st), "infonce")
for bwd in (True, False):
    for _ in range(3):
        run(bwd)
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(reps):
        run(bwd)
    e1.record(); torch.cuda.synchronize()
    ms = e0.elapsed_time(e1) / reps
    flops = (4 if bwd else 2) * K * D * B * HW
    print(json.dumps({"kernel": "infonce_bf16" + ("_fwd_bwd" if bwd else "_fwd"), "B": B, "H": H, "W": W, "ms": round(ms, 4),
                      "TFLOPs": round(flops / ms / 1e9, 1), "Mpix_s": round(B * HW / ms / 1e3, 1)}), flush=True)

# fwd + dX + dText (tensor-core dText: the pair kernel also writes G, then the split-K GEMM)
ws2_bytes = int(L.rc_infonce_workspace_bytes_dt(B, D, HW, K, _lib.RC_BF16))
ws2 = torch.empty(ws2_bytes, device=dev, dtype=torch.uint8)
dt = torch.zeros(K, D, device=dev)
def run_dt():
    _lib.check(L.rc_infonce_bf16(x.data_ptr(), _lib.RC_BF16, B, D, HW, tb.data_ptr(), ttb.data_ptr(), K, y.data_ptr(), w.data_ptr(),
                                 1 / 0.07, lse.data_ptr(), acc[0:].data_ptr(), acc[1:].data_ptr(), acc[3:].data_ptr(), None,
                                 dx.data_ptr(), dt.data_ptr(), acc[2:].data_ptr(), ws2.data_ptr(), ws2_bytes, 0, st), "infonce+dt")
for _ in range(3):
    run_dt()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(reps):
    run_dt()
e1.record(); torch.cuda.synchronize()
ms = e0.elapsed_time(e1) / reps
print(json.dumps({"kernel": "infonce_bf16_fwd_bwd_dtext", "B": B, "ms": round(ms, 4), "TFLOPs_3units": round(6 * K * D * B * HW / ms / 1e9, 1),
                  "Mpix_s": round(B * HW / ms / 1e3, 1)}), flush=True)
