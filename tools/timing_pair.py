"""Per-role barrier wait cycles of the two CTAs of cluster 0 (pair kernel), per tile pair."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ["RANGECLIP_B200_LIB"] = os.path.abspath("rangeclip_b200/librangeclip_b200_timing.so")
from rangeclip_b200 import _lib, ops
import ctypes
_lib.lib().rc_debug_set_timing_buffer.argtypes = [ctypes.c_void_p]      # (a bring-up entry point: not in _lib.PROTOTYPES)
B = int(sys.argv[1]) if len(sys.argv) > 1 else 16
dev = torch.device("cuda:0")
D, H, W, K = 512, 256, 256, 256
g = torch.Generator(device=dev).manual_seed(0)
x = torch.randn(B, D, H, W, device=dev, generator=g).to(torch.bfloat16)
t = torch.nn.functional.normalize(torch.randn(K, D, device=dev, generator=g), dim=1)
y = torch.randint(0, K, (B, H * W), device=dev, generator=g, dtype=torch.int32)
w = torch.ones(B, H * W, device=dev)
buf = torch.zeros(2, 1024, device=dev, dtype=torch.int64)      # [0,128): per-role wait cycles; [256, 640): the event trace of timeline_pair.py
names = {0: {1: "empty(S)", 2: "empty(dX)"}, 1: {3: "s_empty", 4: "xfull(S)", 12: "tfull(S)", 5: "p_full", 6: "acc_empty", 7: "tfull(dX)"},
         2: {8: "s_full", 9: "p_empty", 1: "softmax", 2: "p_store"}, 3: {10: "sc_full", 11: "acc_full", 2: "epi_compute", 3: "tmem_ld", 4: "x_wait+swap", 5: "store_buf_wait", 6: "cursor+fetch",
             7: "math", 8: "staging_sts", 9: "proxy_fence", 12: "tma_issue", 13: "acc_release"}}
roles = ["producer", "mma", "softmax", "epilogue"]
for rep in range(2):
    _lib.lib().rc_debug_set_timing_buffer(buf[rep].data_ptr())
    ops.infonce_raw(x, t, y, w, 1 / 0.07, True, False, "bf16", flags=ops.RC_INFONCE_SS_KERNEL)
    torch.cuda.synchronize()
_lib.lib().rc_debug_set_timing_buffer(None)
pairs = (B * H * W // 128 // 2 + 73) // 74
row = buf[1].tolist()
for cta in range(2):
    for r_, role in enumerate(roles):
        vals = row[(cta * 4 + r_) * 16:(cta * 4 + r_ + 1) * 16]
        if not any(vals):
            continue
        print(f"cta{cta} {role}: lifetime={vals[0] / pairs:.0f} " + ", ".join(f"{names[r_].get(i, i)}={v / pairs:.0f}" for i, v in enumerate(vals) if v and i))
