"""Event timeline of CTA 0 of the pair kernel for tile-pair iterations 40..43 (timing build)."""
import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ["RANGECLIP_B200_LIB"] = os.path.abspath("rangeclip_b200/librangeclip_b200_timing.so")
from rangeclip_b200 import _lib, ops
import ctypes
_lib.lib().rc_debug_set_timing_buffer.argtypes = [ctypes.c_void_p]      # (a bring-up entry point: not in _lib.PROTOTYPES)
B = 32
dev = torch.device("cuda:0")
D, H, W, K = 512, 256, 256, 256
g = torch.Generator(device=dev).manual_seed(0)
x = torch.randn(B, D, H, W, device=dev, generator=g).to(torch.bfloat16)
t = torch.nn.functional.normalize(torch.randn(K, D, device=dev, generator=g), dim=1)
y = torch.randint(0, K, (B, H * W), device=dev, generator=g, dtype=torch.int32)
w = torch.ones(B, H * W, device=dev)
buf = torch.zeros(1024, device=dev, dtype=torch.int64)
for rep in range(2):
    buf.zero_()
    _lib.lib().rc_debug_set_timing_buffer(buf.data_ptr())
    ops.infonce_raw(x, t, y, w, 1 / 0.07, True, False, "bf16", flags=ops.RC_INFONCE_SS_KERNEL)
    torch.cuda.synchronize()
_lib.lib().rc_debug_set_timing_buffer(None)
ev = buf[256:256 + 2 * 4 * 48].view(2, 4, 48).tolist()
names = {0: "mma  S issue start", 1: "mma  S issued", 2: "mma  dX start (P ready)", 3: "mma  dX unit0 start", 4: "mma  dX unit1 start",
         5: "mma  dX unit2 start", 6: "mma  dX unit3 start", 7: "mma  dX issued", 10: "smx  S complete", 11: "smx  exp pass done",
         12: "smx  P buffer free", 13: "smx  P stored", 14: "smx  norms(next) done", 20: "epi  unit0 acc full", 21: "epi  unit0 done",
         22: "epi  unit1 acc full", 23: "epi  unit1 done", 24: "epi  unit2 acc full", 25: "epi  unit2 done", 26: "epi  unit3 acc full",
         27: "epi  unit3 done", 15: "smx  exp pass done (warp 11)", 16: "smx  P stored (warp 11)"}
t0 = min(v for cta in ev for row in cta for v in row if v)
rows = []
for cta in range(2):
    for it, row in enumerate(ev[cta]):
        for i, v in enumerate(row):
            if v:
                rows.append((v - t0, cta, 40 + it, names.get(i, str(i))))
for tt, cta, it, nm in sorted(rows):        # %globaltimer nanoseconds (one clock for both CTAs of the pair)
    print(f"{tt:8d} ns  cta{cta}  iter {it}  {nm}")
