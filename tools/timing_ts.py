"""Where a tile pair's time goes in the TS-mode InfoNCE kernel (csrc/infonce_ts.cu), next to the CTA-pair SS kernel, from the
timing build (make -C rangeclip_b200/csrc timing): per-role barrier wait cycles of the two CTAs of cluster 0, per tile pair,
and the %globaltimer event trace of tile pairs 40..43 of the TS kernel.

    python tools/timing_ts.py [B]          # headline shape D = 512, 256 x 256, K = 256; B images (default 16)
"""
import ctypes
import os
import sys

import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
os.environ["RANGECLIP_B200_LIB"] = os.path.abspath("rangeclip_b200/librangeclip_b200_timing.so")
from rangeclip_b200 import _lib, ops  # noqa: E402

_lib.lib().rc_debug_set_timing_buffer.argtypes = [ctypes.c_void_p]      # (a timing-build entry point: not in _lib.PROTOTYPES)

TS_FLAG, SS_FLAG = 8, 32      # RC_INFONCE_TS_KERNEL (the default), RC_INFONCE_SS_KERNEL
# wait tags / timed sections per role (tags as in the mbar_wait calls of the kernel); index 0 of every role is its lifetime
TS_ROLES = [("text producer", {1: "tempty(S)", 2: "tempty(dX)"}),
            ("mma", {5: "xfull(S)", 6: "tfull(S)", 7: "acc_empty(S)", 9: "p_full", 4: "acc_empty(dX)", 8: "tfull(dX)"}),
            ("softmax", {1: "norms(incl. xf wait)", 11: "xf", 12: "s_full", 2: "exp_pass", 13: "row_exchange", 3: "p_form+store"}),
            ("epilogue", {14: "sc_full", 15: "acc_full", 3: "tmem_ld", 4: "x_box_wait", 2: "math+stmatrix", 5: "store_buf_wait"}),
            ("x producer", {3: "xempty"})]
SS_ROLES = [("producer", {1: "empty(S)", 2: "empty(dX)"}),
            ("mma", {3: "s_empty", 4: "xfull(S)", 12: "tfull(S)", 5: "p_full", 6: "acc_empty", 7: "tfull(dX)"}),
            ("softmax", {8: "s_full", 9: "p_empty", 1: "softmax", 2: "p_store"}),
            ("epilogue", {10: "sc_full", 11: "acc_full", 2: "epi_compute", 3: "tmem_ld", 4: "x_wait+swap", 5: "store_buf_wait",
                          6: "cursor+fetch", 7: "math", 8: "staging_sts", 9: "proxy_fence", 12: "tma_issue", 13: "acc_release"})]
TS_EVENTS = {0: "mma  S issue start (slot free)", 1: "mma  S issued", 2: "mma  dX start (P ready)", 11: "mma  dX issued",
             12: "smx  norms done", 13: "smx  S complete", 14: "smx  exp pass done", 15: "smx  P stored"}
TS_EVENTS.update({3 + b: f"mma  dX blk{b} acc free" for b in range(8)})
TS_EVENTS.update({20 + 2 * b: f"epi  blk{b} acc full" for b in range(8)})
TS_EVENTS.update({21 + 2 * b: f"epi  blk{b} stored" for b in range(8)})


def main():
    B = int(sys.argv[1]) if len(sys.argv) > 1 else 16
    dev = torch.device("cuda:0")
    D, H, W, K = 512, 256, 256, 256
    g = torch.Generator(device=dev).manual_seed(0)
    x = torch.randn(B, D, H, W, device=dev, generator=g).to(torch.bfloat16)
    t = torch.nn.functional.normalize(torch.randn(K, D, device=dev, generator=g), dim=1)
    y = torch.randint(0, K, (B, H * W), device=dev, generator=g, dtype=torch.int32)
    w = torch.ones(B, H * W, device=dev)
    pairs = (B * H * W // 128 // 2 + 73) // 74          # tile pairs of cluster 0 (74 clusters on 148 SMs)
    for name, flags, roles, n_roles in (("SS (infonce_umma_pair_kernel)", SS_FLAG, SS_ROLES, 4), ("TS (infonce_ts_kernel)", TS_FLAG, TS_ROLES, 5)):
        buf = torch.zeros(2, 1024, device=dev, dtype=torch.int64)   # [0, 16 * roles * 2): wait cycles; [256, 640): event trace
        for rep in range(2):                                          # the second launch is the one reported
            _lib.lib().rc_debug_set_timing_buffer(buf[rep].data_ptr())
            ops.infonce_raw(x, t, y, w, 1 / 0.07, True, False, "bf16", flags=flags)
            torch.cuda.synchronize()
        _lib.lib().rc_debug_set_timing_buffer(None)
        row = buf[1].tolist()
        print(f"== {name}: B={B}, {pairs} tile pairs per cluster; cycles per tile pair (SM clock)")
        for cta in range(2):
            for r_, (role, names) in enumerate(roles):
                vals = row[(cta * n_roles + r_) * 16:(cta * n_roles + r_ + 1) * 16]
                if not any(vals):
                    continue
                print(f"  cta{cta} {role}: lifetime={vals[0] / pairs:.0f} " +
                      ", ".join(f"{names.get(i, i)}={v / pairs:.0f}" for i, v in enumerate(vals) if v and i))
        if flags == TS_FLAG:
            ev = buf[1, 256:256 + 2 * 4 * 48].view(2, 4, 48).tolist()
            stamps = [v for cta in ev for r in cta for v in r if v]
            if stamps:
                t0 = min(stamps)
                rows = sorted((v - t0, cta, 40 + it, TS_EVENTS.get(i, str(i)))
                              for cta in range(2) for it, r in enumerate(ev[cta]) for i, v in enumerate(r) if v)
                print("  event trace of cluster 0, tile pairs 40..43 (%globaltimer ns)")
                for tt, cta, it, nm in rows:
                    print(f"    {tt:8d} ns  cta{cta}  pair {it}  {nm}")


if __name__ == "__main__":
    main()
