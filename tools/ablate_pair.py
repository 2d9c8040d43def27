"""Sensitivity of the CTA-pair InfoNCE kernel to its memory traffic classes (bring-up build, RANGECLIP_B200_ABLATE bits; results
are garbage under ablation, only the time counts): 1 no epilogue x loads, 2 no dX stores, 64 no row-norm reads, 256 no text
reloads after the first ring pass.   python tools/ablate_pair.py
RC_AB_FLAGS: rc_infonce_bf16 flags (default 32 = RC_INFONCE_SS_KERNEL, the pair kernel; 0 = the default TS kernel)."""
import json, os, subprocess, sys
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
if len(sys.argv) > 1 and sys.argv[1] == "child":
    sys.path.insert(0, ROOT)
    os.environ["RANGECLIP_B200_LIB"] = os.environ.get("RC_AB_LIB") or os.path.join(ROOT, "rangeclip_b200", "librangeclip_b200_bringup.so")
    import torch
    from rangeclip_b200 import _lib, ops
    dev = torch.device("cuda")
    L = _lib.lib(); st = torch.cuda.current_stream().cuda_stream
    B, D, HW, K = 64, 512, 65536, 256
    g = torch.Generator(device=dev).manual_seed(1)
    x = torch.empty(B, D, HW, device=dev, dtype=torch.bfloat16)
    for b in range(B):
        xb = torch.randn(D, HW, device=dev, generator=g); x[b] = (xb / xb.norm(dim=0, keepdim=True)).to(torch.bfloat16)
    text = torch.nn.functional.normalize(torch.randn(K, D, device=dev, generator=g), dim=1)
    _, tb, ttb = ops.text_prepare(text, None, want_f32=False, want_bf16=True)
    y = torch.randint(0, K, (B * HW,), device=dev, generator=g, dtype=torch.int32)
    w = torch.randint(0, 3, (B * HW,), device=dev, generator=g).float()
    M = B * HW
    acc = torch.zeros(4, device=dev, dtype=torch.float64); lse = torch.empty(M, device=dev)
    dx = torch.empty(B, D, HW, device=dev, dtype=torch.bfloat16)
    wsb = int(L.rc_infonce_workspace_bytes(B, D, HW, K, _lib.RC_BF16)); ws = torch.empty(wsb, device=dev, dtype=torch.uint8)
    _lib.check(L.rc_weight_sum(w.data_ptr(), y.data_ptr(), M, acc[3:].data_ptr(), st), "wsum")
    def run():
        _lib.check(L.rc_infonce_bf16(x.data_ptr(), _lib.RC_BF16, B, D, HW, tb.data_ptr(), ttb.data_ptr(), K, y.data_ptr(), w.data_ptr(), 1 / 0.07,
                                     lse.data_ptr(), acc[0:].data_ptr(), acc[1:].data_ptr(), acc[3:].data_ptr(), None, dx.data_ptr(), None,
                                     acc[2:].data_ptr(), ws.data_ptr(), wsb, int(os.environ.get('RC_AB_FLAGS', 32)), st), "infonce")
    for _ in range(3): run()
    torch.cuda.synchronize()
    ts = []
    for _ in range(7):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(); run(); e1.record(); torch.cuda.synchronize(); ts.append(e0.elapsed_time(e1))
    print(json.dumps({"lib": os.path.basename(os.environ["RANGECLIP_B200_LIB"]), "ablate": int(os.environ.get("RANGECLIP_B200_ABLATE", 0)), "ms_min": min(ts), "ms_med": sorted(ts)[3]}))
elif len(sys.argv) > 1 and sys.argv[1] == "ab":
    # same-box A/B of library variants (make -C rangeclip_b200/csrc variant NAME=.. DEFS=..): python tools/ablate_pair.py ab base x ...
    names = sys.argv[2:]
    for rep in range(2):
        for n in names:
            lib = os.path.join(ROOT, "rangeclip_b200", "librangeclip_b200_bringup.so" if n == "base" else f"librangeclip_b200_var_{n}.so")
            r = subprocess.run([sys.executable, __file__, "child"], env=dict(os.environ, RC_AB_LIB=lib, RANGECLIP_B200_ABLATE="0"), capture_output=True, text=True, timeout=300)
            print(r.stdout.strip() or r.stderr[-400:], flush=True)
else:
    for bits in ([int(v) for v in sys.argv[1:]] or [0, 256, 1, 2, 64, 257, 259, 323, 0]):
        r = subprocess.run([sys.executable, __file__, "child"], env=dict(os.environ, RANGECLIP_B200_ABLATE=str(bits)), capture_output=True, text=True, timeout=300)
        print(r.stdout.strip() or r.stderr[-400:], flush=True)
