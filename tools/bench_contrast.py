import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import bench as BN
from rangeclip_b200 import ops, losses
dev = torch.device("cuda:0")
c = BN.CFG
C, G, K = c["C"], c["G"], c["K"]
g = torch.Generator(device=dev).manual_seed(1)
rest = torch.arange(G + 1, C, device=dev)
contrast = torch.unique(torch.cat([torch.arange(1, G + 1, device=dev), rest[torch.randperm(rest.numel(), device=dev, generator=g)[: K - G]]]))
sets = BN.similarity_sets(contrast.tolist(), G, C)
off, items = losses.similarity_csr(sets, C, False, True, dev)
counts = torch.zeros(C, device=dev, dtype=torch.int32); counts[1:G + 1] = 5
print("csr items", items.numel())
def run(): return ops.contrast_build(counts, off, items, K - G, 0, 256, 7)
for _ in range(3): run()
torch.cuda.synchronize()
e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
e0.record()
for _ in range(20): run()
e1.record(); torch.cuda.synchronize()
print("contrast_build us", e0.elapsed_time(e1) / 20 * 1e3)
