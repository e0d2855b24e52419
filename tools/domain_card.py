import os, sys, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from continuousbayesiannetwork_b200 import synth
from continuousbayesiannetwork_b200.engine import tables_from_spec
dev = "cuda:0"
spec = synth.asia()
t = tables_from_spec(spec, dev)
n = 1 << 26
g = torch.Generator(device=dev).manual_seed(3)
for card in (2, 4, 8, 16, 64, 200):
    col = torch.randint(0, card, (n,), generator=g, device=dev).to(torch.float32) * 0.25
    cols = [col] * 4
    def f(): t.discover_domains(cols)
    f(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(5): f()
    e1.record(); torch.cuda.synchronize()
    s = e0.elapsed_time(e1) / 1e3 / 5
    d = t.discover_domains([col])[0]
    assert d.numel() == card
    print(f"card {card:3d}: {s*1e3:7.3f} ms  {4*n*4/s/1e9:7.1f} GB/s")
