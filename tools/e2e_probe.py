import os, sys, time, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
os.chdir(ROOT)
import pytorchdeeplearing_b200 as b200
from pytorchdeeplearing_b200.graphed import GraphedStep
import oracle
dev = torch.device("cuda", 0)
b200.set_precision("bf16")
torch.manual_seed(0)
model = b200.VNet3d(1, 2).to(dev); model.train()
lossfn = b200.MutilDiceLoss(torch.ones(2, device=dev))
xh, yh = oracle.make_inputs(2, 1, (96, 96, 96), 2, seed=1234)
xh, yh = xh.pin_memory(), yh.pin_memory()
x, y = xh.to(dev), yh.to(dev)
g = GraphedStep(model, lossfn, x, y, warmup=1)
K = 20
def region(fn):
    torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(); fn(); e1.record(); torch.cuda.synchronize()
    return e0.elapsed_time(e1) / K
def a():
    for _ in range(K): g()
def b():
    hl = torch.empty((), dtype=torch.float32).pin_memory()
    for _ in range(K):
        l = g(); hl.copy_(l.detach(), non_blocking=True)
    torch.cuda.synchronize()
def c():
    g.prefetch(xh, yh)
    torch.cuda.synchronize()
    for _ in range(K):
        g._take_prefetched(); g.graph.replay()
def d():
    g.prefetch(xh, yh)
    for i in range(K):
        l = g(prefetched=True)
        if i + 1 < K: g.prefetch(xh, yh)
def e():   # serial H2D on the main stream (old e2e)
    for _ in range(K): g(xh, yh)
for name, fn in (("replay only", a), ("+ async D2H of loss", b), ("+ D2D take", c), ("+ H2D prefetch on copy stream", d), ("H2D on main stream", e)):
    region(fn)
    print(f"{name:34s} {region(fn):.3f} ms/step", flush=True)

# ---- isolate: does an independent H2D copy on another stream overlap a graph replay at all?
cs = torch.cuda.Stream()
sx, sy = torch.empty_like(x), torch.empty_like(y)
def h2d_only():
    for _ in range(K):
        with torch.cuda.stream(cs):
            sx.copy_(xh, non_blocking=True); sy.copy_(yh, non_blocking=True)
    torch.cuda.current_stream().wait_stream(cs)
def replay_plus_free_h2d():
    for _ in range(K):
        g.graph.replay()
        with torch.cuda.stream(cs):
            sx.copy_(xh, non_blocking=True); sy.copy_(yh, non_blocking=True)
    torch.cuda.current_stream().wait_stream(cs)
big = torch.empty(1 << 28, dtype=torch.float32, device=dev)
def memset_plus_free_h2d():      # a plain (non-graph) long kernel instead of the graph
    for _ in range(K):
        for _ in range(8): big.zero_()
        with torch.cuda.stream(cs):
            sx.copy_(xh, non_blocking=True); sy.copy_(yh, non_blocking=True)
    torch.cuda.current_stream().wait_stream(cs)
def memset_only():
    for _ in range(K):
        for _ in range(8): big.zero_()
for name, fn in (("H2D alone (21 MB)", h2d_only), ("replay + independent H2D", replay_plus_free_h2d),
                 ("8 memsets alone", memset_only), ("8 memsets + independent H2D", memset_plus_free_h2d)):
    region(fn)
    print(f"{name:34s} {region(fn):.3f} ms/step", flush=True)
