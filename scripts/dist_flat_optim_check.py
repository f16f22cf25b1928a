"""2-rank NCCL check of flat_adam.FlatAdamW with two parameter groups, global gradient-norm
clipping and the overlapped early bucket (torchrun, 2 GPUs).  Two ranks train a small two-stage
model on disjoint halves of a batch; the result must equal single-process torch.optim.AdamW +
clip_grad_norm_ on the averaged gradients.  Run twice:
  eager:    backward with the early bucket reduced from a tensor hook, then step();
  captured: pack, early all-reduce (side stream), late all-reduce, norm and update captured in one
            CUDA graph over static gradient tensors, replayed every step.
Prints 'dist_flat_optim ok' on rank 0."""
import os, sys
import torch, torch.distributed as dist
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from backtoreality_b200.flat_adam import FlatAdamW

rank, world = int(os.environ["RANK"]), int(os.environ["WORLD_SIZE"])
torch.cuda.set_device(int(os.environ.get("LOCAL_RANK", rank)))
dev = torch.device("cuda", torch.cuda.current_device())
dist.init_process_group("nccl", device_id=dev)
MAX_NORM, STEPS = 0.05, 6


def make():
    torch.manual_seed(0)
    a = torch.nn.Sequential(torch.nn.Linear(16, 32), torch.nn.ReLU()).to(dev)   # "late" stage (first layers)
    b = torch.nn.Sequential(torch.nn.Linear(32, 32), torch.nn.ReLU(), torch.nn.Linear(32, 4)).to(dev)
    return a, b


def groups(a, b):
    # group 0: the first stage; group 1 ("decoder"): its own rate, no weight decay
    return [{"params": list(a.parameters())}, {"params": list(b.parameters()), "lr": 3e-3, "weight_decay": 0.0}]


g = torch.Generator().manual_seed(1)
data = torch.randn(STEPS, 8, 16, generator=g).to(dev)
scale = torch.tensor([0.2, 3.0, 0.5, 4.0, 0.1, 2.0], device=dev)    # some steps clip, some do not


def loss_of(a, b, x, k):
    return b(a(x)).square().mean() * scale[k]


def reference():
    ra, rb = make()
    ropt = torch.optim.AdamW(groups(ra, rb), lr=1e-2, weight_decay=0.05)
    params = list(ra.parameters()) + list(rb.parameters())
    norms = []
    for k in range(STEPS):
        ropt.zero_grad()
        for r in range(world):
            xs = data[k][r * 4:(r + 1) * 4]
            (loss_of(ra, rb, xs, k) / world).backward()
        norms.append(float(torch.nn.utils.clip_grad_norm_(params, MAX_NORM)))
        ropt.step()
    return params, norms


def check(params, norms, ref_params, ref_norms, what):
    err = max(float((p - q).abs().max()) for p, q in zip(params, ref_params))
    assert err < 1e-5, (what, err)
    nerr = max(abs(x - y) / y for x, y in zip(norms, ref_norms))
    assert nerr < 1e-5, (what, norms, ref_norms)
    assert min(ref_norms) < MAX_NORM < max(ref_norms), ref_norms
    return err


ref_params, ref_norms = reference()

# eager: early bucket from the backward hook
a, b = make()
opt = FlatAdamW(groups(a, b), lr=1e-2, weight_decay=0.05, max_grad_norm=MAX_NORM)
opt.set_late(len(list(a.parameters())))
norms = []
for k in range(STEPS):
    opt.zero_grad()
    h = a(data[k][rank * 4:(rank + 1) * 4])
    h.register_hook(lambda gr: opt.reduce_early())
    (b(h).square().mean() * scale[k]).backward()
    assert opt._early_done
    opt.step()
    norms.append(float(opt.last_grad_norm))
err_eager = check(opt.params, norms, ref_params, ref_norms, "eager")

# captured: the whole optimizer step, both all-reduces included, replayed from a graph
a, b = make()
opt = FlatAdamW(groups(a, b), lr=1e-2, weight_decay=0.05, max_grad_norm=MAX_NORM)
opt.set_late(len(list(a.parameters())))
static = [torch.zeros_like(p) for p in opt.params]


def grads_of(k):
    a2, b2 = make()           # gradients at the optimizer's current weights
    with torch.no_grad():
        for p, q in zip(list(a2.parameters()) + list(b2.parameters()), opt.params):
            p.copy_(q)
    loss_of(a2, b2, data[k][rank * 4:(rank + 1) * 4], k).backward()
    return [p.grad for p in list(a2.parameters()) + list(b2.parameters())]


def captured_body():
    for p, s in zip(opt.params, static):
        p.grad = s
    opt.reduce_early()        # params[n_late:]: packed and all-reduced on the side stream
    opt.step()                # the late part, its all-reduce, the norm and the update


norms = []
for x, y in zip(static, grads_of(0)):
    x.copy_(y)
side = torch.cuda.Stream()
side.wait_stream(torch.cuda.current_stream())
with torch.cuda.stream(side):
    captured_body()           # step 0 runs eagerly (warm-up before capture)
torch.cuda.current_stream().wait_stream(side)
norms.append(float(opt.last_grad_norm))
graph = torch.cuda.CUDAGraph()
with torch.cuda.graph(graph):
    captured_body()
for k in range(1, STEPS):
    for x, y in zip(static, grads_of(k)):
        x.copy_(y)
    opt.sync_hparams()
    graph.replay()
    norms.append(float(opt.last_grad_norm))
err_graph = check(opt.params, norms, ref_params, ref_norms, "captured")
if rank == 0:
    print("dist_flat_optim ok, max |dp| eager %.2e captured %.2e, norms %s (max_norm %g)"
          % (err_eager, err_graph, " ".join("%.4f" % x for x in ref_norms), MAX_NORM), flush=True)
torch.cuda.synchronize()
os._exit(0)
