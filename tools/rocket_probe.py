"""Rocket (13+3) solve timing, boxed and unboxed (the library runs both through the group sweep)."""
import importlib, os, sys, time
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
d = importlib.import_module("differentiable-ilqr_b200")
env = importlib.import_module("differentiable-ilqr_b200.env_dx")
lib = importlib.import_module("differentiable-ilqr_b200._lib")
dev = torch.device("cuda:0")
B = int(sys.argv[1]) if len(sys.argv) > 1 else 16384
T = int(sys.argv[2]) if len(sys.argv) > 2 else 100
dtype = torch.float64
g = torch.Generator().manual_seed(0)
dx = env.RocketDx(torch.tensor((0.5, 1.0, 1.0, 1.0, 1.0), dtype=dtype, device=dev))
qv = torch.cat((torch.ones(B, 1, dtype=dtype), 0.1 * torch.randn(B, 3, generator=g, dtype=dtype)), 1)
x0 = torch.cat(((torch.rand(B, 3, generator=g, dtype=dtype) * 2 - 1) * 15,
                torch.rand(B, 3, generator=g, dtype=dtype) * 2 - 1, qv / qv.norm(dim=1, keepdim=True),
                (torch.rand(B, 3, generator=g, dtype=dtype) * 2 - 1) * 0.1), 1).to(dev)
q, p = [t.to(dtype).to(dev) for t in dx.get_true_obj()]
C = torch.diag(q)[None, None].repeat(T, B, 1, 1)
c = p[None, None].repeat(T, B, 1)
for boxed in (True, False):
    kw = dict(u_lower=-20.0, u_upper=20.0) if boxed else {}
    m = d.mpc_explicit.MPC(13, 3, T, lqr_iter=10, verbose=-1, exit_unconverged=False,
                           detach_unconverged=False, linesearch_decay=dx.linesearch_decay,
                           max_linesearch_iter=dx.max_linesearch_iter, eps=dx.mpc_eps, n_batch=B, **kw)
    lib.profile = None
    for _ in range(2):
        with torch.no_grad():
            x, u, _ = m(x0, d.QuadCost(C, c), dx)
    torch.cuda.synchronize()
    lib.profile = {}
    t0 = time.time()
    with torch.no_grad():
        x, u, _ = m(x0, d.QuadCost(C, c), dx)
    torch.cuda.synchronize()
    dt = time.time() - t0
    prof = {k: sum(a.elapsed_time(b) for a, b in v) / len(v) for k, v in lib.profile.items()}
    lib.profile = None
    print("boxed=%s: %.1f ms/solve, qp_iters %s, per call ms %s" % (
        boxed, dt * 1e3, m.last_info.qp_iters[:3], {k: round(v, 2) for k, v in prof.items()}))
