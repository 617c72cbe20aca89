"""Small end-to-end case for compute-sanitizer (memcheck): staged + tail warps +
group sweep + trace replay + factored adjoint + generic adjoint paths."""
import importlib, os, sys
import torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests")); sys.path.insert(0, os.path.join(ROOT, "oracle"))
import port
from common import env_problem, lindx_problem
d = importlib.import_module("differentiable-ilqr_b200")
env = importlib.import_module("differentiable-ilqr_b200.env_dx")
dev = torch.device("cuda:0")
for name, T, B in (("cartpole", 12, 70), ("pendulum", 10, 33), ("rocket", 8, 5)):
    pdx, x0, C, c, kw = env_problem(port, name, T, B, torch.float64, sigma=0.05)
    theta = pdx.params.to(dev).requires_grad_()
    gdx = {"cartpole": env.CartpoleDx, "pendulum": env.PendulumDx, "rocket": env.RocketDx}[name](theta)
    m = d.mpc_explicit.MPC(pdx.n_state, pdx.n_ctrl, T, lqr_iter=4, verbose=-1, exit_unconverged=False,
                           detach_unconverged=False, richardson_passes=3, richardson_tol=None, **kw)
    Cg = C.to(dev).requires_grad_()
    x, u, _ = m(x0.to(dev), d.QuadCost(Cg, c.to(dev)), gdx)
    (x.sum() + u.pow(2).sum()).backward()
    print(name, "ok", float(theta.grad.abs().sum()))
for ns, nc, B in ((4, 2, 40), (5, 1, 31), (16, 4, 3)):
    C, c, F, f, x0 = [t.to(dev) for t in lindx_problem(ns, nc, 8, B, torch.float64)]
    m = d.MPC(ns, nc, 8, lqr_iter=3, verbose=-1, exit_unconverged=False, detach_unconverged=False,
              u_lower=-1.0, u_upper=1.0)
    Cg = C.clone().requires_grad_()
    x, u, _ = m(x0, d.QuadCost(Cg, c), d.LinDx(F, f))
    (x.sum() + u.sum()).backward()
    print("lindx", ns, nc, "ok")
H = torch.eye(3, dtype=torch.float64, device=dev).repeat(9, 1, 1) * 2
print(d.pnqp(H, torch.ones(9, 3, dtype=torch.float64, device=dev), -0.2, 0.3)[3])
torch.cuda.synchronize()
