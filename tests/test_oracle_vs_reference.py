"""The oracle's pnqp and the Cholesky-gain variant of the reference's LQR step against
the reference's outputs, stored in tests/golden by tests/golden/make_golden.py
(pnqp_cases, backup_chol)."""
import pytest
import torch

from common import golden


@pytest.mark.parametrize("n,seed", [(1, 0), (2, 1), (3, 2), (4, 3)])
def test_pnqp_matches_reference(port, n, seed):
    g = golden("ref_pnqp.npz")
    k = "n%d_s%d_" % (n, seed)
    torch.set_default_dtype(torch.float64)
    try:
        for tag, x_init in (("cold", None), ("warm", g[k + "x_init"])):
            o = port.pnqp(g[k + "H"], g[k + "q"], g[k + "lo"], g[k + "hi"], x_init=x_init,
                          n_iter=20)
            assert float((o.x - g[k + tag + "_x"]).abs().max()) == 0.0
            assert torch.equal(o.If, g[k + tag + "_If"])
            assert o.n_iter == int(g[k + tag + "_n_iter"])
    finally:
        torch.set_default_dtype(torch.float32)


def test_backup_variant_cholesky(port):
    """lqr_step_backup's Cholesky(+1e-6 I) gains (used inside the DiLQR backward)."""
    g = golden("ref_backup_chol.npz")
    torch.set_default_dtype(torch.float64)
    try:
        ns, nc, T = 4, 2, 8
        o = port.mpc_forward(g["x0"], port.QuadCost(g["C"], g["c"]), port.LinDx(g["F"], None), ns,
                             nc, T, lqr_iter=1, gain_solve="chol_reg", final_pass=False)
        assert float((o.u - g["u"]).abs().max()) < 1e-13
    finally:
        torch.set_default_dtype(torch.float32)
