"""CPU: host-side logic that needs no kernel - byte accounting of bench.py and the zero-padding that
embeds an (n,m) problem into a compiled (N,M) kernel instance (checked with the oracle)."""
import pytest
import torch

from oracle import lqr_oracle as orc
from tests.helpers import gen_problem, maxdiff, nominal_controls


def test_bytes_per_solve_matches_survey_table():
    """SURVEY.md section 8: 820 / 8788 / 17128 / 17448 / 157928 bytes per solve for configs 1-5."""
    import bench
    assert bench.bytes_per_solve(5, 3, 1) == 820
    assert bench.bytes_per_solve(25, 5, 1) == 8788
    assert bench.bytes_per_solve(20, 8, 2) == 17128
    assert bench.bytes_per_solve(20, 8, 2, tensor_bounds=True) == 17448
    assert bench.bytes_per_solve(50, 16, 4) == 157928


def test_bench_dump_outputs_whole_batch_or_fixed_sample(tmp_path, monkeypatch):
    """`bench.py --dump-outputs`: the whole batch while it fits the size limit, else the same seeded sample of
    problems in every run, taken from every output along its batch axis, within the limit."""
    import numpy as np
    import bench
    T, B, n, m = 4, 64, 3, 2
    g = torch.Generator().manual_seed(1)
    out = dict(new_x=torch.randn(T, B, n, generator=g), new_u=torch.randn(T, B, m, generator=g),
               costs=torch.arange(B, dtype=torch.float32), full_du_norm=torch.randn(B, generator=g),
               alphas=torch.rand(B, generator=g))
    bench.dump_outputs(out, B, str(tmp_path / "all"))
    for k, v in out.items():
        got = np.load(tmp_path / "all" / f"{k}.npy")
        assert got.dtype == np.float32 and np.array_equal(got, v.numpy()), k
    limit = 20 * (T * (n + m) + 3) * 4 + 4096               # room for 20 of the 64 problems
    monkeypatch.setattr(bench, "DUMP_MAX_BYTES", limit)
    for d in ("a", "b"):
        bench.dump_outputs(out, B, str(tmp_path / d))
    idx = np.load(tmp_path / "a" / "costs.npy").astype(np.int64)    # costs[b] == b names the sampled problems
    assert len(idx) == 20 and np.all(np.diff(idx) > 0)
    total = 0
    for k, v in out.items():
        a, b = np.load(tmp_path / "a" / f"{k}.npy"), np.load(tmp_path / "b" / f"{k}.npy")
        assert np.array_equal(a, b) and np.array_equal(a, v.numpy()[idx] if v.dim() == 1 else v.numpy()[:, idx]), k
        total += (tmp_path / "a" / f"{k}.npy").stat().st_size
    assert total <= limit


@pytest.mark.parametrize("shape,bounds", [((3, 3), 0.3), ((6, 1), None), ((5, 3), "tensor")])
def test_padding_embedding_is_exact(shape, bounds):
    """step._Pad: the padded problem solved by the ORACLE equals the original problem (so a padded
    kernel launch computes the same thing); padded controls stay at 0 and free."""
    from mpc.pytorch_b200.step import _Pad
    n, m = shape
    N, M = n + 2, m + 1
    B, T = 4, 6
    C, c, F, f, x0 = gen_problem(90, B, T, n, m, torch.float64, time_varying=True)
    u, ul, uu = nominal_controls(90, B, T, m, torch.float64, bounds)
    x = orc.get_traj(T, u, x0, F, f)
    ref = orc.lqr_step_forward(n, m, T, x0, C, c, F, f, x, u, u_lower=ul, u_upper=uu, coupled=False)
    pad = _Pad(n, m, N, M, torch.device("cpu"))
    if bounds is None:
        lo = hi = None
    else:
        lo = pad.vec_m(ul if torch.is_tensor(ul) else torch.full((T, B, m), ul, dtype=torch.float64), -1.0)
        hi = pad.vec_m(uu if torch.is_tensor(uu) else torch.full((T, B, m), uu, dtype=torch.float64), 1.0)
    got = orc.lqr_step_forward(N, M, T, pad.vec_n(x0), pad.mat_pp(C), pad.vec_p(c), pad.mat_np(F), pad.vec_n(f),
                               pad.vec_n(x), pad.vec_m(u), u_lower=lo, u_upper=hi, coupled=False)
    assert maxdiff(got.new_x[..., :n], ref.new_x) < 1e-10 and maxdiff(got.new_u[..., :m], ref.new_u) < 1e-10
    assert float(got.new_x[..., n:].abs().max()) == 0.0 and float(got.new_u[..., m:].abs().max()) == 0.0
    assert maxdiff(got.costs, ref.costs) < 1e-10
    assert maxdiff(got.Ks[..., :m, :n], ref.Ks) < 1e-10
    if bounds is not None:
        assert torch.equal(got.free_masks[..., :m], ref.free_masks) and bool(got.free_masks[..., m:].all())


def test_reference_full_du_norm_quirk():
    """The reference views a [T,m,B] buffer as [B,T*m] (mpc/lqr_step.py:244-245): identical to the
    per-problem norm only for B == 1; the sum of squares is preserved."""
    from mpc.pytorch_b200.step import reference_full_du_norm
    du = torch.randn(5, 3, 2, dtype=torch.float64)
    q = reference_full_du_norm(du)
    true = du.pow(2).sum((0, 2)).sqrt()
    assert abs(float(q.pow(2).sum() - true.pow(2).sum())) < 1e-12
    assert not torch.allclose(q, true)
    one = torch.randn(5, 1, 2, dtype=torch.float64)
    assert torch.allclose(reference_full_du_norm(one), one.pow(2).sum((0, 2)).sqrt())


def test_linearize_dynamics_methods_agree_on_cpu():
    """linearize_dynamics is pure torch (no kernel): ANALYTIC / AUTO_DIFF / FINITE_DIFF agree to 1e-4 and
    reproduce the dynamics to first order (reference tests/test_mpc.py:747-799)."""
    from mpc.pytorch_b200.solver import MPC, GradMethods
    from tests.cartpole import Cartpole, initial_states

    class CartpoleAnalytic(Cartpole):
        def grad_input(self, x, u):
            xg, ug = x.detach().requires_grad_(True), u.detach().requires_grad_(True)
            with torch.enable_grad():
                y = self.forward(xg, ug)
                rows = [torch.autograd.grad(y[:, j].sum(), [xg, ug], retain_graph=True) for j in range(5)]
            return torch.stack([r[0] for r in rows], 1), torch.stack([r[1] for r in rows], 1)

    T, B = 5, 3
    dx = CartpoleAnalytic()
    x0 = initial_states(B, 2, torch.float64)
    u = 0.5 * torch.randn(T, B, 1, dtype=torch.float64)
    xs = [x0]
    for t in range(T - 1):
        xs.append(dx(xs[t], u[t]))
    x = torch.stack(xs)
    outs = [MPC(5, 1, T, grad_method=gm).linearize_dynamics(x, u, dx, diff=False)
            for gm in (GradMethods.ANALYTIC, GradMethods.AUTO_DIFF, GradMethods.FINITE_DIFF)]
    for F2, f2 in outs[1:]:
        assert maxdiff(F2, outs[0][0]) < 1e-4 and maxdiff(f2, outs[0][1]) < 1e-4
    F, f = outs[0]
    pred = torch.einsum("tbij,tbj->tbi", F, torch.cat((x[:-1], u[:-1]), 2)) + f
    assert maxdiff(pred, x[1:]) < 1e-10                      # exact at the expansion point
    Fd, fd = MPC(5, 1, T, grad_method=GradMethods.AUTO_DIFF).linearize_dynamics(x, u, dx, diff=True)
    assert maxdiff(Fd, F) < 1e-12


def test_approximate_cost_recovers_a_quadratic():
    """approximate_cost (reference mpc/mpc.py:447-487) on a known quadratic returns its C and c."""
    from mpc.pytorch_b200.solver import MPC
    T, B, n, m = 4, 3, 3, 2
    p = n + m
    g = torch.Generator().manual_seed(0)
    L = torch.randn(p, p, generator=g, dtype=torch.float64)
    Cq = L @ L.T + torch.eye(p, dtype=torch.float64)
    cq = torch.randn(p, generator=g, dtype=torch.float64)

    class Quad(torch.nn.Module):
        def forward(self, tau):
            return 0.5 * (tau @ Cq * tau).sum(-1) + tau @ cq

    x = torch.randn(T, B, n, generator=g, dtype=torch.float64)
    u = torch.randn(T, B, m, generator=g, dtype=torch.float64)
    H, lin, costs = MPC(n, m, T).approximate_cost(x, u, Quad(), diff=False)
    assert maxdiff(H, Cq.expand(T, B, p, p)) < 1e-10
    assert maxdiff(lin, cq.expand(T, B, p)) < 1e-10
    tau = torch.cat((x, u), 2)
    assert maxdiff(costs, 0.5 * (tau @ Cq * tau).sum(-1) + tau @ cq) < 1e-10


def test_bench_reference_arm_prints_the_contract_line():
    """`bench.py --impl reference` (CPU arm: the unmodified reference when baseline/_ref travelled, else the
    oracle port) must print one JSON line with the contract keys."""
    import json
    import os
    import subprocess
    import sys
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    out = subprocess.run([sys.executable, os.path.join(root, "bench.py"), "--impl", "reference", "--steps", "1",
                          "--warmup", "1"], capture_output=True, text=True, timeout=240, cwd=root)
    assert out.returncode == 0, out.stderr[-500:]
    line = json.loads(out.stdout.strip().splitlines()[-1])
    for key in ("metric", "value", "unit", "n_gpus", "steps", "warmup", "ms_per_step", "higher_is_better",
                "scaling", "vs_baseline", "dtype", "data", "config", "impl", "cpu_baseline", "e2e"):
        assert key in line, key
    have_ref = os.path.exists(os.path.join(root, "baseline", "_ref", "mpc", "__init__.py"))
    assert line["impl"] == "reference" and line["cpu_baseline"]["kind"] == ("reference" if have_ref else "port")
    assert line["e2e"]["h2d_bytes_per_step"] == 0 and line["value"] > 0
    assert "workload" in line["config"] and "model" not in line["config"]
