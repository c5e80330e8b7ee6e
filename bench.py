#!/usr/bin/env python3
"""bench.py - LQR solves/sec of the B200-native LQR step (BASELINE.json metric).

Workload (default, N=1): BASELINE config 3, "Random LTI batched LQR, n_batch=4096, T=20, n_state=8,
n_ctrl=2" in fp32, unbounded; one *step* = one LQRStepFn.forward over the batch (Riccati sweep +
line-search rollout) = ONE kernel launch.  N>1: every rank owns its own shard (weak scaling, no
collective on the solve path; NCCL only for the barrier and the max-over-ranks).
`--workload config5` measures BASELINE config 5 instead (n_batch=32768 in total, T=50, n=16, m=4,
sharded over the N GPUs: strong scaling).

  value      device-resident throughput: inputs in HBM, rotating over input sets larger than L2; the timed
             region is EXACTLY --steps launches (barrier + synchronize on both sides), max over ranks
  e2e        same metric through the public API LQRStep(...)(x_init,C,c,F,f) with the inputs in
             pinned HOST memory: H2D of the step's inputs and D2H of its results inside the timing
  roofline   algorithmic bytes per launch / kernel time  vs the measured HBM copy peak
  cpu_baseline  the UNMODIFIED reference (baseline/_ref, pip --target install of /root/reference) on the
             host cores when it travelled with the snapshot, else the oracle port (oracle/lqr_oracle.py)
  extra      (N=1) secondary figures of SURVEY.md section 8(d): KKT-adjoint solves/s, box-constrained
             configs 3/4, the config-5 shard with its fp32-FMA fraction

`--impl reference` times the CPU path alone: the unmodified reference when baseline/_ref exists, else the port.
"""
import argparse
import contextlib
import ctypes
import faulthandler
import importlib.util
import io
import json
import os
import statistics
import subprocess
import sys
import threading
import time
import warnings

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

import numpy as np  # noqa: E402
import torch  # noqa: E402

WORKLOADS = {
    "config3": dict(B=4096, T=20, n=8, m=2, scaling="weak",
                    name="config3: random LTI batched LQR, n_batch=4096/GPU, T=20, n_state=8, n_ctrl=2, fp32, unbounded"),
    "config5": dict(B=32768, T=50, n=16, m=4, scaling="strong",
                    name="config5: batch-sharded random LTI LQR, n_batch=32768 total, T=50, n_state=16, n_ctrl=4, fp32, unbounded"),
}
FP32_FMA_PEAK_TFLOPS = 148 * 128 * 2 * 1.965e9 / 1e12      # 148 SMs x 128 FMA lanes x 2 flop x 1.965 GHz = 74.5


def bytes_per_solve(T, n, m, tensor_bounds=False):
    """SURVEY.md section 8(d): every input read once, every output written once (fp32)."""
    p = n + m
    inp = T * p * p + T * p + (T - 1) * n * p + (T - 1) * n + n + T * n + T * m
    if tensor_bounds:
        inp += 2 * T * m
    return 4 * inp + 4 * (T * n + T * m + 2)


def adjoint_bytes_per_solve(T, n, m):
    """SURVEY.md section 8(d) 'adjoint pass bytes': reads C, c_x, F, tau*, r; writes dC, dc, dF, df, dx_init."""
    p = n + m
    rd = T * p * p + T * n + (T - 1) * n * p + 2 * T * p
    wrt = T * p * p + T * p + (T - 1) * n * p + (T - 1) * n + n
    return 4 * (rd + wrt)


def flops_per_solve(T, n, m):
    """SURVEY.md section 8(d) algorithmic flops (one line-search pass)."""
    p = n + m
    bwd = T * (2 * n * n * p + 2 * n * p * p + 2 * n * p + 6 * n * n * m + 2 * m * m * n)
    return bwd + 2 * T * p * p + 2 * T * (2 * m * n + 2 * n * p + 2 * p * p + 2 * p)


def gen_inputs(seed, B, T, n, m, device):
    """Synthetic generator of SURVEY.md section 8(d) (same as tests/helpers.gen_problem, on device)."""
    g = torch.Generator(device=device).manual_seed(seed)
    p = n + m
    L = torch.randn(T, B, p, p, generator=g, device=device) / p ** 0.5
    C = L @ L.transpose(-1, -2) + torch.eye(p, device=device)
    del L
    c = torch.randn(T, B, p, generator=g, device=device)
    A = 0.9 * torch.eye(n, device=device) + 0.1 * torch.randn(B, n, n, generator=g, device=device) / n ** 0.5
    Bm = torch.randn(B, n, m, generator=g, device=device) / n ** 0.5
    F = torch.cat((A, Bm), -1).unsqueeze(0).repeat(T - 1, 1, 1, 1).contiguous()
    f = 0.1 * torch.randn(T - 1, B, n, generator=g, device=device)
    x0 = torch.randn(B, n, generator=g, device=device)
    u = torch.zeros(T, B, m, device=device)
    xs = [x0]
    for t in range(T - 1):
        xs.append(torch.einsum("bij,bj->bi", F[t], torch.cat((xs[t], u[t]), 1)) + f[t])
    x = torch.stack(xs)
    return dict(x_init=x0, C=C.contiguous(), c=c, F=F, f=f, cur_x=x, cur_u=u)


class ClockSampler:
    """nvidia-smi clocks / throttle reasons while the GPU is under this benchmark's load."""
    Q = ("clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,"
         "clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap,utilization.gpu")

    def __init__(self, index):
        self.rows, self.proc, self.index = [], None, index

    def start(self):
        try:
            self.proc = subprocess.Popen(
                ["nvidia-smi", "-i", str(self.index), "--query-gpu=" + self.Q, "--format=csv,noheader,nounits",
                 "-lms", "50"], stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except OSError:
            self.proc = None

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([s.strip() for s in line.split(",")])

    def stop(self):
        if self.proc is None:
            return {"sm_mhz": None, "sm_max_mhz": None, "reasons": ["nvidia-smi unavailable"]}
        self.proc.terminate()
        rows = [r for r in self.rows if len(r) >= 7 and r[0].isdigit()]
        busy = [r for r in rows if r[6].isdigit() and int(r[6]) > 0] or rows
        reasons = set()
        for r in busy:
            for name, v in zip(("hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"), r[2:6]):
                if v.lower().startswith("active"):
                    reasons.add(name)
        return {"sm_mhz": statistics.median(int(r[0]) for r in busy) if busy else None,
                "sm_max_mhz": int(busy[0][1]) if busy else None, "reasons": sorted(reasons),
                "samples": len(busy)}


class RawStepper:
    """Pre-bound C-ABI call (device-resident arm): one ctypes call = one kernel launch."""

    def __init__(self, inp, B, T, n, m, bounds=None, tensor_bounds=None):
        from mpc.pytorch_b200 import _lib
        from mpc.pytorch_b200._lib import Dims, Params, ptr
        dev = inp["C"].device
        self.out = dict(new_x=torch.empty(T, B, n, device=dev), new_u=torch.empty(T, B, m, device=dev),
                        costs=torch.empty(B, device=dev), full_du_norm=torch.empty(B, device=dev),
                        alphas=torch.empty(B, device=dev))
        kind = 0 if bounds is None and tensor_bounds is None else (2 if tensor_bounds is not None else 1)
        self.dims = Dims(B=B, T=T, n=n, m=m, F_T=T - 1, has_f=1, bounds_kind=kind, has_zero_mask=0,
                         has_delta_u=0, max_ls_iter=10, pnqp_max_iter=20, do_rollout=1)
        self.params = Params(u_lo=-(bounds or 0.0), u_hi=(bounds or 0.0), delta_u=0.0, ls_decay=0.2)
        self.fn = _lib.lib().mpcb200_lqr_step_f32
        o = self.out
        lo, hi = tensor_bounds if tensor_bounds is not None else (None, None)
        # long horizons keep their gains in a caller buffer (mpcb200_step_prefers_workspace)
        self.Ks = self.ks = None
        if _lib.lib().mpcb200_step_prefers_workspace(ctypes.byref(self.dims), 4):
            self.Ks = torch.empty(T, B, m, n, device=dev)
            self.ks = torch.empty(T, B, m, device=dev)
        self.args = [ctypes.byref(self.dims), ctypes.byref(self.params), ptr(inp["C"]), ptr(inp["c"]),
                     ptr(inp["F"]), ptr(inp["f"]), ptr(inp["x_init"]), ptr(inp["cur_x"]), ptr(inp["cur_u"]),
                     ptr(lo), ptr(hi), None, ptr(o["new_x"]), ptr(o["new_u"]), ptr(o["costs"]), ptr(o["full_du_norm"]),
                     ptr(o["alphas"]), None, None, None, None, ptr(self.Ks), ptr(self.ks), None]
        self.keep = (inp, lo, hi)

    def __call__(self, stream):
        self.args[-1] = stream
        rc = self.fn(*self.args)
        if rc != 0:
            raise RuntimeError(f"mpcb200_lqr_step_f32 -> {rc}")


class RawAdjoint:
    """Pre-bound one-call KKT adjoint (mpcb200_lqr_adjoint_f32), the C-ABI view of LQRStepFn.backward."""

    def __init__(self, inp, new_x, new_u, B, T, n, m):
        from mpc.pytorch_b200 import _lib
        from mpc.pytorch_b200._lib import Dims, Params, ptr
        dev = inp["C"].device
        p = n + m
        self.dims = Dims(B=B, T=T, n=n, m=m, F_T=T - 1, has_f=1, bounds_kind=0, has_zero_mask=0, has_delta_u=0,
                         max_ls_iter=10, pnqp_max_iter=20, do_rollout=1)
        self.params = Params(u_lo=0.0, u_hi=0.0, delta_u=0.0, ls_decay=0.2)
        L = _lib.lib()
        nbytes = L.mpcb200_adjoint_workspace_bytes(ctypes.byref(self.dims), 4)
        self.buf = dict(ws=torch.empty(nbytes, dtype=torch.uint8, device=dev), wx=torch.randn(T, B, n, device=dev),
                        wu=torch.randn(T, B, m, device=dev), dx_init=torch.empty(B, n, device=dev),
                        dC=torch.empty(T, B, p, p, device=dev), dc=torch.empty(T, B, p, device=dev),
                        dF=torch.empty(T - 1, B, n, p, device=dev), df=torch.empty(T - 1, B, n, device=dev))
        b = self.buf
        self.fn = L.mpcb200_lqr_adjoint_f32
        self.args = [ctypes.byref(self.dims), ctypes.byref(self.params), ptr(inp["C"]), ptr(inp["c"]), ptr(inp["F"]),
                     ptr(new_x), ptr(new_u), ptr(b["wx"]), ptr(b["wu"]), None, None, ptr(b["dx_init"]), ptr(b["dC"]),
                     ptr(b["dc"]), ptr(b["dF"]), ptr(b["df"]), ptr(b["ws"]), ctypes.c_size_t(nbytes), None]
        self.keep = (inp, new_x, new_u)

    def __call__(self, stream):
        self.args[-1] = stream
        rc = self.fn(*self.args)
        if rc != 0:
            raise RuntimeError(f"mpcb200_lqr_adjoint_f32 -> {rc}")


DUMP_MAX_BYTES = 64 * 10**6


def dump_outputs(out, B, path):
    """Writes the arrays one step call returns (new_x, new_u [T,B,.]; costs, full_du_norm, alphas [B]) as float32
    `path/<name>.npy`.  Outputs larger than DUMP_MAX_BYTES are cut to a fixed, seeded sample of the problems (the
    same in every run, kept in batch order), so that the dumps of two builds compare output for output."""
    per_problem = sum(v.numel() // B * v.element_size() for v in out.values())
    keep = min(B, (DUMP_MAX_BYTES - 4096) // per_problem)       # 4 kB left for the .npy headers
    idx = torch.randperm(B, generator=torch.Generator().manual_seed(0))[:keep].sort().values
    os.makedirs(path, exist_ok=True)
    for name, v in out.items():
        v = v.index_select(0 if v.dim() == 1 else 1, idx.to(v.device))
        np.save(os.path.join(path, name + ".npy"), v.cpu().numpy())


# --------------------------------------------------------------------------------------------- CPU arms
def load_unmodified_reference():
    """The reference package as installed by `pip install --target baseline/_ref /root/reference`
    (git-ignored, travels with the gpurun snapshot), imported under an alias so it cannot collide with this
    repo's drop-in `mpc` package.  Returns (mpc module, lqr_step module) or None."""
    pkg_dir = os.path.join(ROOT, "baseline", "_ref", "mpc")
    if not os.path.exists(os.path.join(pkg_dir, "__init__.py")):
        return None
    spec = importlib.util.spec_from_file_location("ref_mpc", os.path.join(pkg_dir, "__init__.py"),
                                                  submodule_search_locations=[pkg_dir])
    pkg = importlib.util.module_from_spec(spec)
    sys.modules["ref_mpc"] = pkg
    spec.loader.exec_module(pkg)
    import ref_mpc.mpc as rmpc          # noqa
    import ref_mpc.lqr_step as rstep    # noqa
    return rmpc, rstep


def _calibrate_threads(one):
    """"All the host threads it can use": the tiny batched ops stop scaling early, so try a few thread
    counts on one step each and keep the fastest."""
    ncpu = os.cpu_count() or 1
    best = None
    for cand in sorted({c for c in (4, 8, 16, 32, 64, ncpu) if c <= ncpu}):
        torch.set_num_threads(cand)
        t0 = time.perf_counter()
        one()
        dt = time.perf_counter() - t0
        if best is None or dt < best[0]:
            best = (dt, cand)
        if dt > 3 * best[0]:
            break
    torch.set_num_threads(best[1])
    return best[1]


def cpu_arm(cfg, steps, warmup, budget_s=20.0, prefer_reference=True):
    """Times the reference's CPU path of the workload on a BOUNDED sample of it:
    (value solves/s, ms/step, cores, kind, steps done, sample description)."""
    from oracle import lqr_oracle as orc
    T, n, m = cfg["T"], cfg["n"], cfg["m"]
    ref = load_unmodified_reference() if prefer_reference else None
    warnings.filterwarnings("ignore")
    # sample size: the whole per-GPU batch for the vectorised port; for the unmodified reference (a Python loop
    # of per-sample pinverse calls, ~1 ms per problem-step) as many problems as keep one step at a few seconds
    B = cfg["B"] if ref is None else min(cfg["B"], 4096 if n <= 8 else 512)
    inp = gen_inputs(3000, B, T, n, m, torch.device("cpu"))

    def make_one(d):
        if ref is not None:
            rmpc, rstep = ref

            def one():  # exactly how the reference's MPC.solve_lqr_subproblem calls it (mpc/mpc.py:342-361)
                with torch.no_grad(), contextlib.redirect_stdout(io.StringIO()):
                    step = rstep.LQRStep(n_state=n, n_ctrl=m, T=T, u_lower=None, u_upper=None, u_zero_I=None,
                                         delta_u=None, linesearch_decay=0.2, max_linesearch_iter=10,
                                         true_cost=rmpc.QuadCost(d["C"], d["c"]),
                                         true_dynamics=rmpc.LinDx(d["F"], d["f"]), delta_space=True,
                                         current_x=d["cur_x"], current_u=d["cur_u"], back_eps=1e-7,
                                         no_op_forward=False)
                    return step(d["x_init"], d["C"], d["c"], d["F"], d["f"])
        else:
            def one():
                return orc.lqr_step_forward(n, m, T, d["x_init"], d["C"], d["c"], d["F"], d["f"],
                                            d["cur_x"], d["cur_u"], coupled=True)
        return one
    if ref is not None:
        kind, what = "reference", "UNMODIFIED reference (baseline/_ref) LQRStep(...)(x_init,C,c,F,f) on torch CPU"
        small = {k: (v[:, :128].contiguous() if v.dim() > 2 else v[:128].contiguous()) for k, v in inp.items()}
        cores = _calibrate_threads(make_one(small))        # thread count chosen on a 128-problem slice
    else:
        kind, what = "port", "oracle port (oracle/lqr_oracle.py, vectorised torch CPU)"
        cores = _calibrate_threads(make_one(inp))
    one = make_one(inp)
    torch.set_num_threads(cores)
    for _ in range(warmup if kind == "port" else 0):
        one()
    t0 = time.perf_counter()
    done = 0
    for _ in range(steps):                 # bounded sample: stop after ~budget_s of CPU work
        one()
        done += 1
        if time.perf_counter() - t0 > budget_s:
            break
    dt = time.perf_counter() - t0
    return (B * done / dt, dt / done * 1e3, cores, kind, done,
            f"{done} x {cfg['name'].split(':')[0]} batch of {B} problems, {what}, {cores} threads")


# --------------------------------------------------------------------------------------------- GPU timing helpers
def time_launches(fns, reps, stream, sh, blocks=3):
    """min/median us per launch of `fns` (rotating) over `blocks` timed blocks of `reps` launches."""
    for i in range(max(3, len(fns))):
        fns[i % len(fns)](sh)
    torch.cuda.synchronize()
    out = []
    for _ in range(blocks):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record(stream)
        for i in range(reps):
            fns[i % len(fns)](sh)
        e1.record(stream)
        torch.cuda.synchronize()
        out.append(e0.elapsed_time(e1) / reps * 1e3)
    return statistics.median(out)


def extras(dev, stream, sh, peak):
    """Secondary figures (SURVEY.md section 8d) on one GPU; each entry: us per launch, solves/s, roofline frac."""
    from mpc.pytorch_b200 import LQRStep, QuadCost, LinDx, _lib
    res = {}

    def entry(us, B, T, n, m, tensor_bounds=False):
        bps = bytes_per_solve(T, n, m, tensor_bounds)
        return {"us_per_launch": round(us, 2), "solves_per_s": B / (us * 1e-6), "bytes_per_solve": bps,
                "hbm_frac": bps * B / (us * 1e-6) / 1e9 / peak}

    # config 3 with box bounds +-0.25, config 4 (B=1024) scalar and tensor bounds
    sets3 = [gen_inputs(3100 + s, 4096, 20, 8, 2, dev) for s in range(4)]
    res["config3_box"] = entry(time_launches([RawStepper(s, 4096, 20, 8, 2, bounds=0.25) for s in sets3], 40, stream, sh),
                               4096, 20, 8, 2)
    sets4 = [gen_inputs(4100 + s, 1024, 20, 8, 2, dev) for s in range(8)]
    res["config4_scalar_bounds"] = entry(
        time_launches([RawStepper(s, 1024, 20, 8, 2, bounds=0.25) for s in sets4], 40, stream, sh), 1024, 20, 8, 2)
    g = torch.Generator(device=dev).manual_seed(7)
    tb = [(-0.5 * torch.rand(20, 1024, 2, generator=g, device=dev), 0.5 * torch.rand(20, 1024, 2, generator=g, device=dev))
          for _ in sets4]
    res["config4_tensor_bounds"] = entry(
        time_launches([RawStepper(s, 1024, 20, 8, 2, tensor_bounds=b) for s, b in zip(sets4, tb)], 40, stream, sh),
        1024, 20, 8, 2, True)
    # KKT adjoint through the public API (LQRStepFn.backward) at config-3 size: solves/s and bytes of section 8(d)
    inp = sets3[0]
    lv = [inp[k].clone().requires_grad_(True) for k in ("x_init", "C", "c", "F", "f")]
    wx, wu = torch.randn_like(inp["cur_x"]), torch.randn_like(inp["cur_u"])

    fn = LQRStep(8, 2, 20, true_cost=QuadCost(lv[1], lv[2]), true_dynamics=LinDx(lv[3], lv[4]),
                 current_x=inp["cur_x"], current_u=inp["cur_u"], no_op_forward=True)
    xo, uo = fn(*lv)

    def adjoint(_sh=None):          # LQRStepFn.backward through autograd, upstream gradients given directly
        return torch.autograd.grad((xo, uo), lv, (wx, wu), retain_graph=True)
    l0 = _lib.launch_count()
    adjoint()
    n_kernels = _lib.launch_count() - l0
    us = time_launches([adjoint], 20, stream, sh)
    ab = adjoint_bytes_per_solve(20, 8, 2)
    res["adjoint_config3_api"] = {"us_per_backward": round(us, 2), "solves_per_s": 4096 / (us * 1e-6),
                                  "bytes_per_solve": ab, "hbm_frac": ab * 4096 / (us * 1e-6) / 1e9 / peak,
                                  "kernels_per_backward": int(n_kernels),
                                  "api": "torch.autograd.grad through LQRStep(no_op_forward=True)(...): the autograd engine + LQRStepFn.backward (Python host path included)"}
    raws = [RawAdjoint(s, s["cur_x"], s["cur_u"], 4096, 20, 8, 2) for s in sets3]
    l0 = _lib.launch_count()
    raws[0](sh)
    n_raw = _lib.launch_count() - l0
    us = time_launches(raws, 20, stream, sh)
    res["adjoint_config3_c_abi"] = {"us_per_backward": round(us, 2), "solves_per_s": 4096 / (us * 1e-6),
                                    "bytes_per_solve": ab, "hbm_frac": ab * 4096 / (us * 1e-6) / 1e9 / peak,
                                    "kernels_per_backward": int(n_raw),
                                    "api": "mpcb200_lqr_adjoint_f32 (prep + fused solve / costate / outer-product kernel), device resident"}
    del raws
    del sets3, sets4, lv
    torch.cuda.empty_cache()
    # config 5 shard of the 8-GPU run (4096 problems, T=50, n=16, m=4): compute bound -> also % of fp32 FMA peak
    s5 = [gen_inputs(5100 + s, 4096, 50, 16, 4, dev) for s in range(2)]
    us = time_launches([RawStepper(s, 4096, 50, 16, 4) for s in s5], 6, stream, sh)
    e = entry(us, 4096, 50, 16, 4)
    e["fp32_fma_frac"] = flops_per_solve(50, 16, 4) * 4096 / (us * 1e-6) / 1e12 / FP32_FMA_PEAK_TFLOPS
    e["fp32_fma_peak_tflops"] = round(FP32_FMA_PEAK_TFLOPS, 1)
    res["config5_shard_4096"] = e
    return res


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=20)
    ap.add_argument("--impl", default="b200", choices=["b200", "reference"])
    ap.add_argument("--workload", default="config3", choices=sorted(WORKLOADS))
    ap.add_argument("--no-extra", action="store_true", help="skip the secondary figures (adjoint, box, config 5)")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="write the outputs of the last timed step to DIR/<name>.npy (float32, at most 64 MB)")
    a = ap.parse_args()
    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local = int(os.environ.get("LOCAL_RANK", "0"))
    if a.steps < 1:
        ap.error("--steps must be at least 1")
    if a.dump_outputs and (a.impl != "b200" or world > 1):
        ap.error("--dump-outputs writes the CUDA step's outputs of a single process (--impl b200, one rank)")
    # watchdog: a hung bench must not eat the box; dumps all Python stacks and exits
    faulthandler.dump_traceback_later(int(os.environ.get("BENCH_WATCHDOG_S", "900")), exit=True)
    cfg = dict(WORKLOADS[a.workload])
    T, n, m = cfg["T"], cfg["n"], cfg["m"]
    B = cfg["B"] if cfg["scaling"] == "weak" else cfg["B"] // max(1, a.gpus)      # problems per GPU
    bps = bytes_per_solve(T, n, m)
    base = {"metric": "LQR solves/sec", "unit": "solves/s", "n_gpus": a.gpus, "steps": a.steps,
            "warmup": a.warmup, "higher_is_better": True, "scaling": cfg["scaling"], "vs_baseline": None,
            "dtype": "f32", "data": "synthetic",
            "config": {"workload": cfg["name"], "n_batch_per_gpu": B, "T": T, "n_state": n, "n_ctrl": m,
                       "parallelism": f"batch-shard x{a.gpus} (no collective on the solve path)"}}

    if a.impl == "reference":
        if rank != 0:
            return
        cfg_ref = dict(cfg, B=B)
        val, ms, cores, kind, done, sample = cpu_arm(cfg_ref, max(1, min(a.steps, 40)), max(1, min(a.warmup, 2)))
        base.update({"impl": "reference", "value": val, "ms_per_step": ms, "steps": done,
                     "cpu_baseline": {"value": val, "unit": "solves/s", "cores": cores, "kind": kind, "sample": sample},
                     "e2e": {"value": val, "unit": "solves/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                     "gpu_launches": 0})
        print(json.dumps(base))
        return

    if not torch.cuda.is_available():
        raise SystemExit("bench.py needs a CUDA device (there is no CPU fallback); use --impl reference for the CPU arm")
    import torch.distributed as dist
    torch.cuda.set_device(local)
    dev = torch.device("cuda", local)
    if world > 1:
        dist.init_process_group("nccl", device_id=dev)

    from mpc.pytorch_b200 import LQRStep, QuadCost, LinDx, _lib
    set_bytes = bps * B
    n_sets = max(2, min(4, int(300e6 // set_bytes) + 1))          # rotate over > 126 MB of inputs (L2)
    sets = [gen_inputs(1000 * 3 + rank * 17 + s, B, T, n, m, dev) for s in range(n_sets)]
    steppers = [RawStepper(s, B, T, n, m) for s in sets]
    stream = torch.cuda.current_stream(dev)
    sh = ctypes.c_void_p(stream.cuda_stream)

    def barrier():
        torch.cuda.synchronize(dev)
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize(dev)

    sampler = ClockSampler(local)
    if rank == 0:
        sampler.start()
    # pre-heat (untimed, before the W warm-up steps): ~0.7 s of the same launches so that the
    # nvidia-smi samples are taken with the SMs at their loaded clocks
    preheat = float(os.environ.get("BENCH_PREHEAT_S", "0.7"))   # set 0 under ncu (every launch is replayed)
    t_end = time.perf_counter() + preheat
    i = 0
    while time.perf_counter() < t_end:
        for _ in range(20):
            steppers[i % n_sets](sh)
            i += 1
        torch.cuda.synchronize(dev)
    for w in range(a.warmup):
        steppers[w % n_sets](sh)
    barrier()
    l0 = _lib.launch_count()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record(stream)
    for k in range(a.steps):
        steppers[k % n_sets](sh)
    e1.record(stream)
    barrier()
    launches = _lib.launch_count() - l0
    ms = e0.elapsed_time(e1)
    if world > 1:
        tms = torch.tensor([ms], device=dev)
        dist.all_reduce(tms, op=dist.ReduceOp.MAX)
        ms = float(tms.item())
    clocks = sampler.stop() if rank == 0 else None
    if a.dump_outputs:
        dump_outputs(steppers[(a.steps - 1) % n_sets].out, B, a.dump_outputs)

    # ---------------- e2e: public API, host buffers, copies inside the timed region
    # Two streams: the copy-in stream feeds double-buffered device inputs while the run stream solves the
    # previous step and copies its results out (H2D and D2H use different DMA engines).  Every step still
    # moves all of its inputs host->device and its results device->host inside the timed region.
    from mpc.pytorch_b200.parallel import numa_local
    with numa_local(dev) as numa:       # staging buffers on the GPU's own socket (first touch while bound there)
        host = [{k: v.cpu().pin_memory() for k, v in s.items()} for s in sets[:2]]
        h_outs = [[torch.empty(T, B, n).pin_memory(), torch.empty(T, B, m).pin_memory(), torch.empty(B).pin_memory()]
                  for _ in range(2)]
    dbufs = [{k: torch.empty_like(v) for k, v in sets[0].items()} for _ in range(2)]
    h2d = sum(v.numel() * v.element_size() for v in host[0].values())
    d2h = sum(v.numel() * v.element_size() for v in h_outs[0])
    s_in, s_run = torch.cuda.Stream(dev), torch.cuda.Stream(dev)
    ev_in = [torch.cuda.Event() for _ in range(2)]
    ev_free = [torch.cuda.Event() for _ in range(2)]

    # LTI variant: the workload's dynamics ARE time invariant (F was materialised with .repeat); declared as such,
    # only one [B,n,n+m] slice crosses PCIe and the kernel reads it through a stride-0 time axis
    with numa_local(dev):
        host_F0 = [h["F"][:1].clone().pin_memory() for h in host]
    dF0 = [torch.empty_like(sets[0]["F"][:1]) for _ in range(2)]

    def e2e_step(k, lti=False):
        i = k % 2
        dbuf, h_out = dbufs[i], h_outs[i]
        with torch.cuda.stream(s_in):
            s_in.wait_event(ev_free[i])                       # the solve that last read dbufs[i] is done
            for key, v in host[i].items():
                if lti and key == "F":
                    dF0[i].copy_(host_F0[i], non_blocking=True)
                else:
                    dbuf[key].copy_(v, non_blocking=True)
            ev_in[i].record(s_in)
        with torch.cuda.stream(s_run):
            s_run.wait_event(ev_in[i])
            Fdev = dF0[i].expand(T - 1, B, n, n + m) if lti else dbuf["F"]
            step = LQRStep(n, m, T, true_cost=QuadCost(dbuf["C"], dbuf["c"]),
                           true_dynamics=LinDx(Fdev, dbuf["f"]),
                           current_x=dbuf["cur_x"], current_u=dbuf["cur_u"])
            nx, nu, _, costs, _, _ = step(dbuf["x_init"], dbuf["C"], dbuf["c"], Fdev, dbuf["f"])
            ev_free[i].record(s_run)
            h_out[0].copy_(nx, non_blocking=True)
            h_out[1].copy_(nu, non_blocking=True)
            h_out[2].copy_(costs, non_blocking=True)

    e2e_steps = min(a.steps, 50 if a.workload == "config3" else 6)     # bounded: a config-5 step moves up to 5 GB over PCIe
    with torch.no_grad(), numa_local(dev):             # the submitting thread runs next to the GPU as well
        for k in range(3):
            e2e_step(k)
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            e2e_step(k)
        torch.cuda.synchronize(dev)
        e2e_s = time.perf_counter() - t0
        for k in range(3):
            e2e_step(k, lti=True)
        barrier()
        t0 = time.perf_counter()
        for k in range(e2e_steps):
            e2e_step(k, lti=True)
        torch.cuda.synchronize(dev)
        e2e_lti_s = time.perf_counter() - t0
    # what the e2e number is bound by: the host->device copy rate of this box, measured with one large pinned copy
    with numa_local(dev):
        hb = torch.zeros(64 << 20, dtype=torch.float32).pin_memory()
    db = torch.empty(64 << 20, dtype=torch.float32, device=dev)
    pcie = 0.0
    for _ in range(3):
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        db.copy_(hb, non_blocking=True)
        e1.record()
        torch.cuda.synchronize(dev)
        pcie = max(pcie, hb.numel() * 4 / (e0.elapsed_time(e1) * 1e-3) / 1e9)
    del hb, db
    if world > 1:
        te = torch.tensor([e2e_s, e2e_lti_s], device=dev)
        dist.all_reduce(te, op=dist.ReduceOp.MAX)
        e2e_s, e2e_lti_s = (float(v) for v in te.tolist())
        dist.barrier()

    if rank != 0:
        if world > 1:
            dist.destroy_process_group()
        return

    peaks_path = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(peaks_path):
        peak, peak_src = float(json.load(open(peaks_path))["hbm_gbs"]), "measured (MEASURED_PEAKS.json hbm_gbs)"
    else:
        peak, peak_src = 6650.0, "fallback (B200_PROFILING.md)"
    achieved = bps * B * a.steps / (ms * 1e-3) / 1e9          # GB/s per GPU (max-over-ranks time)
    traffic = None
    tpath = os.path.join(ROOT, "profiles", "traffic.json")
    if os.path.exists(tpath) and a.workload == "config3":
        traffic = json.load(open(tpath)).get("lqr_step_f32_8_2_dram_bytes_per_launch")
    out = dict(base)
    out.update({
        "value": B * world * a.steps / (ms * 1e-3), "ms_per_step": ms / a.steps,
        "gpu_launches": int(launches), "clocks": clocks,
        "e2e": {"value": B * world * e2e_steps / e2e_s, "unit": "solves/s",
                "h2d_bytes_per_step": int(h2d), "d2h_bytes_per_step": int(d2h), "steps": e2e_steps,
                "h2d_gbs_achieved": round(h2d * e2e_steps / e2e_s / 1e9, 2), "h2d_gbs_measured_peak": round(pcie, 2),
                "bound": "PCIe host->device copy of the step's inputs (single 256 MB pinned copy measured on this box)",
                "numa_local_cpus": len(numa.cpus) if numa.cpus else None,
                "api": "mpc.pytorch_b200.LQRStep(...)(x_init,C,c,F,f), pinned host buffers, copy-in / run streams"},
        "e2e_lti": {"value": B * world * e2e_steps / e2e_lti_s, "unit": "solves/s",
                    "h2d_bytes_per_step": int(h2d - host[0]["F"].numel() * 4 + host_F0[0].numel() * 4),
                    "d2h_bytes_per_step": int(d2h),
                    "note": "same workload with F declared time invariant (stride-0 expand): one slice crosses PCIe"},
        "roofline": {"bound": "hbm", "achieved": achieved, "peak": peak, "unit": "GB/s",
                     "frac": achieved / peak, "traffic": traffic,
                     "traffic_source": "profiles/traffic.json (dram__bytes of one ncu --set full capture, not re-measured in this run)",
                     "peak_source": peak_src, "kernel": f"lqr_step<float,{n},{m}>",
                     "algorithmic_bytes_per_launch": bps * B, "bytes_per_solve": bps},
        "timing": {"l2_policy": f"rotating {n_sets} input sets ({n_sets * bps * B / 1e6:.0f} MB > 126 MB L2)",
                   "preheat_s": preheat, "value_is": f"one timed window of {a.steps} launches, max over ranks"},
    })
    if a.workload == "config5":
        fl = flops_per_solve(T, n, m)
        out["roofline"]["fp32_fma_frac"] = fl * B * a.steps / (ms * 1e-3) / 1e12 / FP32_FMA_PEAK_TFLOPS
        out["roofline"]["fp32_fma_peak_tflops"] = round(FP32_FMA_PEAK_TFLOPS, 1)
        out["roofline"]["flops_per_solve"] = fl
    if world == 1:
        del sets, steppers, host, dbufs
        torch.cuda.empty_cache()
        if not a.no_extra:
            try:
                out["extra"] = extras(dev, stream, sh, peak)
            except Exception as exc:                    # secondary figures must never lose the headline line
                out["extra"] = {"error": repr(exc)}
        cfg_ref = dict(cfg, B=B)
        val, _, cores, kind, _, sample = cpu_arm(cfg_ref, 40, 2, budget_s=12.0)
        out["cpu_baseline"] = {"value": val, "unit": "solves/s", "cores": cores, "kind": kind, "sample": sample}
        if kind == "reference":                         # also the (much faster) vectorised port, for context
            pv, _, pc, _, _, ps = cpu_arm(cfg_ref, 40, 2, budget_s=8.0, prefer_reference=False)
            out["cpu_baseline_port"] = {"value": pv, "unit": "solves/s", "cores": pc, "kind": "port", "sample": ps}
    print(json.dumps(out))
    if world > 1:
        dist.destroy_process_group()


if __name__ == "__main__":
    main()
