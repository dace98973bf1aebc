"""Float64 references for the dense tensor-core path, shared by tests/test_gpu_dense_products.py, and the worker that
test runs in subprocesses under each shared-memory plan of k_gemm_f16x3 (BJX_GEMM_VARIANT) and with programmatic
dependent launch switched off (BJX_GEMM_PDL=0).
usage: dense_products_worker.py out.npz
The worker runs a fixed suite of products and fused trajectories and saves every output plus its worst row-relative
error against float64, so that the test can compare the plans bit for bit and each of them with float64."""
import sys

import numpy as np
import torch

F = np.float32
F64 = torch.float64
WINDOW_LO, WINDOW_HI = 2.0 ** -3, 2.0 ** 15.5   # bjx_gemm.h: the fused epilogue's split is exact for lifted maxima in here


def n_tiles(C, D):
    """Accumulator tiles of one product: 256 rows (a CTA pair) x 256 columns."""
    return -(-C // 256) * -(-D // 256)


def spd(D, seed, lo=-0.5, hi=0.5):
    """(cov, prec) float32, Sigma = Q diag(logspace(lo, hi)) Q^T."""
    from oracle import targets as otargets
    return otargets.correlated_gaussian(D, seed=seed, lo=lo, hi=hi)


def row_err(a, ref):
    """Per row: max |a - ref| / max |ref| (= the smallest rtol with |a - b| <= rtol * max(|b|, rowmax_b) elementwise).
    Rows of `a` with a non-finite entry get inf."""
    a = torch.as_tensor(a).to(ref.device, F64)
    ref = ref.to(F64)
    if ref.ndim == 1:
        a, ref = a[:, None], ref[:, None]
    e = (a - ref).abs().amax(1) / ref.abs().amax(1).clamp_min(1e-300)
    e[~torch.isfinite(a).all(1)] = float("inf")
    return e


def plane_lift(stale):
    """bjx_gemm.h plane_lift in float64: 2^(6 - floor(log2 m)), 1 for m == 0 or non-finite."""
    s = torch.clamp(6 - torch.floor(torch.log2(stale.clamp_min(1e-300))), -126, 126)
    return torch.where((stale > 0) & (stale <= 3.0e38), torch.exp2(s), torch.ones_like(stale))


def out_of_window(new_max, stale_max):
    """Rows whose fused-epilogue split would leave the exact window: what k_planes_fixup must redo."""
    t = new_max * plane_lift(stale_max)
    return (new_max > 0) & ~((t >= WINDOW_LO) & (t < WINDOW_HI))


def lin(x, m):
    """x M^T for a symmetric [D, D] matrix, or x * m for a diagonal one."""
    return x @ m if m.ndim == 2 else x * m


def leapfrog64(q, p, g, eps, imm, prec=None, inv_var=None, mean=None, n=1):
    """n velocity-Verlet steps (integrators.py:104-150) in float64 on the device.  eps scalar or [C].  Target: dense
    Gaussian (prec) or diagonal Gaussian (inv_var, mean).  Returns q, p, g, logp and, per row, the number of fused
    productions (dense metric and dense target only) whose row maximum leaves the window of the previous lift."""
    q, p, g = (t.to(F64).clone() for t in (q, p, g))
    e = torch.as_tensor(eps, dtype=F64, device=q.device)
    e = e[:, None] if e.ndim == 1 else e
    imm = imm.to(F64)

    def grad(x):
        if prec is not None:
            gg = -(x @ prec.to(F64))
            return gg, 0.5 * (x * gg).sum(1)
        d = x - (mean.to(F64) if mean is not None else 0.0)
        gg = -d * inv_var.to(F64)
        return gg, 0.5 * (d * gg).sum(1)

    fused = imm.ndim == 2 and prec is not None
    flagged = torch.zeros(q.shape[0], dtype=torch.int64, device=q.device)
    p = p + 0.5 * e * g
    qm, pm = q.abs().amax(1), p.abs().amax(1)
    logp = None
    for s in range(n):
        q = q + e * lin(p, imm)
        if fused:
            m = q.abs().amax(1)
            flagged += out_of_window(m, qm)
            qm = m
        g, logp = grad(q)
        if s + 1 < n:
            p = p + 0.5 * e * g
            p = p + 0.5 * e * g
            if fused:
                m = p.abs().amax(1)
                flagged += out_of_window(m, pm)
                pm = m
        else:
            p = p + 0.5 * e * g
    return q, p, g, logp, flagged


def dense_gaussian_chains(C, D, seed, dev, scale=1.0):
    """q, p ~ N(0, 1) float32 on the device (torch generator: fast at any size)."""
    gen = torch.Generator(device=dev).manual_seed(seed)
    q = scale * torch.randn(C, D, device=dev, generator=gen)
    p = torch.randn(C, D, device=dev, generator=gen)
    return q, p


def plan_suite(dev="cuda:0"):
    """Products whose bits depend on the plan: fused leapfrogs at one and two column tiles (ragged last tile) with
    several tiles per CTA pair, and the plain products at D = 1024.  Returns {name: array} and {name: error}."""
    from blackjax_b200 import _engine, targets as T
    sms = torch.cuda.get_device_properties(dev).multi_processor_count
    outs, errs = {}, {}
    for D, C, n in ((132, 57000, 3), (260, 28600, 4)):
        assert n_tiles(C, D) >= 3 * (sms // 2), (D, C, n_tiles(C, D), sms)
        cov, prec = spd(D, seed=D)
        tc, pc = torch.from_numpy(cov).to(dev), torch.from_numpy(prec).to(dev)
        eng = _engine.Engine(dev, C, D, T.DenseGaussian(prec))
        eng.set_metric(tc)
        q, p = dense_gaussian_chains(C, D, 100 + D, dev)
        g = (-(q.to(F64) @ pc.to(F64))).float()
        eps = 0.05 + 0.25 * torch.rand(C, device=dev, generator=torch.Generator(device=dev).manual_seed(D))
        q64, p64, g64, l64, _ = leapfrog64(q, p, g, eps, tc, prec=pc, n=n)
        logp = torch.zeros(C, device=dev)
        eng.leapfrog_(q, p, logp, g, eps, n)
        torch.cuda.synchronize()
        for k, a, r in (("q", q, q64), ("p", p, p64), ("g", g, g64)):
            outs[f"lf{D}_{k}"] = a.cpu().numpy()
            errs[f"lf{D}_{k}"] = float(row_err(a, r).max())
        outs[f"lf{D}_logp"] = logp.cpu().numpy()
        eng.close()
    D, C = 1024, 600
    cov, prec = spd(D, seed=1)
    tc, pc = torch.from_numpy(cov).to(dev), torch.from_numpy(prec).to(dev)
    eng = _engine.Engine(dev, C, D, T.DenseGaussian(prec))
    eng.set_metric(tc)
    x, _ = dense_gaussian_chains(C, D, 7, dev)
    x *= torch.pow(10.0, torch.linspace(-6, 6, C, device=dev))[:, None]
    v = eng.velocity(x)
    logp, g = eng.init_state(x)
    torch.cuda.synchronize()
    outs["v1024"], errs["v1024"] = v.cpu().numpy(), float(row_err(v, x.to(F64) @ tc.to(F64)).max())
    outs["g1024"], errs["g1024"] = g.cpu().numpy(), float(row_err(g, -(x.to(F64) @ pc.to(F64))).max())
    eng.close()
    return outs, errs


if __name__ == "__main__":
    o, e = plan_suite()
    np.savez(sys.argv[1], **o, **{"err_" + k: np.float64(v) for k, v in e.items()})
