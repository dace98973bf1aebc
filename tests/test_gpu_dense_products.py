"""The dense tensor-core path (bjx::k_gemm_f16x3 in csrc/bjx_gemm.cu, the row kernels and k_planes_fixup in
csrc/bjx_dense.cu) against float64, row by row, where the kernel's schedule and epilogue branch:

* several accumulator tiles per CTA pair (the persistent grid has about SMs / 2 pairs; every case named "multi" asserts
  at least 3 x SMs / 2 tiles), which is where the double-buffered accumulator, the Cin ring phases and the per-tile row
  factors change between tiles;
* chain counts whose last 256-row tile leaves the second CTA of the pair partly live (C % 256 in [129, 255]);
* ragged last column tiles (D % 256 != 0) with one to four column tiles, and K % 32 != 0 over several K blocks;
* the fused epilogue's operand planes, whose lift comes from the previous production's row maximum, and k_planes_fixup,
  which re-splits rows that left the exact window (origin starts, divergent trajectories, mixed batches);
* the alternative shared-memory plans (BJX_GEMM_VARIANT) and the launch without programmatic dependent launch.

Every comparison is per row against that row's own maximum: |a - b| <= rtol * max(|b|, rowmax_b).  Row scales span
twelve decades in some cases, so a row with a wrong lift or a wrong factor cannot hide behind the array maximum.
The references are float64 on the device (cuBLAS DGEMM) from the same float32 inputs."""
import os
import subprocess
import sys

import numpy as np
import pytest
import torch

import blackjax_b200 as bj
from blackjax_b200 import _engine, targets as T
from oracle import hmc as ohmc
from oracle import prng as oprng
from oracle import targets as otargets

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, os.path.join(ROOT, "tests", "helpers"))
import dense_products_worker as W  # noqa: E402  (float64 references shared with the plan worker)

pytestmark = pytest.mark.gpu
F = np.float32
F64 = torch.float64
DEV = "cuda:0"

# The stated contract of one product: 1e-5 of the output row's maximum (DESIGN.md section 3).
PRODUCT_RTOL = 1e-5


def traj_rtol(n):
    """Tolerance of an n-step fused trajectory.  Its 2n products each add at most PRODUCT_RTOL of their row maximum;
    with the well-conditioned matrices used here (eigenvalues within e^+-0.5, eps <= 0.3) one velocity-Verlet step
    is close to norm-preserving, so those errors add without amplification.  The bound 2n x 1e-5 is doubled for the
    float32 axpys and kicks around the products.  A row with the wrong lift or factor is off by >= 1e-3."""
    return 4 * n * PRODUCT_RTOL + PRODUCT_RTOL


def sms():
    return torch.cuda.get_device_properties(DEV).multi_processor_count


def assert_multi(C, D):
    t = W.n_tiles(C, D)
    assert t >= 3 * (sms() // 2), f"{C} x {D} is {t} tiles: not several per CTA pair on {sms()} SMs"


def check(name, a, ref, rtol):
    e = W.row_err(a, ref)
    worst = float(e.max())
    print(f"  {name}: worst row-relative error {worst:.2e} (rtol {rtol:.1e})")
    assert worst <= rtol, f"{name}: rows {torch.nonzero(e > rtol).flatten()[:8].tolist()} off by up to {worst:.2e}"
    return worst


def tk(keys_np):
    return torch.from_numpy(np.ascontiguousarray(keys_np).view(np.int32)).to(DEV).view(torch.uint32)


def tf(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=F)).to(DEV)


def row_scales(C, seed):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return torch.pow(10.0, -6 + 12 * torch.rand(C, 1, device=DEV, generator=g))


def per_chain_eps(C, seed, lo=0.05, hi=0.3):
    g = torch.Generator(device=DEV).manual_seed(seed)
    return lo + (hi - lo) * torch.rand(C, device=DEV, generator=g)


# One multi-tile chain count per D (C % 256 in [129, 255] where the tile count allows it): 3 x 74 pairs on a B200.
MULTI = {132: 57000, 260: 28600, 264: 28600, 516: 19100, 772: 14300, 1020: 14300, 1024: 16545}
DIMS = (132, 260, 264, 516, 772, 1020, 1024)
COUNTS = (1, 127, 128, 129, 255, 257, 4097)


_MATS = {}


def mats(D):
    if D not in _MATS:
        cov, prec = W.spd(D, seed=D)
        L = np.linalg.cholesky(cov.astype(np.float64))
        msqrt = np.linalg.solve(L.T, np.eye(D)).astype(F)          # L^-T (metrics.py:712-715), float32 like the device
        _MATS[D] = tuple(torch.from_numpy(m).to(DEV) for m in (cov, prec, msqrt))
    return _MATS[D]


def device_normals(C, D, keys, prec):
    """normal(key_c, (D,)) as the dense path draws it (k_dense_normal): a unit diagonal metric makes p = z exactly."""
    eng = _engine.Engine(DEV, C, D, T.DenseGaussian(prec.cpu().numpy()))
    eng.set_metric(torch.ones(D, device=DEV))
    z = eng.sample_momentum(keys)
    eng.close()
    return z


# ---------------------------------------------------------------------------------------------------------
# every building block on the grid of dimensions x chain counts
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", DIMS)
@pytest.mark.parametrize("C", COUNTS + ("multi",))
def test_dense_metric_dense_target_products(D, C):
    """velocity (exact split + plain product), init_state (alpha = -1), sample_momentum (L^-T z) and the fused
    leapfrog (lincomb + double kick + planes) for n = 1, 2, 4, 7 (n >= 4 wraps the three-slot row-maximum ring), with a
    scalar and a per-chain step size."""
    if C == "multi":
        C = MULTI[D]
        assert_multi(C, D)
        assert 129 <= C % 256 <= 255                     # the second CTA of the last row tile is partly live
    assert D == 1024 or (D % 256 != 0 and D % 32 != 0)   # a ragged last column tile and a ragged last K block
    cov, prec, msqrt = mats(D)
    eng = _engine.Engine(DEV, C, D, T.DenseGaussian(prec.cpu().numpy()))
    eng.set_metric(cov)
    print(f"\nD={D} C={C} tiles={W.n_tiles(C, D)} C%256={C % 256} D%256={D % 256}")
    x, p0 = W.dense_gaussian_chains(C, D, seed=C + D, dev=DEV)
    xs = x * row_scales(C, seed=C)
    check("velocity (row scales 1e-6..1e6)", eng.velocity(xs), xs.to(F64) @ cov.to(F64), PRODUCT_RTOL)
    logp, g = eng.init_state(xs)
    g64 = -(xs.to(F64) @ prec.to(F64))
    check("init_state grad", g, g64, PRODUCT_RTOL)
    terms = 0.5 * (xs.to(F64) * g64).abs().sum(1)
    lerr = float(((logp.to(F64) - 0.5 * (xs.to(F64) * g64).sum(1)).abs() / terms.clamp_min(1e-300)).max())
    print(f"  init_state logp: worst error / sum |terms| {lerr:.2e}")
    assert lerr <= 2e-5
    keys = oprng.split(oprng.key(C + D), C)
    p = eng.sample_momentum(tk(keys))
    if C <= 257:
        z = torch.from_numpy(oprng.normal(keys, (D,))).to(DEV)        # the reference's normals (device: within ~1 ulp)
    else:
        z = device_normals(C, D, tk(keys), prec)
    check("sample_momentum L^-T z", p, z.to(F64) @ msqrt.to(F64).T, PRODUCT_RTOL)
    eps_pc = per_chain_eps(C, seed=D)
    for n, eps in ((1, 0.2), (2, eps_pc), (4, 0.3), (7, eps_pc)):
        q, pp = x.clone(), p0.clone()
        gg = (-(q.to(F64) @ prec.to(F64))).float()
        lp = torch.zeros(C, device=DEV)
        q64, p64, g64, l64, _ = W.leapfrog64(q, pp, gg, eps, cov, prec=prec, n=n)
        eng.leapfrog_(q, pp, lp, gg, eps, n)
        tag = "per-chain eps" if isinstance(eps, torch.Tensor) else f"eps {eps}"
        for name, a, r in (("q", q, q64), ("p", pp, p64), ("g", gg, g64)):
            check(f"leapfrog n={n} ({tag}) {name}", a, r, traj_rtol(n))
    eng.close()


@pytest.mark.parametrize("D", DIMS)
@pytest.mark.parametrize("C", (129, 255, "multi"))
@pytest.mark.parametrize("metric, target", [("dense", "diag"), ("diag", "dense")])
def test_mixed_metric_target_leapfrog(D, C, metric, target):
    """Dense metric with a diagonal target (the q-update product with Cin, no planes) and a diagonal metric with a dense
    target (the gradient product alone), n = 3, per-chain step sizes."""
    if C == "multi":
        C = MULTI[D]
        assert_multi(C, D)
    cov, prec, _ = mats(D)
    rs = np.random.default_rng(D)
    if target == "dense":
        tgt, tkw = T.DenseGaussian(prec.cpu().numpy()), dict(prec=prec)
    else:
        s = np.exp(rs.uniform(-0.5, 0.5, D))
        mean = rs.standard_normal(D).astype(F)
        tgt = T.DiagGaussian(s, mean=mean)
        tkw = dict(inv_var=torch.from_numpy(1.0 / s ** 2).to(DEV), mean=tf(mean))
    imm = cov if metric == "dense" else tf(np.exp(rs.uniform(-0.5, 0.5, D)))
    eng = _engine.Engine(DEV, C, D, tgt)
    eng.set_metric(imm)
    q, p = W.dense_gaussian_chains(C, D, seed=3 * D + C, dev=DEV)
    logp, g = eng.init_state(q)
    if target == "dense":
        g = (-(q.to(F64) @ prec.to(F64))).float()
    eps = per_chain_eps(C, seed=C)
    q64, p64, g64, _, _ = W.leapfrog64(q, p, g, eps, imm, n=3, **tkw)
    eng.leapfrog_(q, p, logp, g, eps, 3)
    print(f"\n{metric} metric / {target} target D={D} C={C} tiles={W.n_tiles(C, D)}")
    for name, a, r in (("q", q, q64), ("p", p, p64), ("g", g, g64)):
        check(f"leapfrog n=3 {name}", a, r, traj_rtol(3))
    eng.close()


def test_fused_leapfrog_negative_dominated_rows():
    """Rows whose largest entries are negative, at scales 1e-6 ... 1e6, through the fused leapfrog at one and at
    four column tiles: the epilogue's recorded row maximum (the next production's lift) must be a maximum of |y|."""
    for D, C in ((132, 700), (1024, 700)):
        cov, prec, _ = mats(D)
        eng = _engine.Engine(DEV, C, D, T.DenseGaussian(prec.cpu().numpy()))
        eng.set_metric(cov)
        q, p = W.dense_gaussian_chains(C, D, seed=11, dev=DEV)
        sc = row_scales(C, seed=12)
        q = -(4.0 + q.abs()) * sc
        p = -(4.0 + p.abs()) * sc
        g = (-(q.to(F64) @ prec.to(F64))).float()
        lp = torch.zeros(C, device=DEV)
        q64, p64, g64, _, _ = W.leapfrog64(q, p, g, 0.01, cov, prec=prec, n=4)
        assert (q64.amax(1) < 0.5 * q64.abs().amax(1)).all()       # still dominated by negative entries
        eng.leapfrog_(q, p, lp, g, 0.01, 4)
        print(f"\nnegative-dominated rows D={D} C={C}")
        for name, a, r in (("q", q, q64), ("p", p, p64), ("g", g, g64)):
            check(f"leapfrog n=4 {name}", a, r, traj_rtol(4))
        eng.close()


# ---------------------------------------------------------------------------------------------------------
# bit-exact invariances: a row's arithmetic depends only on that row and the matrix
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", (260, 1024))
def test_batch_embedding_bit_exact(D):
    """64 chains alone (one tile) and the same 64 chains at row offsets 0, 1, 129 and at the end of a multi-tile batch
    give the same bits in every building block and in a fused leapfrog of 4 steps."""
    cov, prec, _ = mats(D)
    tgt = T.DenseGaussian(prec.cpu().numpy())
    Cs, Cb = 64, MULTI[D]
    assert_multi(Cb, D)
    xs, ps = W.dense_gaussian_chains(Cs, D, seed=1, dev=DEV)
    xs = xs * row_scales(Cs, seed=2)
    keys_s = oprng.split(oprng.key(3), Cs)
    eps_s = per_chain_eps(Cs, seed=4)

    def run(eng, x, p, keys, eps):
        v = eng.velocity(x)
        logp, g = eng.init_state(x)
        m = eng.sample_momentum(tk(keys))
        q, pp, lp, gg = x.clone(), p.clone(), logp.clone(), g.clone()
        eng.leapfrog_(q, pp, lp, gg, eps, 4)
        return dict(v=v, logp=logp, g=g, m=m, q=q, p=pp, lp=lp, gg=gg)

    small = _engine.Engine(DEV, Cs, D, tgt)
    small.set_metric(cov)
    ref = run(small, xs, ps, keys_s, eps_s)
    small.close()
    big = _engine.Engine(DEV, Cb, D, tgt)
    big.set_metric(cov)
    xb, pb = W.dense_gaussian_chains(Cb, D, seed=5, dev=DEV)
    keys_b = oprng.split(oprng.key(6), Cb)
    eps_b = per_chain_eps(Cb, seed=7)
    for off in (0, 1, 129, Cb - Cs):
        x, p, k, e = xb.clone(), pb.clone(), keys_b.copy(), eps_b.clone()
        sl = slice(off, off + Cs)
        x[sl], p[sl], k[sl], e[sl] = xs, ps, keys_s, eps_s
        out = run(big, x, p, k, e)
        for name, r in ref.items():
            assert torch.equal(out[name][sl], r), f"offset {off}: {name} differs from the 64 chains alone"
    big.close()


def test_row_poisoning_bit_exact():
    """NaN in one chain's q and inf in another's p change no other chain's bits (multi-tile batch, fused leapfrog and
    the plain products), and the poisoned chains' outputs are non-finite."""
    D, C = 516, MULTI[516]
    assert_multi(C, D)
    cov, prec, _ = mats(D)
    eng = _engine.Engine(DEV, C, D, T.DenseGaussian(prec.cpu().numpy()))
    eng.set_metric(cov)
    x, p = W.dense_gaussian_chains(C, D, seed=8, dev=DEV)
    bad_q, bad_p = 300, C - 2

    def run(x, p):
        v = eng.velocity(p)
        logp, g = eng.init_state(x)
        q, pp = x.clone(), p.clone()
        eng.leapfrog_(q, pp, logp, g, 0.2, 4)
        return dict(v=v, g=g, q=q, p=pp, logp=logp)

    clean = run(x, p)
    xp, pp = x.clone(), p.clone()
    xp[bad_q, 17] = float("nan")
    pp[bad_p, 0] = float("inf")
    pois = run(xp, pp)
    ok = torch.ones(C, dtype=torch.bool, device=DEV)
    ok[[bad_q, bad_p]] = False
    for name in clean:
        assert torch.equal(pois[name][ok], clean[name][ok]), f"{name}: a poisoned row changed another row"
    for name in ("q", "p", "g"):
        for r in (bad_q, bad_p):
            assert not torch.isfinite(pois[name][r]).all(), (name, r)
    assert not torch.isfinite(pois["v"][bad_p]).all()
    eng.close()


# ---------------------------------------------------------------------------------------------------------
# the plane fix-up: rows whose maximum leaves the window of the previous production's lift
# ---------------------------------------------------------------------------------------------------------
def fixup_case(D, q, p, eps, cov, prec, n):
    C = q.shape[0]
    eng = _engine.Engine(DEV, C, D, T.DenseGaussian(prec.cpu().numpy()))
    eng.set_metric(cov)
    g = (-(q.to(F64) @ prec.to(F64))).float()
    lp = torch.zeros(C, device=DEV)
    q64, p64, g64, _, flagged = W.leapfrog64(q, p, g, eps, cov, prec=prec, n=n)
    eng.leapfrog_(q, p, lp, g, eps, n)
    torch.cuda.synchronize()
    eng.close()
    return (q, p, g), (q64, p64, g64), flagged


def test_fixup_origin_start():
    """Chains started at q = 0: the first q production is lifted by 1 (previous maximum 0) and its rows, of size
    eps |M^-1 p|, leave the window for the small step sizes.  Per-chain eps from 1e-6 to 1 over one step, and from 1e-6
    to 0.1 over four (the ring of row maxima wraps).  The step sizes stop short of the values where the rotation between
    q and p (M^-1 P = I here) brings a whole row of q or p back near zero after n steps: there the row's own maximum is
    not the scale of its rounding."""
    D, C = 260, 4097
    cov, prec, _ = mats(D)
    for n, top in ((1, 0.0), (4, -1.0)):
        _, p = W.dense_gaussian_chains(C, D, seed=20, dev=DEV)
        eps = torch.logspace(-6, top, C, device=DEV)
        q = torch.zeros(C, D, device=DEV)
        (q, p, g), (q64, p64, g64), flagged = fixup_case(D, q, p, eps, cov, prec, n=n)
        print(f"\norigin start n={n}: {int((flagged > 0).sum())} of {C} rows re-split by the fix-up")
        assert (flagged > 0).sum() >= C // 4
        for name, a, r in (("q", q, q64), ("p", p, p64), ("g", g, g64)):
            check(f"origin start n={n} {name}", a, r, traj_rtol(n))


def test_fixup_divergent_trajectory():
    """M^-1 = I against a target with precision eigenvalues up to 1e4 at eps = 0.4: the stiff modes grow by more than
    2^10 per step, so every production leaves the window of the previous lift, and the rows stay finite for the 6 steps
    compared.  Per row against float64: the dynamics is linear, so the relative error stays at the products' level."""
    D, C = 264, 1000
    stiff, _ = W.spd(D, seed=9, lo=0.0, hi=4.0)                       # eigenvalues 1 ... 1e4
    prec = torch.from_numpy(stiff).to(DEV)
    cov = torch.eye(D, device=DEV)
    q, p = W.dense_gaussian_chains(C, D, seed=21, dev=DEV)
    n = 6
    q64a, _, _, _, _ = W.leapfrog64(q, p, (-(q.to(F64) @ prec.to(F64))).float(), 0.4, cov, prec=prec, n=n - 1)
    q64b, _, _, _, _ = W.leapfrog64(q, p, (-(q.to(F64) @ prec.to(F64))).float(), 0.4, cov, prec=prec, n=n)
    growth = float((q64b.abs().amax(1) / q64a.abs().amax(1)).min())
    (q, p, g), (q64, p64, g64), flagged = fixup_case(D, q, p, 0.4, cov, prec, n=n)
    print(f"\ndivergent: growth per step >= {growth:.3g}, rows re-split per trajectory min {int(flagged.min())}, "
          f"max |q| {float(q64.abs().max()):.3g}")
    assert growth > 2.0 ** 10
    assert bool(torch.isfinite(q64).all()) and float(p64.abs().max()) < 1e30
    assert int(flagged.min()) >= n
    for name, a, r in (("q", q, q64), ("p", p, p64), ("g", g, g64)):
        check(f"divergent n={n} {name}", a, r, traj_rtol(n))


@pytest.mark.parametrize("n", (1, 3))
def test_fixup_mixed_batch(n):
    """Fix-up rows (origin starts at a step size of 1e-6) at positions 0, 31, 32, 255, 256 and the last, between stable
    rows: k_planes_fixup's warp-per-32-rows loop must redo exactly those rows and leave the neighbours alone.
    With n = 1 the gradient is taken from the re-split planes themselves (without the fix-up its rows are off by ~1e-2).
    The stable rows must come out bit for bit as in a batch without fix-up rows: a re-split of a neighbour (exact lift
    instead of the epilogue's) would change its product bits."""
    D, C = 516, 1000
    cov, prec, _ = mats(D)
    q0, p0 = W.dense_gaussian_chains(C, D, seed=22, dev=DEV)
    rows = [0, 31, 32, 255, 256, C - 1]
    stable = torch.ones(C, dtype=torch.bool, device=DEV)
    stable[rows] = False
    eps = torch.full((C,), 0.2, device=DEV)
    (qs, ps, gs), _, flagged = fixup_case(D, q0.clone(), p0.clone(), eps, cov, prec, n=n)
    assert int(flagged.sum()) == 0
    q = q0.clone()
    q[rows] = 0.0
    eps[rows] = 1e-6
    (q, p, g), (q64, p64, g64), flagged = fixup_case(D, q, p0.clone(), eps, cov, prec, n=n)
    hit = torch.nonzero(flagged > 0).flatten().tolist()
    print(f"\nmixed batch n={n}: rows re-split {hit}")
    assert hit == rows
    for name, a, r in (("q", q, q64), ("p", p, p64), ("g", g, g64)):
        check(f"mixed batch n={n} {name}", a, r, traj_rtol(n))
    for name, a, b in (("q", q, qs), ("p", p, ps), ("g", g, gs)):
        assert torch.equal(a[stable], b[stable]), f"{name}: a stable row changed next to the fix-up rows"


def test_dense_hmc_divergent_chains_vs_oracle():
    """A dense HMC transition with eps = 30 on a third of the chains (they diverge) and 0.1 on the rest, against the
    float32 oracle: divergence and acceptance flags identical (acceptance up to ties), rejected chains return q_in
    bit for bit, and the stable chains still match."""
    D, C, L = 260, 300, 5
    cov, prec = W.spd(D, seed=13)
    tgt, otgt = T.DenseGaussian(prec), otargets.DenseGaussian(prec)
    rs = np.random.default_rng(14)
    q = (0.5 * rs.standard_normal((C, D))).astype(F)
    eps = np.full(C, 0.1, F)
    eps[::3] = 30.0
    keys = oprng.split(oprng.key(15), C)
    onew, oinfo = ohmc.hmc_kernel(keys, ohmc.init(q, otgt), otgt, eps, ohmc.Metric(cov), L)
    new, info = bj.hmc.build_kernel(full_info=True)(tk(keys), bj.hmc.init(tf(q), tgt), tgt, tf(eps), tf(cov), L)
    torch.cuda.synchronize()
    div, acc = info.is_divergent.cpu().numpy().astype(bool), info.is_accepted.cpu().numpy().astype(bool)
    print(f"\neps=30 chains: {int(div[::3].sum())} of {len(div[::3])} divergent; oracle {int(oinfo.is_divergent[::3].sum())}")
    assert div[::3].all() and np.array_equal(div, oinfo.is_divergent)
    u = oprng.uniform(oprng.split(keys, 2)[:, 1])
    tie = np.abs(u - oinfo.acceptance_rate) < 2e-3
    assert ((acc == oinfo.is_accepted) | tie).all()
    pos = new.position.cpu().numpy()
    assert np.array_equal(pos[~acc], q[~acc])
    stable = (eps < 1) & (acc == oinfo.is_accepted)
    err = np.abs(pos[stable] - onew.position[stable]).max(1) / np.abs(onew.position[stable]).max(1)
    print(f"  stable chains: worst row-relative error vs oracle {err.max():.2e}")
    assert err.max() < 3e-5


# ---------------------------------------------------------------------------------------------------------
# shared-memory plans and programmatic dependent launch
# ---------------------------------------------------------------------------------------------------------
def test_gemm_plans_and_pdl(tmp_path):
    """The worker's product suite (fused leapfrogs at D = 132 and 260, several tiles per pair; plain products at
    D = 1024) under each plan.  PDL on and off are bit-identical; the default plan and variant 2 share BK = 32 and so
    the MMA order, as do variants 1 and 3 with BK = 64; every plan is within tolerance of float64."""
    worker = os.path.join(ROOT, "tests", "helpers", "dense_products_worker.py")
    runs = {"default": {}, "pdl0": {"BJX_GEMM_PDL": "0"}, "v1": {"BJX_GEMM_VARIANT": "1"},
            "v2": {"BJX_GEMM_VARIANT": "2"}, "v3": {"BJX_GEMM_VARIANT": "3"}}
    res = {}
    for name, extra in runs.items():
        out = str(tmp_path / f"{name}.npz")
        env = dict(os.environ, PYTHONPATH=ROOT, **extra)
        env.pop("BJX_GEMM_DEBUG", None)
        if name == "default":
            env.pop("BJX_GEMM_VARIANT", None)
            env.pop("BJX_GEMM_PDL", None)
        subprocess.run([sys.executable, worker, out], check=True, env=env, timeout=600)
        res[name] = dict(np.load(out))
    for name, r in res.items():
        errs = {k[4:]: float(v) for k, v in r.items() if k.startswith("err_")}
        print(f"\nplan {name}: " + "  ".join(f"{k} {v:.2e}" for k, v in errs.items()))
        for k, v in errs.items():
            assert v <= (PRODUCT_RTOL if k.endswith("1024") else traj_rtol(4)), (name, k, v)
    keys = [k for k in res["default"] if not k.startswith("err_")]
    for a, b in (("default", "pdl0"), ("default", "v2"), ("v1", "v3")):
        for k in keys:
            assert np.array_equal(res[a][k], res[b][k]), f"{a} and {b} differ in {k}"


# ---------------------------------------------------------------------------------------------------------
# the dense path's dimension limit
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("D", (1028, 2048, 4096))
def test_dense_beyond_1024_dims_refused(D):
    """The float32 accumulator of the tensor-core products truncates at each of its 3K/16 steps, so the per-product
    error grows linearly in K and passes the 1e-5 contract beyond K = 1024 (DESIGN.md section 3).  Dense targets and
    dense metrics above 1024 dims are refused up front instead of running less accurate than stated."""
    C = 8
    cov = prec = np.eye(D, dtype=F)
    with pytest.raises(bj.BjxError, match="1024"):
        _engine.Engine(DEV, C, D, T.DenseGaussian(prec))
    eng = _engine.Engine(DEV, C, D, T.DiagGaussian(np.ones(D, F)))
    with pytest.raises(bj.BjxError, match="1024"):
        eng.set_metric(tf(cov))
    eng.close()
    if D == 1028:
        q = tf(0.1 * np.random.default_rng(0).standard_normal((C, D)))
        tgt = T.DiagGaussian(np.ones(D, F))
        for algo in (bj.hmc, bj.nuts):
            with pytest.raises(bj.BjxError, match="1024"):
                algo.build_kernel()(bj.random.key(0, DEV), algo.init(q, tgt), tgt, 0.1, tf(cov), 4)
