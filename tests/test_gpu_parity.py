"""GPU parity tests: the CUDA path (through the C ABI, via the blackjax_b200 API) against the CPU
oracle on the same seeded inputs, plus size-independent properties at BASELINE.json's full shapes.

Tolerances (stated per BASELINE.md section 4): PRNG integers and uniform variates bit-exact; one
transition from an identical (state, key) within 1e-5 relative (abs floor 1e-5 x typical scale);
discrete decisions (accept, direction, turning, tree size) identical except where the deciding float
comparison is within float32 rounding of a tie.
"""
import numpy as np
import pytest
import torch

import blackjax_b200 as bj
from blackjax_b200 import _engine, targets as T
from oracle import adaptation as oadapt
from oracle import hmc as ohmc
from oracle import nuts as onuts
from oracle import prng as oprng
from oracle import targets as otargets

pytestmark = pytest.mark.gpu
F = np.float32
DEV = "cuda:0"


def tk(keys_np):
    """numpy uint32 keys -> torch uint32 CUDA tensor."""
    return torch.from_numpy(np.ascontiguousarray(keys_np).view(np.int32)).to(DEV).view(torch.uint32)


def tf(a):
    return torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32)).to(DEV)


def npy(t):
    return t.detach().cpu().numpy()


def close(a, b, rtol=1e-5, scale=None, floor_frac=None):
    """Elementwise: |a - b| <= rtol * max(|b|, floor) for every element.
    * state vectors (no ``scale``): floor = 5 % of max |b|.  Elements above it are held to rtol relative to THEMSELVES,
      smaller ones to rtol * floor (their rounding noise comes from terms of the size of the large elements).
    * reductions (``scale`` given: energies, log-densities, acceptance rates): floor = scale, the magnitude of the terms
      that were summed -- a sum of D terms that cancels to a small value is not accurate relative to that value.
    * floor_frac = 1 without scale (``dclose``): outputs of the tensor-core products, whose error is absolute in the row.
    Non-finite entries must match exactly (inf with inf, NaN with NaN)."""
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    fin = np.isfinite(b)
    assert np.array_equal(np.isnan(a), np.isnan(b)) and np.array_equal(a[~fin & ~np.isnan(b)], b[~fin & ~np.isnan(b)])
    if not fin.any():
        return
    if floor_frac is None:
        floor_frac = 1.0 if scale is not None else 0.05
    s = np.max(np.abs(b[fin])) if scale is None else scale
    floor = floor_frac * max(s, 1e-30)
    err = np.abs(a[fin] - b[fin]) / np.maximum(np.abs(b[fin]), floor)
    assert np.all(err <= rtol), f"worst elementwise error {np.max(err):.3e} > rtol {rtol:.1e} (floor {floor:.3e})"


def dclose(a, b, rtol=1e-5, scale=None):
    """close() relative to the array maximum: for quantities that come out of the dense path's tensor-core products."""
    close(a, b, rtol=rtol, scale=scale, floor_frac=1.0)


# ---------------------------------------------------------------------------------------------------------
# PRNG: bit-exact
# ---------------------------------------------------------------------------------------------------------
def test_prng_bit_exact():
    k0 = bj.random.key(0, DEV)
    assert npy(bj.random.split(k0)).tolist() == [[1797259609, 2579123966], [928981903, 3453687069]]
    keys = oprng.split(oprng.key(123), 257)
    dk = tk(keys)
    assert (npy(bj.random.split(dk, 3)) == oprng.split(keys, 3)).all()
    assert (npy(bj.random.fold_in(dk, 77)) == oprng.fold_in(keys, 77)).all()
    assert (npy(bj.random.bits(dk, (33,))) == oprng.random_bits(keys, (33,))).all()
    assert (npy(bj.random.uniform(dk, (33,))) == oprng.uniform(keys, (33,))).all()
    n_dev = npy(bj.random.normal(dk, (130,)))
    n_ref = oprng.normal(keys, (130,))
    assert np.max(np.abs(n_dev - n_ref)) < 2e-6
    assert float(npy(bj.random.normal(bj.random.key(42, DEV)))) == pytest.approx(-0.028304616, abs=1e-7)


# ---------------------------------------------------------------------------------------------------------
# building blocks
# ---------------------------------------------------------------------------------------------------------
def make_target(kind, D, rs):
    if kind == "std":
        return T.StdNormal(D), otargets.StdNormal(D)
    if kind == "diag":
        s = np.exp(rs.uniform(-1, 1, D))
        mean = rs.standard_normal(D).astype(F)
        return T.DiagGaussian(s, mean=mean, logp_offset=0.25), otargets.DiagGaussian(s, mean=mean, logp_offset=0.25)
    if kind == "funnel":
        return T.Funnel(D), otargets.Funnel(D)
    if kind == "dense":
        A = rs.standard_normal((D, D))
        P = A @ A.T / D + np.eye(D)
        return T.DenseGaussian(P), otargets.DenseGaussian(P)
    if kind == "banana":
        return T.Banana(), otargets.Banana()
    raise ValueError(kind)


SHAPES = [("std", 100), ("diag", 1024), ("diag", 516), ("diag", 7), ("diag", 97), ("funnel", 128),
          ("funnel", 10), ("funnel", 260), ("dense", 6), ("dense", 64), ("banana", 2), ("std", 1)]


@pytest.mark.parametrize("kind, D", SHAPES)
def test_init_state_matches_oracle(kind, D):
    rs = np.random.default_rng(1)
    tgt, otgt = make_target(kind, D, rs)
    C = 37
    q = rs.standard_normal((C, D)).astype(F)
    st = bj.hmc.init(tf(q), tgt)
    lp, g = otgt(q)
    close(npy(st.logdensity), lp, rtol=2e-6, scale=np.max(np.abs(lp)) + 1)
    close(npy(st.logdensity_grad), g, rtol=2e-6)


@pytest.mark.parametrize("D, dense", [(100, False), (1024, False), (7, False), (6, True), (64, True)])
def test_sample_momentum_matches_oracle(D, dense):
    rs = np.random.default_rng(2)
    C = 33
    if dense:
        A = rs.standard_normal((D, D))
        imm = (A @ A.T / D + np.eye(D)).astype(F)
    else:
        imm = np.exp(rs.uniform(-2, 2, D)).astype(F)
    tgt = T.StdNormal(D)
    eng = _engine.Engine(DEV, C, D, tgt)
    eng.set_metric(tf(imm))
    keys = oprng.split(oprng.key(5), C)
    p = npy(eng.sample_momentum(tk(keys)))
    ref = ohmc.Metric(imm).sample_momentum(keys, D)
    close(p, ref, rtol=3e-6)
    # kinetic energy through bjx_energy
    e = npy(eng.energy(tf(ref), tf(np.zeros(C, F))))
    close(e, ohmc.Metric(imm).kinetic_energy(ref), rtol=2e-6)


def test_dense_metric_factorisation_identity():
    # tests/mcmc/test_metrics.py:158-179: p = L^-T z for M^-1 = [[2/3, .5], [.5, 3/4]]
    imm = np.array([[2 / 3, 0.5], [0.5, 3 / 4]], F)
    eng = _engine.Engine(DEV, 1, 2, T.StdNormal(2))
    eng.set_metric(tf(imm))
    p = npy(eng.sample_momentum(tk(oprng.key(0)[None])))
    L = np.linalg.cholesky(imm.astype(np.float64))
    z = oprng.normal(oprng.key(0), (2,)).astype(np.float64)
    close(p[0], np.linalg.solve(L.T, z), rtol=3e-6)
    with pytest.raises(ValueError, match="wrong number of dimensions"):
        eng.set_metric(torch.ones(2, 2, 2, device=DEV))


def test_momentum_identity_diag_quarter():
    # tests/mcmc/test_metrics.py:124-142: M^-1 = [1/4] -> p = 2 * normal(key)
    eng = _engine.Engine(DEV, 1, 1, T.StdNormal(1))
    eng.set_metric(tf(np.array([0.25], F)))
    p = npy(eng.sample_momentum(tk(oprng.key(0)[None])))
    assert abs(p[0, 0] - 2.0 * float(oprng.normal(oprng.key(0)))) < 1e-6


def test_velocity_verlet_mvn_golden():
    # tests/mcmc/test_integrators.py:74-103 golden end state through bjx_leapfrog (dense metric + dense target)
    from test_oracle_kat import COV6, P6_END, P6_INIT, Q6_END, Q6_INIT
    tgt = T.DenseGaussian(np.linalg.inv(COV6))
    eng = _engine.Engine(DEV, 1, 6, tgt)
    eng.set_metric(tf(COV6))
    q = tf(Q6_INIT)
    p = tf(P6_INIT)
    logp, g = eng.init_state(q)
    eng.leapfrog_(q, p, logp, g, 0.005, 16)
    np.testing.assert_allclose(npy(q)[0], Q6_END, atol=3e-6)
    np.testing.assert_allclose(npy(p)[0], P6_END, atol=3e-6)


@pytest.mark.parametrize("kind, D", [("std", 100), ("diag", 1024), ("diag", 97), ("funnel", 128), ("dense", 6)])
def test_leapfrog_matches_oracle(kind, D):
    rs = np.random.default_rng(3)
    tgt, otgt = make_target(kind, D, rs)
    C = 19
    imm = np.exp(rs.uniform(-1, 1, D)).astype(F)
    q = (0.3 * rs.standard_normal((C, D))).astype(F)
    p = rs.standard_normal((C, D)).astype(F)
    eng = _engine.Engine(DEV, C, D, tgt)
    eng.set_metric(tf(imm))
    dq, dp = tf(q), tf(p)
    logp, g = eng.init_state(dq)
    eps = F(0.05)
    eng.leapfrog_(dq, dp, logp, g, float(eps), 7)
    lp0, g0 = otgt(q)
    q1, p1, lp1, g1 = ohmc.static_integration(otgt, ohmc.Metric(imm), q, p, lp0, g0, eps, 7)
    if kind in ("std", "diag"):  # purely elementwise dynamics: bit-identical to the oracle's emulated FMAs
        for a, b in ((npy(dq), q1), (npy(dp), p1), (npy(g), g1)):
            assert (a == b).mean() > 0.999          # (float64 emulation of an FMA double-rounds w.p. ~2^-29)
            close(a, b, rtol=1e-6)
    else:
        close(npy(dq), q1)
        close(npy(dp), p1)
        close(npy(g), g1)
    close(npy(logp), lp1, rtol=3e-6, scale=np.max(np.abs(lp1)) + 1)


# ---------------------------------------------------------------------------------------------------------
# HMC transition (teacher-forced: identical state + key on both sides)
# ---------------------------------------------------------------------------------------------------------
def run_hmc_case(kind, D, C, L, eps, imm_kind="diag", per_chain_eps=False, seed=11):
    rs = np.random.default_rng(seed)
    tgt, otgt = make_target(kind, D, rs)
    if imm_kind == "diag":
        imm = np.exp(rs.uniform(-0.5, 0.5, D)).astype(F)
    elif imm_kind == "ones":
        imm = np.ones(D, F)
    elif imm_kind == "dense":
        A = rs.standard_normal((D, D))
        imm = (A @ A.T / D + np.eye(D)).astype(F)
    else:  # per-chain diagonal
        imm = np.exp(rs.uniform(-0.5, 0.5, (C, D))).astype(F)
    q = (0.5 * rs.standard_normal((C, D))).astype(F)
    keys = oprng.split(oprng.key(seed), C)
    eps_np = (eps * np.exp(rs.uniform(-0.3, 0.3, C))).astype(F) if per_chain_eps else F(eps)
    ometric = oadapt._PerChainDiag(imm) if imm_kind == "per_chain" else ohmc.Metric(imm)
    ostate = ohmc.init(q, otgt)
    onew, oinfo = ohmc.hmc_kernel(keys, ostate, otgt, eps_np, ometric, L)

    kernel = bj.hmc.build_kernel(full_info=True)
    state = bj.hmc.init(tf(q), tgt)
    step = tf(eps_np) if per_chain_eps else float(eps_np)
    new, info = kernel(tk(keys), state, tgt, step, tf(imm), L)
    torch.cuda.synchronize()
    # energies and acceptance probability
    close(npy(info.energy), oinfo.energy, rtol=1e-5, scale=np.max(np.abs(oinfo.energy)) + 1)
    close(npy(info.acceptance_rate), oinfo.acceptance_rate, rtol=1e-4, scale=1.0)
    close(npy(info.momentum), oinfo.momentum, rtol=3e-6)
    close(npy(info.proposal.position), oinfo.proposal[0])
    close(npy(info.proposal.momentum), oinfo.proposal[1])
    # accept decisions: identical except within rounding of a tie
    u = oprng.uniform(oprng.split(keys, 2)[:, 1])
    acc_dev = npy(info.is_accepted)
    tie = np.abs(u - oinfo.acceptance_rate) < 1e-5
    assert ((acc_dev == oinfo.is_accepted) | tie).all()
    assert (npy(info.is_divergent) == oinfo.is_divergent).all()
    same = acc_dev == oinfo.is_accepted
    close(npy(new.position)[same], onew.position[same])
    close(npy(new.logdensity_grad)[same], onew.logdensity_grad[same])
    close(npy(new.logdensity)[same], onew.logdensity[same], rtol=1e-5, scale=np.max(np.abs(onew.logdensity)) + 1)
    return acc_dev.mean()


def test_hmc_config1_iso_gaussian_1024x100():
    # BASELINE config 1: HMC, 100-D isotropic Gaussian, 1024 chains, diag mass, 10 leapfrog steps
    rate = run_hmc_case("std", 100, 1024, 10, 0.2, imm_kind="ones")
    assert 0.5 < rate <= 1.0


@pytest.mark.parametrize("kind, D, C, L, eps, imm_kind, pce", [
    ("diag", 1024, 64, 10, 0.05, "diag", False),
    ("diag", 516, 33, 5, 0.1, "diag", True),
    ("diag", 97, 40, 8, 0.1, "per_chain", True),
    ("diag", 7, 40, 8, 0.2, "diag", False),
    ("funnel", 128, 96, 10, 0.05, "ones", False),
    ("funnel", 10, 50, 20, 0.1, "diag", False),
    ("dense", 6, 30, 10, 0.1, "dense", False),
    ("dense", 64, 20, 5, 0.05, "dense", False),
    ("banana", 2, 64, 12, 0.1, "dense", False),
    ("std", 1, 64, 30, 3.9, "ones", False),     # tests/mcmc/test_sampling.py:1055-1119 HMC settings
    ("std", 100, 64, 10, 30.0, "ones", False),  # wildly unstable step: divergences / NaN energies -> reject
])
def test_hmc_transition_matches_oracle(kind, D, C, L, eps, imm_kind, pce):
    run_hmc_case(kind, D, C, L, eps, imm_kind, pce)


@pytest.mark.parametrize("algo", ["hmc", "nuts", "mhmc"])
def test_shared_step_key_equals_explicit_split(algo):
    # a single key [2] == jax.random.split(key, C_global) per-chain keys; chain_offset selects this process's shard
    tgt = T.Funnel(32)
    C, Cg, off = 96, 256, 100
    q = 0.1 * torch.randn(C, 32, device=DEV)
    imm = torch.ones(32, device=DEV)
    key = bj.random.key(31, DEV)
    explicit = bj.random.split(key, Cg)[off:off + C]
    mod = {"hmc": bj.hmc, "nuts": bj.nuts, "mhmc": bj.mhmc}[algo]
    args = (0.1, imm) if algo == "nuts" else (0.1, imm, 7)
    a, ia = mod.build_kernel()(explicit, mod.init(q.clone(), tgt), tgt, *args)
    b, ib = mod.build_kernel(chain_offset=off)(key, mod.init(q.clone(), tgt), tgt, *args)
    assert torch.equal(a.position, b.position) and torch.equal(ia.acceptance_rate, ib.acceptance_rate)
    c, _ = mod.build_kernel(chain_offset=0)(key, mod.init(q.clone(), tgt), tgt, *args)
    assert not torch.equal(a.position, c.position)


@pytest.mark.parametrize("multinomial", [False, True])
def test_native_sampler_equals_python_loop(multinomial):
    # bjx_hmc_sample == run_inference_algorithm's loop (util.py:200-211): same keys, same draws, history and all
    tgt = T.DiagGaussian(np.logspace(-0.3, 0.3, 40))
    C, T_ = 300, 12
    imm = torch.ones(40, device=DEV)
    st0 = bj.hmc.init(torch.randn(C, 40, device=DEV), tgt)
    key = bj.random.key(77, DEV)
    alg = (bj.mhmc if multinomial else bj.hmc)(tgt, 0.2, imm, 9)
    st, hist = bj.run_inference_algorithm(key, alg, T_, initial_state=st0, transform=lambda s, i: (s.position, i.acceptance_rate))
    fin, positions, acc = bj.sample_hmc_native(key, st0, tgt, 0.2, imm, 9, T_, multinomial=multinomial)
    assert torch.equal(fin.position, st.position) and torch.equal(fin.logdensity_grad, st.logdensity_grad)
    assert torch.equal(positions[-1], st.position) and torch.equal(positions[3], hist[3][0])
    assert torch.equal(acc[5], hist[5][1])
    fin2, pos2, _ = bj.sample_hmc_native(key, st0, tgt, 0.2, imm, 9, T_, multinomial=multinomial, thin=4)
    assert pos2.shape[0] == 3 and torch.equal(pos2[0], positions[3]) and torch.equal(pos2[2], positions[11])
    assert torch.equal(st0.position, st0.position.clone())      # input state untouched (native path works on a copy)


def test_potential_scale_reduction_on_device_history():
    from oracle import diagnostics as odiag
    tgt = T.DiagGaussian(np.logspace(-0.3, 0.3, 24))
    C, T_ = 64, 200
    imm = torch.ones(24, device=DEV)
    st0 = bj.hmc.init(torch.randn(C, 24, device=DEV), tgt)
    _, hist, _ = bj.sample_hmc_native(bj.random.key(5, DEV), st0, tgt, 0.3, imm, 8, T_)
    rhat = npy(bj.diagnostics.potential_scale_reduction(hist, tgt))
    ref = odiag.potential_scale_reduction(npy(hist), chain_axis=1, sample_axis=0)
    np.testing.assert_allclose(rhat, ref, rtol=2e-5)
    assert np.all(rhat < 1.05)                       # the chains start in the typical set and mix
    hist[:, : C // 2] += 3.0                         # shift half the chains: R-hat must flag it
    assert np.all(npy(bj.diagnostics.potential_scale_reduction(hist, tgt)) > 1.2)


@pytest.mark.parametrize("C, T_, D", [(64, 200, 24), (1, 501, 5), (7, 64, 132), (3, 33, 1)])
def test_effective_sample_size_on_device_history(C, T_, D):
    """blackjax/diagnostics.py:159-305 on the device vs the oracle, on autocorrelated draws (AR(1) per dim with a
    different coefficient each, incl. anti-correlated ones) plus the degenerate columns of tests/test_diagnostics.py:91-116."""
    from oracle import diagnostics as odiag
    rs = np.random.default_rng(C * 1000 + T_)
    phi = np.linspace(-0.6, 0.95, D)
    x = np.zeros((T_, C, D), F)
    e = rs.standard_normal((T_, C, D)).astype(F)
    for t in range(1, T_):
        x[t] = phi * x[t - 1] + e[t]
    if D >= 5:
        x[:, :, 1] = 0.0                                    # constant
        x[:, :, 2] = np.arange(C, dtype=F)[None, :]         # constant per chain, different means
        x[:, :, 3] = 1e-30 * e[:, :, 3]                      # numerically constant
    tgt = T.StdNormal(D)
    ess = npy(bj.diagnostics.effective_sample_size(tf(x), tgt))
    ref = np.atleast_1d(odiag.effective_sample_size(x, chain_axis=1, sample_axis=0))
    if D >= 5:
        np.testing.assert_array_equal(ess[1:4], 0.0)
        np.testing.assert_array_equal(ref[1:4], 0.0)
    # the truncation points of Geyer's sequences are discontinuous in the autocorrelations: allow a few columns to land
    # on the other side of a float32-level tie, require the rest to agree tightly
    rel = np.abs(ess - ref) / np.maximum(np.abs(ref), 1e-30)
    rel[ref == 0] = np.abs(ess[ref == 0])
    assert np.mean(rel < 2e-3) >= 0.9, (ess, ref)
    assert np.all(rel < 0.2), (ess, ref)


def test_effective_sample_size_iid_and_hmc_history():
    tgt = T.DiagGaussian(np.logspace(-0.3, 0.3, 24))
    C, T_ = 256, 100
    iid = torch.randn(T_, C, 24, device=DEV)
    ess = npy(bj.diagnostics.effective_sample_size(iid, tgt))
    np.testing.assert_allclose(ess, C * T_, rtol=0.1)
    st0 = bj.hmc.init(torch.randn(C, 24, device=DEV), tgt)
    _, hist, _ = bj.sample_hmc_native(bj.random.key(5, DEV), st0, tgt, 0.3, torch.ones(24, device=DEV), 8, T_)
    ess = npy(bj.diagnostics.effective_sample_size(hist, tgt))
    assert np.all(ess > 0.05 * C * T_) and np.all(np.isfinite(ess))


def test_hmc_inplace_and_out_of_place_agree():
    tgt = T.StdNormal(64)
    q = torch.randn(128, 64, device=DEV)
    keys = bj.random.split(bj.random.key(3, DEV), 128)
    st = bj.hmc.init(q.clone(), tgt)
    imm = torch.ones(64, device=DEV)
    a, ia = bj.hmc.build_kernel()(keys, st, tgt, 0.3, imm, 5)
    st2 = bj.hmc.init(q.clone(), tgt)
    b, ib = bj.hmc.build_kernel(inplace=True)(keys, st2, tgt, 0.3, imm, 5)
    assert torch.equal(a.position, b.position) and torch.equal(a.logdensity_grad, b.logdensity_grad)
    assert b.position.data_ptr() == st2.position.data_ptr()
    assert torch.equal(st.position, q)  # the out-of-place call left its input untouched


# ---------------------------------------------------------------------------------------------------------
# large-D dense path: tensor-core GEMMs (float32-accurate operand split) for M^-1 p, -P x, L^-T z
# ---------------------------------------------------------------------------------------------------------
def dense_problem(D, C, seed=31, metric="dense", target="dense"):
    rs = np.random.default_rng(seed)
    cov, prec = otargets.correlated_gaussian(D, seed=seed, lo=-0.5, hi=0.5)
    if target == "dense":
        tgt, otgt = T.DenseGaussian(prec), otargets.DenseGaussian(prec)
    else:
        s = np.exp(rs.uniform(-0.5, 0.5, D))
        tgt, otgt = T.DiagGaussian(s), otargets.DiagGaussian(s)
    imm = cov if metric == "dense" else np.exp(rs.uniform(-0.5, 0.5, D)).astype(F)
    q = (0.5 * rs.standard_normal((C, D))).astype(F)
    return tgt, otgt, imm, q


@pytest.mark.parametrize("D, C, metric, target", [(256, 100, "dense", "dense"), (512, 37, "dense", "dense"),
                                                  (256, 64, "diag", "dense"), (256, 64, "dense", "diag"),
                                                  (132, 21, "dense", "dense")])   # D % 8 != 0: padded operand planes
def test_dense_path_building_blocks(D, C, metric, target):
    tgt, otgt, imm, q = dense_problem(D, C, metric=metric, target=target)
    eng = _engine.Engine(DEV, C, D, tgt)
    eng.set_metric(tf(imm))
    om = ohmc.Metric(imm)
    dq = tf(q)
    logp, g = eng.init_state(dq)
    lp0, g0 = otgt(q)
    dclose(npy(g), g0, rtol=1e-5)
    dclose(npy(logp), lp0, rtol=1e-5, scale=np.max(np.abs(lp0)) + 1)
    keys = oprng.split(oprng.key(9), C)
    p = eng.sample_momentum(tk(keys))
    p_ref = om.sample_momentum(keys, D)
    dclose(npy(p), p_ref, rtol=1e-5)
    e = eng.energy(tf(p_ref), logp)
    dclose(npy(e), -lp0 + om.kinetic_energy(p_ref), rtol=1e-5, scale=np.max(np.abs(lp0)) + D)
    dclose(npy(eng.velocity(tf(p_ref))), om.velocity(p_ref), rtol=1e-5)
    dp = tf(p_ref)
    eng.leapfrog_(dq, dp, logp, g, 0.05, 4)
    q1, p1, lp1, g1 = ohmc.static_integration(otgt, om, q, p_ref, lp0, g0, F(0.05), 4)
    dclose(npy(dq), q1, rtol=2e-5)
    dclose(npy(dp), p1, rtol=2e-5)
    dclose(npy(g), g1, rtol=2e-5)
    dclose(npy(logp), lp1, rtol=2e-5, scale=np.max(np.abs(lp1)) + 1)


def test_dense_velocity_row_scaling_and_non_finite_rows():
    """The fp16 operand split is only float32-accurate because every row is lifted by a power of two first
    (bjx_dense.cu k_rows_split2): rows of magnitude 1e-6 ... 1e6 must all come out at float32 accuracy relative to
    their own scale, matrices of any magnitude too, and a NaN / inf row must poison only itself."""
    D, C = 256, 40
    rs = np.random.default_rng(5)
    for mat_scale in (1e-5, 1.0, 3e4):
        A = rs.standard_normal((D, D))
        imm = ((A @ A.T / D + np.eye(D)) * mat_scale).astype(F)
        tgt = T.DiagGaussian(np.ones(D, F))
        eng = _engine.Engine(DEV, C, D, tgt)
        eng.set_metric(tf(imm))
        p = rs.standard_normal((C, D)).astype(F)
        p *= (10.0 ** rs.uniform(-6, 6, size=(C, 1))).astype(F)
        p[3, 7] = np.nan
        p[5, 0] = np.inf
        v = npy(eng.velocity(tf(p)))
        ok = np.ones(C, bool)
        ok[[3, 5]] = False
        ref = p[ok].astype(np.float64) @ imm.astype(np.float64)
        err = np.abs(v[ok] - ref).max(axis=1) / np.abs(ref).max(axis=1)
        assert err.max() < 3e-6, (mat_scale, err.max())
        assert not np.isfinite(v[3]).any() or np.isnan(v[3]).any()
        assert np.isnan(v[3]).all() and not np.isfinite(v[5]).all()
        eng.close()


@pytest.mark.parametrize("D, C, L, pce", [(256, 96, 6, False), (384, 40, 4, True), (256, 8203, 3, False),
                                          (256, 8200, 2, True),      # 33 row tiles, rank 1 of the last one dead
                                          (132, 33, 5, True)])       # padded operand planes
def test_dense_hmc_transition_matches_oracle(D, C, L, pce):
    tgt, otgt, imm, q = dense_problem(D, C)
    keys = oprng.split(oprng.key(17), C)
    rs = np.random.default_rng(3)
    eps_np = (0.08 * np.exp(rs.uniform(-0.2, 0.2, C))).astype(F) if pce else F(0.08)
    onew, oinfo = ohmc.hmc_kernel(keys, ohmc.init(q, otgt), otgt, eps_np, ohmc.Metric(imm), L)
    kernel = bj.hmc.build_kernel(full_info=True)
    st = bj.hmc.init(tf(q), tgt)
    new, info = kernel(tk(keys), st, tgt, tf(eps_np) if pce else float(eps_np), tf(imm), L)
    torch.cuda.synchronize()
    dclose(npy(info.momentum), oinfo.momentum, rtol=1e-5)
    dclose(npy(info.proposal.position), oinfo.proposal[0], rtol=3e-5)
    dclose(npy(info.proposal.momentum), oinfo.proposal[1], rtol=3e-5)
    dclose(npy(info.energy), oinfo.energy, rtol=3e-5, scale=np.max(np.abs(oinfo.energy)) + D)
    dclose(npy(info.acceptance_rate), oinfo.acceptance_rate, rtol=2e-3, scale=1.0)
    u = oprng.uniform(oprng.split(keys, 2)[:, 1])
    tie = np.abs(u - oinfo.acceptance_rate) < 2e-3
    acc = npy(info.is_accepted)
    assert ((acc == oinfo.is_accepted) | tie).all()
    same = acc == oinfo.is_accepted
    dclose(npy(new.position)[same], onew.position[same], rtol=3e-5)
    dclose(npy(new.logdensity_grad)[same], onew.logdensity_grad[same], rtol=3e-5)


def test_dense_unsupported_combinations_fail_loudly():
    # a dense metric beyond 128 dims runs on the tensor-core path, whose gradient kernels cover the Gaussian targets
    # (NUTS there is built since round 2: tests/test_gpu_round2.py::test_dense_path_nuts_matches_oracle)
    _, _, imm, q = dense_problem(256, 8)
    tgt = T.Funnel(256)
    st = bj.hmc.init(tf(q), tgt)
    with pytest.raises(bj.BjxError, match="large-D dense path supports"):
        bj.hmc.build_kernel()(bj.random.key(0, DEV), st, tgt, 0.1, tf(imm), 5)
    with pytest.raises(bj.BjxError):
        bj.nuts.build_kernel()(bj.random.key(0, DEV), st, tgt, 0.1, tf(imm), 5)


def test_fullsize_dense_config2_65536x1024():
    # BASELINE config 2 shape: 1024-D correlated Gaussian, 65536 chains, dense mass matrix.  Size-independent
    # properties: energy conservation of the symplectic integrator, time reversibility, and linearity of the
    # dynamics (Gaussian target + Gaussian kinetic energy => the flow map is linear in (q, p)).
    C, D = 65536, 1024
    cov, prec = otargets.correlated_gaussian(D, seed=0)
    tgt = T.DenseGaussian(prec)
    eng = _engine.Engine(DEV, C, D, tgt)
    eng.set_metric(tf(cov))
    g_ = torch.Generator(device=DEV).manual_seed(0)
    q0 = 0.1 * torch.randn(C, D, device=DEV, generator=g_)
    p0 = eng.sample_momentum(bj.random.split(bj.random.key(1, DEV), C))
    q, p = q0.clone(), p0.clone()
    logp, g = eng.init_state(q)
    e0 = eng.energy(p, logp)
    eng.leapfrog_(q, p, logp, g, 0.5, 3)
    e1 = eng.energy(p, logp)
    assert float((e1 - e0).abs().max() / e0.abs().mean()) < 0.2          # eps=0.5 is near the stability limit
    p.neg_()
    eng.leapfrog_(q, p, logp, g, 0.5, 3)
    assert float((q - q0).abs().max()) < 2e-3 * float(q0.abs().max() + p0.abs().max())
    # linearity: flow(2 q0, 2 p0) == 2 flow(q0, p0)
    qa, pa = q0.clone(), p0.clone()
    la, ga = eng.init_state(qa)
    eng.leapfrog_(qa, pa, la, ga, 0.5, 2)
    qb, pb = 2 * q0, 2 * p0
    lb, gb = eng.init_state(qb)
    eng.leapfrog_(qb, pb, lb, gb, 0.5, 2)
    torch.testing.assert_close(qb, 2 * qa, rtol=1e-4, atol=1e-4 * float(qa.abs().max()))


# ---------------------------------------------------------------------------------------------------------
# SURVEY 8f item 1: multinomial HMC (blackjax.mhmc; hmc.py:181-248, trajectory.py:170-232)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("kind, D, C, L, eps, imm_kind", [
    ("std", 100, 96, 10, 0.2, "ones"), ("diag", 516, 40, 12, 0.08, "diag"), ("funnel", 64, 64, 16, 0.1, "ones"),
    ("banana", 2, 64, 10, 0.1, "dense"), ("std", 1, 32, 100, 1000.0, "ones")])
def test_multinomial_hmc_matches_oracle(kind, D, C, L, eps, imm_kind):
    rs = np.random.default_rng(12)
    tgt, otgt = make_target(kind, D, rs)
    if imm_kind == "ones":
        imm = np.ones(D, F)
    elif imm_kind == "diag":
        imm = np.exp(rs.uniform(-0.5, 0.5, D)).astype(F)
    else:
        A = rs.standard_normal((D, D))
        imm = (A @ A.T / D + np.eye(D)).astype(F)
    q = (0.5 * rs.standard_normal((C, D))).astype(F)
    keys = oprng.split(oprng.key(14), C)
    onew, oinfo = ohmc.mhmc_kernel(keys, ohmc.init(q, otgt), otgt, F(eps), imm, L)
    kernel = bj.mhmc.build_kernel(full_info=True)
    new, info = kernel(tk(keys), bj.mhmc.init(tf(q), tgt), tgt, float(eps), tf(imm), L)
    torch.cuda.synchronize()
    assert bool(info.is_accepted.all())
    assert (npy(info.is_divergent) == oinfo.is_divergent).all()
    # the multinomial selection index must agree (same uniforms); chains whose draw sits on a tie may differ
    same = np.all(np.isclose(npy(new.position), onew.position, rtol=1e-4, atol=1e-5), axis=1)
    assert same.mean() >= 0.95
    close(npy(info.acceptance_rate)[same], oinfo.acceptance_rate[same], rtol=1e-4, scale=1.0)
    fin = np.isfinite(oinfo.energy) & same
    close(npy(info.energy)[fin], oinfo.energy[fin], rtol=1e-5, scale=np.max(np.abs(oinfo.energy[fin])) + 1)
    close(npy(new.logdensity_grad)[same], onew.logdensity_grad[same], rtol=1e-4)
    close(npy(info.proposal.momentum)[same], oinfo.proposal[1][same], rtol=1e-4)
    assert torch.equal(info.proposal.position, new.position)


def test_mhmc_api_and_sampling():
    # tests/mcmc/test_multinomial_hmc.py:21-55,95-152
    assert bj.multinomial_hmc is bj.mhmc
    tgt = T.StdNormal(1)
    alg = bj.mhmc(tgt, 0.5, torch.ones(1, device=DEV), 20)
    st = alg.init(torch.zeros(4096, 1, device=DEV))
    keys = bj.random.split(bj.random.key(0, DEV), 60)
    for t in range(60):
        st, info = alg.step(keys[t], st)
    assert abs(float(st.position.mean())) < 0.3 and abs(float(st.position.std()) - 1.0) < 0.3
    explicit = bj.hmc.build_kernel(build_proposal=bj.mcmc.hmc.multinomial_hmc_proposal)
    a, _ = explicit(keys[0], st, tgt, 0.5, torch.ones(1, device=DEV), 20)
    b, _ = bj.mhmc.build_kernel()(keys[0], st, tgt, 0.5, torch.ones(1, device=DEV), 20)
    assert torch.equal(a.position, b.position)


# ---------------------------------------------------------------------------------------------------------
# SURVEY 8f item 4 (first piece): dynamic HMC -- per-chain random trajectory lengths (mcmc/dynamic_hmc.py)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("shape, lo, hi", [((), 1, 10), ((5,), 0, 100), ((3,), -7, 7), ((), 4, 4), ((2,), 0, 1 << 20)])
def test_randint_bit_exact(shape, lo, hi):
    keys = oprng.split(oprng.key(21), 257)
    ref = oprng.randint(keys, shape, lo, hi)
    out = bj.random.randint(tk(keys), shape, lo, hi).cpu().numpy()
    assert out.dtype == np.int32 and out.shape == ref.shape
    np.testing.assert_array_equal(out, ref)
    assert out.min() >= lo and (out.max() < hi or hi <= lo)


@pytest.mark.parametrize("kind, D, multinomial", [("std", 100, False), ("diag", 1024, False), ("funnel", 64, False),
                                                  ("dense", 6, False), ("diag", 97, True)])
def test_dynamic_hmc_matches_oracle(kind, D, multinomial):
    rs = np.random.default_rng(31)
    tgt, otgt = make_target(kind, D, rs)
    C, eps = 48, 0.11
    imm = np.exp(rs.uniform(-0.5, 0.5, D)).astype(F)
    q = (0.4 * rs.standard_normal((C, D))).astype(F)
    keys = oprng.split(oprng.key(8), C)
    rga = oprng.split(oprng.key(9), C)
    onew, oinfos, onext, osteps = ohmc.dynamic_hmc_kernel(keys, ohmc.init(q, otgt), rga, otgt, F(eps), imm,
                                                          multinomial=multinomial)
    alg = bj.dmhmc if multinomial else bj.dhmc
    kernel = alg.build_kernel()
    state = alg.init(tf(q), tgt, tk(rga))
    new, info = kernel(tk(keys), state, tgt, float(eps), tf(imm))
    torch.cuda.synchronize()
    np.testing.assert_array_equal(info.num_integration_steps.cpu().numpy(), osteps)     # bit-exact step counts
    assert len(set(osteps.tolist())) > 3                                                # the chains really differ
    np.testing.assert_array_equal(new.random_generator_arg.cpu().numpy().view(np.uint32), onext)
    oacc = np.array([i.is_accepted[0] for i in oinfos])
    orate = np.array([i.acceptance_rate[0] for i in oinfos])
    if multinomial:
        same = np.all(np.isclose(npy(new.position), onew.position, rtol=1e-4, atol=1e-5), axis=1)
        assert same.mean() >= 0.9
    else:
        assert (npy(info.is_accepted) == oacc).all()
        same = np.ones(C, bool)
    close(npy(info.acceptance_rate)[same], orate[same], rtol=1e-4, scale=1.0)
    close(npy(new.position)[same], onew.position[same], rtol=1e-5 if not multinomial else 1e-4)
    close(npy(new.logdensity)[same], onew.logdensity[same], rtol=1e-5, scale=np.max(np.abs(onew.logdensity)) + 1)


def test_dynamic_hmc_top_level_api_samples():
    # tests/mcmc/test_sampling.py dynamic HMC usage: the step-count keys evolve, the sampler mixes
    assert bj.dynamic_hmc is bj.dhmc
    tgt = T.DiagGaussian(np.array([1.0, 2.0], F))
    alg = bj.dhmc(tgt, 0.5, torch.ones(2, device=DEV))
    st = alg.init(torch.zeros(8192, 2, device=DEV), bj.random.key(3, DEV))
    assert st.random_generator_arg.shape == (8192, 2)
    keys = bj.random.split(bj.random.key(0, DEV), 80)
    for t in range(80):
        prev = st.random_generator_arg
        st, info = alg.step(keys[t], st)
        assert not torch.equal(prev, st.random_generator_arg)
    assert int(info.num_integration_steps.min()) >= 1 and int(info.num_integration_steps.max()) <= 9
    std = st.position.std(0).cpu().numpy()
    np.testing.assert_allclose(std, [1.0, 2.0], rtol=0.1)
    with pytest.raises(bj.BjxError):                       # per-chain step counts are a row-kernel feature
        big = T.DiagGaussian(np.ones(2048, F))
        k = bj.dhmc.build_kernel()
        s0 = bj.dhmc.init(torch.zeros(16, 2048, device=DEV), big, bj.random.split(bj.random.key(1, DEV), 16))
        k(keys[0], s0, big, 0.1, torch.ones(2048, device=DEV))


# ---------------------------------------------------------------------------------------------------------
# SURVEY 8f item 2: the other palindromic integrators (coefficient tables, integrators.py:335-369)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("name", ["mclachlan", "yoshida", "omelyan"])
@pytest.mark.parametrize("kind, D", [("diag", 100), ("funnel", 64), ("dense", 6)])
def test_general_integrators_match_oracle(name, kind, D):
    from blackjax_b200.mcmc import integrators as I
    coef = getattr(I, name)
    ocoef = getattr(ohmc, name.upper())
    assert tuple(F(c) for c in coef) == tuple(F(c) for c in ocoef)
    rs = np.random.default_rng(6)
    tgt, otgt = make_target(kind, D, rs)
    C = 21
    imm = np.exp(rs.uniform(-0.5, 0.5, D)).astype(F)
    q = (0.3 * rs.standard_normal((C, D))).astype(F)
    p = rs.standard_normal((C, D)).astype(F)
    eng = _engine.Engine(DEV, C, D, tgt)
    eng.set_metric(tf(imm))
    eng.set_integrator(coef)
    dq, dp = tf(q), tf(p)
    logp, g = eng.init_state(dq)
    eng.leapfrog_(dq, dp, logp, g, 0.1, 4)
    lp0, g0 = otgt(q)
    q1, p1, lp1, g1 = ohmc.static_integration(otgt, ohmc.Metric(imm), q, p, lp0, g0, F(0.1), 4, ocoef)
    close(npy(dq), q1)
    close(npy(dp), p1)
    close(npy(g), g1)
    close(npy(logp), lp1, rtol=1e-5, scale=np.max(np.abs(lp1)) + 1)
    # whole transitions through the public API
    keys = oprng.split(oprng.key(8), C)
    onew, oinfo = ohmc.hmc_kernel(keys, ohmc.init(q, otgt), otgt, F(0.1), imm, 5, coefficients=ocoef)
    new, info = bj.hmc.build_kernel(integrator=coef, full_info=True)(tk(keys), bj.hmc.init(tf(q), tgt), tgt, 0.1, tf(imm), 5)
    close(npy(info.proposal.position), oinfo.proposal[0])
    close(npy(info.acceptance_rate), oinfo.acceptance_rate, rtol=1e-4, scale=1.0)
    if kind != "dense":
        onew, oinfo = onuts.nuts_kernel(keys, ohmc.init(q, otgt), otgt, F(0.2), imm, 6, coefficients=ocoef)
        new, info = bj.nuts.build_kernel(integrator=name)(tk(keys), bj.nuts.init(tf(q), tgt), tgt, 0.2, tf(imm), 6)
        same = npy(info.num_integration_steps) == oinfo.num_integration_steps
        assert same.mean() >= 0.9
        close(npy(new.position)[same], onew.position[same], rtol=1e-4)
    eng.set_integrator(I.velocity_verlet)


def test_integrator_validation():
    from blackjax_b200.mcmc import integrators as I
    with pytest.raises(ValueError):
        I.as_coefficients((0.5, 1.0))
    with pytest.raises(ValueError):
        I.as_coefficients((0.3, 1.0, 0.5))
    with pytest.raises(ValueError):
        bj.hmc.build_kernel(integrator="leapfrogz")


# ---------------------------------------------------------------------------------------------------------
# rows larger than a warp's registers (1024 < D <= 18432): CTA-per-chain kernels, incl. BASELINE config 5's target
# ---------------------------------------------------------------------------------------------------------
def big_problem(kind, D, seed=41):
    rs = np.random.default_rng(seed)
    if kind == "diag":
        s = np.exp(rs.uniform(-0.5, 0.5, D))
        return T.DiagGaussian(s), otargets.DiagGaussian(s)
    if kind == "funnel":
        return T.Funnel(D), otargets.Funnel(D)
    x, bits = T.HierLogit.synthetic_data(D - 4, seed=1)
    return T.HierLogit(x, bits), otargets.HierLogit(x, bits)


@pytest.mark.parametrize("kind, D, C", [("diag", 2048, 40), ("funnel", 1500, 24), ("hier", 1504, 24), ("hier", 10000, 6)])
def test_big_rows_match_oracle(kind, D, C):
    tgt, otgt = big_problem(kind, D)
    rs = np.random.default_rng(5)
    q = (0.3 * rs.standard_normal((C, D))).astype(F)
    imm = np.exp(rs.uniform(-0.3, 0.3, D)).astype(F)
    eng = _engine.Engine(DEV, C, D, tgt)
    eng.set_metric(tf(imm))
    om = ohmc.Metric(imm)
    dq = tf(q)
    logp, g = eng.init_state(dq)
    lp0, g0 = otgt(q)
    close(npy(g), g0, rtol=1e-5)
    close(npy(logp), lp0, rtol=1e-5, scale=np.max(np.abs(lp0)) + 1)
    keys = oprng.split(oprng.key(2), C)
    p_ref = om.sample_momentum(keys, D)
    close(npy(eng.sample_momentum(tk(keys))), p_ref, rtol=3e-6)
    close(npy(eng.energy(tf(p_ref), logp)), -lp0 + om.kinetic_energy(p_ref), rtol=1e-5, scale=np.max(np.abs(lp0)) + D)
    dp = tf(p_ref)
    eps = F(0.01)
    eng.leapfrog_(dq, dp, logp, g, float(eps), 5)
    q1, p1, lp1, g1 = ohmc.static_integration(otgt, om, q, p_ref, lp0, g0, eps, 5)
    close(npy(dq), q1, rtol=1e-5)
    close(npy(dp), p1, rtol=2e-5)
    close(npy(g), g1, rtol=2e-5)
    close(npy(logp), lp1, rtol=1e-5, scale=np.max(np.abs(lp1)) + 1)
    # one whole transition, teacher-forced
    onew, oinfo = ohmc.hmc_kernel(keys, ohmc.init(q, otgt), otgt, eps, om, 6)
    st = bj.hmc.init(tf(q), tgt)
    new, info = bj.hmc.build_kernel(full_info=True)(tk(keys), st, tgt, float(eps), tf(imm), 6)
    torch.cuda.synchronize()
    close(npy(info.proposal.position), oinfo.proposal[0], rtol=1e-5)
    close(npy(info.energy), oinfo.energy, rtol=1e-5, scale=np.max(np.abs(oinfo.energy)) + D)
    u = oprng.uniform(oprng.split(keys, 2)[:, 1])
    tie = np.abs(u - oinfo.acceptance_rate) < 1e-3
    acc = npy(info.is_accepted)
    assert ((acc == oinfo.is_accepted) | tie).all()
    same = acc == oinfo.is_accepted
    close(npy(new.position)[same], onew.position[same], rtol=1e-5)
    with pytest.raises(bj.BjxError, match="dim <= 1024"):
        bj.nuts.build_kernel()(tk(keys), st, tgt, 0.01, tf(imm), 3)


@pytest.mark.parametrize("D, C, inplace", [(1504, 7, False), (1504, 1, True), (2052, 5, True)])
def test_hier_logit_two_chains_per_cta_transition(D, C, inplace):
    # k_big2_hmc_hier (two chains per CTA, momentum in registers): odd chain counts (the last CTA's second slot idles),
    # per-chain step sizes and per-chain diagonal metrics, in place and out of place, against the oracle
    tgt, otgt = big_problem("hier", D)
    rs = np.random.default_rng(17)
    q = (0.3 * rs.standard_normal((C, D))).astype(F)
    imm = np.exp(rs.uniform(-0.3, 0.3, (C, D))).astype(F)
    eps = (0.01 * np.exp(rs.uniform(-0.3, 0.3, C))).astype(F)
    keys = oprng.split(oprng.key(3), C)
    L = 5
    onew, oinfo = ohmc.hmc_kernel(keys, ohmc.init(q, otgt), otgt, eps, oadapt._PerChainDiag(imm), L)
    st = bj.hmc.init(tf(q), tgt)
    q_before = st.position.clone()
    new, info = bj.hmc.build_kernel(full_info=True, inplace=inplace)(tk(keys), st, tgt, tf(eps), tf(imm), L)
    torch.cuda.synchronize()
    close(npy(info.momentum), oinfo.momentum, rtol=3e-6)
    close(npy(info.proposal.position), oinfo.proposal[0], rtol=1e-5)
    close(npy(info.proposal.momentum), oinfo.proposal[1], rtol=2e-5)
    close(npy(info.energy), oinfo.energy, rtol=1e-5, scale=np.max(np.abs(oinfo.energy)) + D)
    close(npy(info.acceptance_rate), oinfo.acceptance_rate, rtol=2e-2, scale=1.0)
    u = oprng.uniform(oprng.split(keys, 2)[:, 1])
    acc = npy(info.is_accepted)
    assert ((acc == oinfo.is_accepted) | (np.abs(u - oinfo.acceptance_rate) < 2e-2)).all()
    same = acc == oinfo.is_accepted
    close(npy(new.position)[same], onew.position[same], rtol=1e-5)
    close(npy(new.logdensity_grad)[same], onew.logdensity_grad[same], rtol=2e-5)
    close(npy(new.logdensity)[same], onew.logdensity[same], rtol=1e-5, scale=np.max(np.abs(onew.logdensity)) + 1)
    rej = ~acc
    assert torch.equal(new.position[torch.from_numpy(rej).to(DEV)], q_before[torch.from_numpy(rej).to(DEV)])


def hier_logit_typical_start(C, D, device, seed=0):
    """A start in the typical set (the data-generating values + N(0, 0.7^2) group effects).  The origin is NOT usable:
    with every alpha_g == mu the log_tau gradient is -G, tau collapses and the centred model's funnel makes any
    fixed step size unstable -- the start/step SURVEY 8d pencilled in (q0 = 0, eps = 0.02) gives acceptance 0."""
    g_ = torch.Generator(device=device).manual_seed(seed)
    q0 = torch.empty(C, D, device=device)
    q0[:, 0], q0[:, 1], q0[:, 2], q0[:, 3] = 0.5, float(np.log(0.7)), 1.0, -0.5
    q0[:, 4:] = 0.5 + 0.7 * torch.randn(C, D - 4, device=device, generator=g_)
    return q0


def test_fullsize_config5_hier_logit_10000d():
    # BASELINE config 5 target/shape per chain (D = 10000); 8192 chains here (the config shards 1M chains over 8 GPUs).
    # Properties: reversibility and energy conservation of the integrator; sanity of the accept statistics.
    C, D, L, eps = 8192, 10000, 20, 0.005
    x, bits = T.HierLogit.synthetic_data(D - 4, seed=1)
    tgt = T.HierLogit(x, bits)
    imm = torch.ones(D, device=DEV)
    q0 = hier_logit_typical_start(C, D, DEV)
    st = bj.hmc.init(q0, tgt)
    eng = _engine.get_engine(q0, tgt)
    eng.set_metric(imm)
    p0 = eng.sample_momentum(bj.random.split(bj.random.key(3, DEV), C))
    q, p, logp, g = q0.clone(), p0.clone(), st.logdensity.clone(), st.logdensity_grad.clone()
    e0 = eng.energy(p, logp)
    eng.leapfrog_(q, p, logp, g, eps, L)
    e1 = eng.energy(p, logp)
    assert float((e1 - e0).abs().max()) < 5.0              # O(eps^2) energy error on energies of order 1e4
    p.neg_()
    eng.leapfrog_(q, p, logp, g, eps, L)
    assert float((q - q0).abs().max()) < 1e-3
    new, info = bj.hmc.build_kernel()(bj.random.key(4, DEV), st, tgt, eps, imm, L)
    assert 0.3 < float(info.acceptance_rate.mean()) <= 1.0
    assert bool(info.is_accepted.any())


# ---------------------------------------------------------------------------------------------------------
# NUTS
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("step_size, diverge, turn, doublings",
                         [(1e-10, False, False, 10), (1.0, False, True, 2), (1e5, True, True, 1)])
def test_nuts_expansion_outcomes_kat(step_size, diverge, turn, doublings):
    # tests/mcmc/test_trajectory.py:193-260 through bjx_nuts_step
    tgt = T.StdNormal(1)
    imm = torch.ones(1, device=DEV)
    k = oprng.key(0)[None]
    p0 = ohmc.Metric(np.ones(1, F)).sample_momentum(k, 1)
    st = bj.nuts.init(torch.zeros(1, 1, device=DEV), tgt)
    kern = bj.nuts.build_kernel()
    _, info = kern(None, st, tgt, step_size, imm, 10, _momentum=tf(p0), _key_integrator=tk(k))
    assert bool(info.is_divergent[0]) == diverge
    assert bool(info.is_turning[0]) == turn
    assert int(info.num_trajectory_expansions[0]) == doublings


def run_nuts_case(kind, D, C, eps, imm_kind="ones", max_doublings=10, seed=21, min_match=0.97):
    rs = np.random.default_rng(seed)
    tgt, otgt = make_target(kind, D, rs)
    if imm_kind == "ones":
        imm = np.ones(D, F)
    elif imm_kind == "diag":
        imm = np.exp(rs.uniform(-0.5, 0.5, D)).astype(F)
    else:
        A = rs.standard_normal((D, D))
        imm = (A @ A.T / D + np.eye(D)).astype(F)
    q = (0.1 * rs.standard_normal((C, D))).astype(F)
    keys = oprng.split(oprng.key(seed), C)
    ostate = ohmc.init(q, otgt)
    onew, oinfo = onuts.nuts_kernel(keys, ostate, otgt, F(eps), imm, max_doublings)
    kern = bj.nuts.build_kernel(full_info=True, max_tree_depth=max_doublings)
    st = bj.nuts.init(tf(q), tgt)
    new, info = kern(tk(keys), st, tgt, float(eps), tf(imm), max_doublings)
    torch.cuda.synchronize()
    close(npy(info.momentum), oinfo.momentum, rtol=3e-6)
    n_dev, n_ref = npy(info.num_integration_steps), oinfo.num_integration_steps
    same = ((n_dev == n_ref) & (npy(info.num_trajectory_expansions) == oinfo.num_trajectory_expansions)
            & (npy(info.is_turning) == oinfo.is_turning) & (npy(info.is_divergent) == oinfo.is_divergent))
    pos_same = np.all(np.isclose(npy(new.position), onew.position, rtol=1e-4, atol=1e-5), axis=1)
    frac = float(np.mean(same & pos_same))
    # discrete tree decisions sit on float comparisons (U-turn dot products, multinomial draws): chains whose
    # deciding comparison is within rounding of a tie may legitimately differ; everything else must agree.
    assert frac >= min_match, f"only {frac:.3f} of chains match the oracle"
    ok = same & pos_same
    close(npy(info.acceptance_rate)[ok], oinfo.acceptance_rate[ok], rtol=1e-4, scale=1.0)
    close(npy(info.energy)[ok], oinfo.energy[ok], rtol=1e-5, scale=np.max(np.abs(oinfo.energy)) + 1)
    close(npy(new.logdensity_grad)[ok], onew.logdensity_grad[ok], rtol=1e-4)
    close(npy(info.trajectory_leftmost_state.position)[ok], oinfo.trajectory_leftmost_state[0][ok], rtol=1e-4)
    close(npy(info.trajectory_rightmost_state.momentum)[ok], oinfo.trajectory_rightmost_state[1][ok], rtol=1e-4)
    return n_dev


@pytest.mark.parametrize("kind, D, C, eps, imm_kind, md", [
    ("std", 1, 64, 1.0, "ones", 10),          # tests/mcmc/test_sampling.py:1174-1186 NUTS settings
    ("std", 100, 64, 0.2, "ones", 10),
    ("diag", 64, 48, 0.15, "diag", 10),
    ("diag", 97, 32, 0.15, "diag", 6),        # scalar layout
    ("funnel", 128, 64, 0.1, "ones", 10),     # BASELINE config 3 target/shape (fewer chains)
    ("funnel", 10, 64, 0.3, "ones", 10),
    ("banana", 2, 64, 0.1, "dense", 10),      # dense metric through the small in-warp path
    ("dense", 6, 32, 0.2, "dense", 8),
    ("std", 8, 64, 1e-4, "ones", 4),          # never turns: hits max depth
    ("std", 8, 32, 1e4, "ones", 10),          # diverges on the first leaf
])
def test_nuts_transition_matches_oracle(kind, D, C, eps, imm_kind, md):
    run_nuts_case(kind, D, C, eps, imm_kind, md)


def test_nuts_step_count_stats():
    n = run_nuts_case("std", 16, 256, 0.5, "ones", 10)
    assert n.min() >= 1 and n.max() <= 1023


# ---------------------------------------------------------------------------------------------------------
# window adaptation
# ---------------------------------------------------------------------------------------------------------
def test_dual_averaging_and_welford_kernels():
    from blackjax_b200._lib import check, lib, ptr
    C, D = 50, 12
    rs = np.random.default_rng(4)
    eng = _engine.Engine(DEV, C, D, T.StdNormal(D))
    st = torch.empty(C, 5, device=DEV)
    eps0 = tf(np.exp(rs.uniform(-1, 1, C)))
    eps = torch.empty(C, device=DEV)
    check(lib().bjx_da_init(eng.h, ptr(st), ptr(eps0), ptr(eps)), eng.h)
    o = [oadapt.da_init(e) for e in npy(eps0)]
    for it in range(12):
        acc = rs.uniform(0, 1, C).astype(F)
        dacc = tf(acc)
        check(lib().bjx_da_update(eng.h, ptr(st), ptr(dacc), 0.8, ptr(eps)), eng.h)
        o = [oadapt.da_update(s, a, 0.8) for s, a in zip(o, acc)]
        close(npy(eps), [np.exp(s.log_step_size) for s in o], rtol=1e-5)
    fin = torch.empty(C, device=DEV)
    check(lib().bjx_da_final(eng.h, ptr(st), ptr(fin)), eng.h)
    close(npy(fin), [oadapt.da_final(s) for s in o], rtol=1e-5)
    check(lib().bjx_da_reset(eng.h, ptr(st), ptr(eps)), eng.h)
    close(npy(eps), [np.exp(oadapt.da_init(oadapt.da_final(s)).log_step_size) for s in o], rtol=1e-5)
    # Welford
    mean = torch.zeros(C, D, device=DEV)
    m2 = torch.zeros(C, D, device=DEV)
    ws = [oadapt.welford_init(D) for _ in range(C)]
    for n in range(1, 9):
        x = rs.standard_normal((C, D)).astype(F)
        dx = tf(x)
        check(lib().bjx_welford_update(eng.h, ptr(dx), ptr(mean), ptr(m2), n), eng.h)
        ws = [oadapt.welford_update(w, xi) for w, xi in zip(ws, x)]
    close(npy(mean), np.stack([w.mean for w in ws]), rtol=1e-5)
    close(npy(m2), np.stack([w.m2 for w in ws]), rtol=1e-5)
    imm = torch.empty(C, D, device=DEV)
    check(lib().bjx_welford_final(eng.h, ptr(mean), ptr(m2), 8, ptr(imm)), eng.h)
    close(npy(imm), np.stack([oadapt.welford_final(w) for w in ws]), rtol=1e-5)
    assert float(mean.abs().max()) == 0.0
    # pooled block
    x = rs.standard_normal((C, D)).astype(F) * 3 + 1
    acc = rs.uniform(0, 1, C).astype(F)
    out = torch.empty(2 + 2 * D, device=DEV)
    dx, dacc = tf(x), tf(acc)   # keep both alive: the caching allocator would hand a freed block to the next tensor
    check(lib().bjx_pooled_stats(eng.h, ptr(dx), ptr(dacc), ptr(out)), eng.h)
    o = npy(out)
    assert o[1] == C
    close(o[0], acc.sum(), rtol=1e-5)
    close(o[2:2 + D], x.mean(0), rtol=1e-5)
    close(o[2 + D:], ((x - x.mean(0)) ** 2).sum(0), rtol=1e-4)


@pytest.mark.parametrize("algo", ["hmc", "nuts"])
def test_window_adaptation_per_chain_matches_oracle(algo):
    """Per-chain warm-up (what ``jax.vmap(warmup.run)`` computes), checked TEACHER-FORCED: at every one of the
    60 warm-up steps the oracle is restarted from the device's current (state, step size, inverse mass matrix,
    dual-averaging state, Welford accumulators) and must reproduce the device's next values.  (Free-running
    chains cannot be compared element-wise: early dual-averaging iterates put the integrator in its unstable
    regime, which amplifies float32 rounding differences exponentially -- BASELINE.md section 4.)"""
    from blackjax_b200._lib import check, lib, ptr
    D, C, T_ = 8, 16, 60
    scale = np.logspace(-0.5, 0.5, D)
    tgt, otgt = T.DiagGaussian(scale), otargets.DiagGaussian(scale)
    rs = np.random.default_rng(9)
    q = rs.standard_normal((C, D)).astype(F)
    ckeys = oprng.split(oprng.key(77), C)
    keys_np = oprng.split(ckeys, T_)                      # [C,T,2]  util.py:203 per chain
    if algo == "hmc":
        okern = lambda k, s, e, m: ohmc.hmc_kernel(k, s, otgt, e, m, 8)
        extra, alg = dict(num_integration_steps=8), bj.hmc
    else:
        okern = lambda k, s, e, m: onuts.nuts_kernel(k, s, otgt, e, m, 6)
        extra, alg = dict(max_num_doublings=6), bj.nuts
    kern = alg.build_kernel()
    state = alg.init(tf(q), tgt)
    eng = _engine.get_engine(state.position, tgt)
    da_state = torch.empty(C, 5, device=DEV)
    eps = torch.full((C,), 1.0, device=DEV)
    check(lib().bjx_da_init(eng.h, ptr(da_state), ptr(eps), ptr(eps)), eng.h)
    imm = torch.ones(C, D, device=DEV)
    w_mean, w_m2, w_n = torch.zeros(C, D, device=DEV), torch.zeros(C, D, device=DEV), 0
    eps_trace, ok_frac = [], []
    for t, (stage, wend) in enumerate(bj.build_schedule(T_)):
        ost = ohmc.HMCState(npy(state.position), npy(state.logdensity), npy(state.logdensity_grad))
        oeps, oimm = npy(eps).copy(), npy(imm).copy()
        onew, oinfo = okern(keys_np[:, t], ost, oeps, oadapt._PerChainDiag(oimm))
        state, info = kern(tk(keys_np[:, t]), state, tgt, eps, imm, **extra)
        torch.cuda.synchronize()
        if algo == "hmc":
            ok = npy(info.is_accepted) == oinfo.is_accepted
        else:
            ok = npy(info.num_integration_steps) == oinfo.num_integration_steps
            ok &= np.all(np.isclose(npy(state.position), onew.position, rtol=1e-4, atol=1e-5), axis=1)
        ok_frac.append(ok.mean())   # decisions on float ties may differ for single chains at wild warm-up step sizes
        assert ok.mean() >= 0.7
        close(npy(state.position)[ok], onew.position[ok], rtol=1e-4)
        close(npy(info.acceptance_rate)[ok], oinfo.acceptance_rate[ok], rtol=1e-4, scale=1.0)
        st_np, acc_np = npy(da_state).copy(), npy(info.acceptance_rate)
        odas = [oadapt.da_update(oadapt.DAState(F(r[0]), F(r[1]), int(r[2]), F(r[3]), F(r[4])), a, 0.8)
                for r, a in zip(st_np, acc_np)]
        if stage == 1:
            w_n += 1
            check(lib().bjx_welford_update(eng.h, ptr(state.position), ptr(w_mean), ptr(w_m2), w_n), eng.h)
        check(lib().bjx_da_update(eng.h, ptr(da_state), ptr(info.acceptance_rate), 0.8, ptr(eps)), eng.h)
        close(npy(eps), [np.exp(s.log_step_size) for s in odas], rtol=1e-5)
        if wend:
            m2_np, mean_np = npy(w_m2).copy(), npy(w_mean).copy()
            new_imm = torch.empty_like(imm)
            check(lib().bjx_welford_final(eng.h, ptr(w_mean), ptr(w_m2), w_n, ptr(new_imm)), eng.h)
            close(npy(new_imm), np.stack([oadapt.welford_final(oadapt.Welford(mean_np[c], m2_np[c], w_n))
                                          for c in range(C)]), rtol=1e-5)
            imm, w_n = new_imm, 0
            check(lib().bjx_da_reset(eng.h, ptr(da_state), ptr(eps)), eng.h)
        eps_trace.append(npy(eps).copy())
    assert np.mean(ok_frac) >= 0.97
    fin = torch.empty(C, device=DEV)
    check(lib().bjx_da_final(eng.h, ptr(da_state), ptr(fin)), eng.h)
    # the packaged driver runs exactly this loop: identical bits
    warm = bj.window_adaptation(alg, tgt, **extra)
    (st2, params), _ = warm.run(tk(ckeys), tf(q), T_)
    assert torch.equal(params["step_size"], fin)
    assert torch.equal(params["inverse_mass_matrix"], imm)
    assert torch.equal(st2.position, state.position)
    # and it adapts: the pooled step size lands in a sane range for this target (stable below 2*min scale)
    assert 0.05 < float(np.median(npy(fin))) < 2.5


def test_window_adaptation_shared_matches_oracle_and_recovers_scales():
    D, C, T_ = 16, 256, 120
    scale = np.logspace(-0.5, 0.5, D)
    tgt, otgt = T.DiagGaussian(scale), otargets.DiagGaussian(scale)
    rs = np.random.default_rng(10)
    q = rs.standard_normal((C, D)).astype(F)
    okern = lambda k, s, t, e, m, **kw: onuts.nuts_kernel(k, s, t, e, m, 5)
    ost, oeps, oimm, ohist = oadapt.window_adaptation_run(okern, otgt, oprng.key(5), q, T_, shared=True)
    warm = bj.window_adaptation(bj.nuts, tgt, shared=True, max_num_doublings=5)
    (st, params), hist = warm.run(bj.random.key(5, DEV), tf(q), T_)
    # pooled statistics over 256 chains damp single-chain decision flips: the two runs track closely
    assert abs(params["step_size"] / float(oeps) - 1) < 0.05
    np.testing.assert_allclose(npy(params["inverse_mass_matrix"]), oimm, rtol=0.1)
    np.testing.assert_allclose(npy(params["inverse_mass_matrix"]), scale ** 2, rtol=0.35)
    np.testing.assert_allclose(np.array(hist[:20]), ohist[:20], rtol=2e-3)


def test_window_adaptation_shared_dense_recovers_covariance():
    # welford_dense recipe, chain-pooled (staged_adaptation.py:906-966 with a dense metric core): the adapted dense
    # inverse mass matrix must recover the target covariance; the oracle run tracks it.
    D, C, T_ = 6, 512, 150
    from test_oracle_kat import COV6
    cov = COV6
    tgt, otgt = T.DenseGaussian(np.linalg.inv(cov)), otargets.DenseGaussian(np.linalg.inv(cov))
    rs = np.random.default_rng(11)
    q = rs.standard_normal((C, D)).astype(F)
    okern = lambda k, s, t, e, m, **kw: onuts.nuts_kernel(k, s, t, e, m, 6)
    ost, oeps, oimm, ohist = oadapt.window_adaptation_run(okern, otgt, oprng.key(6), q, T_, shared=True,
                                                          is_mass_matrix_diagonal=False)
    warm = bj.window_adaptation(bj.nuts, tgt, is_mass_matrix_diagonal=False, shared=True, max_num_doublings=6)
    (st, params), hist = warm.run(bj.random.key(6, DEV), tf(q), T_)
    imm = npy(params["inverse_mass_matrix"])
    assert imm.shape == (D, D)
    np.testing.assert_allclose(imm, cov, rtol=0.25, atol=0.25)
    np.testing.assert_allclose(imm, oimm, rtol=0.15, atol=0.15)
    assert abs(params["step_size"] / float(oeps) - 1) < 0.15
    np.testing.assert_allclose(np.array(hist[:10]), ohist[:10], rtol=5e-3)
    # the pooled dense block itself, against numpy
    from blackjax_b200._lib import check, lib, ptr
    eng = _engine.get_engine(st.position, tgt, max_tree_depth=6)
    out = torch.empty(2 + D + D * D, device=DEV)
    acc = torch.rand(C, device=DEV)
    check(lib().bjx_pooled_stats_dense(eng.h, ptr(st.position), ptr(acc), ptr(out)), eng.h)
    x = npy(st.position).astype(np.float64)
    o = npy(out)
    close(o[2:2 + D], x.mean(0), rtol=1e-5)
    close(o[2 + D:].reshape(D, D), (x - x.mean(0)).T @ (x - x.mean(0)), rtol=1e-4)
    # per-chain dense adaptation ([C, D, D] metrics in the warp kernels) stops at 64 dims; beyond, the pooled recipe above
    with pytest.raises(NotImplementedError):
        bj.window_adaptation(bj.nuts, T.StdNormal(100), is_mass_matrix_diagonal=False).run(
            bj.random.key(0, DEV), torch.zeros(4, 100, device=DEV), 30)


# ---------------------------------------------------------------------------------------------------------
# committed golden fixtures (tests/golden/hmc_nuts_golden.npz, generated by the oracle -- see make_golden.py)
# ---------------------------------------------------------------------------------------------------------
def test_device_matches_committed_golden():
    import os
    G = np.load(os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "hmc_nuts_golden.npz"))
    # A: HMC config-1 shape
    tgt = T.StdNormal(100)
    new, info = bj.hmc.build_kernel(full_info=True)(tk(G["A_keys"]), bj.hmc.init(tf(G["A_q"]), tgt), tgt, 0.2,
                                                    torch.ones(100, device=DEV), 10)
    assert (npy(info.is_accepted) == G["A_accepted"]).all()
    close(npy(new.position), G["A_pos"])
    close(npy(info.energy), G["A_energy"], rtol=1e-5, scale=np.max(np.abs(G["A_energy"])))
    close(npy(info.acceptance_rate), G["A_acc"], rtol=1e-4, scale=1.0)
    close(npy(info.momentum), G["A_momentum"], rtol=3e-6)
    # B: NUTS funnel
    tgt = T.Funnel(16)
    new, info = bj.nuts.build_kernel(max_tree_depth=8)(tk(G["B_keys"]), bj.nuts.init(tf(G["B_q"]), tgt), tgt, 0.2,
                                                       torch.ones(16, device=DEV), 8)
    assert (npy(info.num_integration_steps) == G["B_n"]).all()
    assert (npy(info.num_trajectory_expansions) == G["B_depth"]).all()
    assert (npy(info.is_turning) == G["B_turn"]).all() and (npy(info.is_divergent) == G["B_div"]).all()
    close(npy(new.position), G["B_pos"], rtol=1e-4)
    close(npy(info.acceptance_rate), G["B_acc"], rtol=1e-4, scale=1.0)
    # C: multinomial HMC
    tgt = T.DiagGaussian(G["C_scale"])
    new, info = bj.mhmc.build_kernel()(tk(G["C_keys"]), bj.mhmc.init(tf(G["C_q"]), tgt), tgt, 0.15, tf(G["C_imm"]), 7)
    close(npy(new.position), G["C_pos"], rtol=1e-4)
    close(npy(info.acceptance_rate), G["C_acc"], rtol=1e-4, scale=1.0)
    # D: NUTS, dense metric, banana
    tgt = T.Banana()
    new, info = bj.nuts.build_kernel(max_tree_depth=6)(tk(G["D_keys"]), bj.nuts.init(tf(G["D_q"]), tgt), tgt, 0.1,
                                                       tf(G["D_imm"]), 6)
    assert (npy(info.num_integration_steps) == G["D_n"]).all()
    close(npy(new.position), G["D_pos"], rtol=1e-4)


# ---------------------------------------------------------------------------------------------------------
# free-running chains, compared distributionally (tests/mcmc/test_sampling.py:1343-1471: multi-chain MCSE test on a
# correlated 2-D normal, HMC & NUTS, diagonal & dense mass matrix)
# ---------------------------------------------------------------------------------------------------------
@pytest.mark.parametrize("algo", ["hmc", "nuts", "mhmc"])
@pytest.mark.parametrize("dense_metric", [False, True])
def test_multichain_moments_correlated_normal(algo, dense_metric):
    cov = np.array([[1.0, 0.6 * np.sqrt(2.0)], [0.6 * np.sqrt(2.0), 2.0]])       # corr 0.6, variances (1, 2)
    tgt = T.DenseGaussian(np.linalg.inv(cov))
    C, T_ = 4096, 250
    imm = tf(cov.astype(F)) if dense_metric else tf(np.array([1.0, 2.0], F))
    if algo == "hmc":
        alg = bj.hmc(tgt, 0.45, imm, 12)
    elif algo == "mhmc":
        alg = bj.mhmc(tgt, 0.45, imm, 12)
    else:
        alg = bj.nuts(tgt, 0.45, imm)
    st = alg.init(torch.zeros(C, 2, device=DEV))
    keys = bj.random.split(bj.random.key(8456, DEV), T_)
    s1 = torch.zeros(2, dtype=torch.float64, device=DEV)
    s2 = torch.zeros(2, 2, dtype=torch.float64, device=DEV)
    n = 0
    for t in range(T_):
        st, info = alg.step(keys[t], st)
        if t >= 50:
            x = st.position.double()
            s1 += x.sum(0)
            s2 += x.T @ x
            n += C
    mean = (s1 / n).cpu().numpy()
    c = (s2 / n).cpu().numpy() - np.outer(mean, mean)
    # 4096 chains x 200 kept draws; autocorrelation leaves an effective sample size well above 1e5
    assert np.all(np.abs(mean) < 0.02), mean
    np.testing.assert_allclose(np.diag(c), [1.0, 2.0], rtol=0.03)
    assert abs(c[0, 1] / np.sqrt(c[0, 0] * c[1, 1]) - 0.6) < 0.02


# ---------------------------------------------------------------------------------------------------------
# full BASELINE sizes: size-independent properties
# ---------------------------------------------------------------------------------------------------------
def test_fullsize_leapfrog_reversibility_and_energy_65536x1024():
    C, D, L = 65536, 1024, 50
    s = np.logspace(-0.5, 0.5, D)
    tgt = T.DiagGaussian(s)
    eng = _engine.Engine(DEV, C, D, tgt)
    imm = torch.from_numpy((s ** 2).astype(F)).to(DEV)
    eng.set_metric(imm)
    g_ = torch.Generator(device=DEV).manual_seed(0)
    q0 = torch.randn(C, D, device=DEV, generator=g_) * torch.from_numpy(s.astype(F)).to(DEV)
    p0 = eng.sample_momentum(bj.random.split(bj.random.key(1, DEV), C))
    q, p = q0.clone(), p0.clone()
    logp, g = eng.init_state(q)
    e0 = eng.energy(p, logp)
    eng.leapfrog_(q, p, logp, g, 0.1, L)
    e1 = eng.energy(p, logp)
    # symplectic integrator: energy error O(eps^2) and bounded
    assert float((e1 - e0).abs().max() / e0.abs().mean()) < 5e-3
    # time reversibility: flip momentum, integrate back, recover the start (float32 round-off only)
    p.neg_()
    eng.leapfrog_(q, p, logp, g, 0.1, L)
    assert float((q - q0).abs().max()) < 5e-4 * float(q0.abs().max())
    assert float((p + p0).abs().max()) < 5e-4 * float(p0.abs().max())
    # n_steps composition: 50 one-step launches == one 50-step launch, bit for bit
    qa, pa = q0.clone(), p0.clone()
    la, ga = eng.init_state(qa)
    qb, pb = q0.clone(), p0.clone()
    lb, gb = eng.init_state(qb)
    eng.leapfrog_(qa, pa, la, ga, 0.1, 5)
    for _ in range(5):
        eng.leapfrog_(qb, pb, lb, gb, 0.1, 1)
    assert torch.equal(qa, qb) and torch.equal(pa, pb) and torch.equal(ga, gb)


def test_fullsize_hmc_65536x1024_detailed_balance_stats():
    C, D, L = 65536, 1024, 50
    tgt = T.StdNormal(D)
    imm = torch.ones(D, device=DEV)
    g_ = torch.Generator(device=DEV).manual_seed(1)
    q = torch.randn(C, D, device=DEV, generator=g_)
    st = bj.hmc.init(q, tgt)
    kern = bj.hmc.build_kernel()
    keys = bj.random.split(bj.random.key(2, DEV), 3)
    acc = []
    for t in range(3):
        st, info = kern(keys[t], st, tgt, 0.12, imm, L)
        acc.append(float(info.acceptance_rate.mean()))
        # accepted rows moved, rejected rows kept the old state (checked through the log-density identity)
        lp = -0.5 * (st.position.double() ** 2).sum(1)
        assert float((lp - st.logdensity.double()).abs().max()) < 1e-2
    assert 0.6 < np.mean(acc) < 0.999
    # stationary: started from the target, the second moment stays 1 within Monte-Carlo error
    assert abs(float(st.position.var()) - 1.0) < 5e-3


def test_fullsize_nuts_funnel_65536x128():
    # BASELINE config 3: NUTS, Neal's funnel D=128, 65536 chains, diag mass, max_tree_depth=10
    C, D = 65536, 128
    tgt = T.Funnel(D)
    imm = torch.ones(D, device=DEV)
    q = 0.1 * bj.random.normal(bj.random.split(bj.random.key(0, DEV), C), (D,))
    st = bj.nuts.init(q, tgt)
    kern = bj.nuts.build_kernel()
    st2, info = kern(bj.random.key(1, DEV), st, tgt, 0.1, imm, 10)
    n = info.num_integration_steps
    d = info.num_trajectory_expansions
    assert int(n.min()) >= 1 and int(n.max()) <= 1023
    # a tree of depth d holds between 2^(d-1) and 2^d - 1 leaves (last sub-tree may stop early)
    assert bool(((n <= (2 ** d.long()) - 1) & (n >= 2 ** (d.long() - 1))).all())
    ar = info.acceptance_rate
    # exp(logaddexp-accumulated log sum)/n can exceed 1 by float32 rounding when every leaf has min(w,0)=0
    assert bool(((ar >= 0) & (ar <= 1 + 1e-5)).all())
    # returned state is self-consistent: logdensity/grad are those of the returned position
    lp, g = _engine.get_engine(st2.position, tgt).init_state(st2.position)
    assert float((lp - st2.logdensity).abs().max()) < 1e-2 * (1 + float(lp.abs().max()) * 1e-3)
    torch.testing.assert_close(g, st2.logdensity_grad, rtol=1e-4, atol=1e-3)
    # identical keys + identical state => identical result (determinism, no atomics in the data path)
    st3, info3 = kern(bj.random.key(1, DEV), st, tgt, 0.1, imm, 10)
    assert torch.equal(st2.position, st3.position) and torch.equal(n, info3.num_integration_steps)
