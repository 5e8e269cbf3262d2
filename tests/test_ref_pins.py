"""The CPU oracle against vectors produced by the reference's OWN source.

tests/golden/ref_*.npz were written by oracle/tf_shim/make_ref_golden.py: zhusuan/hmc.py and
zhusuan/sgmcmc.py of the reference checkout, imported unmodified and executed on the NumPy
stand-in for the TF-1.x graph API (oracle/tf_shim/tensorflow.py), with every random draw
injected.  The state machine (step-size search hmc.py:279-333, dual averaging hmc.py:56-90, mass
estimator hmc.py:93-158, the SG-MCMC update rules sgmcmc.py:183-470) therefore comes from the
reference's code, not from the restatement in oracle/.  Here:

* oracle/hmc.py and oracle/sgmcmc.py must reproduce those vectors (float32: bit-exact for the
  element-wise models, rounding of the matmul summation order for the dense one);
* the committed files must equal, bit for bit, the reference run whose digests are stored in
  tests/golden/ref_digests.json (and, where ZHUSUAN_REFERENCE names a checkout of the original
  ZhuSuan, a fresh run of it).

CPU only.
"""
import os
import sys

import numpy as np
import pytest

from oracle import hmc as OH
from oracle import models as OM
from oracle import sgmcmc as OS

HERE = os.path.dirname(os.path.abspath(__file__))
GOLD = os.path.join(HERE, "golden")
SHIM = os.path.join(os.path.dirname(HERE), "oracle", "tf_shim")
REF = os.environ.get("ZHUSUAN_REFERENCE", "")
have_ref = bool(REF) and os.path.isfile(os.path.join(REF, "zhusuan", "hmc.py"))


def _model(g):
    if "P" in g.files:
        return OM.DenseGaussian(g["P"].astype(np.float32), g["mu"], float(g["const"]))
    return OM.DiagGaussian(np.zeros_like(g["std"]), g["std"])


@pytest.mark.parametrize("name,tol", [("ref_hmc_diag", 0.0), ("ref_hmc_dense32", 3e-5),
                                      ("ref_hmc_dense64", 3e-5)])
def test_oracle_hmc_reproduces_reference_run(name, tol):
    g = np.load(os.path.join(GOLD, name + ".npz"))
    model = _model(g)
    h = OH.HMC(step_size=float(g["cfg_step_size"]), n_leapfrogs=int(g["cfg_n_leapfrogs"]),
               adapt_step_size=True, target_acceptance_rate=float(g["cfg_target_acceptance_rate"]),
               adapt_mass=True, mass_collect_iters=int(g["cfg_mass_collect_iters"]),
               mass_decay=float(g["cfg_mass_decay"]))
    q = [g["q0"].copy()]
    n_live = 0
    for i in range(g["q"].shape[0]):
        adapt = i < int(g["n_adapt"])
        q, info = h.step(q, model.logp, model.grad, [g["noise_p"][i]], g["noise_u"][i],
                         adapt_step_size=adapt, adapt_mass=adapt)
        cmp = lambda a, b, what: np.testing.assert_allclose(
            a, b, rtol=tol, atol=tol * 1e-1, err_msg="%s iteration %d %s" % (name, i, what))
        np.testing.assert_array_equal(info.if_accept.astype(np.int32), g["accept"][i])
        cmp(info.init_momentum[0], g["p0"][i], "p0")
        cmp(info.orig_log_prob, g["lp0"][i], "lp0")
        cmp(info.orig_hamiltonian, g["h0"][i], "h0")
        cmp(info.acceptance_rate, g["acc"][i], "acc")
        cmp(info.log_prob, g["lp"][i], "lp")
        cmp(np.float32(info.updated_step_size), g["step_size"][i], "step_size")
        np.testing.assert_allclose(q[0], g["q"][i], rtol=tol * 30, atol=tol,
                                   err_msg="%s iteration %d q" % (name, i))
        live = g["acc"][i] > 1e-6        # a diverged proposal's energy is chaotic in float32
        cmp(info.hamiltonian[live], g["h1"][i][live], "h1")
        n_live += int(live.sum())
    # the fixture exercises both regimes: diverging step-size overshoots and healthy iterations
    assert 0.3 * g["acc"].size < n_live < g["acc"].size


SG = {
    "sgld": (OS.SGLD, dict(learning_rate=0.01)),
    "psgld": (OS.PSGLD, dict(learning_rate=0.01)),
    "sghmc1": (OS.SGHMC, dict(learning_rate=0.01, friction=0.3, variance_estimate=0.02,
                              n_iter_resample_v=3, second_order=False)),
    "sghmc2": (OS.SGHMC, dict(learning_rate=0.01, friction=0.3, variance_estimate=0.02,
                              n_iter_resample_v=3, second_order=True)),
    "sgnht1v": (OS.SGNHT, dict(learning_rate=0.01, variance_extra=0.1, tune_rate=2.,
                               n_iter_resample_v=4, second_order=False, use_vector_alpha=True)),
    "sgnht2v": (OS.SGNHT, dict(learning_rate=0.01, variance_extra=0.1, tune_rate=2.,
                               n_iter_resample_v=4, second_order=True, use_vector_alpha=True)),
    "sgnht1s": (OS.SGNHT, dict(learning_rate=0.01, variance_extra=0.1, tune_rate=2.,
                               n_iter_resample_v=None, second_order=False,
                               use_vector_alpha=False)),
    "sgnht2s": (OS.SGNHT, dict(learning_rate=0.01, variance_extra=0.1, tune_rate=2.,
                               n_iter_resample_v=None, second_order=True,
                               use_vector_alpha=False)),
}


@pytest.mark.parametrize("name", sorted(SG))
def test_oracle_sgmcmc_reproduces_reference_run(name):
    g = np.load(os.path.join(GOLD, "ref_sgmcmc.npz"))
    model = OM.DiagGaussian(g["mean"], g["std"])
    cls, kw = SG[name]
    s = cls(**kw)
    q = [g["q0"].copy()]
    if hasattr(s, "init_v"):
        s.init_v([g[name + "_v0"]])
    tol = 1e-6 if name == "psgld" else 0.0      # x**2 (reference) vs x*x: one rounding
    for t in range(g[name + "_q"].shape[0]):
        if hasattr(s, "init_v"):
            q, info = s.step(q, model.grad, [g[name + "_resample"][t]], [g[name + "_noise"][t]])
        else:
            q, info = s.step(q, model.grad, [g[name + "_noise"][t]])
        np.testing.assert_allclose(q[0], g[name + "_q"][t], rtol=tol, atol=tol)
        if name + "_mean_k" in g.files:
            np.testing.assert_allclose(np.asarray(info["mean_k"][0], np.float32),
                                       g[name + "_mean_k"][t], rtol=1e-6)
        if name + "_alpha" in g.files:
            np.testing.assert_allclose(np.asarray(info["alpha"][0], np.float32).reshape(-1),
                                       g[name + "_alpha"][t].reshape(-1), rtol=1e-6)
    # the schedule of momentum re-draws is the reference's own (t % n == 0, counted from 0)
    n = kw.get("n_iter_resample_v")
    want = [2 if (n and t % n == 0) else 1 for t in range(g[name + "_q"].shape[0])]
    assert g[name + "_n_used"].tolist() == want


def test_oracle_ais_reproduces_reference_run():
    """class AIS of zhusuan/evaluation.py:57-172 driving the reference's HMC (prior draws, HMC noise
    injected): per-chain log-weights and the bound."""
    from oracle import evaluation as OE
    g = np.load(os.path.join(GOLD, "ref_ais.npz"))
    x, s = g["x"], float(g["s"])
    c, f32 = -0.5 * np.log(2 * np.pi), np.float32
    lp = lambda q: (c - 0.5 * q[0].astype(np.float64) ** 2).sum(-1).astype(f32)
    gp = lambda q: [(-q[0]).astype(f32)]
    lj = lambda q: (lp(q).astype(np.float64) + (c - np.log(s) - 0.5 * (
        (x - q[0].astype(np.float64)) / s) ** 2).sum(-1)).astype(f32)
    gj = lambda q: [(-q[0] + (x - q[0]) / (s * s)).astype(f32)]
    oh = OH.HMC(step_size=0.2, n_leapfrogs=3, adapt_step_size=True, target_acceptance_rate=0.7)
    nt, na = int(g["n_temperatures"]), int(g["n_adapt"])
    oa = OE.AIS(lp, gp, lj, gj, oh, n_temperatures=nt, n_adapt=na)
    est, lw = oa.run([[g["init"][0]], [g["init"][1]]],
                     lambda k: ([g["noise_p"][k]], g["noise_u"][k]), adapt_flags=(True, False))
    np.testing.assert_allclose(lw, g["log_weights"], rtol=1e-5, atol=5e-6)
    assert abs(est - float(g["bound"])) < 5e-6
    np.testing.assert_allclose([oa.schedule(t) for t in range(nt + 1)], g["schedule"], rtol=1e-12)


def test_reference_run_equals_oracle_made_fixtures():
    """The round-1 fixtures (written by the oracle) and the reference-run ones share seeds and
    configurations: same inputs, same outputs."""
    for a, b, tol in (("hmc_diag", "ref_hmc_diag", 0.0), ("hmc_dense", "ref_hmc_dense32", 3e-5)):
        o, r = np.load(os.path.join(GOLD, a + ".npz")), np.load(os.path.join(GOLD, b + ".npz"))
        np.testing.assert_array_equal(o["noise_p"], r["noise_p"])
        np.testing.assert_array_equal(o["q0"], r["q0"])
        np.testing.assert_array_equal(o["accept"], r["accept"])
        for k in ("acc", "step_size", "lp", "lp0", "h0", "p0"):
            np.testing.assert_allclose(o[k], r[k], rtol=tol, atol=tol * 1e-1, err_msg=a + " " + k)
        np.testing.assert_allclose(o["q"], r["q"], rtol=tol * 30, atol=tol)


def test_committed_vectors_are_what_the_reference_code_produces():
    """tests/golden/ref_digests.json: digests of every array of the reference's own run
    (make_ref_golden.py::reference_digests).  Every committed ref_*.npz must hold exactly those
    arrays, bit for bit; where ZHUSUAN_REFERENCE names a checkout of the original ZhuSuan, its
    source is run again and must reproduce the same digests."""
    import json
    want = json.load(open(os.path.join(GOLD, "ref_digests.json")))
    # ref_hmc_diag: the model of examples/toy_examples/gaussian.py built with the reference's own
    # meta_bayesian_net / BayesianNet.normal / Normal.log_prob; dense32 / dense64: a callable
    assert sorted(want) == ["ref_ais", "ref_bnn_sghmc", "ref_hmc_dense32", "ref_hmc_dense64",
                            "ref_hmc_diag", "ref_lntm_hmc", "ref_sgmcmc", "ref_vae"]
    sys.path.insert(0, SHIM)
    saved = {k: sys.modules.get(k) for k in ("tensorflow", "zhusuan")}
    try:
        import make_ref_golden as M
        for name, digests in want.items():
            g = np.load(os.path.join(GOLD, name + ".npz"))
            assert sorted(g.files) == sorted(digests), name
            for k in g.files:
                assert M.array_digest(g[k]) == digests[k], name + " " + k
        if have_ref:
            assert M.reference_digests() == want
            import zhusuan.hmc
            assert os.path.realpath(zhusuan.hmc.__file__).startswith(os.path.realpath(REF))
    finally:
        sys.path.remove(SHIM)
        for k in [m for m in sys.modules if m == "tensorflow" or m.startswith("zhusuan")]:
            del sys.modules[k]
        for k, v in saved.items():
            if v is not None:
                sys.modules[k] = v


def _vae_terms_torch(g, eps, reparameterized, dtype):
    """An independent restatement (torch autograd, CPU) of the VAE the fixture was produced on
    (iwae.py:23-44): returns the weights (leaf tensors), log_joint [K, N] and log q [K, N]."""
    import torch
    names = [str(n) for n in g["names"]]
    w = {n: torch.tensor(g["w_" + n], dtype=dtype, requires_grad=True) for n in names}
    x = torch.tensor(g["x"], dtype=dtype)
    e = torch.tensor(eps, dtype=dtype)
    c = -0.5 * np.log(2 * np.pi)
    relu = torch.relu
    h = relu(x @ w["q0_w"] + w["q0_b"])
    h = relu(h @ w["q1_w"] + w["q1_b"])
    mean, logstd = h @ w["q2_w"] + w["q2_b"], h @ w["q3_w"] + w["q3_b"]
    if reparameterized:
        z = mean + torch.exp(logstd) * e
    else:                                   # Normal._sample with stop_gradient (univariate.py:163-165)
        z = (mean + torch.exp(logstd) * e).detach()
    log_q = (c - logstd - 0.5 * torch.exp(-2 * logstd) * (z - mean) ** 2).sum(-1)
    log_pz = (c - 0.5 * z ** 2).sum(-1)
    h = relu(z @ w["g0_w"] + w["g0_b"])
    h = relu(h @ w["g1_w"] + w["g1_b"])
    logits = h @ w["g2_w"] + w["g2_b"]
    log_px = -(torch.clamp(logits, min=0) - logits * x +
               torch.log1p(torch.exp(-logits.abs()))).sum(-1)
    return w, log_pz + log_px, log_q


def test_reference_run_vae_objectives_against_independent_autograd():
    """tests/golden/ref_vae.npz = the reference's own framework / distributions / variational code
    (importance_weighted_objective, elbo, .sgvb(), .reinforce()) on the NumPy TF stand-in.  Its
    values AND its tf.gradients results must agree with torch autograd on a restatement of the
    same model -- this vouches for the stand-in's reverse-mode differentiation."""
    import torch
    g = np.load(os.path.join(GOLD, "ref_vae.npz"))
    names = [str(n) for n in g["names"]]
    K = g["eps"].shape[0]
    w, lj, lq = _vae_terms_torch(g, g["eps"], True, torch.float64)
    np.testing.assert_allclose(lj.detach().numpy(), g["log_joint"], rtol=2e-6, atol=2e-6)
    np.testing.assert_allclose(-lq.detach().numpy(), g["entropy"], rtol=2e-6, atol=2e-6)
    bound = torch.logsumexp(lj - lq, 0) - np.log(K)
    np.testing.assert_allclose(bound.detach().numpy(), g["iw_bound"], rtol=2e-6)
    cost = -bound.mean()
    grads = torch.autograd.grad(cost, [w[n] for n in names], retain_graph=True)
    for n, gr in zip(names, grads):
        np.testing.assert_allclose(gr.numpy(), g["iw_grad_" + n], rtol=2e-4, atol=2e-6, err_msg=n)
    ecost = -(lj - lq).mean(0).mean()
    np.testing.assert_allclose(float(ecost), float(g["elbo_cost"]), rtol=2e-6)
    grads = torch.autograd.grad(ecost, [w[n] for n in names])
    for n, gr in zip(names, grads):
        np.testing.assert_allclose(gr.numpy(), g["elbo_grad_" + n], rtol=2e-4, atol=2e-6,
                                   err_msg=n)
    # REINFORCE, three steps: baseline = the moving mean BEFORE the step's update; update =
    # TF's zero-debiased assign_moving_average (oracle/variational.py)
    from oracle import variational as OV
    state, mm_prev = None, 0.0
    for t in range(3):
        w, lj, lq = _vae_terms_torch(g, g["rf_eps"][t], False, torch.float64)
        signal = (lj - lq).detach()
        cost = (-lj - (signal - mm_prev) * lq).mean(0).mean()
        np.testing.assert_allclose(float(cost), float(g["rf_cost"][t]), rtol=2e-5)
        grads = torch.autograd.grad(cost, [w[n] for n in names[:8]])
        for n, gr in zip(names[:8], grads):
            np.testing.assert_allclose(gr.numpy(), g["rf_grad_" + n][t], rtol=5e-4, atol=5e-5,
                                       err_msg="step %d %s" % (t, n))
        mm_prev, state = OV.zero_debiased_moving_average(state, float(signal.mean()), 0.8)
        np.testing.assert_allclose(mm_prev, float(g["rf_moving_mean"][t]), rtol=2e-6)
    # VIMCO (monte_carlo.py:166-227) and self-normalised importance (inclusive_kl.py:119-151)
    w, lj, lq = _vae_terms_torch(g, g["eps"], False, torch.float64)
    lw = lj - lq
    lwd = lw.detach()
    mean_except = (lwd.sum(0, keepdim=True) - lwd) / (K - 1)
    x_ex = lwd.t().unsqueeze(1).repeat(1, K, 1)                       # [N, k, j] = lw[j, n]
    idx = torch.arange(K)
    x_ex[:, idx, idx] = mean_except.t()
    control = (torch.logsumexp(x_ex, -1) - np.log(K)).t()             # [K, N]
    lme = torch.logsumexp(lw, 0) - np.log(K)
    signal = lme.detach().unsqueeze(0) - control
    cost = (-(lq * signal).sum(0) - lme).mean()
    np.testing.assert_allclose(float(cost.detach()), float(g["vimco_cost"]), rtol=2e-6)
    grads = torch.autograd.grad(cost, [w[n] for n in names], retain_graph=True)
    for n, gr in zip(names, grads):
        np.testing.assert_allclose(gr.numpy(), g["vimco_grad_" + n], rtol=5e-4, atol=5e-6,
                                   err_msg="vimco " + n)
    wt = torch.softmax(lwd, 0)
    cost = (-(wt * lq).sum(0)).mean()
    np.testing.assert_allclose(float(cost.detach()), float(g["importance_cost"]), rtol=2e-6)
    grads = torch.autograd.grad(cost, [w[n] for n in names[:8]])
    for n, gr in zip(names[:8], grads):
        np.testing.assert_allclose(gr.numpy(), g["importance_grad_" + n], rtol=5e-4, atol=5e-6,
                                   err_msg="importance " + n)


def test_oracle_bnn_sghmc_reproduces_reference_run():
    """tests/golden/ref_bnn_sghmc.npz: config 4's model (bnn_sgmcmc.py:19-35, log_joint 74-77) on
    the reference's BayesianNet + SGHMC classes (second order, momentum re-draws at t = 0, 3).
    oracle/models.py::BNN (hand-derived gradient) + oracle/sgmcmc.py::SGHMC must follow it."""
    g = np.load(os.path.join(GOLD, "ref_bnn_sghmc.npz"))
    ls0, ls1 = g["logstd0"], g["logstd1"]

    class M(OM.BNN):                      # per-weight prior log-stddevs (bnn_sgmcmc.py:71)
        def grad(self, qs):
            g0, g1 = OM.BNN.grad(self, qs)
            g0 = g0 + np.exp(-2 * self.ls0) * qs[0] - np.exp(-2 * ls0) * qs[0]
            g1 = g1 + np.exp(-2 * self.ls1) * qs[1] - np.exp(-2 * ls1) * qs[1]
            return [g0, g1]
    for dtype, tol in ((np.float32, 2e-5), (np.float64, 2e-5)):
        om = M(g["x"].astype(dtype), g["y"].astype(dtype), int(g["n_train"]), dtype=dtype)
        s = OS.SGHMC(dtype=dtype, learning_rate=float(g["cfg_learning_rate"]),
                     friction=float(g["cfg_friction"]),
                     variance_estimate=float(g["cfg_variance_estimate"]),
                     n_iter_resample_v=int(g["cfg_n_iter_resample_v"]), second_order=True)
        s.init_v([g["v0_0"].astype(dtype), g["v0_1"].astype(dtype)])
        q = [g["w0_init"].astype(dtype), g["w1_init"].astype(dtype)]
        for t in range(g["w0"].shape[0]):
            q, info = s.step(q, om.grad, [g["resample0"][t], g["resample1"][t]],
                             [g["noise0"][t], g["noise1"][t]])
            np.testing.assert_allclose(q[0], g["w0"][t], rtol=tol * 10, atol=tol)
            np.testing.assert_allclose(q[1], g["w1"][t], rtol=tol * 10, atol=tol)
            np.testing.assert_allclose(info["mean_k"][0], g["mean_k0"][t], rtol=1e-3)
            np.testing.assert_allclose(info["mean_k"][1], g["mean_k1"][t], rtol=1e-3)
    assert g["n_used"].tolist() == [4, 2, 2, 4, 2]


def test_oracle_lntm_hmc_follows_reference_run():
    """tests/golden/ref_lntm_hmc.npz: config 5's E-step (lntm_mcem.py:33-48, e_obj 97-98) on the
    reference's BayesianNet, UnnormalizedMultinomial and HMC (two chain axes).  The oracle's dense
    restatement (oracle/models.py::LNTM, analytic gradient) driving oracle/hmc.py must follow it:
    identical accept decisions away from u ~ acc, state and step sizes to float32 rounding."""
    g = np.load(os.path.join(GOLD, "ref_lntm_hmc.npz"))
    om = OM.LNTM(g["x"], g["beta"], g["eta_mean"], g["eta_logstd"], dtype=np.float32)
    oh = OH.HMC(step_size=float(g["cfg_step_size"]), n_leapfrogs=int(g["cfg_n_leapfrogs"]),
                adapt_step_size=True, target_acceptance_rate=float(g["cfg_target_acceptance_rate"]))
    q = [g["eta0"].copy()]
    for i in range(g["eta"].shape[0]):
        with np.errstate(all="ignore"):
            q, info = oh.step(q, om.logp, om.grad, [g["noise_p"][i]], g["noise_u"][i], True, False)
        np.testing.assert_allclose(info.orig_log_prob, g["lp0"][i], rtol=2e-5, atol=2e-4)
        np.testing.assert_allclose(info.acceptance_rate, g["acc"][i], rtol=2e-3, atol=2e-4)
        np.testing.assert_allclose(np.float32(info.updated_step_size), g["step_size"][i],
                                   rtol=2e-4)
        near = np.abs(g["noise_u"][i] - g["acc"][i]) < 1e-3
        np.testing.assert_allclose(q[0][~near], g["eta"][i][~near], rtol=1e-3, atol=1e-4)
        q = [g["eta"][i].copy()]             # continue from the reference's state


@pytest.mark.parametrize("name", ["hmc_dense64", "hmc_dense1024"])
def test_reference_hmc_itself_passes_the_l50_protocol(name):
    """The L = 50 adaptive fixtures the benchmarked CUDA kernels are replayed against
    (tests/golden/hmc_dense64.npz, hmc_dense1024.npz: written by the float32 oracle, with a
    float64 re-evaluation of every iteration) versus THE REFERENCE'S OWN hmc.py run on the TF
    stand-in under the same protocol (tests/golden/ref_<name>_l50.npz, written by
    make_ref_golden.py::write_reference_hmc_big), at the benchmark's shape (D = 1024, L = 50,
    both step-size searches, mass != 1): every accept decision, the step-size trajectory
    exactly, Hamiltonians within 1e-6 of float64."""
    o = np.load(os.path.join(GOLD, "ref_%s_l50.npz" % name))
    g = np.load(os.path.join(GOLD, name + ".npz"))
    accept = (g["noise_u"] < o["acc"]).astype(np.int32)
    np.testing.assert_array_equal(accept, g["accept"])
    np.testing.assert_array_equal(np.asarray(o["step_size"], np.float32), g["step_size"])
    np.testing.assert_allclose(o["h0"], g["h0_64"], rtol=1e-6)
    live = g["acc64"] > 1e-6
    assert 0.4 * live.size < live.sum() < live.size      # healthy and diverging iterations
    np.testing.assert_allclose(o["h1"][live], g["h1_64"][live], rtol=1e-6)
    np.testing.assert_allclose(o["acc"], g["acc64"], atol=1e-3)
    np.testing.assert_allclose(o["acc"], g["acc"], atol=1e-3)           # the float32 oracle's
    np.testing.assert_allclose(o["lp0"], g["lp0"], rtol=1e-6)
