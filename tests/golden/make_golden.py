"""Generates tests/golden/*.npz from the CPU oracle (run from the repo root:
``python tests/golden/make_golden.py``).

The reference holds NO golden vectors for an HMC trajectory, accept decision,
step-size / mass adaptation or any SG-MCMC update (tests/test_mcmc.py is
statistical only) and TensorFlow cannot be installed here, so these vectors
are oracle-generated ("parity unpinned" by the reference, see
oracle/__init__.py).  They freeze the oracle: tests/test_oracle_hmc.py checks
the oracle still reproduces them, and the GPU parity tests replay the same
injected noise through the CUDA path.
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle import hmc as OH            # noqa: E402
from oracle import sgmcmc as OS         # noqa: E402
from oracle import models as OM         # noqa: E402

HERE = os.path.dirname(os.path.abspath(__file__))


def run_hmc(model, q0, n_iters, n_adapt, rng, **kw):
    h = OH.HMC(**kw)
    q = [q0.copy()]
    rec = {k: [] for k in ("noise_p", "noise_u", "q", "acc", "accept",
                           "step_size", "eps_used", "mass", "lp", "h0", "h1",
                           "lp0", "p0")}
    for i in range(n_iters):
        npz = rng.standard_normal(q0.shape).astype(np.float32)
        nu = rng.random(q0.shape[0]).astype(np.float32)
        adapt = i < n_adapt
        q, info = h.step(q, model.logp, model.grad, [npz], nu,
                         adapt_step_size=adapt, adapt_mass=adapt)
        rec["noise_p"].append(npz)
        rec["noise_u"].append(nu)
        rec["q"].append(q[0].copy())
        rec["acc"].append(info.acceptance_rate)
        rec["accept"].append(info.if_accept.astype(np.int32))
        rec["step_size"].append(np.float32(info.updated_step_size))
        rec["eps_used"].append(np.float32(info.step_size_used))
        rec["mass"].append(info.mass[0].reshape(-1))
        rec["lp"].append(info.log_prob)
        rec["h0"].append(info.orig_hamiltonian)
        rec["h1"].append(info.hamiltonian)
        rec["lp0"].append(info.orig_log_prob)
        rec["p0"].append(info.init_momentum[0])
    out = {k: np.stack(v) for k, v in rec.items()}
    out["n_search_iters"] = np.int32(h.n_search_iters)
    return out


def make_hmc_diag():
    rng = np.random.Generator(np.random.PCG64(101))
    D, C = 12, 16
    std = (1.0 / (1.0 + np.arange(D))).astype(np.float32)   # gaussian.py:29
    model = OM.DiagGaussian(np.zeros(D, np.float32), std)
    q0 = (0.1 * rng.standard_normal((C, D))).astype(np.float32)
    cfg = dict(step_size=1e-3, n_leapfrogs=5, adapt_step_size=True,
               target_acceptance_rate=0.9, adapt_mass=True,
               mass_collect_iters=4, mass_decay=0.99)
    out = run_hmc(model, q0, n_iters=14, n_adapt=9, rng=rng, **cfg)
    out.update(q0=q0, std=std, n_adapt=np.int32(9),
               **{"cfg_" + k: np.float32(v) for k, v in cfg.items()})
    np.savez_compressed(os.path.join(HERE, "hmc_diag.npz"), **out)


def make_hmc_dense():
    rng = np.random.Generator(np.random.PCG64(202))
    D, C = 32, 24
    P, const = OM.make_dense_gaussian_problem(D, seed=2)
    mu = (0.5 * rng.standard_normal(D)).astype(np.float32)
    model = OM.DenseGaussian(P.astype(np.float32), mu, const)
    q0 = rng.standard_normal((C, D)).astype(np.float32)
    cfg = dict(step_size=0.05, n_leapfrogs=4, adapt_step_size=True,
               target_acceptance_rate=0.8, adapt_mass=True,
               mass_collect_iters=3, mass_decay=0.99)
    out = run_hmc(model, q0, n_iters=12, n_adapt=10, rng=rng, **cfg)
    out.update(q0=q0, P=P, mu=mu, const=np.float64(const), n_adapt=np.int32(10),
               **{"cfg_" + k: np.float32(v) for k, v in cfg.items()})
    np.savez_compressed(os.path.join(HERE, "hmc_dense.npz"), **out)


def make_sgmcmc():
    rng = np.random.Generator(np.random.PCG64(303))
    D, C, T = 8, 6, 5
    std = (0.5 + 0.1 * np.arange(D)).astype(np.float32)
    model = OM.DiagGaussian(np.linspace(-1, 1, D).astype(np.float32), std)
    q0 = rng.standard_normal((C, D)).astype(np.float32)
    nz = lambda: rng.standard_normal((C, D)).astype(np.float32)
    out = {"q0": q0, "std": std, "mean": model.mean}
    samplers = {
        "sgld": (OS.SGLD, dict(learning_rate=0.01)),
        "psgld": (OS.PSGLD, dict(learning_rate=0.01)),
        "sghmc1": (OS.SGHMC, dict(learning_rate=0.01, friction=0.3,
                                  variance_estimate=0.02,
                                  n_iter_resample_v=3, second_order=False)),
        "sghmc2": (OS.SGHMC, dict(learning_rate=0.01, friction=0.3,
                                  variance_estimate=0.02,
                                  n_iter_resample_v=3, second_order=True)),
        "sgnht1v": (OS.SGNHT, dict(learning_rate=0.01, variance_extra=0.1,
                                   tune_rate=2., n_iter_resample_v=4,
                                   second_order=False, use_vector_alpha=True)),
        "sgnht2v": (OS.SGNHT, dict(learning_rate=0.01, variance_extra=0.1,
                                   tune_rate=2., n_iter_resample_v=4,
                                   second_order=True, use_vector_alpha=True)),
        "sgnht1s": (OS.SGNHT, dict(learning_rate=0.01, variance_extra=0.1,
                                   tune_rate=2., n_iter_resample_v=None,
                                   second_order=False,
                                   use_vector_alpha=False)),
        "sgnht2s": (OS.SGNHT, dict(learning_rate=0.01, variance_extra=0.1,
                                   tune_rate=2., n_iter_resample_v=None,
                                   second_order=True, use_vector_alpha=False)),
    }
    for name, (cls, kw) in samplers.items():
        s = cls(**kw)
        q = [q0.copy()]
        v0 = nz()
        if hasattr(s, "init_v"):
            s.init_v([v0])
        qs, ns, rs, mk, al = [], [], [], [], []
        for t in range(T):
            n, r = nz(), nz()
            if isinstance(s, (OS.SGHMC, OS.SGNHT)):
                q, info = s.step(q, model.grad, [r], [n])
            else:
                q, info = s.step(q, model.grad, [n])
            qs.append(q[0].copy()); ns.append(n); rs.append(r)
            if "mean_k" in info:
                mk.append(np.asarray(info["mean_k"][0], np.float32))
            if "alpha" in info:
                al.append(np.asarray(info["alpha"][0], np.float32))
        out[name + "_v0"] = v0
        out[name + "_q"] = np.stack(qs)
        out[name + "_noise"] = np.stack(ns)
        out[name + "_resample"] = np.stack(rs)
        if mk:
            out[name + "_mean_k"] = np.stack(mk)
        if al:
            out[name + "_alpha"] = np.stack(al)
    np.savez_compressed(os.path.join(HERE, "sgmcmc.npz"), **out)
    return samplers


# ---------------------------------------------------------------------------
# Large dense-Gaussian replays for the tensor-core kernels (impl 2 = fp16-split per-pass kernel,
# impl 4 / 5 = trajectory-fused kernels): D = 64 and the benchmark's D = 1024, L = 50, step-size +
# mass adaptation, mass != 1 after `mass_collect_iters`, both step-size searches, iterations whose
# trajectories diverge (non-finite -> acceptance 0, hmc.py:56-59) and healthy ones.
#
# Protocol.  Fifty leapfrog steps at a step size near the stability limit amplify a 1-ulp
# perturbation of q by ~2-3x per ITERATION, so NO float32 implementation (not even this oracle on
# another CPU's BLAS) can track a chained multi-iteration run bit for bit: in round 2 the SIMT
# fp32 kernel drifted from the oracle by 1e-3 after 14 chained iterations.  The replay therefore
# restarts every iteration from a prescribed state: q_in(i) = mu + chol(Sigma) z_i with z_i from
# the oracle's Philox (nothing is stored: `big_state` regenerates it), while the sampler's OWN
# state -- t, step size, dual-averaging variables, EWMV mean / variance -- carries over.  That is
# exactly one `sess.run(sample_op)` per iteration after the caller assigned the latent variable.
#
# Stored per iteration: the float32 oracle's outputs AND a float64 re-evaluation of the same
# iteration from the float32 inputs (`acc64`, `h0_64`, `h1_64`); the distance between the two is
# the rounding noise floor of a float32 HMC at this size (|H| ~ D, so acc = exp(H0 - H1) carries
# ~|H| * 2^-23 of absolute error).  Uniforms within `u_guard` of the float64 acceptance are pushed
# away at generation time, so the accept decisions of a correct implementation are unambiguous.
# ---------------------------------------------------------------------------
BIG = {
    "hmc_dense64": dict(D=64, C=160, L=50, iters=16, n_adapt=12, mci=4, seed=11, eps0=0.05,
                        u_guard=4e-3),
    "hmc_dense1024": dict(D=1024, C=320, L=50, iters=16, n_adapt=12, mci=4, seed=12, eps0=0.05,
                          u_guard=2e-2),
}
STREAM_P, STREAM_U, STREAM_Q, STREAM_MU = 1, 2, 9, 10
_BIG_CACHE = {}


def big_problem(cfg):
    """(P float64, const, mu float32, chol(Sigma) float64) of a BIG config, derived from seeds."""
    key = (cfg["D"], cfg["seed"])
    if key not in _BIG_CACHE:
        from oracle import philox as PH
        D, seed = cfg["D"], cfg["seed"]
        P, const = OM.make_dense_gaussian_problem(D, seed=2)
        mu = (0.5 * PH.normal_matrix(seed, STREAM_MU, 0, 0, 1, D)[0]).astype(np.float32)
        chol = np.linalg.cholesky(np.linalg.inv(P))
        _BIG_CACHE[key] = (P, const, mu, chol)
    return _BIG_CACHE[key]


def big_state(cfg, i):
    """q_in of iteration i (0-based): a posterior draw mu + chol(Sigma) z_i, float32 [C, D]."""
    from oracle import philox as PH
    P, const, mu, chol = big_problem(cfg)
    z = PH.normal_matrix(cfg["seed"], STREAM_Q, i + 1, 0, cfg["C"], cfg["D"]).astype(np.float64)
    return (mu.astype(np.float64) + z @ chol.T).astype(np.float32)


def big_noise(cfg, i):
    """Momentum noise [C, D] of iteration i (0-based) of a BIG config."""
    from oracle import philox as PH
    return PH.normal_matrix(cfg["seed"], STREAM_P, i + 1, 0, cfg["C"], cfg["D"])


def _iteration_f64(model64, q_in, noise_p, mass, eps, L):
    """One HMC proposal + acceptance in float64 from float32 inputs (hmc.py:347-372, 46-61)."""
    h = OH.HMC(step_size=float(eps), n_leapfrogs=L, dtype=np.float64)
    mass = np.asarray(mass, np.float64)
    p = np.asarray(noise_p, np.float64) * np.sqrt(mass)
    q = [np.asarray(q_in, np.float64)]
    cq, cp = q, [p]
    eps = np.float64(eps)
    with np.errstate(all="ignore"):
        for k in range(L + 1):
            cq, cp = h._leapfrog_integrator(cq, cp, eps if k > 0 else 0.0,
                                            eps if 0 < k < L else eps / 2, model64.grad, [mass])
        h0, h1, lp0, lp1, acc = h._acceptance(q, [p], cq, cp, model64.logp, [mass], [[1]])
    return h0, h1, acc, cq[0]


def make_hmc_dense_big(name):
    import copy
    from oracle import philox as PH
    cfg = BIG[name]
    D, C, L = cfg["D"], cfg["C"], cfg["L"]
    P, const, mu, chol = big_problem(cfg)
    P32 = P.astype(np.float32)
    m32 = OM.DenseGaussian(P32, mu, const)
    m64 = OM.DenseGaussian(P32.astype(np.float64), mu.astype(np.float64), const,
                           dtype=np.float64)
    h = OH.HMC(step_size=cfg["eps0"], n_leapfrogs=L, adapt_step_size=True, adapt_mass=True,
               mass_collect_iters=cfg["mci"])
    keys = ("noise_u", "acc", "accept", "step_size", "eps_used", "mass", "lp", "lp0", "h0",
            "h1", "acc64", "h0_64", "h1_64", "q_sub", "q_rowsum", "n_pushed")
    rec = {k: [] for k in keys}
    stride = D // 16
    for i in range(cfg["iters"]):
        q_in = big_state(cfg, i)
        npz = big_noise(cfg, i)
        nu = PH.uniform_vector(cfg["seed"], STREAM_U, i + 1, 0, C)
        adapt = i < cfg["n_adapt"]
        # provisional run to learn this iteration's acceptance, then push borderline uniforms away
        h_try = copy.deepcopy(h)
        with np.errstate(all="ignore"):
            _, info_try = h_try.step([q_in.copy()], m32.logp, m32.grad, [npz], nu, adapt, adapt)
        _, _, acc64, _ = _iteration_f64(m64, q_in, npz, info_try.mass[0].reshape(-1),
                                        info_try.step_size_used, L)
        g = np.float32(cfg["u_guard"])
        a = acc64.astype(np.float32)
        near = (np.abs(nu - a) < g) | (np.abs(nu - info_try.acceptance_rate) < g)
        pushed = nu.copy()
        lo_ok = a - 2 * g > 0
        pushed[near & lo_ok] = (a - 2 * g)[near & lo_ok]          # accept side
        pushed[near & ~lo_ok] = np.minimum(a + 2 * g, np.float32(0.999999))[near & ~lo_ok]
        nu = pushed.astype(np.float32)
        with np.errstate(all="ignore"):
            q_out, info = h.step([q_in.copy()], m32.logp, m32.grad, [npz], nu, adapt, adapt)
        h0_64, h1_64, acc64, _ = _iteration_f64(m64, q_in, npz, info.mass[0].reshape(-1),
                                                     info.step_size_used, L)
        assert not np.any(np.abs(nu - info.acceptance_rate) < g / 2)
        assert np.array_equal(nu < acc64.astype(np.float32), info.if_accept)
        rec["noise_u"].append(nu)
        rec["acc"].append(info.acceptance_rate)
        rec["accept"].append(info.if_accept.astype(np.int32))
        rec["step_size"].append(np.float32(info.updated_step_size))
        rec["eps_used"].append(np.float32(info.step_size_used))
        rec["mass"].append(info.mass[0].reshape(-1))
        rec["lp"].append(info.log_prob)
        rec["lp0"].append(info.orig_log_prob)
        rec["h0"].append(info.orig_hamiltonian)
        rec["h1"].append(info.hamiltonian)
        rec["acc64"].append(acc64)
        rec["h0_64"].append(h0_64)
        rec["h1_64"].append(h1_64)
        rec["q_sub"].append(q_out[0][:, ::stride].copy())
        rec["q_rowsum"].append(q_out[0].astype(np.float64).sum(1))
        rec["n_pushed"].append(np.int32(near.sum()))
    out = {k: np.stack(v) for k, v in rec.items()}
    out["n_search_iters"] = np.int32(h.n_search_iters)
    out["P_checksum"] = np.float64(np.abs(P).sum())
    out["q0_checksum"] = np.float64(np.abs(big_state(cfg, 0).astype(np.float64)).sum())
    for k, v in cfg.items():
        out["cfg_" + k] = np.float64(v)
    np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
    return out


SGMCMC_CONFIGS = None

if __name__ == "__main__":
    which = sys.argv[1:] or ["diag", "dense", "sgmcmc"] + list(BIG)
    if "diag" in which:
        make_hmc_diag()
    if "dense" in which:
        make_hmc_dense()
    if "sgmcmc" in which:
        make_sgmcmc()
    for name in BIG:
        if name in which:
            make_hmc_dense_big(name)
    for f in sorted(os.listdir(HERE)):
        if f.endswith(".npz"):
            print(f, os.path.getsize(os.path.join(HERE, f)), "bytes")
