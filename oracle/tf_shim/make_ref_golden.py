"""Golden vectors produced by THE REFERENCE'S OWN SOURCE (zhusuan/hmc.py, zhusuan/sgmcmc.py),
executed unmodified on the NumPy TensorFlow stand-in of this directory (TEST INFRASTRUCTURE ONLY).

    python oracle/tf_shim/make_ref_golden.py        ->  tests/golden/ref_*.npz

Needs /root/reference (it is not on the GPU box: the fixtures are committed).  Every random draw
of the reference (tf.random_normal hmc.py:22 / sgmcmc.py:196-365, tf.random_uniform hmc.py:485) is
replaced by injected arrays, which are stored next to the outputs; the per-iteration booleans are
fed through placeholders exactly as the reference's examples do (hmc.py:228-231).
"""
import hashlib
import importlib
import json
import os
import sys
import types

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
REF = os.environ.get("ZHUSUAN_REFERENCE", "/root/reference")
GOLD = os.path.join(ROOT, "tests", "golden")


def load_reference():
    """Register the shim as `tensorflow`, then import zhusuan.hmc / zhusuan.sgmcmc from the
    reference checkout WITHOUT running zhusuan/__init__.py (which pulls in the whole package)."""
    if HERE not in sys.path:
        sys.path.insert(0, HERE)
    for m in [k for k in sys.modules if k == "tensorflow" or k.startswith("tensorflow.")]:
        del sys.modules[m]
    tf = importlib.import_module("tensorflow")
    assert tf.__version__.endswith("numpy-shim")
    pkg = types.ModuleType("zhusuan")
    pkg.__path__ = [os.path.join(REF, "zhusuan")]
    for m in [k for k in sys.modules if k == "zhusuan" or k.startswith("zhusuan.")]:
        del sys.modules[m]
    sys.modules["zhusuan"] = pkg
    hmc = importlib.import_module("zhusuan.hmc")
    sgmcmc = importlib.import_module("zhusuan.sgmcmc")
    assert os.path.realpath(hmc.__file__).startswith(os.path.realpath(REF))
    return tf, hmc, sgmcmc


def dense_problem(D, seed):
    """Sigma = A A^T / D + 0.1 I rescaled to unit diagonal (the benchmark's target family)."""
    rng = np.random.Generator(np.random.PCG64(seed))
    A = rng.standard_normal((D, D))
    S = A @ A.T / D + 0.1 * np.eye(D)
    d = 1.0 / np.sqrt(np.diag(S))
    S = S * d[:, None] * d[None, :]
    P = np.linalg.inv(S)
    P = 0.5 * (P + P.T)
    _, logdet = np.linalg.slogdet(S)
    return P, -0.5 * (D * np.log(2 * np.pi) + logdet)


def run_reference_hmc(kind, D, C, cfg, n_iters, n_adapt, seed):
    tf, hmc_mod, _ = load_reference()
    rng = np.random.Generator(np.random.PCG64(seed))
    out = {}
    if kind == "dense":
        P, const = dense_problem(D, seed=2)
        mu = (0.5 * rng.standard_normal(D)).astype(np.float32)
        P32 = P.astype(np.float32)
        Pt, mut = tf.constant(P32), tf.constant(mu)

        def log_joint(obs):                      # a callable log-joint (hmc.py:412-416)
            xc = obs["x"] - mut
            return -0.5 * tf.reduce_sum(xc * tf.matmul(xc, Pt), axis=-1) + np.float32(const)
        q0 = rng.standard_normal((C, D)).astype(np.float32)
        out.update(P=P, mu=mu, const=np.float64(const))
    else:
        # the model of examples/toy_examples/gaussian.py:15-20, built with the REFERENCE'S OWN
        # meta_bayesian_net / BayesianNet.normal / Normal.log_prob (framework/bn.py,
        # framework/meta_bn.py, distributions/univariate.py run on the stand-in too)
        fw = importlib.import_module("zhusuan.framework")
        std = (1.0 / (1.0 + np.arange(D))).astype(np.float32)      # gaussian.py:29

        @fw.meta_bayesian_net()
        def gaussian(n_x, stdev, n_particles):
            bn = fw.BayesianNet()
            bn.normal('x', tf.zeros([n_x]), std=stdev, n_samples=n_particles, group_ndims=1)
            return bn
        log_joint = gaussian(D, std, C)
        q0 = (0.1 * rng.standard_normal((C, D))).astype(np.float32)
        out.update(std=std)
    adapt_step = tf.placeholder(tf.bool, shape=[], name="adapt_step_size")
    adapt_mass = tf.placeholder(tf.bool, shape=[], name="adapt_mass")
    x = tf.Variable(q0, name="x", dtype=tf.float32)
    sampler = hmc_mod.HMC(step_size=cfg["step_size"], n_leapfrogs=cfg["n_leapfrogs"],
                          adapt_step_size=adapt_step,
                          target_acceptance_rate=cfg["target_acceptance_rate"],
                          adapt_mass=adapt_mass, mass_collect_iters=cfg["mass_collect_iters"],
                          mass_decay=cfg["mass_decay"])
    sample_op, info = sampler.sample(log_joint, observed={}, latent={"x": x})
    sess = tf.Session()
    rec = {k: [] for k in ("noise_p", "noise_u", "q", "acc", "accept", "step_size", "lp", "h0",
                           "h1", "lp0", "p0")}
    for i in range(n_iters):
        npz = rng.standard_normal((C, D)).astype(np.float32)
        nu = rng.random(C).astype(np.float32)
        tf.set_noise(normal=[npz], uniform=[nu])
        adapt = i < n_adapt
        _, r = sess.run([sample_op, info], feed_dict={adapt_step: adapt, adapt_mass: adapt})
        rec["noise_p"].append(npz)
        rec["noise_u"].append(nu)
        rec["q"].append(np.array(x.value))
        rec["acc"].append(r.acceptance_rate)
        rec["accept"].append((nu < r.acceptance_rate).astype(np.int32))
        rec["step_size"].append(np.float32(r.updated_step_size))
        rec["lp"].append(r.log_prob)
        rec["h0"].append(r.orig_hamiltonian)
        rec["h1"].append(r.hamiltonian)
        rec["lp0"].append(r.orig_log_prob)
        rec["p0"].append(r.init_momentum["x"])
        np.testing.assert_array_equal(r.samples["x"], x.value)
    out.update({k: np.stack(v) for k, v in rec.items()})
    out.update(q0=q0, n_adapt=np.int32(n_adapt),
               **{"cfg_" + k: np.float32(v) for k, v in cfg.items()})
    return out


def run_reference_sgmcmc(seed=303):
    """The eight SG-MCMC configurations of tests/golden/make_golden.py, on the reference classes."""
    tf, _, sg = load_reference()
    rng = np.random.Generator(np.random.PCG64(seed))
    D, C, T = 8, 6, 5
    std = (0.5 + 0.1 * np.arange(D)).astype(np.float32)
    mean = np.linspace(-1, 1, D).astype(np.float32)
    q0 = rng.standard_normal((C, D)).astype(np.float32)
    nz = lambda: rng.standard_normal((C, D)).astype(np.float32)
    out = {"q0": q0, "std": std, "mean": mean}
    ls, mu = np.log(std).astype(np.float32), mean
    configs = {
        "sgld": (sg.SGLD, dict(learning_rate=0.01)),
        "psgld": (sg.PSGLD, dict(learning_rate=0.01)),
        "sghmc1": (sg.SGHMC, dict(learning_rate=0.01, friction=0.3, variance_estimate=0.02,
                                  n_iter_resample_v=3, second_order=False)),
        "sghmc2": (sg.SGHMC, dict(learning_rate=0.01, friction=0.3, variance_estimate=0.02,
                                  n_iter_resample_v=3, second_order=True)),
        "sgnht1v": (sg.SGNHT, dict(learning_rate=0.01, variance_extra=0.1, tune_rate=2.,
                                   n_iter_resample_v=4, second_order=False,
                                   use_vector_alpha=True)),
        "sgnht2v": (sg.SGNHT, dict(learning_rate=0.01, variance_extra=0.1, tune_rate=2.,
                                   n_iter_resample_v=4, second_order=True,
                                   use_vector_alpha=True)),
        "sgnht1s": (sg.SGNHT, dict(learning_rate=0.01, variance_extra=0.1, tune_rate=2.,
                                   n_iter_resample_v=None, second_order=False,
                                   use_vector_alpha=False)),
        "sgnht2s": (sg.SGNHT, dict(learning_rate=0.01, variance_extra=0.1, tune_rate=2.,
                                   n_iter_resample_v=None, second_order=True,
                                   use_vector_alpha=False)),
    }
    for name, (cls, kw) in configs.items():
        lst, mut = tf.constant(ls), tf.constant(mu)

        def log_joint(obs):
            x = obs["x"]
            c = np.float32(-0.5 * np.log(2 * np.pi))
            return tf.reduce_sum(c - lst - 0.5 * tf.exp(-2 * lst) * tf.square(x - mut), axis=-1)
        x = tf.Variable(q0.copy(), name="x", dtype=tf.float32)
        v0 = nz()
        tf.set_noise(normal=[v0] * 4)          # the momentum initialisers (Variable initial values)
        sampler = cls(**kw)
        sample_op, info = sampler.sample(log_joint, observed={}, latent={"x": x})
        sess = tf.Session()
        qs, draws, mk, al = [], [], [], []
        for t in range(T):
            pool = [nz() for _ in range(4)]          # consumed in evaluation order
            tf.set_noise(normal=list(pool))
            _, r = sess.run([sample_op, info])
            used = 4 - len(tf._NOISE["normal"])
            qs.append(np.array(x.value))
            draws.append(np.stack(pool))
            out.setdefault(name + "_n_used", []).append(used)
            if hasattr(r, "mean_k"):
                mk.append(np.asarray(r.mean_k["x"], np.float32))
            if hasattr(r, "alpha"):
                al.append(np.asarray(r.alpha["x"], np.float32))
        out[name + "_v0"] = v0
        out[name + "_q"] = np.stack(qs)
        draws = np.stack(draws)
        used = np.asarray(out.pop(name + "_n_used"), np.int32)
        # consumption order inside one run: the momentum re-draw (sgmcmc.py:306-309, 446-449)
        # is evaluated before the injected noise of the update, so a 2-draw step is
        # (resample, noise) and a 1-draw step is (noise,)
        two = (used == 2)[:, None, None]
        out[name + "_resample"] = np.where(two, draws[:, 0], 0).astype(np.float32)
        out[name + "_noise"] = np.where(two, draws[:, 1], draws[:, 0]).astype(np.float32)
        out[name + "_n_used"] = used
        if mk:
            out[name + "_mean_k"] = np.stack(mk)
        if al:
            out[name + "_alpha"] = np.stack(al)
    return out


def run_reference_ais(seed=4):
    """zhusuan/evaluation.py:57-172 (class AIS) driving the reference's HMC: z ~ N(0, I),
    x | z ~ N(z, s^2 I).  `zhusuan.variational` (imported by evaluation.py for
    is_loglikelihood only) is stubbed: AIS does not touch it."""
    tf, hmc_mod, _ = load_reference()
    stub = types.ModuleType("zhusuan.variational")
    stub.ImportanceWeightedObjective = None
    sys.modules["zhusuan.variational"] = stub
    ev = importlib.import_module("zhusuan.evaluation")
    assert os.path.realpath(ev.__file__).startswith(os.path.realpath(REF))
    rng = np.random.RandomState(seed)
    n_chains, n_data, d, s = 8, 3, 2, 0.8
    nt, na = 12, 3
    x_np = (rng.standard_normal((n_data, d)) * 1.2).astype(np.float32)
    init = [rng.standard_normal((n_chains, n_data, d)).astype(np.float32) for _ in range(2)]
    noises = [(rng.standard_normal((n_chains, n_data, d)).astype(np.float32),
               rng.random_sample((n_chains, n_data)).astype(np.float32))
              for _ in range(na + nt)]
    c = np.float32(-0.5 * np.log(2 * np.pi))
    xt = tf.constant(x_np)

    def normal_lp(x, mean, std):        # Normal._log_prob (univariate.py:174-181), group_ndims 1
        logstd = np.float32(np.log(std))
        return tf.reduce_sum(c - logstd - np.float32(0.5 * np.exp(-2 * np.log(std)))
                             * tf.square(x - mean), axis=-1)

    class _Net(object):                 # the two BayesianNet methods AIS calls
        def __init__(self, obs): self.obs = obs
        def log_joint(self): return normal_lp(self.obs["z"], 0.0, 1.0)
        def get(self, names): return [tf.random_normal([n_chains, n_data, d]) for _ in names]

    class _Proposal(object):
        def observe(self, **obs): return _Net(obs)

    def log_joint(obs):
        return normal_lp(obs["z"], 0.0, 1.0) + normal_lp(obs["x"], obs["z"], s)
    z = tf.Variable(np.zeros((n_chains, n_data, d), np.float32), name="z", dtype=tf.float32)
    hmc = hmc_mod.HMC(step_size=0.2, n_leapfrogs=3, adapt_step_size=True,
                      target_acceptance_rate=0.7)
    ais = ev.AIS(log_joint, _Proposal(), hmc, observed={"x": xt}, latent={"z": z},
                 n_temperatures=nt, n_adapt=na)
    # consumption order of AIS.run: prior draw, n_adapt x (p, u), prior draw, nt x (p, u)
    normal = [init[0]] + [n[0] for n in noises[:na]] + [init[1]] + [n[0] for n in noises[na:]]
    tf.set_noise(normal=normal, uniform=[n[1] for n in noises])
    captured = {}
    orig = ais._get_lower_bound
    ais._get_lower_bound = lambda lw: captured.setdefault("lw", np.array(lw)) is None or orig(lw)
    est = ais.run(tf.Session(), {})
    assert not tf._NOISE["normal"] and not tf._NOISE["uniform"]
    return dict(x=x_np, s=np.float32(s), init=np.stack(init),
                noise_p=np.stack([n[0] for n in noises]), noise_u=np.stack([n[1] for n in noises]),
                log_weights=captured["lw"].astype(np.float32), bound=np.float64(est),
                z_final=np.array(z.value), n_temperatures=np.int32(nt), n_adapt=np.int32(na),
                schedule=np.array([ais._get_schedule_t(t) for t in range(nt + 1)]))


def run_reference_variational(seed=77):
    """The VAE of examples/variational_autoencoders/iwae.py:23-44 (smaller layers) on the
    REFERENCE'S OWN framework + distributions + variational code: importance_weighted_objective /
    elbo with .sgvb() (iwae.py:72-75), and elbo(...).reinforce() over three steps (moving-mean
    baseline state).  tf.layers.dense weights are Glorot-uniform draws of the given generator."""
    tf, _, _ = load_reference()
    fw = importlib.import_module("zhusuan.framework")
    var = importlib.import_module("zhusuan.variational")
    rng = np.random.Generator(np.random.PCG64(seed))
    tf.reset_default_graph()
    tf.set_init_rng(rng)
    N, x_dim, z_dim, H, K = 6, 10, 4, 8, 5

    @fw.meta_bayesian_net(scope="gen", reuse_variables=True)
    def build_gen(n, x_dim, z_dim, n_particles):
        bn = fw.BayesianNet()
        z_mean = tf.zeros([n, z_dim])
        z = bn.normal("z", z_mean, std=1., group_ndims=1, n_samples=n_particles)
        h = tf.layers.dense(z, H, activation=tf.nn.relu)
        h = tf.layers.dense(h, H, activation=tf.nn.relu)
        x_logits = tf.layers.dense(h, x_dim)
        bn.bernoulli("x", x_logits, group_ndims=1)
        return bn

    def q_net(reparameterized):
        @fw.reuse_variables(scope="q_net")
        def build_q_net(x, z_dim, n_particles):
            bn = fw.BayesianNet()
            h = tf.layers.dense(tf.cast(x, tf.float32), H, activation=tf.nn.relu)
            h = tf.layers.dense(h, H, activation=tf.nn.relu)
            z_mean = tf.layers.dense(h, z_dim)
            z_logstd = tf.layers.dense(h, z_dim)
            bn.normal("z", z_mean, logstd=z_logstd, group_ndims=1, n_samples=n_particles,
                      is_reparameterized=reparameterized)
            return bn
        return build_q_net
    x_np = (rng.random((N, x_dim)) < 0.4).astype(np.int32)
    x = tf.constant(x_np)
    model = build_gen(N, x_dim, z_dim, K)
    build_q = q_net(True)
    variational = build_q(x, z_dim, K)
    iw = var.importance_weighted_objective(model, {'x': x}, variational=variational, axis=0)
    el = var.elbo(model, {'x': x}, variational=variational, axis=0)
    q_vars = tf.trainable_variables()                 # the four q-net layers (built first)
    iw_cost, el_cost = tf.reduce_mean(iw.sgvb()), tf.reduce_mean(el.sgvb())
    lj, ent = iw._log_joint_term(), iw._entropy_term()        # builds the generator
    all_vars = tf.trainable_variables()
    names = ["q%d_%s" % (i // 2, "wb"[i % 2]) for i in range(len(q_vars))] + \
            ["g%d_%s" % (i // 2, "wb"[i % 2]) for i in range(len(all_vars) - len(q_vars))]
    eps = rng.standard_normal((K, N, z_dim)).astype(np.float32)
    sess = tf.Session()
    out = {"x": x_np, "eps": eps, "names": np.array(names)}
    for nme, v in zip(names, all_vars):
        out["w_" + nme] = np.array(v.value)
    tf.set_noise(normal=[eps])
    r = sess.run([iw, iw_cost, lj, ent] + tf.gradients(iw_cost, all_vars))
    out.update(iw_bound=r[0], iw_cost=r[1], log_joint=r[2], entropy=r[3])
    for nme, g in zip(names, r[4:]):
        out["iw_grad_" + nme] = g
    tf.set_noise(normal=[eps])
    r = sess.run([el, el_cost] + tf.gradients(el_cost, all_vars))
    out.update(elbo_bound=r[0], elbo_cost=r[1])
    for nme, g in zip(names, r[2:]):
        out["elbo_grad_" + nme] = g
    # ---- score-function estimator with the moving-mean baseline, three consecutive steps -------
    variational_sf = q_net(False)
    # the SAME q-net weights: reuse_variables templates own their variables, so copy them over
    bn_sf = variational_sf(x, z_dim, K)
    sf_vars = tf.trainable_variables()[len(all_vars):]
    for dst, src in zip(sf_vars, q_vars):
        dst.load(src.value)
    el_sf = var.elbo(model, {'x': x}, variational=bn_sf, axis=0)
    rf_cost = tf.reduce_mean(el_sf.reinforce())
    rf_grads = tf.gradients(rf_cost, sf_vars)
    mm = tf.get_variable('moving_mean')
    eps_sf = rng.standard_normal((3, K, N, z_dim)).astype(np.float32)
    costs, mms, grads = [], [], []
    for t in range(3):
        tf.set_noise(normal=[eps_sf[t]])
        r = sess.run([rf_cost] + rf_grads)
        costs.append(r[0])
        grads.append(r[1:])
        mms.append(np.array(mm.value))
    out.update(rf_eps=eps_sf, rf_cost=np.array(costs), rf_moving_mean=np.array(mms))
    for i, nme in enumerate(names[:len(q_vars)]):
        out["rf_grad_" + nme] = np.stack([g[i] for g in grads])
    # ---- VIMCO (monte_carlo.py:166-227) and the self-normalised importance estimator of the
    # inclusive KL (inclusive_kl.py:119-151) on the same non-reparameterised q-net ----------------
    gen_vars = all_vars[len(q_vars):]
    iw_sf = var.importance_weighted_objective(model, {'x': x}, variational=bn_sf, axis=0)
    vm_cost = tf.reduce_mean(iw_sf.vimco())
    kl_sf = var.klpq(model, {'x': x}, variational=bn_sf, axis=0)
    im_cost = tf.reduce_mean(kl_sf.importance())
    tf.set_noise(normal=[eps])
    r = sess.run([vm_cost] + tf.gradients(vm_cost, sf_vars + gen_vars))
    out["vimco_cost"] = r[0]
    for nme, gr in zip(names, r[1:]):
        out["vimco_grad_" + nme] = gr
    tf.set_noise(normal=[eps])
    r = sess.run([im_cost] + tf.gradients(im_cost, sf_vars))
    out["importance_cost"] = r[0]
    for nme, gr in zip(names[:len(q_vars)], r[1:]):
        out["importance_grad_" + nme] = gr
    return out


def run_reference_bnn_sghmc(seed=707):
    """Config 4's model, examples/bayesian_neural_nets/bnn_sgmcmc.py:19-35 + its log_joint
    override (74-77), on the reference's BayesianNet and SGHMC classes: per-weight prior
    log-stddevs, second-order SGHMC with a momentum re-draw at t = 0 and t = 3, five steps."""
    tf, _, sg = load_reference()
    fw = importlib.import_module("zhusuan.framework")
    rng = np.random.Generator(np.random.PCG64(seed))
    tf.reset_default_graph()
    C, n_in, H, B, n_train = 9, 4, 37, 23, 500
    x_np = rng.standard_normal((B, n_in)).astype(np.float32)
    y_np = rng.standard_normal(B).astype(np.float32)
    layer_sizes = [n_in, H, 1]
    ls_np = [(0.1 * rng.standard_normal((H, n_in + 1))).astype(np.float32),
             (0.1 * rng.standard_normal((1, H + 1))).astype(np.float32)]
    w_np = [rng.uniform(-2, 2, (C, H, n_in + 1)).astype(np.float32),
            rng.uniform(-2, 2, (C, 1, H + 1)).astype(np.float32)]

    @fw.meta_bayesian_net(scope="bnn", reuse_variables=True)
    def build_bnn(x, layer_sizes, logstds, n_particles):
        bn = fw.BayesianNet()
        h = tf.tile(x[None, ...], [n_particles, 1, 1])
        for i, (n_i, n_o) in enumerate(zip(layer_sizes[:-1], layer_sizes[1:])):
            w = bn.normal("w" + str(i), tf.zeros([n_o, n_i + 1]),
                          logstd=logstds[i], group_ndims=2, n_samples=n_particles)
            h = tf.concat([h, tf.ones(tf.shape(h)[:-1])[..., None]], -1)
            h = tf.einsum("imk,ijk->ijm", w, h) / tf.sqrt(
                tf.cast(tf.shape(h)[2], tf.float32))
            if i < len(layer_sizes) - 2:
                h = tf.nn.relu(h)
        y_mean = bn.deterministic("y_mean", tf.squeeze(h, 2))
        y_logstd = -0.95
        bn.normal("y", y_mean, logstd=y_logstd)
        return bn
    x, y = tf.constant(x_np), tf.constant(y_np)
    w_names = ["w0", "w1"]
    wv = [tf.Variable(w, name=n) for w, n in zip(w_np, w_names)]
    logstds = [tf.constant(a) for a in ls_np]
    model = build_bnn(x, layer_sizes, logstds, C)

    def log_joint(bn):                                            # bnn_sgmcmc.py:74-77
        log_pws = bn.cond_log_prob(w_names)
        log_py_xw = bn.cond_log_prob('y')
        return tf.add_n(log_pws) + tf.reduce_mean(log_py_xw, 1) * n_train
    model.log_joint = log_joint
    kw = dict(learning_rate=1e-4, friction=0.2, variance_estimate=0.01, n_iter_resample_v=3,
              second_order=True)
    v0 = [rng.standard_normal(w.shape).astype(np.float32) for w in w_np]
    tf.set_noise(normal=[v0[0], v0[1]] * 2)
    sgmcmc = sg.SGHMC(**kw)
    sample_op, info = sgmcmc.sample(model, observed={'y': y}, latent=dict(zip(w_names, wv)))
    sess = tf.Session()
    out = dict(x=x_np, y=y_np, logstd0=ls_np[0], logstd1=ls_np[1], w0_init=w_np[0],
               w1_init=w_np[1], n_train=np.int32(n_train), v0_0=v0[0], v0_1=v0[1],
               **{"cfg_" + k: np.float32(v) for k, v in kw.items()})
    rec = {k: [] for k in ("w0", "w1", "noise0", "noise1", "resample0", "resample1", "mean_k0",
                           "mean_k1", "n_used")}
    for t in range(5):
        pool = [rng.standard_normal(w_np[k % 2].shape).astype(np.float32) for k in range(4)]
        tf.set_noise(normal=list(pool))
        _, r = sess.run([sample_op, info])
        used = 4 - len(tf._NOISE["normal"])
        # consumption order inside a run: [re-draw of v for w0, w1,] then the update noise of
        # w0, w1 (latents are visited in dictionary order, sgmcmc.py:105-107)
        if used == 4:
            rs, nz = pool[:2], pool[2:]
        else:
            assert used == 2
            rs, nz = [np.zeros_like(pool[0]), np.zeros_like(pool[1])], pool[:2]
        rec["n_used"].append(used)
        for k in range(2):
            rec["w%d" % k].append(np.array(wv[k].value))
            rec["noise%d" % k].append(nz[k])
            rec["resample%d" % k].append(rs[k])
            rec["mean_k%d" % k].append(np.float32(r.mean_k["w%d" % k]))
    out.update({k: np.stack(v) for k, v in rec.items()})
    return out


def run_reference_lntm_hmc(seed=909):
    """Config 5's E-step: the model of examples/topic_models/lntm_mcem.py:33-48 with the e_obj
    log-joint override (97-98) on the reference's BayesianNet, sampled by the reference's HMC
    with two chain axes [chains, docs] (69-70, 99-105), adaptive step size, injected noise."""
    tf, hmc_mod, _ = load_reference()
    fw = importlib.import_module("zhusuan.framework")
    rng = np.random.Generator(np.random.PCG64(seed))
    tf.reset_default_graph()
    K, V, C, Dn = 32, 120, 6, 5
    log_delta = 10.0
    x_np = rng.poisson(0.1, (Dn, V)).astype(np.float32)
    x_np[0] = 0                                              # a padding document (71-74)
    beta_np = rng.standard_normal((K, V)).astype(np.float32)
    mean_np = (0.2 * rng.standard_normal(K)).astype(np.float32)
    logstd_np = (0.1 * rng.standard_normal(K)).astype(np.float32)
    eta0 = (0.1 * rng.standard_normal((C, Dn, K))).astype(np.float32)

    @fw.meta_bayesian_net(scope='lntm')
    def lntm(n_chains, n_docs, n_topics, n_vocab, eta_mean, eta_logstd):
        bn = fw.BayesianNet()
        eta_mean = tf.tile(tf.expand_dims(eta_mean, 0), [n_docs, 1])
        eta = bn.normal('eta', eta_mean, logstd=eta_logstd, n_samples=n_chains, group_ndims=1)
        theta = tf.nn.softmax(eta)
        beta = bn.normal('beta', tf.zeros([n_topics, n_vocab]), logstd=log_delta, group_ndims=1)
        phi = tf.nn.softmax(beta)
        doc_word = tf.matmul(tf.reshape(theta, [-1, n_topics]), phi)
        doc_word = tf.reshape(doc_word, [n_chains, n_docs, n_vocab])
        bn.unnormalized_multinomial('x', tf.log(doc_word), normalize_logits=False,
                                    dtype=tf.float32)
        return bn

    def e_obj(bn):
        return bn.cond_log_prob('eta') + bn.cond_log_prob('x')
    cfg = dict(step_size=0.02, n_leapfrogs=6, target_acceptance_rate=0.6)
    hmc = hmc_mod.HMC(adapt_step_size=True, **cfg)
    eta = tf.Variable(eta0, name='eta')
    model = lntm(C, Dn, K, V, tf.constant(mean_np), tf.constant(logstd_np))
    model.log_joint = e_obj
    sample_op, info = hmc.sample(model, observed={'x': tf.constant(x_np),
                                                  'beta': tf.constant(beta_np)},
                                 latent={'eta': eta})
    sess = tf.Session()
    rec = {k: [] for k in ("noise_p", "noise_u", "eta", "acc", "step_size", "lp", "lp0", "h0",
                           "h1")}
    for i in range(8):
        npz = rng.standard_normal(eta0.shape).astype(np.float32)
        nu = rng.random((C, Dn)).astype(np.float32)
        tf.set_noise(normal=[npz], uniform=[nu])
        with np.errstate(all="ignore"):
            _, r = sess.run([sample_op, info])
        rec["noise_p"].append(npz); rec["noise_u"].append(nu)
        rec["eta"].append(np.array(eta.value)); rec["acc"].append(r.acceptance_rate)
        rec["step_size"].append(np.float32(r.updated_step_size))
        rec["lp"].append(r.log_prob); rec["lp0"].append(r.orig_log_prob)
        rec["h0"].append(r.orig_hamiltonian); rec["h1"].append(r.hamiltonian)
    out = {k: np.stack(v) for k, v in rec.items()}
    out.update(x=x_np, beta=beta_np, eta_mean=mean_np, eta_logstd=logstd_np, eta0=eta0,
               **{"cfg_" + k: np.float32(v) for k, v in cfg.items()})
    return out


def run_reference_hmc_big(name):
    """The L = 50 adaptive protocol of tests/golden/make_golden.py (BIG: every iteration starts
    from a prescribed posterior draw, the sampler's adaptation state carries over) executed by the
    reference's own HMC -- the source of truth the BIG fixtures (written by the float32 oracle
    with a float64 re-evaluation) are compared with in tests/test_ref_pins.py.  Returns the
    per-iteration outputs; nothing is written."""
    tf, hmc_mod, _ = load_reference()
    sys.path.insert(0, GOLD)
    import make_golden as MG
    cfg = dict(MG.BIG[name])
    g = np.load(os.path.join(GOLD, name + ".npz"))
    D, C, L = cfg["D"], cfg["C"], cfg["L"]
    P, const, mu, _ = MG.big_problem(cfg)
    Pt, mut = tf.constant(P.astype(np.float32)), tf.constant(mu)

    def log_joint(obs):
        xc = obs["x"] - mut
        return -0.5 * tf.reduce_sum(xc * tf.matmul(xc, Pt), axis=-1) + np.float32(const)
    adapt_step = tf.placeholder(tf.bool, shape=[], name="adapt_step_size")
    adapt_mass = tf.placeholder(tf.bool, shape=[], name="adapt_mass")
    x = tf.Variable(MG.big_state(cfg, 0), name="x", dtype=tf.float32)
    sampler = hmc_mod.HMC(step_size=cfg["eps0"], n_leapfrogs=L, adapt_step_size=adapt_step,
                          adapt_mass=adapt_mass, mass_collect_iters=cfg["mci"])
    sample_op, info = sampler.sample(log_joint, observed={}, latent={"x": x})
    sess = tf.Session()
    rec = {k: [] for k in ("acc", "step_size", "lp", "lp0", "h0", "h1", "q")}
    for i in range(cfg["iters"]):
        x.load(MG.big_state(cfg, i))                  # the caller assigns the latent variable
        tf.set_noise(normal=[MG.big_noise(cfg, i)], uniform=[g["noise_u"][i]])
        adapt = i < cfg["n_adapt"]
        with np.errstate(all="ignore"):
            _, r = sess.run([sample_op, info], feed_dict={adapt_step: adapt, adapt_mass: adapt})
        rec["acc"].append(r.acceptance_rate); rec["step_size"].append(r.updated_step_size)
        rec["lp"].append(r.log_prob); rec["lp0"].append(r.orig_log_prob)
        rec["h0"].append(r.orig_hamiltonian); rec["h1"].append(r.hamiltonian)
        rec["q"].append(np.array(x.value))
    return {k: np.stack(v) for k, v in rec.items()}


# per-iteration outputs of run_reference_hmc_big kept in tests/golden/ref_<name>_l50.npz (the
# chain states are left out: [iters, C, D] would not fit a fixture at D = 1024)
BIG_KEYS = ("acc", "step_size", "lp0", "h0", "h1")


def write_reference_hmc_big():
    for name in ("hmc_dense64", "hmc_dense1024"):
        o = run_reference_hmc_big(name)
        np.savez_compressed(os.path.join(GOLD, "ref_%s_l50.npz" % name),
                            **{k: o[k] for k in BIG_KEYS})
        print("ref_%s_l50 step sizes" % name, o["step_size"].tolist())


HMC_CASES = {
    "ref_hmc_diag": ("diag", 12, 16, dict(step_size=1e-3, n_leapfrogs=5,
                                          target_acceptance_rate=0.9, mass_collect_iters=4,
                                          mass_decay=0.99), 14, 9, 101),
    "ref_hmc_dense32": ("dense", 32, 24, dict(step_size=0.05, n_leapfrogs=4,
                                              target_acceptance_rate=0.8, mass_collect_iters=3,
                                              mass_decay=0.99), 12, 10, 202),
    "ref_hmc_dense64": ("dense", 64, 40, dict(step_size=0.05, n_leapfrogs=6,
                                              target_acceptance_rate=0.8, mass_collect_iters=3,
                                              mass_decay=0.99), 16, 12, 404),
}


def array_digest(a):
    """SHA-256 of an array's dtype, shape and bytes: equal digests = bit-identical arrays."""
    a = np.ascontiguousarray(a)
    h = hashlib.sha256(("%s %s " % (a.dtype.str, a.shape)).encode())
    h.update(a.tobytes())
    return h.hexdigest()


def reference_digests():
    """{fixture: {array: array_digest}} of a fresh run of every tests/golden/ref_*.npz that main()
    writes (the L = 50 runs aside) -> tests/golden/ref_digests.json, so that the committed
    fixtures can be checked against what the reference's code produced without its checkout."""
    runs = {name: (lambda c=c: run_reference_hmc(*c)) for name, c in HMC_CASES.items()}
    runs.update(ref_vae=run_reference_variational, ref_lntm_hmc=run_reference_lntm_hmc,
                ref_bnn_sghmc=run_reference_bnn_sghmc, ref_ais=run_reference_ais,
                ref_sgmcmc=run_reference_sgmcmc)
    return {name: {k: array_digest(v) for k, v in sorted(run().items())}
            for name, run in runs.items()}


def main():
    for name, (kind, D, C, cfg, n_iters, n_adapt, seed) in HMC_CASES.items():
        out = run_reference_hmc(kind, D, C, cfg, n_iters, n_adapt, seed)
        np.savez_compressed(os.path.join(GOLD, name + ".npz"), **out)
        print(name, "acc mean per iteration", np.round(out["acc"].mean(1), 3).tolist())
    out = run_reference_variational()
    np.savez_compressed(os.path.join(GOLD, "ref_vae.npz"), **out)
    print("ref_vae iw bound", out["iw_bound"].tolist(), "reinforce costs", out["rf_cost"].tolist(),
          "moving mean", out["rf_moving_mean"].tolist())
    out = run_reference_lntm_hmc()
    np.savez_compressed(os.path.join(GOLD, "ref_lntm_hmc.npz"), **out)
    print("ref_lntm_hmc acc mean", np.round(out["acc"].mean((1, 2)), 3).tolist(), "step",
          out["step_size"].tolist())
    out = run_reference_bnn_sghmc()
    np.savez_compressed(os.path.join(GOLD, "ref_bnn_sghmc.npz"), **out)
    print("ref_bnn_sghmc draws per step", out["n_used"].tolist(), "mean_k", out["mean_k0"].tolist())
    out = run_reference_ais()
    np.savez_compressed(os.path.join(GOLD, "ref_ais.npz"), **out)
    print("ref_ais bound", float(out["bound"]))
    out = run_reference_sgmcmc()
    np.savez_compressed(os.path.join(GOLD, "ref_sgmcmc.npz"), **out)
    print("ref_sgmcmc draws per step", {k: out[k].tolist() for k in out if k.endswith("_n_used")})
    write_reference_hmc_big()
    with open(os.path.join(GOLD, "ref_digests.json"), "w") as f:
        json.dump(reference_digests(), f, indent=1, sort_keys=True)
        f.write("\n")


if __name__ == "__main__":
    main()
