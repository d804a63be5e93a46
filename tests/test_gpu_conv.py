"""GPU parity of the conv dynamics (SURVEY 8f n3, the cifar10 config's node core) against the CPU oracle,
through the C ABI: f(u, p, t), its pullback, and the whole layer (solve + local regulariser + adjoint).

Tolerances: states / regulariser 1e-4 relative, gradients 1e-3 relative (BASELINE.json); f itself 2e-5."""
import numpy as np
import pytest

import __graft_entry__ as entry
import oracle as orc
from oracle.lrnde_conv_oracle import ConvLayer, ConvNet, cifar10_node_core, glorot_uniform_conv_params

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    entry.build()
    return entry.load_package()


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


def _pair(pkg, layers, W, H, td):
    onet = ConvNet([ConvLayer(*l) for l in layers], W, H, time_dependent=td)
    chain = pkg.ConvChain(*[pkg.Conv(*l) for l in layers], width=W, height=H)
    return onet, (pkg.TDConvChain(chain) if td else chain)


SHAPES = [
    # layers (in, out, batchnorm, act), W, H, td, B
    ([(1, 1, False, "identity")], 4, 4, False, 1),                                          # bare convolution
    ([(2, 5, True, "gelu"), (5, 4, True, "gelu"), (4, 2, False, "identity")], 8, 4, True, 3),
    ([(3, 24, True, "gelu"), (24, 20, False, "tanh"), (20, 3, False, "identity")], 12, 7, True, 5),   # 64-wide tiles, masks
    ([(8, 64, True, "gelu"), (64, 64, True, "gelu"), (64, 8, False, "identity")], 32, 32, True, 2),  # the cifar10 core
    ([(2, 17, True, "gelu"), (17, 2, False, "identity")], 16, 40, False, 2),                 # several row tiles
    # tensor-core engine (csrc/lrnde_conv_tc.cu: channel counts multiples of 8, <= 64): partial 16-channel chunks, the
    # 16-wide instantiation with statistics, swapped / narrow weight-gradient operands, a row count that is not a
    # multiple of the split
    ([(8, 16, True, "gelu"), (16, 24, True, "tanh"), (24, 8, False, "identity")], 32, 6, True, 3),
    ([(8, 64, True, "gelu"), (64, 64, True, "gelu"), (64, 8, False, "identity")], 32, 32, True, 5),  # images split over CTAs
    ([(8, 32, False, "tanh"), (32, 8, False, "identity")], 32, 8, False, 2),                 # no BatchNorm, no time channel
    ([(8, 64, True, "gelu"), (64, 8, False, "identity")], 16, 16, True, 2),                  # width 16: SIMT weight gradient
    ([(16, 16, False, "identity")], 32, 3, True, 2),                                         # one layer, time channel
]


@pytest.mark.parametrize("layers,W,H,td,B", SHAPES)
def test_conv_dynamics_matches_oracle(pkg, layers, W, H, td, B):
    rng = np.random.default_rng(0)
    onet, chain = _pair(pkg, layers, W, H, td)
    ps = glorot_uniform_conv_params(onet, rng, jitter=0.2)
    assert pkg.nparams(chain) == onet.nparams
    u = rng.standard_normal((onet.state_dims, B)).astype(np.float32)
    layer = pkg.NeuralODE(chain)
    got = layer.dynamics(u, ps, 0.37)
    want = onet.f(u.astype(np.float64), ps.astype(np.float64), 0.37)
    assert got.shape == want.shape
    assert rel(got, want) < 2e-5, rel(got, want)


@pytest.mark.parametrize("layers,W,H,td,B", SHAPES)
def test_conv_vjp_matches_oracle(pkg, layers, W, H, td, B):
    rng = np.random.default_rng(1)
    onet, chain = _pair(pkg, layers, W, H, td)
    ps = glorot_uniform_conv_params(onet, rng, jitter=0.2)
    u = rng.standard_normal((onet.state_dims, B)).astype(np.float32)
    lam = rng.standard_normal((onet.state_dims, B)).astype(np.float32)
    a, dps = pkg.NeuralODE(chain).dynamics_vjp(u, ps, 0.61, lam)
    wa, wdps = onet.vjp(u.astype(np.float64), ps.astype(np.float64), 0.61, lam.astype(np.float64))
    assert rel(a, wa) < 1e-4, rel(a, wa)
    for (wo, go), L in zip(onet.offsets, onet.layers):          # per parameter block: weights, then scale / bias
        n = 9 * (L.in_ch + (1 if td else 0)) * L.out_ch
        assert rel(dps[wo:wo + n], wdps[wo:wo + n]) < 1e-4
        if L.batchnorm:
            assert rel(dps[go:go + 2 * L.out_ch], wdps[go:go + 2 * L.out_ch]) < 1e-4


def test_tensor_core_and_simt_conv_engines_agree(pkg, monkeypatch):
    """The tcgen05 engine (3xTF32) against the FP32 SIMT direct convolutions of the same library on the cifar10 core:
    f, the data gradient and every parameter gradient (LRNDE_CONV_TC=0 selects the SIMT engine per call)."""
    rng = np.random.default_rng(11)
    layers, W, H, B = [(8, 64, True, "gelu"), (64, 64, True, "gelu"), (64, 8, False, "identity")], 32, 32, 7
    onet, chain = _pair(pkg, layers, W, H, True)
    ps = glorot_uniform_conv_params(onet, rng, jitter=0.2)
    u = rng.standard_normal((onet.state_dims, B)).astype(np.float32)
    lam = rng.standard_normal((onet.state_dims, B)).astype(np.float32)
    layer = pkg.NeuralODE(chain)
    f_tc = layer.dynamics(u, ps, 0.3)
    a_tc, d_tc = layer.dynamics_vjp(u, ps, 0.3, lam)
    monkeypatch.setenv("LRNDE_CONV_TC", "0")
    f_si = layer.dynamics(u, ps, 0.3)
    a_si, d_si = layer.dynamics_vjp(u, ps, 0.3, lam)
    assert rel(f_tc, f_si) < 1e-5, rel(f_tc, f_si)
    assert rel(a_tc, a_si) < 1e-5, rel(a_tc, a_si)
    assert rel(d_tc, d_si) < 1e-5, rel(d_tc, d_si)


def test_conv_model_validation(pkg):
    with pytest.raises(pkg.LrndeError):                          # width not a multiple of 4
        pkg.NeuralODE(pkg.ConvChain(pkg.Conv(1, 1), width=6, height=6)).dynamics(np.zeros((36, 1), np.float32),
                                                                              np.zeros(9, np.float32), 0.0)
    with pytest.raises(pkg.LrndeError):                          # last layer must be a plain Conv
        pkg.NeuralODE(pkg.ConvChain(pkg.Conv(1, 1, True, "gelu"), width=4, height=4)).dynamics(
            np.zeros((16, 1), np.float32), np.zeros(11, np.float32), 0.0)


@pytest.mark.parametrize("mode,reg_type", [("unbiased", "error_estimate"), ("unbiased", "stiffness_estimate"),
                                           ("none", "error_estimate")])
def test_conv_neural_ode_layer_matches_oracle(pkg, mode, reg_type):
    """The layer functor on conv dynamics: same accepted / rejected step sequence and NFE, states and
    regulariser 1e-4, gradients 1e-3 (cotangents on u(t2) and on reg_val)."""
    layers, W, H, B = [(2, 6, True, "gelu"), (6, 6, True, "gelu"), (6, 2, False, "identity")], 8, 8, 4
    rng = np.random.default_rng(2)
    onet, chain = _pair(pkg, layers, W, H, True)
    ps = glorot_uniform_conv_params(onet, rng, jitter=0.1)
    x = rng.standard_normal((onet.state_dims, B)).astype(np.float32)
    kw = dict(regularize=mode, regularize_type=reg_type, abstol=1e-3, reltol=1e-3, maxiters=1000)
    onode = orc.NeuralODE(onet, **kw)
    gnode = pkg.NeuralODE(chain, **kw)
    ost = onode.initialstates(np.random.default_rng(5))
    gst = gnode.initialstates(np.random.default_rng(5))
    osol, ost2, aux = onode.forward(x, ps, ost)
    # Float64 twin of the oracle: where the embedded error estimate of the regulariser's step (taken at the
    # conservative initial dt, perform_step.jl:4) is Float32 rounding noise, two Float32 implementations agree
    # only up to that noise (DESIGN.md section 2); the twin measures it
    o64 = orc.NeuralODE(onet, dtype=np.float64, **kw)
    osol64, ost64, aux64 = o64.forward(x.astype(np.float64), ps.astype(np.float64),
                                       o64.initialstates(np.random.default_rng(5)))
    gsol, gst2 = gnode(x, ps, gst)
    assert gst2["nfe"] == ost2["nfe"]
    t, dt, eest, acc = gsol.step_log(0)
    assert int(acc.sum()) == aux["sol"].naccept and int((~acc).sum()) == aux["sol"].nreject
    assert len(gsol.u) == len(osol.u)
    for g, w in zip(gsol.u, osol.u):
        assert rel(g, w) < 1e-4, rel(g, w)
    if mode != "none":
        r32, r64 = float(ost2["reg_val"]), float(ost64["reg_val"])
        assert abs(float(gst2["reg_val"]) - r32) <= 1e-4 * abs(r32) + 10 * abs(r32 - r64) + 1e-12
    cot = rng.standard_normal(gsol.u[-1].shape).astype(np.float32)
    d_us = [None] * len(gsol.u)
    d_us[-1] = cot
    od = [np.zeros_like(u) for u in osol.u]
    od[-1] = cot
    # adjoint alone (bar: 1e-3), then with the regulariser's cotangent (noise-aware bar from the twin)
    gdx, gdps = gnode.backward(gsol, d_us, 0.0)
    odx, odps = onode.backward(aux, od, np.float32(0.0), ps)
    assert rel(gdx, odx) < 1e-3, rel(gdx, odx)
    assert rel(gdps, odps) < 1e-3, rel(gdps, odps)
    if mode != "none":
        gsol2, _ = gnode(x, ps, gst)
        gdx2, gdps2 = gnode.backward(gsol2, d_us, 2.5)
        odx2, odps2 = onode.backward(aux, od, np.float32(2.5), ps)
        od64 = [np.zeros_like(u) for u in osol64.u]
        od64[-1] = cot.astype(np.float64)
        _, odps64 = o64.backward(aux64, od64, np.float64(2.5), ps.astype(np.float64))
        assert rel(gdx2, odx2) < 1e-3                              # d reg / d x == 0 (test/runtests.jl:129)
        assert rel(gdps2, odps2) < 1e-3 + 3 * rel(odps2, odps64), (rel(gdps2, odps2), rel(odps2, odps64))


def test_cifar10_core_training_iteration_properties(pkg):
    """Full-size node core (32x32x8 state, 47 560 parameters, batch 16): the reference's NeuralODE property
    test (test/runtests.jl:118-131) -- finite outputs, reg_val > 0, finite non-zero parameter gradient --
    plus linearity of the pullback in its cotangent (size-independent)."""
    rng = np.random.default_rng(3)
    onet = cifar10_node_core()
    chain = pkg.TDConvChain(pkg.ConvChain(pkg.Conv(8, 64, True, "gelu"), pkg.Conv(64, 64, True, "gelu"),
                                          pkg.Conv(64, 8), width=32, height=32))
    ps = glorot_uniform_conv_params(onet, rng)
    x = rng.standard_normal((onet.state_dims, 16)).astype(np.float32)
    node = pkg.NeuralODE(chain, regularize="unbiased", abstol=1e-4, reltol=1e-4, maxiters=10_000)
    st = node.initialstates(np.random.default_rng(0))
    sol, st2 = node(x, ps, st)
    assert sol.retcode == "Success" and st2["nfe"] > 0 and float(st2["reg_val"]) > 0
    assert all(np.isfinite(u).all() for u in sol.u)
    cot = rng.standard_normal(sol.u[-1].shape).astype(np.float32)
    dx1, dps1 = node.backward(sol, [None, cot], 0.0)
    assert np.isfinite(dps1).all() and np.abs(dps1).max() > 0 and np.isfinite(dx1).all()
    sol2, _ = node(x, ps, st)
    dx2, dps2 = node.backward(sol2, [None, 2.0 * cot], 0.0)
    assert rel(dps2, 2.0 * np.asarray(dps1)) < 1e-3


# ------------------------------------------------------------------ st.model: BatchNorm running statistics
def _bn_case(pkg, seed=4):
    layers, W, H, B = [(2, 6, True, "gelu"), (6, 20, True, "gelu"), (20, 2, False, "identity")], 8, 8, 4
    rng = np.random.default_rng(seed)
    onet, chain = _pair(pkg, layers, W, H, True)
    ps = glorot_uniform_conv_params(onet, rng, jitter=0.1)
    x = rng.standard_normal((onet.state_dims, B)).astype(np.float32)
    return onet, chain, ps, x, rng


def test_closure_call_updates_running_statistics(pkg):
    """One ``dudt`` call = one Lux.apply of the BatchNorm layers in training mode: momentum 0.1, unbiased variance."""
    from oracle.lrnde_conv_oracle import initial_conv_state
    onet, chain, ps, x, _ = _bn_case(pkg)
    node = pkg.NeuralODE(chain)
    st = node.initialstates(np.random.default_rng(0))
    assert np.array_equal(st["model"]["running"], initial_conv_state(onet))
    du, mst = node.dynamics(x, ps, 0.2, model_state=st["model"])
    onet.running, onet.track = initial_conv_state(onet, np.float64), True
    want = onet.f(x.astype(np.float64), ps.astype(np.float64), 0.2)
    assert rel(du, want) < 2e-5
    assert rel(mst["running"], onet.running) < 1e-5
    assert np.array_equal(st["model"]["running"], initial_conv_state(onet))     # the input state is not mutated


def test_testmode_uses_running_statistics(pkg):
    onet, chain, ps, x, rng = _bn_case(pkg)
    running = (np.abs(rng.standard_normal(onet.nstate)) + 0.5).astype(np.float32)
    node = pkg.NeuralODE(chain)
    mst = dict(running=running, training=False)
    du, mst2 = node.dynamics(x, ps, 0.2, model_state=mst)
    onet.running, onet.testmode = running.astype(np.float64), True
    assert rel(du, onet.f(x.astype(np.float64), ps.astype(np.float64), 0.2)) < 2e-5
    assert np.array_equal(mst2["running"], running)
    lam = rng.standard_normal(x.shape).astype(np.float32)
    a, dps = node.dynamics_vjp(x, ps, 0.2, lam, model_state=mst)
    wa, wdps = onet.vjp(x.astype(np.float64), ps.astype(np.float64), 0.2, lam.astype(np.float64))
    assert rel(a, wa) < 1e-4 and rel(dps, wdps) < 1e-4


def test_layer_returns_the_state_of_the_closure(pkg):
    """st'.model = the closure's st_ when the solve returns (neural_ode.jl:44-53): one update per f evaluation of
    the MAIN solve -- f(u0, t0) twice (initialize! and the initial-dt heuristic), the initial-dt probe, six per
    attempt -- and none for the regulariser's evaluations."""
    from oracle.lrnde_conv_oracle import initial_conv_state
    onet, chain, ps, x, _ = _bn_case(pkg)

    def oracle_state(maxiters):
        onet.running, onet.track = initial_conv_state(onet), True
        sol = orc.solve_tsit5(lambda u, t: onet.f(u, ps, t), x, np.float32(0), np.float32(1), abstol=1e-3,
                              reltol=1e-3, maxiters=maxiters)
        return sol, onet.running.copy()

    def gpu_state(mode, maxiters):
        node = pkg.NeuralODE(chain, regularize=mode, abstol=1e-3, reltol=1e-3, maxiters=maxiters)
        sol, st2 = node(x, ps, node.initialstates(np.random.default_rng(5)))
        assert st2["model"]["training"] is True
        return sol, st2["model"]["running"]

    # exactly one attempt (3 + 6 closure calls): the call counting, to rounding
    _, want1 = oracle_state(1)
    gsol1, got1 = gpu_state("none", 1)
    assert gsol1.retcode == "MaxIters" and rel(got1, want1) < 1e-5, rel(got1, want1)
    # whole solve: same number of attempts; the step sizes of two Float32 implementations agree to ~1e-3 at
    # this tolerance (the embedded estimate is a cancellation), and the layer-1 statistics move with the stage
    # times through the time channel, hence the looser bar
    osol, want = oracle_state(1000)
    gsol, got = gpu_state("none", 1000)
    assert gsol.stats.naccept == osol.naccept and gsol.stats.nreject == osol.nreject
    assert rel(got, want) < 5e-3, rel(got, want)
    # the regulariser's integrator evaluates the same closure but AFTER solve returned st_: bitwise the same state
    _, got_reg = gpu_state("unbiased", 1000)
    assert np.array_equal(got_reg, got)


def test_testmode_layer_matches_oracle(pkg):
    """Lux.testmode(st): the solve and its adjoint with BatchNorm normalising by the running statistics."""
    onet, chain, ps, x, rng = _bn_case(pkg)
    running = (np.abs(rng.standard_normal(onet.nstate)) + 0.5).astype(np.float32)
    kw = dict(regularize="none", abstol=1e-3, reltol=1e-3, maxiters=1000)
    onet.running, onet.testmode = running.copy(), True
    onode, gnode = orc.NeuralODE(onet, **kw), pkg.NeuralODE(chain, **kw)
    osol, ost2, aux = onode.forward(x, ps, onode.initialstates(np.random.default_rng(5)))
    gst = gnode.initialstates(np.random.default_rng(5))
    gst["model"] = dict(running=running, training=False)
    gsol, gst2 = gnode(x, ps, gst)
    assert gst2["nfe"] == ost2["nfe"] and rel(gsol.u[-1], osol.u[-1]) < 1e-4
    assert np.array_equal(gst2["model"]["running"], running)
    cot = rng.standard_normal(gsol.u[-1].shape).astype(np.float32)
    gdx, gdps = gnode.backward(gsol, [cot], 0.0)
    odx, odps = onode.backward(aux, [cot], np.float32(0.0), ps)
    assert rel(gdx, odx) < 1e-3 and rel(gdps, odps) < 1e-3


# ------------------------------------------------------------------ layers either side of the cifar10 NeuralODE
@pytest.mark.parametrize("cin,cout,act,W,H,B", [(3, 5, "identity", 32, 32, 3), (8, 1, "gelu", 32, 32, 4),
                                                 (3, 5, "identity", 8, 8, 2), (20, 24, "tanh", 12, 5, 3)])
def test_conv2d_layer_matches_oracle(pkg, cin, cout, act, W, H, B):
    from oracle.lrnde_conv_oracle import conv2d, conv2d_vjp
    rng = np.random.default_rng(11)
    x = rng.standard_normal((W, H, cin, B)).astype(np.float32)
    ps = (0.3 * rng.standard_normal(9 * cin * cout + cout)).astype(np.float32)
    dy = rng.standard_normal((W, H, cout, B)).astype(np.float32)
    y = pkg.conv2d_forward(x, ps, cout, act)
    assert y.shape == (W, H, cout, B)
    assert rel(y, conv2d(x.astype(np.float64), ps.astype(np.float64), cout, act)) < 2e-5
    d_x, d_ps = pkg.conv2d_backward(x, ps, dy, act)
    wdx, wdps = conv2d_vjp(x.astype(np.float64), ps.astype(np.float64), dy.astype(np.float64), act)
    assert rel(d_x, wdx) < 1e-4 and rel(d_ps, wdps) < 1e-4


@pytest.mark.parametrize("training", [True, False])
def test_batchnorm_layer_matches_oracle(pkg, training):
    from oracle.lrnde_conv_oracle import batchnorm, batchnorm_vjp
    rng = np.random.default_rng(12)
    W, H, C, B = 32, 32, 8, 5
    x = (1.5 * rng.standard_normal((W, H, C, B)) + 0.3).astype(np.float32)
    ps = np.concatenate([1 + 0.2 * rng.standard_normal(C), 0.2 * rng.standard_normal(C)]).astype(np.float32)
    run = np.concatenate([0.1 * rng.standard_normal(C), 0.5 + rng.random(C)]).astype(np.float32)
    dy = rng.standard_normal(x.shape).astype(np.float32)
    y, st2 = pkg.batchnorm_forward(x, ps, dict(running=run, training=training))
    wy, wrun = batchnorm(x.astype(np.float64), ps.astype(np.float64), "identity", run.astype(np.float64), training)
    assert rel(y, wy) < 2e-5 and rel(st2["running"], wrun) < 1e-5
    d_x, d_ps = pkg.batchnorm_backward(x, ps, dy, dict(running=run, training=training))
    wdx, wdps = batchnorm_vjp(x.astype(np.float64), ps.astype(np.float64), dy.astype(np.float64), "identity",
                              run.astype(np.float64), training)
    assert rel(d_x, wdx) < 1e-4 and rel(d_ps, wdps) < 1e-4


def test_cifar10_model_end_to_end(pkg):
    """The whole Chain of experiments/src/construct.jl:212-227 at a reduced width (8x8 images, hidden 16):
    AugmenterLayer(Conv 3=>5) -> BatchNorm(8) -> NeuralODE(conv core, :unbiased) -> diffeqsol_to_array ->
    Conv(8=>1, gelu) -> Flatten -> Dense(64=>10) -> logitcrossentropy + w_reg * reg_val, forward and reverse,
    against the oracle pipeline: loss 1e-4, every gradient block 1e-3 (regulariser term: noise-aware, see above)."""
    from oracle.lrnde_conv_oracle import (augmenter, augmenter_vjp, batchnorm, batchnorm_vjp, conv2d, conv2d_vjp)
    import ctypes as C
    rng = np.random.default_rng(13)
    W = H = 8
    B, NC = 6, 10
    core = [(8, 16, True, "gelu"), (16, 16, True, "gelu"), (16, 8, False, "identity")]
    onet, chain = _pair(pkg, core, W, H, True)
    x = rng.standard_normal((W, H, 3, B)).astype(np.float32)
    labels = rng.integers(0, NC, B).astype(np.int32)
    p_aug = (0.3 * rng.standard_normal(9 * 3 * 5 + 5)).astype(np.float32)
    p_bn = np.concatenate([np.ones(8), np.zeros(8)]).astype(np.float32)
    p_node = glorot_uniform_conv_params(onet, rng, jitter=0.1)
    p_cls = (0.3 * rng.standard_normal(9 * 8 + 1)).astype(np.float32)
    p_head = np.concatenate([(0.2 * rng.standard_normal(NC * W * H)), np.zeros(NC)]).astype(np.float32)
    kw = dict(regularize="unbiased", abstol=1e-3, reltol=1e-3, maxiters=1000)
    w_reg = 0.0      # the regulariser's own gradient is covered (noise-aware) by the layer test above

    # ---- oracle pipeline
    a0 = augmenter(x, p_aug, 5)
    a1, _ = batchnorm(a0, p_bn)
    onode = orc.NeuralODE(onet, **kw)
    osol, ost2, aux = onode.forward(a1.reshape((-1, B), order="F"), p_node, onode.initialstates(np.random.default_rng(5)))
    u2 = osol.u[-1].reshape((W, H, 8, B), order="F")     # Julia reshapes are column-major
    c = conv2d(u2, p_cls, 1, "gelu")
    flat = c.reshape((W * H, B), order="F")                # FlattenLayer
    Wh, bh = p_head[:NC * W * H].reshape((NC, W * H), order="F"), p_head[NC * W * H:]
    logits = Wh @ flat + bh[:, None]
    lse = np.log(np.exp(logits - logits.max(0)).sum(0)) + logits.max(0)
    oloss = float(np.mean(lse - logits[labels, np.arange(B)]))
    sm = np.exp(logits - lse)
    sm[labels, np.arange(B)] -= 1
    dlog = sm / B
    od_head = np.concatenate([(dlog @ flat.T).ravel(order="F"), dlog.sum(1)])
    d_c = (Wh.T @ dlog).reshape((W, H, 1, B), order="F")
    d_u2, od_cls = conv2d_vjp(u2, p_cls, d_c, "gelu")
    cots = [np.zeros_like(u) for u in osol.u]
    cots[-1] = d_u2.reshape((-1, B), order="F").astype(np.float32)
    d_a1, od_node = onode.backward(aux, cots, np.float32(w_reg), p_node)
    d_a0, od_bn = batchnorm_vjp(a0, p_bn, d_a1.reshape((W, H, 8, B), order="F"))
    _, od_aug = augmenter_vjp(x, p_aug, d_a0)

    # ---- the same Chain through libLRNDE
    aug = pkg.AugmenterLayer(3, 5)
    g0 = aug(x, p_aug)
    g1, _ = pkg.batchnorm_forward(g0, p_bn, dict(running=np.concatenate([np.zeros(8), np.ones(8)]), training=True))
    gnode = pkg.NeuralODE(chain, **kw)
    gsol, gst2 = gnode(np.ascontiguousarray(g1.transpose(3, 2, 1, 0)).reshape(B, -1).T, p_node,
                       gnode.initialstates(np.random.default_rng(5)))
    assert gst2["nfe"] == ost2["nfe"]
    gu2 = np.ascontiguousarray(np.asarray(gsol.u[-1]).T).reshape(B, 8, H, W).transpose(3, 2, 1, 0)
    gc = pkg.conv2d_forward(gu2, p_cls, 1, "gelu")
    gflat = np.ascontiguousarray(gc.transpose(3, 2, 1, 0)).reshape(B, W * H)      # batch-major == column-major [D, B]
    loss = C.c_float()
    gd_flat = np.empty((B, W * H), np.float32)
    gd_head = np.empty(p_head.size, np.float32)
    lib = pkg.lib()
    ctx = gnode.ctx
    rc = lib.lrnde_head_ce(ctx._h, p_head.ctypes.data, gflat.ctypes.data, labels.ctypes.data, B, W * H, NC, 1,
                           C.byref(loss), gd_flat.ctypes.data, gd_head.ctypes.data)
    assert rc == 0
    assert abs(loss.value - oloss) < 1e-4 * abs(oloss)
    gd_c = gd_flat.reshape(B, 1, H, W).transpose(3, 2, 1, 0)
    gd_u2, gd_cls = pkg.conv2d_backward(gu2, p_cls, gd_c, "gelu")
    gcot = np.ascontiguousarray(gd_u2.transpose(3, 2, 1, 0)).reshape(B, -1).T
    gd_a1, gd_node = gnode.backward(gsol, [None] * (len(gsol.u) - 1) + [gcot], w_reg)
    gd_a1 = np.ascontiguousarray(np.asarray(gd_a1).T).reshape(B, 8, H, W).transpose(3, 2, 1, 0)
    gd_a0, gd_bn = pkg.batchnorm_backward(g0, p_bn, gd_a1, dict(running=None, training=True))
    _, gd_aug = aug.backward(x, p_aug, gd_a0)
    for name, got, want in (("head", gd_head, od_head), ("classifier conv", gd_cls, od_cls), ("node core", gd_node, od_node),
                            ("batchnorm", gd_bn, od_bn), ("augmenter", gd_aug, od_aug)):
        assert rel(got, want) < 1e-3, (name, rel(got, want))


def test_device_resident_tensors_match_host_buffers(pkg):
    """Zero-copy path (torch CUDA tensors, host_buffers = 0) of the conv dynamics and the side layers gives the
    results of the host-buffer path bit for bit, including st'.model."""
    import torch
    onet, chain, ps, x, rng = _bn_case(pkg)
    dev = torch.device("cuda", 0)
    node = pkg.NeuralODE(chain, regularize="unbiased", abstol=1e-3, reltol=1e-3, maxiters=1000)
    st = node.initialstates(np.random.default_rng(5))
    sol_h, st_h = node(x, ps, st)
    cot = rng.standard_normal(sol_h.u[-1].shape).astype(np.float32)
    dx_h, dps_h = node.backward(sol_h, [None, cot], 1.0)
    xt, pt = torch.from_numpy(x).to(dev), torch.from_numpy(ps).to(dev)
    sol_d, st_d = node(xt, pt, st)
    dx_d, dps_d = node.backward(sol_d, [None, torch.from_numpy(cot).to(dev)], 1.0)
    assert st_d["nfe"] == st_h["nfe"] and float(st_d["reg_val"]) == float(st_h["reg_val"])
    assert np.array_equal(sol_d.u[-1].cpu().numpy(), np.asarray(sol_h.u[-1]))
    assert np.array_equal(st_d["model"]["running"].cpu().numpy(), st_h["model"]["running"])
    assert np.array_equal(dps_d.cpu().numpy(), np.asarray(dps_h)) and np.array_equal(dx_d.cpu().numpy(), np.asarray(dx_h))
    # side layers
    xi = rng.standard_normal((8, 8, 3, 4)).astype(np.float32)
    pa = (0.3 * rng.standard_normal(9 * 3 * 5 + 5)).astype(np.float32)
    y_h = pkg.conv2d_forward(xi, pa, 5)
    y_d = pkg.conv2d_forward(torch.from_numpy(xi).to(dev), torch.from_numpy(pa).to(dev), 5)
    assert np.array_equal(y_d.cpu().numpy(), y_h)
    bn_ps = np.concatenate([np.ones(3), np.zeros(3)]).astype(np.float32)
    state = dict(running=np.concatenate([np.zeros(3), np.ones(3)]).astype(np.float32), training=True)
    b_h, s_h = pkg.batchnorm_forward(xi, bn_ps, state)
    b_d, s_d = pkg.batchnorm_forward(torch.from_numpy(xi).to(dev), torch.from_numpy(bn_ps).to(dev), state)
    assert np.array_equal(b_d.cpu().numpy(), b_h) and np.array_equal(s_d["running"].cpu().numpy(), s_h["running"])
    # the pullbacks; d_y is passed as the very tensor the library reads (the wrappers' WHCN -> BCHW conversion is a
    # no-op on a permuted contiguous tensor), so it must come back untouched although both calls transform a copy
    # of it in place
    def whcn_view(a):
        return torch.from_numpy(np.ascontiguousarray(a.transpose(3, 2, 1, 0))).to(dev).permute(3, 2, 1, 0)
    gy = rng.standard_normal((8, 8, 5, 4)).astype(np.float32)
    gy_d = whcn_view(gy)
    gy_before = gy_d.clone()
    cx_h, cp_h = pkg.conv2d_backward(xi, pa, gy, activation="gelu")
    cx_d, cp_d = pkg.conv2d_backward(torch.from_numpy(xi).to(dev), torch.from_numpy(pa).to(dev), gy_d, activation="gelu")
    assert np.array_equal(cx_d.cpu().numpy(), cx_h) and np.array_equal(cp_d.cpu().numpy(), cp_h)
    assert torch.equal(gy_d, gy_before)
    gb = rng.standard_normal(xi.shape).astype(np.float32)
    gb_d = whcn_view(gb)
    gb_before = gb_d.clone()
    bx_h, bp_h = pkg.batchnorm_backward(xi, bn_ps, gb, activation="relu")
    bx_d, bp_d = pkg.batchnorm_backward(torch.from_numpy(xi).to(dev), torch.from_numpy(bn_ps).to(dev), gb_d, activation="relu")
    assert np.array_equal(bx_d.cpu().numpy(), bx_h) and np.array_equal(bp_d.cpu().numpy(), bp_h)
    assert torch.equal(gb_d, gb_before)


@pytest.mark.parametrize("mode,kwargs", [("unbiased", dict(saveat=[0.25, 0.6, 1.0])), ("biased", {}), ("none", dict(saveat=[0.5, 1.0]))])
def test_conv_layer_saveat_and_biased_modes(pkg, mode, kwargs):
    """saveat with cotangents on every saved state (lambda jumps at interior stops of the adjoint) and the :biased
    mode (t1 drawn from the accepted step times, every step saved) on conv dynamics: same saves, same NFE, states
    1e-4, adjoint gradients 1e-3."""
    layers, W, H, B = [(2, 6, True, "gelu"), (6, 6, True, "gelu"), (6, 2, False, "identity")], 8, 8, 3
    rng = np.random.default_rng(21)
    onet, chain = _pair(pkg, layers, W, H, True)
    ps = glorot_uniform_conv_params(onet, rng, jitter=0.1)
    x = rng.standard_normal((onet.state_dims, B)).astype(np.float32)
    kw = dict(regularize=mode, abstol=1e-3, reltol=1e-3, maxiters=1000, **kwargs)
    onode, gnode = orc.NeuralODE(onet, **kw), pkg.NeuralODE(chain, **kw)
    osol, ost2, aux = onode.forward(x, ps, onode.initialstates(np.random.default_rng(9)))
    gsol, gst2 = gnode(x, ps, gnode.initialstates(np.random.default_rng(9)))
    assert gst2["nfe"] == ost2["nfe"] and len(gsol.u) == len(osol.u)
    if mode == "biased":
        # the saves sit at the accepted step times, and two Float32 implementations agree on the step sizes only to
        # ~1e-2 at this tolerance (the embedded estimate is a cancellation, DESIGN.md section 2): compare the times
        # loosely, the final state and the pullback of a cotangent on u(t2) at the usual bars
        assert np.allclose(np.asarray(gsol.t, np.float32), np.asarray(osol.t, np.float32), rtol=3e-2, atol=1e-6)
        assert rel(gsol.u[-1], osol.u[-1]) < 1e-4
        cots = [np.zeros_like(u) for u in osol.u]
        cots[-1] = rng.standard_normal(osol.u[-1].shape).astype(np.float32)
    else:
        assert np.allclose(np.asarray(gsol.t, np.float32), np.asarray(osol.t, np.float32), rtol=1e-5, atol=1e-6)
        for g, w in zip(gsol.u, osol.u):
            assert rel(g, w) < 1e-4
        cots = [rng.standard_normal(u.shape).astype(np.float32) for u in osol.u]
    gdx, gdps = gnode.backward(gsol, cots, 0.0)
    odx, odps = onode.backward(aux, cots, np.float32(0.0), ps)
    assert rel(gdx, odx) < 1e-3 and rel(gdps, odps) < 1e-3
