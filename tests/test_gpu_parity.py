"""GPU parity suite: libLRNDE.so (through the Python mirror of the Lux layer API, i.e. through
the C ABI) against the CPU oracle on the same seeded inputs, against the committed golden
fixtures, and -- at full benchmark sizes -- through size-independent properties.

Tolerances are BASELINE.json's: identical accepted/rejected step sequence and NFE, final
states and regulariser within 1e-4 relative, gradients within 1e-3 relative."""
import importlib.util
import os

import numpy as np
import pytest

import __graft_entry__ as entry
import oracle as orc

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")
PRECS = ["fp32", "tf32x3"]
PRECS_SMALL = ["fp32", "tf32x3", "smem"]     # "smem": the shared-memory engine (networks that fit one SM)
NOISE_TF32X3 = 1.0    # measured on B200: |reg_gpu - reg32| / |reg32 - reg64| <= 2.8 on every fixture for tf32x3 (fp32: <= 3.7), inside the 10x allowance of the fp32 engine: the 3xTF32 engines need no extra factor


@pytest.fixture(scope="module")
def pkg():
    entry.build()
    return entry.load_package()


def _cases():
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLD, "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    return mg.CASES


def _chain(pkg, layers, td, input_act):
    c = pkg.Chain(*[pkg.Dense(i, o, a) for (i, o, a) in layers], input_activation=input_act)
    return pkg.TDChain(c) if td else c


def _omodel(layers, td, input_act):
    return orc.MLP([orc.Dense(*l) for l in layers], time_dependent=td, input_act=input_act)


def rel(a, b):
    a, b = np.asarray(a, np.float64), np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


# f(u, p, t) and its pullback, call by call against Float64: tests/test_gpu_dense_rhs.py


def _check_controller_replay(pkg, t, dt, eest, acc, t0, tend, stops, maxiters):
    """The device controller, fed its own measured EEst sequence, must take bit-for-bit the
    decisions the oracle's controller takes (the host build of the same header is pinned to the
    oracle in tests/test_hostlogic.py)."""
    import ctypes as C
    L = C.CDLL(os.path.join(entry.PKG_DIR, "liblrnde_hostcheck.so"))
    f32, i32 = C.c_float, C.c_int32
    L.lrhc_replay.restype = i32
    L.lrhc_replay.argtypes = [f32, f32, C.c_void_p, i32, f32, f32, i32, i32, C.c_void_p, i32,
                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    n = len(t)
    if n == 0:
        return
    ee = np.ascontiguousarray(eest, np.float32)
    to, dto, ao = np.zeros(n + 4, np.float32), np.zeros(n + 4, np.float32), np.zeros(n + 4, np.uint8)
    st = np.array(stops, np.float32)
    rc = C.c_int32()
    dtmin = max(np.spacing(np.float32(abs(t0))), np.spacing(np.float32(abs(tend))))
    k = L.lrhc_replay(t0, tend, st.ctypes.data, len(st), float(dt[0]), float(dtmin), maxiters, 0,
                      ee.ctypes.data, n, to.ctypes.data, dto.ctypes.data, ao.ctypes.data, C.byref(rc))
    assert k == n, (k, n)
    assert to[:n].tobytes() == np.asarray(t, np.float32).tobytes()
    assert dto[:n].tobytes() == np.asarray(dt, np.float32).tobytes()
    assert np.array_equal(ao[:n].astype(bool), acc)


# ------------------------------------------------------------------ golden fixtures
GOLDEN = ["tiny_td_gelu", "tiny_plain_biased", "mid_tanh_stiff", "latent_saveat", "mnist_b16",
          "eval_mode", "mid_x3_err", "mid_x3_stiff", "gelu3_x3_biased"]


@pytest.mark.parametrize("prec", PRECS_SMALL)
@pytest.mark.parametrize("loop_mode", [0, 1])
@pytest.mark.parametrize("name", GOLDEN)
def test_layer_matches_golden(pkg, name, loop_mode, prec):
    """Tolerance policy.  Each fixture carries the Float64 twin of the Float32 oracle run.  Where
    the two agree (truncation-dominated error estimates: the *_x3_* cases) the GPU is held to
    BASELINE.json's bars: identical accept/reject sequence and NFE, states / regulariser 1e-4,
    gradients 1e-3.  Where Float32 rounding noise dominates the embedded error estimate (the
    controller is still growing dt from the conservative initial step; the regulariser reads
    EEst at exactly such a step) the Float32 oracle itself is 10-1000x away from Float64 in
    EEst / reg_val, so a second Float32 implementation is held to: same decisions up to the
    measured Float32-vs-Float64 gap, states 1e-4, adjoint gradients 1e-3."""
    layers, td, input_act, B, kw, seed, d_reg = _cases()[name]
    if prec == "smem" and name == "mnist_b16":
        pytest.skip("the mnist network does not fit shared memory: tcgen05 path only")
    g = np.load(os.path.join(GOLD, name + ".npz"))
    want, want64 = g["step_log"], g["step_log64"]
    n64 = min(len(want), len(want64))
    dev_t = float(np.abs(want[:n64, 0] - want64[:n64, 0]).max())
    strict = len(want) == len(want64) and dev_t < 1e-3
    strict_bwd = strict and int(g["n_bwd64"]) == len(g["bwd_step_log"])
    # 3xTF32 keeps fp32-level products but drops the lo*lo term and rounds the lo parts: its
    # rounding noise is a few times the FP32 FMA's, so noise-regime allowances scale with it
    # measured on B200 (LRNDE_TEST_VERBOSE=1 prints the ratios): |reg_gpu - reg32| / |reg32 - reg64| stays below
    # NOISE_TF32X3 on every noise-regime fixture; fp32 / smem do the oracle's arithmetic and get 1
    noise = 1.0 if prec in ("fp32", "smem") else NOISE_TF32X3
    layer = pkg.NeuralODE(_chain(pkg, layers, td, input_act), precision=prec, loop_mode=loop_mode, **kw)
    st = layer.initialstates(np.random.default_rng(seed + 100))
    if name == "eval_mode":
        st["training"] = False
    if kw.get("regularize") == "biased":
        # the index sampling of rand(rng, sol.t[1:end-1]) is host-RNG specific: pin the index
        ncand = len(g["t"]) - 1

        class _R:
            def random(self, dtype=None):
                return np.float32((1 + 0.5) / ncand)
        st["rng"] = _R()
    sol, st2 = layer(g["x"], g["ps"], st, keep_tape=True)
    assert sol.retcode == "Success"
    t, dt, eest, acc = sol.step_log(0)
    _check_controller_replay(pkg, t, dt, eest, acc, 0.0, 1.0, [], kw.get("maxiters", 1000))
    if strict:
        assert len(t) == len(want), (len(t), len(want))
        assert np.array_equal(acc, want[:, 3].astype(bool))     # same accept/reject sequence
        assert st2["nfe"] == int(g["nfe"])
        np.testing.assert_allclose(t, want[:, 0], rtol=0, atol=max(5e-4, 5 * dev_t))
        np.testing.assert_allclose(dt, want[:, 1], rtol=2e-2)
        np.testing.assert_allclose(eest, want[:, 2], rtol=0.1)
    else:
        # noise regime: the number of steps follows the implementation's rounding-noise level
        assert 0.5 * len(want) <= len(t) <= 2.0 * len(want) + 3, (len(t), len(want))
    assert len(sol.u) == g["u"].shape[0] or kw.get("regularize") == "biased"
    if kw.get("regularize") != "biased":
        np.testing.assert_allclose(np.array(sol.t), g["t"], rtol=1e-6)
        for i in range(len(sol.u)):
            assert rel(sol.u[i], g["u"][i]) < 1e-4, (i, rel(sol.u[i], g["u"][i]))
    assert rel(sol.u[-1], g["u"][-1]) < 1e-4
    reg32, reg64 = float(g["reg_val"]), float(g["reg_val64"])
    if name != "eval_mode":
        tol = 1e-4 * abs(reg32) + 10 * noise * abs(reg32 - reg64) + 1e-12   # 2nd term: pure-noise regime
        if os.environ.get("LRNDE_TEST_VERBOSE"):
            print(f"[noise] {name} {prec} loop{loop_mode}: |reg_gpu-reg32|/|reg32-reg64| = "
                  f"{abs(float(st2['reg_val']) - reg32) / (abs(reg32 - reg64) + 1e-30):.3g} strict={strict}")
        assert abs(float(st2["reg_val"]) - reg32) <= tol, (float(st2["reg_val"]), reg32, reg64)
        if kw.get("regularize") != "biased" or strict:
            assert abs(sol.stats.t1_used - float(g["t1"])) < 1e-4
            assert abs(sol.stats.dt_reg - float(g["dt_reg"])) <= 1e-3 * float(g["dt_reg"])
    else:
        assert st2["reg_val"] == 0
    if kw.get("regularize") == "biased":
        cots = [None] * (len(sol.u) - 1) + [g["cot"][-1]]
    else:
        cots = [g["cot"][i] if g["cot_mask"][i] else None for i in range(len(sol.u))]
    stride = int(g["d_ps_stride"])
    # adjoint part only (d_reg = 0): well defined in every regime
    d_x0, d_ps0 = layer.backward(sol, cots, 0.0)
    bt, bdt, beest, bacc = sol.step_log(1)
    t1u = np.float32(sol.stats.t1_used)
    stops = sorted({np.float32(x) for x in sol.t if 0.0 < float(x) < 1.0} |
                   ({t1u} if name != "eval_mode" and 0.0 < float(t1u) < 1.0 else set()), reverse=True)
    _check_controller_replay(pkg, bt, bdt, beest, bacc, 1.0, 0.0, stops, kw.get("maxiters", 1000))
    assert rel(d_x0, g["d_x"]) < 1e-3 + 3 * float(g["d_x_rel64"]), rel(d_x0, g["d_x"])
    assert rel(np.asarray(d_ps0)[::stride], g["d_ps0"]) < 1e-3 + 3 * float(g["d_ps0_rel64"])
    assert abs(np.linalg.norm(np.asarray(d_ps0, np.float64)) / float(g["d_ps0_norm"]) - 1) < \
        1e-3 + 3 * float(g["d_ps0_rel64"])
    # with the regulariser cotangent
    d_x, d_ps = layer.backward(sol, cots, float(g["d_reg"]))
    bt, bdt, beest, bacc = sol.step_log(1)
    bw = g["bwd_step_log"]
    if strict_bwd and prec in ("fp32", "tf32x3"):     # tf32x3: the latent-space adjoint on the two-layer fixtures
        assert len(bt) == len(bw), (len(bt), len(bw))
        assert np.array_equal(bacc, bw[:, 3].astype(bool))
        assert sol.bwd_stats.nf_bwd == int(g["nf_bwd"])
    assert np.array_equal(np.asarray(d_x), np.asarray(d_x0))        # d reg / d x == 0 (runtests.jl:129)
    assert rel(np.asarray(d_ps)[::stride], g["d_ps"]) < 1e-3 + 10 * noise * float(g["d_ps_rel64"])   # measured: <= 3.1 x the gap
    assert sol.stats.gpu_launches > 0 and sol.bwd_stats.gpu_launches > 0


# ------------------------------------------------------------------ the reference's property tests
@pytest.mark.parametrize("mode", ["none", "unbiased", "biased"])
@pytest.mark.parametrize("td", [True, False])
def test_reference_property_suite(pkg, mode, td):
    """test/runtests.jl:4-331 (ODE items) through the GPU layer."""
    inner = pkg.Chain(pkg.Dense(2, 4, "gelu"), pkg.Dense(4, 2))
    inner = pkg.TDChain(inner) if td else inner
    rng = np.random.default_rng(0)
    node = pkg.NeuralODE(inner, regularize=mode, tspan=(0.0, 1.0))
    ps = node.initialparameters(rng)
    W2 = rng.uniform(-1, 1, (2, 2)).astype(np.float32)
    x = rng.standard_normal((2, 1)).astype(np.float32)
    st = node.initialstates(np.random.default_rng(0))
    sol, st2 = node(x, ps, st)
    y = W2 @ pkg.diffeqsol_to_array(sol)
    assert y.dtype == np.float32 and y.shape == (2, 1)                  # :21
    assert (st2["reg_val"] == 0) if mode == "none" else (st2["reg_val"] != 0)   # :22, :118
    assert set(st2) == {"model", "nfe", "reg_val", "rng", "training"} and st2["nfe"] > 0
    if mode == "unbiased":
        assert len(sol.u) == 2 and sol.t[-1] == np.float32(1.0)         # neural_ode.jl:108
    d_last = W2.T @ np.ones((2, 1), np.float32)
    d_x, d_ps = node.backward(sol, [None] * (len(sol.u) - 1) + [d_last], 0.0)
    assert np.all(np.isfinite(d_x)) and np.all(d_x != 0)                # :24-26
    assert np.all(np.isfinite(d_ps)) and np.all(d_ps != 0)              # :27-29
    if mode != "none":
        d_x2, d_ps2 = node.backward(sol, [None] * len(sol.u), 1.0)
        assert np.all(d_x2 == 0)                                        # :129 (=== nothing)
        assert np.all(np.isfinite(d_ps2)) and np.any(d_ps2 != 0)        # :130-131
    # eval mode falls back to the vanilla solve (:66)
    sol_e, st_e = node(x, ps, dict(st, training=False))
    assert st_e["reg_val"] == 0 and len(sol_e.u) == 1


def test_rng_state_contract(pkg):
    inner = pkg.TDChain(pkg.Chain(pkg.Dense(2, 4, "tanh"), pkg.Dense(4, 2)))
    node = pkg.NeuralODE(inner, regularize="unbiased")
    ps = node.initialparameters(np.random.default_rng(0))
    x = np.ones((2, 3), np.float32)
    st = node.initialstates(np.random.default_rng(0))
    _, st2 = node(x, ps, st)
    _, st3 = node(x, ps, st)
    assert st3["reg_val"] == st2["reg_val"]          # same rng state -> same t1 (:69)
    _, st4 = node(x, ps, st2)
    assert st4["reg_val"] != st2["reg_val"]          # the returned rng has advanced (:83)


# ------------------------------------------------------------------ edge cases
def test_maxiters_and_retcodes(pkg):
    inner = pkg.Chain(pkg.Dense(2, 4, "tanh"), pkg.Dense(4, 2))
    rng = np.random.default_rng(0)
    ps = pkg.glorot_uniform(inner, rng) * 8
    x = rng.standard_normal((2, 5)).astype(np.float32)
    node = pkg.NeuralODE(inner, regularize="none", maxiters=3, abstol=1e-9, reltol=1e-9)
    sol, st2 = node(x, ps, node.initialstates(np.random.default_rng(0)))
    assert sol.retcode == "MaxIters" and sol.stats.naccept + sol.stats.nreject == 3
    om = orc.MLP([orc.Dense(2, 4, "tanh"), orc.Dense(4, 2)], time_dependent=False)
    osol = orc.solve_tsit5(lambda u, t: om.f(u, ps, t), x, 0.0, 1.0, abstol=1e-9, reltol=1e-9, maxiters=3)
    assert osol.retcode == orc.RETCODE_MAXITERS
    assert np.all(np.isfinite(sol.u[-1]))        # what exists is returned, like the reference
    xnan = x.copy()
    xnan[0, 0] = np.nan
    sol, _ = pkg.NeuralODE(inner, regularize="none")(xnan, ps, node.initialstates(np.random.default_rng(0)))
    assert sol.retcode != "Success"


def test_tape_growth(pkg):
    """More accepted steps than the initial tape capacity (96 slots): the tape is regrown and
    the solve resumes with the same step sequence."""
    inner = pkg.Chain(pkg.Dense(3, 8, "tanh"), pkg.Dense(8, 3))
    rng = np.random.default_rng(1)
    ps = pkg.glorot_uniform(inner, rng) * 6
    x = rng.standard_normal((3, 4)).astype(np.float32)
    kw = dict(abstol=1e-9, reltol=1e-9, maxiters=5000)
    node = pkg.NeuralODE(inner, regularize="none", precision="fp32", **kw)
    sol, st2 = node(x, ps, node.initialstates(np.random.default_rng(0)), keep_tape=True)
    om = orc.MLP([orc.Dense(3, 8, "tanh"), orc.Dense(8, 3)], time_dependent=False)
    osol = orc.solve_tsit5(lambda u, t: om.f(u, ps, t), x, 0.0, 1.0, **kw)
    assert osol.naccept > 100
    assert sol.retcode == "Success"
    # abstol = reltol = 1e-9 is far below Float32 resolution: the step count is set by the
    # rounding-noise level of the implementation, not by the dynamics
    assert abs(sol.stats.naccept - osol.naccept) <= osol.naccept // 4
    assert rel(sol.u[-1], osol.us[-1]) < 1e-4
    d_x, d_ps = node.backward(sol, [np.ones_like(x)], 0.0)
    assert np.all(np.isfinite(d_x)) and np.all(np.isfinite(d_ps))


@pytest.mark.parametrize("prec", PRECS)
def test_mnist_ode_b128_reference_tolerance(pkg, prec):
    """BASELINE configs[0]: abstol = reltol = 1.4e-8 is below Float32 eps, so EEst is partly
    rounding noise and exact step identity between two Float32 implementations is not defined;
    the contract checked here is step-count closeness and state parity."""
    layers = [(784, 100, "tanh"), (100, 784, "identity")]
    om = _omodel(layers, True, None)
    rng = np.random.default_rng(0)
    ps = orc.glorot_uniform_params(om, rng)
    x = rng.random((784, 128), dtype=np.float32)
    kw = dict(abstol=1.4e-8, reltol=1.4e-8, maxiters=10000)
    node = pkg.NeuralODE(_chain(pkg, layers, True, None), regularize="unbiased", save_start=False,
                         precision=prec, **kw)
    st = node.initialstates(np.random.default_rng(7))
    sol, st2 = node(x, ps, st)
    on = orc.NeuralODE(om, regularize="unbiased", save_start=False, **kw)
    osol, ost2, aux = on.forward(x, ps, on.initialstates(np.random.default_rng(7)))
    assert sol.retcode == "Success"
    # the Float64 twin gives the truncation-determined step count (10 here); Float32 rounding noise in
    # sum btilde_i k_i can only push EEst up, i.e. add steps (the numpy Float32 oracle takes 40).  An
    # implementation with less noise in the error estimate (the hidden-space engine forms sum btilde_i h_i
    # before the GEMM: 19 steps) lies between the two
    on64 = orc.NeuralODE(om, regularize="unbiased", save_start=False, dtype=np.float64, **kw)
    osol64, ost64, aux64 = on64.forward(x.astype(np.float64), ps.astype(np.float64), on64.initialstates(np.random.default_rng(7)))
    assert aux64["sol"].naccept <= sol.stats.naccept <= 1.5 * aux["sol"].naccept, \
        (aux64["sol"].naccept, sol.stats.naccept, aux["sol"].naccept)
    assert rel(sol.u[-1], osol.u[-1]) < 1e-4
    assert rel(sol.u[-1], osol64.u[-1]) < 1e-4
    assert rel(sol.u[0], osol.u[0]) < 1e-4
    c = rng.standard_normal((784, 128)).astype(np.float32) / 128
    d_x, d_ps = node.backward(sol, [None, c], 2.5)
    o_dx, o_dps = on.backward(aux, [None, c], 2.5, ps)
    assert rel(d_x, o_dx) < 1e-3
    # the regulariser gradient is rounding-noise dominated at this tolerance; compare the part
    # that is defined (the adjoint) tightly and the total loosely
    d_x0, d_ps0 = node.backward(sol, [None, c], 0.0)
    o_dx0, o_dps0 = on.backward(aux, [None, c], 0.0, ps)
    assert rel(d_ps0, o_dps0) < 1e-3, rel(d_ps0, o_dps0)
    # the regulariser value and the total gradient against the Float64 twin of the oracle, within the measured
    # Float32-vs-Float64 gap of the oracle itself (both are rounding noise of the same step at this tolerance)
    _, o_dps64 = on64.backward(aux64, [None, c.astype(np.float64)], 2.5, ps.astype(np.float64))
    reg_gpu, reg32, reg64 = float(st2["reg_val"]), float(ost2["reg_val"]), float(ost64["reg_val"])
    gap_reg = abs(reg32 - reg64)
    gap_dps = rel(o_dps, o_dps64)
    noise = 1.0 if prec == "fp32" else NOISE_TF32X3
    print("reg gpu/oracle32/oracle64", reg_gpu, reg32, reg64, "d_ps rel vs f64: gpu", rel(d_ps, o_dps64), "oracle32", gap_dps)
    assert abs(reg_gpu - reg64) <= 10 * noise * gap_reg + 1e-4 * abs(reg64), (reg_gpu, reg32, reg64)
    assert rel(d_ps, o_dps64) <= 1e-3 + 10 * noise * gap_dps, (rel(d_ps, o_dps64), gap_dps)


# ------------------------------------------------------------------ full-size properties
@pytest.mark.parametrize("prec", PRECS)
def test_full_size_batch_replication_property(pkg, prec):
    """At benchmark size the oracle is too slow; use a size-independent property instead:
    solving the batch [x, x] must reproduce solve(x) (the RMS norm is replication invariant, so
    the step sequence is identical) and the parameter gradient must double."""
    layers = [(784, 100, "tanh"), (100, 784, "identity")]
    chain = _chain(pkg, layers, True, None)
    rng = np.random.default_rng(0)
    B = 4096
    x = rng.random((784, B), dtype=np.float32)
    node = pkg.NeuralODE(chain, regularize="unbiased", abstol=1e-6, reltol=1e-6, maxiters=10000,
                         save_start=False, precision=prec)
    ps = node.initialparameters(rng)
    st = node.initialstates(np.random.default_rng(3))
    c = rng.standard_normal((784, B)).astype(np.float32) / B
    sol1, st1 = node(x, ps, st)
    dx1, dps1 = node.backward(sol1, [None, c], 1.5)
    x2 = np.concatenate([x, x], axis=1)
    c2 = np.concatenate([c, c], axis=1)
    sol2, st2 = node(x2, ps, st)
    dx2, dps2 = node.backward(sol2, [None, c2], 1.5)
    assert st1["nfe"] == st2["nfe"]
    assert rel(sol2.u[-1][:, :B], sol1.u[-1]) < 1e-5 and rel(sol2.u[-1][:, B:], sol1.u[-1]) < 1e-5
    # the K-chunk order of the tcgen05 kernels is rotated per CTA, so a sample and its replica
    # are summed in different orders: bit-identical in fp32 mode only
    assert abs(float(st1["reg_val"]) / float(st2["reg_val"]) - 1) < (1e-4 if prec == "fp32" else 5e-3)
    assert rel(dx2[:, :B], dx1) < 1e-3


@pytest.mark.parametrize("prec", PRECS_SMALL)
def test_physionet_latent_ode_shape(pkg, prec):
    """BASELINE configs[2] shape on the path: the latent-ODE decoder dynamics
    (experiments/src/construct.jl:235-243: tanh.(u) then 8 x Dense(20<->40, tanh), not time
    dependent), 49 observation times as saveat, batch 256, unbiased regulariser; cotangents
    arrive at every saved time (49 lambda jumps in the adjoint).  Weights x2 keep the case
    truncation-dominated so the oracle comparison is meaningful."""
    layers = [(20, 40, "tanh"), (40, 20, "tanh")] * 4
    om = _omodel(layers, False, "tanh")
    rng = np.random.default_rng(5)
    ps = (orc.glorot_uniform_params(om, rng) * 2 + 0.05 * rng.standard_normal(om.nparams)).astype(np.float32)
    B = 256
    x = rng.standard_normal((20, B)).astype(np.float32)
    saveat = np.sort(np.concatenate([[0.0], rng.uniform(0.02, 1.0, 47), [1.0]])).astype(np.float32)
    kw = dict(regularize="unbiased", abstol=1e-4, reltol=1e-4, maxiters=10000, saveat=list(saveat))
    node = pkg.NeuralODE(_chain(pkg, layers, False, "tanh"), precision=prec, **kw)
    on = orc.NeuralODE(om, **kw)
    st = node.initialstates(np.random.default_rng(2))
    sol, st2 = node(x, ps, st)
    osol, ost2, aux = on.forward(x, ps, on.initialstates(np.random.default_rng(2)))
    assert len(sol.u) == 49 and np.allclose(np.array(sol.t), saveat)
    ts = pkg.diffeqsol_to_timeseries(sol)
    assert ts.shape == (20, 49, B)                                  # src/utils.jl:43-45
    assert st2["nfe"] == ost2["nfe"]
    for i in (0, 1, 17, 48):
        assert rel(sol.u[i], osol.u[i]) < 1e-4
    assert abs(float(st2["reg_val"]) / float(ost2["reg_val"]) - 1) < (1e-3 if prec in ("fp32", "smem") else 2e-2)
    cots = [(rng.standard_normal((20, B)) / B).astype(np.float32) for _ in range(49)]
    d_x, d_ps = node.backward(sol, cots, 0.0)
    o_dx, o_dps = on.backward(aux, cots, 0.0, ps)
    assert rel(d_x, o_dx) < 1e-3 and rel(d_ps, o_dps) < 1e-3
    bt, bdt, bee, bacc = sol.step_log(1)
    for s in saveat[1:-1]:
        assert np.any(np.abs(bt + bdt - s) < 1e-6) or np.any(np.abs(bt - s) < 1e-6)   # jumps are tstops


# ------------------------------------------------------------------ SOSRI step + head
def test_sosri_step_matches_oracle(pkg):
    import ctypes as C
    from importlib import import_module
    L = pkg.lib()
    rng = np.random.default_rng(0)
    D, B = 32, 128
    drift = pkg.Chain(pkg.Dense(32, 64, "tanh"), pkg.Dense(64, 32))
    diff = pkg.Chain(pkg.Dense(32, 32))
    od = orc.MLP([orc.Dense(32, 64, "tanh"), orc.Dense(64, 32)], time_dependent=False)
    og = orc.MLP([orc.Dense(32, 32)], time_dependent=False)
    psd = orc.glorot_uniform_params(od, rng)
    psg = orc.glorot_uniform_params(og, rng) * 0.3
    u0 = rng.standard_normal((D, B)).astype(np.float32)
    t, dt = np.float32(0.3), np.float32(0.05)
    dW = (rng.standard_normal((D, B)) * np.sqrt(dt)).astype(np.float32)
    dZ = (rng.standard_normal((D, B)) * np.sqrt(dt)).astype(np.float32)
    want_u, want_reg, _, _ = orc.perform_step_sosri_reg(
        lambda u, tt: od.f(u, psd, tt), lambda u, tt: og.f(u, psg, tt), u0, t, dt, dW, dZ, 0.14, 0.14,
        delta=1.0 / 6.0)
    node = pkg.NeuralODE(drift, regularize="none", abstol=0.14, reltol=0.14)
    ctx = node.ctx
    o, _ = node._opts("none", 0.0, 0.0, False, True)
    u = np.empty((B, D), np.float32)
    reg = C.c_float()
    cT = lambda a: np.ascontiguousarray(a.T)
    a_u0, a_dW, a_dZ = cT(u0), cT(dW), cT(dZ)
    pkg._lib.check(L.lrnde_sosri_step(ctx._h, ctx.model_handle(drift), ctx.model_handle(diff), C.byref(o),
                                      psd.ctypes.data, psg.ctypes.data, a_u0.ctypes.data,
                                      a_dW.ctypes.data, a_dZ.ctypes.data, float(t), float(dt),
                                      1.0 / 6.0, B, u.ctypes.data, C.byref(reg)))
    assert rel(u.T, want_u) < 1e-5
    assert abs(reg.value / float(want_reg) - 1) < 1e-4


def test_head_ce_matches_numpy(pkg):
    import ctypes as C
    L = pkg.lib()
    rng = np.random.default_rng(0)
    D, B, Cn = 784, 128, 10
    W = (rng.standard_normal((Cn, D)) * 0.05).astype(np.float32)
    b = (rng.standard_normal(Cn) * 0.1).astype(np.float32)
    u = rng.standard_normal((D, B)).astype(np.float32)
    y = rng.integers(0, Cn, B).astype(np.int32)
    z = (W.astype(np.float64) @ u + b[:, None])
    lse = np.log(np.exp(z - z.max(0)).sum(0)) + z.max(0)
    want = float(np.mean(lse - z[y, np.arange(B)]))
    sm = np.exp(z - lse)
    sm[y, np.arange(B)] -= 1
    dz = sm / B
    want_du, want_dW, want_db = W.T.astype(np.float64) @ dz, dz @ u.T, dz.sum(1)
    Wc = np.concatenate([W.ravel(order="F"), b])
    ub = np.ascontiguousarray(u.T)
    loss = C.c_float()
    du = np.empty((B, D), np.float32)
    dWc = np.empty(Cn * D + Cn, np.float32)
    ctx = pkg.default_context(0)
    pkg._lib.check(L.lrnde_head_ce(ctx._h, Wc.ctypes.data, ub.ctypes.data, y.ctypes.data, B, D, Cn, 1,
                                   C.byref(loss), du.ctypes.data, dWc.ctypes.data))
    assert abs(loss.value - want) < 1e-5 * abs(want)
    assert rel(du.T, want_du) < 1e-4
    assert rel(dWc[:Cn * D].reshape((Cn, D), order="F"), want_dW) < 1e-4
    assert rel(dWc[Cn * D:], want_db) < 1e-4


# ------------------------------------------------------------------ kernel instantiations
def test_lean_wide_and_cluster_instantiations_agree(pkg, monkeypatch):
    """MlpEval::dense picks, per launch, the lean instantiation (no scalar fallback / activation switch
    in the hot loops), the wide RESIDENT schedule (128 samples per CTA) and the 4-CTA cluster multicast.
    Each can be switched off by an environment variable read per call; all combinations must give the
    same forward states, step sequence and gradients on the mnist_ode shape (tanh / identity, K % 4 == 0,
    batch large enough for the wide schedule), and the general path is also exercised by the
    gelu / sigmoid / relu / odd-K cases of this suite."""
    layers = [(784, 100, "tanh"), (100, 784, "identity")]
    om = _omodel(layers, True, None)
    rng = np.random.default_rng(11)
    ps = (orc.glorot_uniform_params(om, rng) * 2).astype(np.float32)
    B = 6208                                         # 97 tiles of 64: ragged against 128, above the wide threshold
    x = rng.random((784, B)).astype(np.float32)
    # tight tolerances: the adjoint is itself an adaptive solve, so at 1e-3 two summation orders (the
    # chunk rotation depends on the cluster id) may differ by the discretisation error
    kw = dict(regularize="unbiased", abstol=1e-6, reltol=1e-6, maxiters=1000, save_start=False)
    cot = (rng.standard_normal((784, B)) / B).astype(np.float32)
    res = {}
    for name, env in [("default", {}), ("general", {"LRNDE_NO_LEAN": "1"}), ("narrow", {"LRNDE_NO_WIDE": "1"}),
                      ("nocluster", {"LRNDE_NO_CLUSTER": "1"}),
                      ("plain", {"LRNDE_NO_LEAN": "1", "LRNDE_NO_WIDE": "1", "LRNDE_NO_CLUSTER": "1"})]:
        for k in ("LRNDE_NO_LEAN", "LRNDE_NO_WIDE", "LRNDE_NO_CLUSTER"):
            monkeypatch.delenv(k, raising=False)
        for k, v in env.items():
            monkeypatch.setenv(k, v)
        node = pkg.NeuralODE(_chain(pkg, layers, True, None), precision="tf32x3", **kw)
        sol, st2 = node(x, ps, node.initialstates(np.random.default_rng(2)))
        d_x, d_ps = node.backward(sol, [None, cot], 0.0)   # the regulariser's gradient is Float32 noise at this tolerance
        t, dt, ee, acc = sol.step_log(0)
        res[name] = (np.array(sol.u[-1]), st2["nfe"], float(st2["reg_val"]), np.array(d_x), np.array(d_ps), acc.copy(), dt.copy())
        sol.free()
    ref = res["plain"]
    for name, r in res.items():
        assert r[1] == ref[1] and np.array_equal(r[5], ref[5]), name          # same NFE and step sequence
        assert np.allclose(r[6], ref[6], rtol=1e-2), name          # EEst carries Float32 noise at this tolerance
        assert rel(r[0], ref[0]) < 1e-5, (name, rel(r[0], ref[0]))
        assert abs(r[2] / ref[2] - 1) < 1e-3, name
        assert rel(r[3], ref[3]) < 3e-4 and rel(r[4], ref[4]) < 3e-4, (name, rel(r[3], ref[3]), rel(r[4], ref[4]))
    # lean vs general and wide vs narrow do the same arithmetic in the same order per output element
    assert res["default"][0].tobytes() == res["general"][0].tobytes()
    assert res["default"][0].tobytes() == res["narrow"][0].tobytes()


def test_return_last_only_is_the_fused_sol_to_arr(pkg):
    """lrnde_opts.last_only: only sol.u[end] crosses the boundary (src/utils.jl:37 fused); states, the
    regulariser, NFE and the gradients are those of the full call with a zero cotangent on u(t1)."""
    layers = [(16, 12, "tanh"), (12, 16, "identity")]
    om = _omodel(layers, True, None)
    rng = np.random.default_rng(4)
    ps = (orc.glorot_uniform_params(om, rng) * 3).astype(np.float32)
    x = rng.standard_normal((16, 37)).astype(np.float32)
    kw = dict(regularize="unbiased", abstol=1e-3, reltol=1e-3, save_start=False)
    cot = (rng.standard_normal((16, 37)) / 37).astype(np.float32)
    full = pkg.NeuralODE(_chain(pkg, layers, True, None), precision="tf32x3", **kw)
    last = pkg.NeuralODE(_chain(pkg, layers, True, None), precision="tf32x3", return_last_only=True, **kw)
    s1, st1 = full(x, ps, full.initialstates(np.random.default_rng(2)))
    s2, st2 = last(x, ps, last.initialstates(np.random.default_rng(2)))
    assert len(s1.u) == 2 and len(s2.u) == 1 and s2.t[0] == np.float32(1.0)
    assert np.asarray(s2.u[0]).tobytes() == np.asarray(s1.u[1]).tobytes()
    assert st1["nfe"] == st2["nfe"] and st1["reg_val"] == st2["reg_val"]
    dx1, dp1 = full.backward(s1, [None, cot], 0.7)
    dx2, dp2 = last.backward(s2, [cot], 0.7)
    assert np.asarray(dx1).tobytes() == np.asarray(dx2).tobytes() and np.asarray(dp1).tobytes() == np.asarray(dp2).tobytes()
    s1.free(); s2.free()


# ------------------------------------------------------------------ latent-space engines vs the per-layer engines
@pytest.mark.parametrize("shape", [(16, 12, 37), (784, 100, 96)])
def test_latent_space_engines_match_the_layer_engines(pkg, shape):
    """The hidden-space schedule (csrc/lrnde_fused.cu forward attempts with the lean tape, csrc/lrnde_adjoint.cu
    adjoint attempts) against the per-layer tcgen05 kernels (LRNDE_NO_FUSED=1: one GEMM per layer, D-dimensional
    tape and adjoint) on a truncation-dominated case: same accept / reject sequences forward and backward, same NFE,
    states, regulariser and gradients."""
    Dd, Hh, B = shape
    layers = [(Dd, Hh, "tanh"), (Hh, Dd, "identity")]
    om = _omodel(layers, True, None)
    rng = np.random.default_rng(11)
    ps = (orc.glorot_uniform_params(om, rng) * (3 if Dd < 100 else 5)).astype(np.float32)
    x = (rng.standard_normal((Dd, B)) if Dd < 100 else rng.random((Dd, B))).astype(np.float32)
    cot = [(rng.standard_normal((Dd, B)) / B).astype(np.float32) for _ in range(2)]
    kw = dict(regularize="unbiased", abstol=1e-3, reltol=1e-3, save_start=False, precision="tf32x3")
    out = {}
    for mode in ("latent", "layers"):
        if mode == "layers":
            os.environ["LRNDE_NO_FUSED"] = "1"
        try:
            node = pkg.NeuralODE(_chain(pkg, layers, True, None), **kw)
            sol, st2 = node(x, ps, node.initialstates(np.random.default_rng(3)))
            d_x, d_ps = node.backward(sol, cot, 0.9)
            out[mode] = dict(u=[np.asarray(u).copy() for u in sol.u], reg=float(st2["reg_val"]), nfe=st2["nfe"],
                             log=sol.step_log(0), blog=sol.step_log(1), d_x=np.asarray(d_x).copy(),
                             d_ps=np.asarray(d_ps).copy(), nfb=sol.bwd_stats.nf_bwd)
            sol.free()
        finally:
            os.environ.pop("LRNDE_NO_FUSED", None)
    a, b = out["latent"], out["layers"]
    assert a["nfe"] == b["nfe"] and a["nfb"] == b["nfb"]
    assert np.array_equal(a["log"][3], b["log"][3]) and np.array_equal(a["blog"][3], b["blog"][3])
    np.testing.assert_allclose(a["log"][1], b["log"][1], rtol=2e-3)          # dt sequence
    for ua, ub in zip(a["u"], b["u"]):
        assert rel(ua, ub) < 2e-5, rel(ua, ub)
    assert abs(a["reg"] - b["reg"]) <= 2e-3 * abs(b["reg"]), (a["reg"], b["reg"])
    assert rel(a["d_x"], b["d_x"]) < 3e-4 and rel(a["d_ps"], b["d_ps"]) < 3e-4, (rel(a["d_x"], b["d_x"]), rel(a["d_ps"], b["d_ps"]))


def test_save_start_in_unbiased_mode_prepends_u0(pkg):
    """NeuralODE(...; save_start = true) splats into solve (neural_ode.jl:51): sol.u = [u0, u(t1), u(t2)], and a
    cotangent on u0 flows straight into d_x."""
    layers = [(16, 12, "tanh"), (12, 16, "identity")]
    om = _omodel(layers, True, None)
    rng = np.random.default_rng(5)
    ps = (orc.glorot_uniform_params(om, rng) * 3).astype(np.float32)
    x = rng.standard_normal((16, 9)).astype(np.float32)
    kw = dict(regularize="unbiased", abstol=1e-3, reltol=1e-3, save_start=True)
    node = pkg.NeuralODE(_chain(pkg, layers, True, None), precision="tf32x3", **kw)
    on = orc.NeuralODE(om, **kw)
    sol, st2 = node(x, ps, node.initialstates(np.random.default_rng(2)))
    osol, ost2, aux = on.forward(x, ps, on.initialstates(np.random.default_rng(2)))
    assert len(sol.u) == len(osol.u) == 3 and float(sol.t[0]) == 0.0
    assert np.array_equal(np.asarray(sol.u[0]), x)
    for i in range(3):
        assert rel(sol.u[i], osol.u[i]) < 1e-4
    cots = [(rng.standard_normal((16, 9)) / 9).astype(np.float32) for _ in range(3)]
    d_x, d_ps = node.backward(sol, cots, 0.0)
    o_dx, o_dps = on.backward(aux, cots, 0.0, ps)
    assert rel(d_x, o_dx) < 1e-3 and rel(d_ps, o_dps) < 1e-3
    sol.free()


def test_biased_mode_sizes_the_states_from_the_solve(pkg):
    """:biased with the experiments' maxiters = 10_000 (ADVICE r1): the saved states are fetched after the solve
    (lrnde_ode_saved_states), one block per accepted step, instead of reserving maxiters + 2 blocks."""
    layers = [(784, 100, "tanh"), (100, 784, "identity")]
    om = _omodel(layers, True, None)
    rng = np.random.default_rng(0)
    ps = (orc.glorot_uniform_params(om, rng) * 5).astype(np.float32)
    B = 512
    x = rng.random((784, B), dtype=np.float32)
    node = pkg.NeuralODE(_chain(pkg, layers, True, None), regularize="biased", abstol=1e-4, reltol=1e-4,
                         maxiters=10_000, precision="tf32x3")
    sol, st2 = node(x, ps, node.initialstates(np.random.default_rng(1)))
    assert len(sol.u) == sol.stats.naccept + 1 and sol.stats.naccept < 200        # u0 and every accepted step
    assert np.array_equal(np.asarray(sol.u[0]), x) and float(sol.t[-1]) == 1.0
    assert any(abs(float(t) - sol.stats.t1_used) < 1e-7 for t in sol.t[:-1])      # t1 is one of the step times
    d_x, d_ps = node.backward(sol, [None] * (len(sol.u) - 1) + [np.ones_like(x) / B], 1.0)
    assert np.isfinite(np.asarray(d_ps)).all() and float(np.abs(np.asarray(d_ps)).max()) > 0
    sol.free()


def test_default_stream_work_is_ordered_before_the_library(pkg):
    """ADVICE r1 (high): buffers prepared on torch's default stream right before the call.  The ctx of a NULL stream
    handle runs on a blocking stream (ordered with stream 0), so a pending host-to-device copy behind a long kernel
    queue must be complete when the library reads x."""
    import torch
    dev = torch.device("cuda", 0)
    layers = [(784, 100, "tanh"), (100, 784, "identity")]
    om = _omodel(layers, True, None)
    rng = np.random.default_rng(0)
    ps = torch.from_numpy((orc.glorot_uniform_params(om, rng) * 3).astype(np.float32)).to(dev)
    B = 2048
    xh = torch.from_numpy(rng.random((B, 784), dtype=np.float32)).pin_memory()
    ctx = pkg.Context(0, torch.cuda.current_stream(dev).cuda_stream)     # handle 0 -> NULL -> the library's own stream
    node = pkg.NeuralODE(_chain(pkg, layers, True, None), regularize="none", abstol=1e-3, reltol=1e-3, precision="tf32x3",
                         ctx=ctx)
    st = node.initialstates(np.random.default_rng(1))
    xd = xh.to(dev)
    torch.cuda.synchronize()
    ref, _ = node(xd.t(), ps, st)
    want = ref.u[-1].clone()
    big = torch.randn((8192, 8192), device=dev)
    xd2 = torch.zeros_like(xd)
    torch.cuda.synchronize()
    for _ in range(8):
        big = big @ big * 1e-4            # ~100 ms of queued work on stream 0
    xd2.copy_(xh, non_blocking=True)      # queued behind it
    sol, _ = node(xd2.t(), ps, st)        # must not read xd2 before the copy has landed
    torch.cuda.synchronize()
    assert torch.equal(sol.u[-1], want)


def test_head_ce_rejects_labels_outside_the_class_range(pkg):
    import ctypes as C
    import torch
    dev = torch.device("cuda", 0)
    ctx = pkg.default_context(0)
    B, Dd, Cn = 16, 8, 10
    Wc = torch.randn(Cn * Dd + Cn, device=dev)
    u = torch.randn((B, Dd), device=dev)
    y = torch.arange(1, B + 1, device=dev, dtype=torch.int32)      # 1-based labels as Julia's onecold gives: 10 is out of range
    loss = C.c_float()
    rc = pkg.lib().lrnde_head_ce(ctx._h, Wc.data_ptr(), u.data_ptr(), y.data_ptr(), B, Dd, Cn, 0, C.byref(loss), None, None)
    assert rc == -1 and b"0-based" in pkg.lib().lrnde_last_error()


def test_classifier_grad_is_the_layer_by_layer_iteration(pkg):
    """lrnde_classifier_grad (host buffers: x, labels, ps, Wc in; loss, d_ps, d_Wc out) against the same iteration
    assembled from lrnde_ode_forward + lrnde_head_ce + lrnde_ode_backward on device buffers."""
    import ctypes as C
    import torch
    dev = torch.device("cuda", 0)
    ctx = pkg.default_context(0)
    Dd, Hh, Cn, B = 784, 100, 10, 256
    layers = [(Dd, Hh, "tanh"), (Hh, Dd, "identity")]
    om = _omodel(layers, True, None)
    rng = np.random.default_rng(2)
    ps = (orc.glorot_uniform_params(om, rng) * 3).astype(np.float32)
    Wc = np.concatenate([rng.uniform(-0.1, 0.1, Cn * Dd), np.zeros(Cn)]).astype(np.float32)
    x = rng.random((B, Dd), dtype=np.float32)
    y = rng.integers(0, Cn, B).astype(np.int32)
    chain = _chain(pkg, layers, True, None)
    node = pkg.NeuralODE(chain, regularize="unbiased", save_start=False, abstol=1e-3, reltol=1e-3, precision="tf32x3",
                         return_last_only=True, ctx=ctx)
    st = node.initialstates(np.random.default_rng(4))
    # layer by layer on the device
    pst, Wct, xt, yt = (torch.from_numpy(a).to(dev) for a in (ps, Wc, x, y))
    sol, st2 = node(xt.t(), pst, st)
    loss = C.c_float()
    d_u = torch.empty((B, Dd), device=dev)
    d_Wc = torch.empty_like(Wct)
    pkg._lib.check(pkg.lib().lrnde_head_ce(ctx._h, Wct.data_ptr(), sol.u[-1].t().data_ptr(), yt.data_ptr(), B, Dd, Cn, 0,
                                           C.byref(loss), d_u.data_ptr(), d_Wc.data_ptr()))
    d_x, d_ps = node.backward(sol, [d_u.t()], 2.5)
    # fused, host buffers
    import copy
    o, _ = node._opts("unbiased", 0.0, 0.0, True, True)
    o.t1 = float(np.float32(copy.deepcopy(st["rng"]).random(dtype=np.float32)))
    stats = pkg._lib.Stats()
    loss2 = C.c_float()
    g_ps, g_wc = np.empty_like(ps), np.empty_like(Wc)
    pkg._lib.check(pkg.lib().lrnde_classifier_grad(ctx._h, ctx.model_handle(chain), C.byref(o), ps.ctypes.data, Wc.ctypes.data,
                                                   x.ctypes.data, y.ctypes.data, B, Cn, 2.5, 1.0, C.byref(loss2),
                                                   g_ps.ctypes.data, g_wc.ctypes.data, C.byref(stats)))
    assert stats.nfe == st2["nfe"] and abs(loss2.value - loss.value) <= 1e-6 * abs(loss.value)
    assert abs(stats.reg_val - float(st2["reg_val"])) <= 1e-6 * abs(float(st2["reg_val"]))
    assert rel(g_ps, d_ps.cpu().numpy()) < 1e-6 and rel(g_wc, d_Wc.cpu().numpy()) < 1e-6
    sol.free()
    # input pipeline: the batch staged by lrnde_prefetch_inputs (pinned host memory, copy stream) gives the same bits
    xp = torch.from_numpy(x).pin_memory()
    yp = torch.from_numpy(y).pin_memory()
    pkg._lib.check(pkg.lib().lrnde_prefetch_inputs(ctx._h, xp.data_ptr(), yp.data_ptr(), B, Dd))
    g_ps2, g_wc2 = np.empty_like(ps), np.empty_like(Wc)
    loss3 = C.c_float()
    pkg._lib.check(pkg.lib().lrnde_classifier_grad(ctx._h, ctx.model_handle(chain), C.byref(o), ps.ctypes.data, Wc.ctypes.data,
                                                   xp.data_ptr(), yp.data_ptr(), B, Cn, 2.5, 1.0, C.byref(loss3),
                                                   g_ps2.ctypes.data, g_wc2.ctypes.data, C.byref(stats)))
    assert loss3.value == loss2.value and np.array_equal(g_ps2, g_ps) and np.array_equal(g_wc2, g_wc)
