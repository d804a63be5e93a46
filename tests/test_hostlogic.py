"""CPU suite for the host side of libLRNDE: the scalar step-size logic that the device
controller runs (csrc/lrnde_controller.h, re-exported by liblrnde_hostcheck.so) is pinned
bit-for-bit against the oracle, so is the save plan of a forward call (csrc/lrnde_saveplan.h),
the golden fixtures are re-derived from the oracle, and the
CUDA library loads and exports every symbol include/lrnde.h declares (no compute here)."""
import ctypes as C
import os
import re

import numpy as np
import pytest

import __graft_entry__ as entry
import oracle as orc
from oracle.lrnde_oracle import TSIT5, _tab

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
GOLD = os.path.join(ROOT, "tests", "golden")


@pytest.fixture(scope="module")
def hc():
    entry.build()
    L = C.CDLL(os.path.join(entry.PKG_DIR, "liblrnde_hostcheck.so"))
    f32, i32 = C.c_float, C.c_int32
    L.lrhc_fastpow.restype = f32
    L.lrhc_fastpow.argtypes = [f32, f32, i32]
    L.lrhc_spacing.restype = f32
    L.lrhc_spacing.argtypes = [f32]
    L.lrhc_interp_weights.argtypes = [f32, C.c_void_p]
    for n in ("lrhc_tsit5_a", "lrhc_tsit5_c", "lrhc_tsit5_btilde"):
        getattr(L, n).restype = f32
    L.lrhc_tsit5_a.argtypes = [i32, i32]
    L.lrhc_tsit5_c.argtypes = [i32]
    L.lrhc_tsit5_btilde.argtypes = [i32]
    L.lrhc_locate.argtypes = [C.c_void_p, i32, i32, f32]
    L.lrhc_locate.restype = i32
    L.lrhc_initdt.restype = f32
    L.lrhc_initdt.argtypes = [f32, f32, f32, i32, f32, f32, i32, C.c_void_p]
    L.lrhc_replay.restype = i32
    L.lrhc_replay.argtypes = [f32, f32, C.c_void_p, i32, f32, f32, i32, i32, C.c_void_p, i32,
                              C.c_void_p, C.c_void_p, C.c_void_p, C.c_void_p]
    L.lrhc_save_plan.restype = i32
    L.lrhc_save_plan.argtypes = [i32, f32, f32, f32, f32, C.c_void_p, i32, i32, i32, C.c_void_p, i32,
                                 C.c_void_p, C.c_void_p, i32, C.c_void_p, C.c_void_p]
    return L


def test_fastpow_bit_exact(hc):
    rng = np.random.default_rng(0)
    xs = np.concatenate([10.0 ** rng.uniform(-12, 6, 4000), [1.0, 1e-4, 0.5, 2.0, 1e-30, 3e38]])
    for y in (np.float32(0.14), np.float32(0.08)):
        for x in xs.astype(np.float32):
            want = orc.fastpow(np.float32(x), y)
            got = np.float32(hc.lrhc_fastpow(float(x), float(y), 0))
            assert got.tobytes() == np.float32(want).tobytes(), (x, y, got, want)
    assert hc.lrhc_fastpow(0.0, 0.14, 0) == 0.0
    assert abs(hc.lrhc_fastpow(0.3, 0.14, 1) / 0.3 ** 0.14 - 1) < 1e-6


def test_tableau_and_interpolant_bit_exact(hc):
    tab = TSIT5
    for row in range(6):
        for i, v in enumerate(tab.a[row + 1]):
            assert np.float32(hc.lrhc_tsit5_a(row, i)) == v
        assert np.float32(hc.lrhc_tsit5_c(row)) == tab.c[row + 1]
    for i in range(7):
        assert np.float32(hc.lrhc_tsit5_btilde(i)) == tab.btilde[i]
    b = np.zeros(7, np.float32)
    for th in np.random.default_rng(1).uniform(-0.1, 1.1, 200).astype(np.float32):
        hc.lrhc_interp_weights(float(th), b.ctypes.data)
        want = np.array(tab.interp_weights(th), np.float32)
        assert b.tobytes() == want.tobytes()


def test_spacing_and_locate(hc):
    for x in (0.0, 1.0, 0.3, 1e-8, 123.0):
        assert np.float32(hc.lrhc_spacing(x)) == np.spacing(np.float32(x))
    ts = np.array([0.0, 0.1, 0.25, 0.6, 1.0], np.float32)
    sol = orc.ODESolution(ts=list(ts), us=[None] * 5, ks=[None] * 4, dts=[0] * 4, step_log=[],
                          nf=0, naccept=4, nreject=0, retcode=0, tdir=1, dtype=np.dtype(np.float32))
    for tv in (0.0, 0.05, 0.1, 0.100001, 0.25, 0.59, 0.6, 0.99, 1.0):
        assert hc.lrhc_locate(ts.ctypes.data, 4, 1, float(np.float32(tv))) == sol.locate(np.float32(tv))
    back = ts[::-1].copy()
    solb = orc.ODESolution(ts=list(back), us=[None] * 5, ks=[None] * 4, dts=[0] * 4, step_log=[],
                           nf=0, naccept=4, nreject=0, retcode=0, tdir=-1, dtype=np.dtype(np.float32))
    for tv in (1.0, 0.7, 0.6, 0.3, 0.0):
        assert hc.lrhc_locate(back.ctypes.data, 4, -1, float(np.float32(tv))) == solb.locate(np.float32(tv))


def _replay(hc, sol, t0, tend, stops, dt0, maxiters=1000, pow_mode=0):
    log = sol.step_log
    n = len(log)
    eest = np.array([e for (_, _, e, _) in log], np.float32)
    t = np.zeros(n + 4, np.float32)
    dt = np.zeros(n + 4, np.float32)
    acc = np.zeros(n + 4, np.uint8)
    stops = np.array(stops, np.float32)
    rc = C.c_int32()
    dtmin = max(np.spacing(np.float32(abs(t0))), np.spacing(np.float32(abs(tend))))
    k = hc.lrhc_replay(t0, tend, stops.ctypes.data, len(stops), float(dt0), float(dtmin), maxiters,
                       pow_mode, eest.ctypes.data, n, t.ctypes.data, dt.ctypes.data,
                       acc.ctypes.data, C.byref(rc))
    return k, t[:k], dt[:k], acc[:k].astype(bool), rc.value


@pytest.mark.parametrize("case", ["fwd", "bwd_tstops", "rejects", "maxiters"])
def test_controller_replay_is_bit_exact(hc, case):
    """Feeding the oracle's measured EEst sequence through the C controller must reproduce the
    oracle's (t, dt, accepted) of every attempt exactly."""
    A = np.array([[-0.5, 20.0], [-20.0, -0.5]], np.float32)
    f = lambda u, t: (A @ u + np.float32(np.sin(7 * t))).astype(np.float32)
    u0 = np.array([[1.0], [0.0]], np.float32)
    kw = dict(abstol=1e-6, reltol=1e-5, maxiters=1000)
    t0, tend, stops = 0.0, 1.0, []
    if case == "bwd_tstops":
        t0, tend, stops = 1.0, 0.0, [0.6, 0.25]
    if case == "rejects":
        f = lambda u, t: (A @ u * np.float32(1 + 30 * (t > 0.5))).astype(np.float32)
    if case == "maxiters":
        kw["maxiters"] = 7
    sol = orc.solve_tsit5(f, u0, t0, tend, tstops=stops, **kw)
    if case == "rejects":
        assert sol.nreject > 0
    dt0 = sol.step_log[0][1]
    # the very first dt may have been clamped by the header; recover the initdt value
    dt_init, _ = orc.ode_initdt(f, u0, t0, 1 if tend > t0 else -1, abs(tend - t0), kw["abstol"],
                                kw["reltol"],
                                dtmin=max(np.spacing(np.float32(t0)), np.spacing(np.float32(tend))))
    k, t, dt, acc, rc = _replay(hc, sol, t0, tend, stops, dt_init, kw["maxiters"])
    assert k == len(sol.step_log) and rc == sol.retcode
    want_t = np.array([s[0] for s in sol.step_log], np.float32)
    want_dt = np.array([s[1] for s in sol.step_log], np.float32)
    want_acc = np.array([s[3] for s in sol.step_log])
    assert t.tobytes() == want_t.tobytes()
    assert dt.tobytes() == want_dt.tobytes()
    assert np.array_equal(acc, want_acc)
    assert np.float32(dt0) == dt[0]


def test_initdt_matches_oracle(hc):
    rng = np.random.default_rng(3)
    for trial in range(20):
        u0 = rng.standard_normal((3, 4)).astype(np.float32)
        M = rng.standard_normal((3, 3)).astype(np.float32) * (10.0 ** rng.uniform(-2, 2))
        f = lambda u, t: (M @ u).astype(np.float32)
        tol = 10.0 ** rng.uniform(-8, -2)
        tdir = 1 if trial % 2 == 0 else -1
        dtmax, dtmin = np.float32(1.0), np.spacing(np.float32(1.0))
        want, _ = orc.ode_initdt(f, u0, 0.0, tdir, dtmax, tol, tol, dtmin=dtmin)
        T = np.float32
        sk = T(tol) + np.abs(u0) * T(tol)
        f0 = f(u0, 0.0)
        d0, d1 = orc.rms(u0 / sk), orc.rms(f0 / sk)
        dt0 = np.float32(0)
        ref = C.c_float()
        # two-phase: first get dt0 (needs d2 = 0 placeholder), then the real d2
        hc.lrhc_initdt(float(d0), float(d1), 0.0, 0, float(dtmax), float(dtmin), tdir, C.byref(ref))
        dt0 = T(ref.value)
        f1 = f(u0 + dt0 * f0, T(0) + dt0)
        d2 = orc.rms((f1 - f0) / sk)
        got = T(hc.lrhc_initdt(float(d0), float(d1), float(d2), int(np.array_equal(f0, f1)),
                               float(dtmax), float(dtmin), tdir, None))
        # 10^x / log10 go through libm here and numpy's own kernels in the oracle: a few ulps
        assert abs(float(got) - float(want)) <= 2e-6 * abs(float(want)), (trial, got, want)


# accepted times of a solve on tspan (0, 1): all the save plan reads of the solve
_FTS = np.array([0.0, 0.05, 0.17, 0.4, 0.63, 0.9, 1.0], np.float32)


def _fake_solution(fts=_FTS):
    """An oracle ODESolution that accepted the steps fts (zero stages: interpolating it is cheap)."""
    z = np.zeros((2, 1), np.float32)
    n = len(fts) - 1
    return orc.ODESolution(ts=list(fts), us=[z + np.float32(i) for i in range(n + 1)], ks=[[z] * 7] * n,
                           dts=list(np.diff(fts)), step_log=[], nf=0, naccept=n, nreject=0, retcode=0, tdir=1,
                           dtype=np.dtype(np.float32))


def _solve_kwargs(saveat, save_start):
    kw = {} if saveat is None else dict(saveat=saveat)
    if save_start is not None:
        kw["save_start"] = save_start
    return kw


def _oracle_forward(mode, saveat, save_start):
    """The oracle NeuralODE.forward on _fake_solution: (full saved times, returned times, t1)."""
    model = orc.MLP([orc.Dense(2, 4, "tanh"), orc.Dense(4, 2)], time_dependent=True)
    layer = orc.NeuralODE(model, regularize=mode, **_solve_kwargs(saveat, save_start))
    layer._solve = lambda x, ps: _fake_solution()
    ps = orc.glorot_uniform_params(model, np.random.default_rng(0))
    out, _, aux = layer.forward(np.zeros((2, 1), np.float32), ps, layer.initialstates(np.random.default_rng(1)))
    full = out.t if mode == "none" else aux["out_full"].t
    return list(full), list(out.t), aux.get("t1")


def _save_plan(hc, mode, saveat, save_start, last_only, t1=0.0, u01=0.0, nsave=None):
    """lrnde_opts as the NeuralODE layer fills them, through lr_save_plan on _FTS: (times, blocks, t1, nout)."""
    pkg = entry.load_package()
    layer = pkg.NeuralODE(pkg.Chain(pkg.Dense(2, 4, "tanh"), pkg.Dense(4, 2)), regularize=mode,
                          return_last_only=last_only, **_solve_kwargs(saveat, save_start))
    o, _keep = layer._opts(mode, t1, u01, keep_tape=True, host=True)
    if nsave is not None:
        o.nsave = nsave
    cap = len(_FTS) + max(o.nsave, 0) + 3
    times, out = np.zeros(cap, np.float32), np.zeros(cap, np.int32)
    t1_out, nout = C.c_float(), C.c_int32()
    n = hc.lrhc_save_plan(o.reg_mode, o.t0, o.t2, o.t1, o.u01, C.cast(o.saveat, C.c_void_p), o.nsave, o.save_start,
                          o.last_only, _FTS.ctypes.data, len(_FTS), times.ctypes.data, out.ctypes.data, cap,
                          C.byref(t1_out), C.byref(nout))
    assert 0 < n <= cap
    return times[:n], out[:n], np.float32(t1_out.value), nout.value


def _returned(times, out, nout):
    """The times of the output blocks 0 .. nout-1, in block order (each block written once)."""
    blocks = sorted((int(b), t) for t, b in zip(times, out) if b >= 0)
    assert [b for b, _ in blocks] == list(range(nout))
    return np.array([t for _, t in blocks], np.float32)


@pytest.mark.parametrize("last_only", [False, True], ids=["all", "last_only"])
@pytest.mark.parametrize("save_start", [None, False, True], ids=["start_unset", "start0", "start1"])
@pytest.mark.parametrize("saveat", [None, [0.25, 0.5, 0.9], [0.0, 0.4, 1.0]], ids=["no_saveat", "saveat", "saveat_t0"])
@pytest.mark.parametrize("mode", ["none", "unbiased", "biased"])
def test_save_plan_matches_oracle(hc, mode, saveat, save_start, last_only):
    """The saved times, the returned blocks and t1 of a forward call (lrnde_saveplan.h) are those of the oracle's
    NeuralODE.forward; :biased draws t1 with its own RNG there, so the library's rule is checked instead:
    t1 = times[clamp(floor(u01 * ncand), 0, ncand - 1)] over the ncand = len(times) - 1 candidates times[:-1]."""
    full, ret, t1_orc = _oracle_forward(mode, saveat, save_start)
    want_ret = np.array(ret[-1:] if last_only else ret, np.float32)
    for u01 in ((0.0, 0.37, 0.9999999) if mode == "biased" else (0.0,)):
        t1_in = t1_orc if mode == "unbiased" else 0.0
        times, out, t1, nout = _save_plan(hc, mode, saveat, save_start, last_only, t1=t1_in, u01=u01)
        assert times.tobytes() == np.array(full, np.float32).tobytes(), (times, full)
        assert _returned(times, out, nout).tobytes() == want_ret.tobytes(), (times, out, ret)
        if mode == "biased":
            ncand = len(times) - 1
            idx = min(ncand - 1, max(0, int(np.floor(np.float32(u01) * np.float32(ncand)))))
            assert t1 == times[idx] and t1_orc in list(times[:-1])
        else:
            assert t1 == np.float32(t1_in)


@pytest.mark.parametrize("save_start", [False, True], ids=["start0", "start1"])
@pytest.mark.parametrize("mode", ["none", "unbiased"])
def test_save_plan_every_step(hc, mode, save_start):
    """nsave == -1 saves every accepted step (the oracle's saveat = [] path) in any mode; t1 is not appended."""
    times, out, t1, nout = _save_plan(hc, mode, None, save_start, False, t1=0.3, nsave=-1)
    layer = orc.NeuralODE(orc.MLP([orc.Dense(2, 2)]), regularize=mode, save_start=save_start)
    want = np.array(layer._saves(_fake_solution(), None, all_steps=True).t, np.float32)
    assert times.tobytes() == want.tobytes()
    assert _returned(times, out, nout).tobytes() == want.tobytes()
    assert t1 == np.float32(0.3)


def test_library_exports_every_header_symbol():
    entry.build()
    pkg = entry.load_package()
    hdr = open(os.path.join(ROOT, "include", "lrnde.h")).read()
    hdr = re.sub(r"/\*.*?\*/", "", hdr, flags=re.S)
    names = set(re.findall(r"\b(lrnde_[a-z0-9_]+)\s*\(", hdr))
    assert names, "no prototypes found"
    L = C.CDLL(pkg.LIB_PATH)
    for n in sorted(names):
        assert hasattr(L, n), f"libLRNDE.so does not export {n}"
    assert names == set(pkg.SYMBOLS), names ^ set(pkg.SYMBOLS)
    assert pkg.lib().lrnde_version() >= 100


def test_no_cpu_fallback_without_device():
    """On a box without a GPU the product path must fail loudly, never route to the oracle."""
    import torch
    if torch.cuda.is_available():
        pytest.skip("GPU present")
    pkg = entry.load_package()
    with pytest.raises(pkg.LrndeError):
        pkg.Context(0)
    src = ""
    for fn in os.listdir(entry.PKG_DIR):
        if fn.endswith(".py"):
            src += open(os.path.join(entry.PKG_DIR, fn)).read()
    assert "import oracle" not in src and "from oracle" not in src


def test_layer_constructor_validation_mirrors_reference():
    pkg = entry.load_package()
    chain = pkg.Chain(pkg.Dense(2, 4, "tanh"), pkg.Dense(4, 2))
    with pytest.raises(ValueError):
        pkg.NeuralODE(chain, regularize="bogus")                 # utils.jl:53-58
    with pytest.raises(ValueError):
        pkg.NeuralODE(chain, regularize_type="bogus")
    assert pkg.NeuralODE(chain, regularize=True).regularize == "unbiased"   # neural_ode.jl:14-16
    assert pkg.NeuralODE(chain, regularize=False).regularize == "none"
    st = pkg.NeuralODE(chain).initialstates(np.random.default_rng(0))
    assert st["nfe"] == -1 and st["reg_val"] == 0 and st["training"] is True   # :27-31
    assert pkg.nparams(pkg.TDChain(chain)) == 4 * 3 + 4 + 2 * 5 + 2
    ps = pkg.glorot_uniform(pkg.TDChain(chain), np.random.default_rng(0))
    om = orc.MLP([orc.Dense(2, 4, "tanh"), orc.Dense(4, 2)], time_dependent=True)
    assert np.array_equal(ps, orc.glorot_uniform_params(om, np.random.default_rng(0)))


@pytest.mark.parametrize("name", ["tiny_td_gelu", "tiny_plain_biased", "mid_tanh_stiff",
                                  "latent_saveat", "eval_mode", "mid_x3_err", "mid_x3_stiff",
                                  "gelu3_x3_biased"])
def test_oracle_reproduces_golden(name):
    import importlib.util
    spec = importlib.util.spec_from_file_location("make_golden", os.path.join(GOLD, "make_golden.py"))
    mg = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(mg)
    got = mg.build(name)
    want = np.load(os.path.join(GOLD, name + ".npz"))
    assert int(got["nfe"]) == int(want["nfe"])
    assert np.array_equal(got["step_log"][:, 3], want["step_log"][:, 3])
    np.testing.assert_allclose(got["u"], want["u"], rtol=1e-5, atol=1e-6)
    np.testing.assert_allclose(got["reg_val"], want["reg_val"], rtol=1e-4)
    np.testing.assert_allclose(got["d_ps"], want["d_ps"], rtol=1e-3, atol=1e-6)
