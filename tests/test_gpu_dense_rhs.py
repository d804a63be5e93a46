"""The dense right-hand side f(u, p, t) and its pullback (J_u^T lam, J_p^T lam), one call per engine, against the
Float64 oracle with an elementwise rounding-error bound.

The adjoint of every dense config evaluates the pullback several times per attempt; the full-solve tests see it only
through max-normalised gradients at the end of an adaptive solve.  Here one f call and one pullback call on fixed
inputs are compared element by element with oracle.MLP.f / MLP.vjp in Float64, so every difference is rounding, and
rounding is bounded by a Float64 "magnitude pass" over the same chain:

  forward    E_pre_l = g(K) |W_l| [|x_{l-1}|; |t|; 1] + rss(W_l[:, :in], E_{l-1})  (K = in + td + 1)
             E_l     = D(act_l) E_pre_l + c1 u max(|y_l|, 1)                        (the input activation is layer 0)
  reverse    E_delta_L = |lam| (K2(act_L) E_pre_L + c1 u)                           (K2 bounds |act''|)
             E_dW_l    = g(B) |delta_l| |x~_l|^T + E_delta_l |x~_l|^T + |delta_l| E_x~_l^T
             E_g_{l-1} = g(out) |W_l|^T |delta_l| + rss(W_l^T, E_delta_l), then through act'_{l-1} like the forward
  with g(n) = c0 sqrt(n) u, u = 2^-24 (probabilistic GEMM bound), D(act) = max |act'| over [pre -+ E_pre] (at most
  Lip(act)), and rss(W, E) = sqrt(W^2 E^2): the rounding errors of different elements are independent, so the
  propagated error adds in quadrature.  A worst-case |W| E (and a global Lip) compounds per layer: on the 8-layer
  physionet decoder it puts the bound 10^6 above the error, where no kernel defect could reach it.

LRNDE_TEST_VERBOSE=1 prints the worst |err| / bound per case and per precision."""
import functools
import os

import numpy as np
import pytest

import __graft_entry__ as entry
import oracle as orc
from oracle.lrnde_oracle import _act, _act_grad

pytestmark = pytest.mark.gpu

U = 2.0 ** -24
# (c0, c1): twice the worst |err| / bound measured with (1, 1) on a B200 (1000 W) over every element of every case
# below.  LRNDE_TEST_VERBOSE=1 prints the worst per precision; with these constants, on the same B200: fp32 0.50,
# smem 0.50, tf32x3 0.50, auto 0.22
C_FP32 = (1.2, 1.2)      # fp32 (SIMT GEMMs), smem (shared-memory engine): 0.60 with (1, 1), dps of the 2x4 gelu net, B = 1
C_TF32X3 = (3.5, 3.5)    # tcgen05 3xTF32: 1.76 with (1, 1), dps of the 16x16 net, B = 1 (one product off by 3.5 u)
# The thinnest fp32 / smem margin is the gelu output under cancellation at B = 1: numpy's own Float32 evaluation of the
# oracle reaches 0.96 of C_FP32 there, so a change to how lrnde_act.cuh rounds gelu may need this row re-measured.
# "auto" routes to the smem engine for small batches of nets that fit (there it is held ~3x looser than the smem rows)
# and to tcgen05 3xTF32 otherwise (mnist_ode, the 200x150 net, B = 20011): its constant is chosen for the latter.
CONST = {"fp32": C_FP32, "smem": C_FP32, "tf32x3": C_TF32X3, "auto": C_TF32X3}
# relu samples within the widest forward bound of the kink are excluded (their derivative is not defined by rounding)
C_KINK = tuple(max(c[i] for c in CONST.values()) for i in (0, 1))
LIP = {"identity": 1.0, "tanh": 1.0, "sigmoid": 0.25, "relu": 1.0, "gelu": 1.13}      # max |act'|
K2 = {"identity": 0.0, "tanh": 0.77, "sigmoid": 0.0963, "relu": 0.0, "gelu": 0.80}    # max |act''| (relu: kink excluded)
PRECS = ["fp32", "tf32x3", "smem", "auto"]
TIMES = [0.37, -2.5]           # at t = -2.5 the time column carries a large, negative share of every pre-activation

TANH2 = [(20, 40, "tanh"), (40, 20, "tanh")] * 4
MNIST = [(784, 100, "tanh"), (100, 784, "identity")]
SMALL = [(16, 12, "tanh"), (12, 16, "identity")]
# layers (in, out, act), td, input activation, B, fused -- and the branch of MlpEval (csrc/lrnde_api.cu) each row
# reaches.  fused: under tf32x3 / auto, f may run on the hidden-space FusedEngine (lrf_shape: 2 layers, identity
# output, no input activation, H + td + 1 <= 128); those cases also run f with LRNDE_NO_FUSED=1 (per-layer GEMMs)
SHAPES = [
    # tcgen05 weight gradient transposed (layer 1: out 12 < in+td+1 18) and normal (layer 2), lambda formed in the
    # data-gradient GEMM's prologue (identity output), a 32-sample chunk plus a ragged 5; f: hidden-space FusedEngine
    (SMALL, True, None, 37, True),
    # L == 1 with identity: y materialised by lincomb_kernel; one sample in a 32-sample chunk
    ([(16, 16, "identity")], False, None, 1, False),
    # L == 1, non-identity: delta_L by dact_mul_kernel; chunk of 32 + 1
    ([(16, 16, "tanh")], True, None, 33, False),
    # physionet decoder: input-activation derivative read from ybuf, general (non-lean) weight gradient with in_act,
    # general dense with in_act; 8 layers of the smem engine under smem / auto
    (TANH2, False, "tanh", 256, False),
    (TANH2, False, "tanh", 1000, False),
    # K % 4 != 0: general dense and general weight gradient; gelu and its derivative; fused f (Kaug 72)
    ([(33, 70, "gelu"), (70, 33, "identity")], True, None, 65, True),
    # min(out, in+td+1) > 128 on both layers: SIMT wgrad_nt_kernel (16-rounded split) under tf32x3 and auto;
    # sigmoid, relu (kink exclusion); too large for shared memory
    ([(200, 150, "sigmoid"), (150, 200, "relu")], False, None, 300, False),
    # fused f eligibility edge: H + td + 1 = 128 (FusedEngine) and 129 (per-layer GEMMs)
    ([(64, 126, "tanh"), (126, 64, "identity")], True, None, 129, True),
    ([(64, 127, "tanh"), (127, 64, "identity")], True, None, 129, False),
    # mnist_ode: resident layer-2 GEMM, ring layer-1 GEMM, no cluster (2 tiles of 64); tcgen05 wgrad in 4 chunks of 32
    (MNIST, True, None, 128, True),
    # mnist_ode at batch 77: a ragged 64-sample tile, wgrad chunks 32 + 32 + 13
    (MNIST, True, None, 77, True),
    # mnist_ode: wide (128 samples per CTA) and cluster forward and data GEMMs, uS = 21 chunks of 800 with a ragged
    # last chunk of 411
    (MNIST, True, None, 16411, True),
    # smem engine tile S shrunk to 8 (ceil(100 / 16) < 148 / 2)
    (SMALL, True, None, 100, True),
    # smem engine with two tiles per CTA (626 tiles of 32 > 4 * 148); tcgen05 / SIMT above the auto smem threshold
    (SMALL, True, None, 20011, True),
    # one sample, gelu through the fused f and a 2-row output
    ([(2, 4, "gelu"), (4, 2, "identity")], True, None, 1, True),
    # input activation on a 3-wide state, tanh output (dact_mul_kernel), 7 samples
    ([(3, 5, "tanh"), (5, 3, "tanh")], False, "tanh", 7, False),
    # 4 layers with td: tanh, sigmoid and relu (kink exclusion) derivatives between general GEMMs, 130 samples
    ([(20, 40, "tanh"), (40, 20, "tanh"), (20, 40, "sigmoid"), (40, 20, "relu")], True, None, 130, False),
]
MNIST_B128 = 9


@pytest.fixture(scope="module")
def pkg():
    entry.build()
    return entry.load_package()


WORST = {}      # precision -> (worst |err| / bound, case)


@pytest.fixture(scope="module", autouse=True)
def _report_worst():
    yield
    if os.environ.get("LRNDE_TEST_VERBOSE"):
        for prec, (r, case) in sorted(WORST.items()):
            print(f"[bound] worst |err|/bound {prec}: {r:.3g} ({case})")


def _shape_id(row):
    layers, td, input_act, B, _ = row
    net = "-".join(f"{i}x{o}{a[:4]}" for i, o, a in layers)
    return f"{net}{'-td' if td else ''}{'-in' + input_act if input_act else ''}-B{B}"


def _chain(pkg, layers, td, input_act):
    c = pkg.Chain(*[pkg.Dense(i, o, a) for (i, o, a) in layers], input_activation=input_act)
    return pkg.TDChain(c) if td else c


def _rss(W, E):
    """Propagated rounding error W E of independent element errors E: root of the sum of squares."""
    return np.sqrt(np.square(W) @ np.square(E))


def _dact_max(act, pre, Epre):
    """max |act'| over [pre - Epre, pre + Epre] (first order in Epre for the smooth activations)."""
    if act == "relu":
        return (pre + Epre > 0).astype(np.float64)
    return np.minimum(LIP[act], np.abs(_act_grad(act, pre, _act(act, pre))) + K2[act] * Epre)


def _forward_bound(om, u, ps, t, c0, c1):
    """Per layer (x~ = [x; t; 1], its bound, W_aug = [W | b], pre, pre's bound), and the bound of f."""
    B = u.shape[1]
    td = 1 if om.time_dependent else 0
    x, E = u, np.zeros_like(u)
    if om.input_act is not None:
        x = _act(om.input_act, u)
        E = c1 * U * np.maximum(np.abs(x), 1.0)
    layers = []
    for L, (W, b) in zip(om.layers, om.unpack(ps)):
        Wa = np.concatenate([W, b[:, None]], axis=1)
        xt = np.concatenate([x] + ([np.full((1, B), t)] if td else []) + [np.ones((1, B))], axis=0)
        Ext = np.concatenate([E, np.zeros((td + 1, B))], axis=0)
        pre = Wa @ xt
        Epre = c0 * np.sqrt(Wa.shape[1]) * U * (np.abs(Wa) @ np.abs(xt)) + _rss(W[:, :L.in_dims], E)
        x = _act(L.act, pre)
        E = _dact_max(L.act, pre, Epre) * Epre + c1 * U * np.maximum(np.abs(x), 1.0)
        layers.append((xt, Ext, Wa, pre, Epre))
    return layers, E


def _reverse_bound(om, u, layers, lam, c0, c1):
    """Bounds of a = J_u^T lam and of dps = J_p^T lam (oracle parameter layout)."""
    B = u.shape[1]
    g, Eg = lam, np.zeros_like(lam)
    Edps = np.zeros(om.nparams)
    for L, (wo, bo), (xt, Ext, Wa, pre, Epre) in reversed(list(zip(om.layers, om.offsets, layers))):
        d = g * _act_grad(L.act, pre, _act(L.act, pre))
        Ed = Eg * _dact_max(L.act, pre, Epre) + np.abs(g) * (K2[L.act] * Epre + c1 * U)
        EdW = c0 * np.sqrt(B) * U * (np.abs(d) @ np.abs(xt).T) + Ed @ np.abs(xt).T + np.abs(d) @ Ext.T
        Edps[wo:bo] = EdW[:, :-1].ravel(order="F")
        Edps[bo:bo + L.out_dims] = EdW[:, -1]
        Win = Wa[:, :L.in_dims]
        Eg = c0 * np.sqrt(L.out_dims) * U * (np.abs(Win).T @ np.abs(d)) + _rss(Win.T, Ed)
        g = Win.T @ d
    if om.input_act is not None:      # the input itself is exact: only the derivative's own rounding
        Eg = Eg * np.abs(_act_grad(om.input_act, u, _act(om.input_act, u))) + np.abs(g) * c1 * U
    return Eg, Edps


@functools.lru_cache(maxsize=1)
def _reference(row, t):
    """Inputs and Float64 oracle results (f, a, dps) of SHAPES[row] at time t."""
    layers, td, input_act, B, _ = SHAPES[row]
    om = orc.MLP([orc.Dense(*l) for l in layers], time_dependent=td, input_act=input_act)
    rng = np.random.default_rng(row)
    # Glorot x2 plus jitter: every activation in its non-linear range, non-zero biases
    ps = (orc.glorot_uniform_params(om, rng) * 2 + 0.05 * rng.standard_normal(om.nparams)).astype(np.float32)
    u = rng.standard_normal((om.state_dims, B)).astype(np.float32)
    lam = rng.standard_normal((om.state_dims, B)).astype(np.float32)
    t64 = float(np.float32(t))              # the library takes t as a Float32
    u64, ps64 = u.astype(np.float64), ps.astype(np.float64)
    kinked = np.zeros(B, bool)
    if any(L.act == "relu" for L in om.layers):
        fl, _ = _forward_bound(om, u64, ps64, t64, *C_KINK)
        for L, (_, _, _, pre, Epre) in zip(om.layers, fl):
            if L.act == "relu":
                kinked |= np.any(np.abs(pre) <= Epre, axis=0)
        assert kinked.mean() < 0.01, f"{kinked.sum()} of {B} samples within the forward bound of a relu kink"
    lam[:, kinked] = 0.0                    # a zero cotangent column drops the sample from a and dps exactly
    a, dps = om.vjp(u64, ps64, t64, lam.astype(np.float64))
    return dict(om=om, u=u, ps=ps, lam=lam, t=t64, nkinked=int(kinked.sum()), f=om.f(u64, ps64, t64), a=a, dps=dps)


@functools.lru_cache(maxsize=2)
def _bound(row, t, c0, c1):
    """Elementwise bounds of f, a and dps of SHAPES[row] at time t for the constants (c0, c1)."""
    ref = _reference(row, t)
    u64 = ref["u"].astype(np.float64)
    layers, Ef = _forward_bound(ref["om"], u64, ref["ps"].astype(np.float64), ref["t"], c0, c1)
    Ea, Edps = _reverse_bound(ref["om"], u64, layers, ref["lam"].astype(np.float64), c0, c1)
    return dict(f=Ef, a=Ea, dps=Edps)


def _param_block(om, k):
    """(layer, block name, index in the block) of parameter k."""
    for l, (L, (wo, bo)) in enumerate(zip(om.layers, om.offsets)):
        if wo <= k < bo:
            i, j = (k - wo) % L.out_dims, (k - wo) // L.out_dims
            return l + 1, ("W[:, :in]" if j < L.in_dims else "W time column"), (i, j)
        if bo <= k < bo + L.out_dims:
            return l + 1, "b", (k - bo,)
    raise IndexError(k)


def _excess(name, got, want, bound, om=None):
    """Worst |got - want| / bound and a report of where it is."""
    got = np.asarray(got, np.float64)
    assert got.shape == want.shape, (name, got.shape, want.shape)
    err = np.abs(got - want)
    with np.errstate(divide="ignore", invalid="ignore"):
        ratio = np.where(err == 0, 0.0, err / bound)
    ratio[~np.isfinite(got)] = np.inf
    k = int(np.argmax(ratio))
    r = float(ratio.flat[k])
    if name != "dps":
        idx = np.unravel_index(k, want.shape)
        return r, (f"{name}: worst at (row {idx[0]}, sample {idx[1]}): got {got[idx]:.9g} want {want[idx]:.9g} "
                   f"|err| {err[idx]:.3g} bound {bound[idx]:.3g} |err|/bound {r:.3g}")
    lines = []
    for l, (L, (wo, bo)) in enumerate(zip(om.layers, om.offsets)):
        nin = L.out_dims * L.in_dims
        for block, sl in (("W[:, :in]", slice(wo, wo + nin)), ("W time column", slice(wo + nin, bo)),
                          ("b", slice(bo, bo + L.out_dims))):
            if sl.stop > sl.start:
                kb = sl.start + int(np.argmax(ratio[sl]))
                if ratio[kb] > 1 or kb == k:
                    lb, _, ij = _param_block(om, kb)
                    lines.append(f"dps layer {lb} {block}{list(ij)}: got {got[kb]:.9g} want {want[kb]:.9g} "
                                 f"|err| {err[kb]:.3g} bound {bound[kb]:.3g} |err|/bound {ratio[kb]:.3g}")
    return r, "\n".join(lines)


def _check(pkg, row, t, prec, consts, fused_off=None):
    """Worst |err| / bound of f (and, given fused_off, of f with LRNDE_NO_FUSED), a and dps of one precision."""
    layers, td, input_act, B, _ = SHAPES[row]
    ref = _reference(row, t)
    bound = _bound(row, t, *consts)
    node = pkg.NeuralODE(_chain(pkg, layers, td, input_act), precision=prec)
    try:
        f = node.dynamics(ref["u"], ref["ps"], t)
    except pkg._lib.LrndeError as e:
        if prec == "smem" and "does not fit" in str(e):
            pytest.skip(f"the library reports that the network does not fit shared memory: {e}")
        raise
    a, dps = node.dynamics_vjp(ref["u"], ref["ps"], t, ref["lam"])
    got = {"f": f, "a": a, "dps": dps}
    if fused_off is not None:
        fused_off.setenv("LRNDE_NO_FUSED", "1")
        got["f (LRNDE_NO_FUSED)"] = node.dynamics(ref["u"], ref["ps"], t)
        fused_off.delenv("LRNDE_NO_FUSED")
    res = {}
    for name, val in got.items():
        key = name.split()[0]
        res[name] = _excess(key, val, ref[key], bound[key], ref["om"])
    return res, ref["nkinked"]


@pytest.mark.parametrize("row,t,prec", [(r, t, p) for r in range(len(SHAPES)) for t in TIMES for p in PRECS],
                         ids=[f"{_shape_id(SHAPES[r])}-t{t}-{p}" for r in range(len(SHAPES)) for t in TIMES
                              for p in PRECS])
def test_dense_rhs_within_float64_bound(pkg, monkeypatch, row, t, prec):
    """f, J_u^T lam and J_p^T lam of one call each, elementwise within the rounding bound of the Float64 oracle."""
    fused = SHAPES[row][4] and prec in ("tf32x3", "auto")
    res, nkinked = _check(pkg, row, t, prec, CONST[prec], fused_off=monkeypatch if fused else None)
    worst = max(r for r, _ in res.values())
    case = f"{_shape_id(SHAPES[row])} t={t}"
    if os.environ.get("LRNDE_TEST_VERBOSE"):
        print(f"[bound] {case} {prec}: " + " ".join(f"{k}={r:.3g}" for k, (r, _) in res.items()) +
              (f" (relu kink: {nkinked} samples excluded)" if nkinked else ""))
    if worst > WORST.get(prec, (-1.0, ""))[0]:
        WORST[prec] = (worst, case)
    bad = [msg for r, msg in res.values() if r > 1]
    assert not bad, f"{case} {prec}:\n" + "\n".join(bad)


def test_single_pass_tf32_breaks_the_tf32x3_bound(pkg):
    """The bar is tight enough to catch a 3xTF32 path that falls back to one pass (or loses a hi*lo term): single-pass
    TF32 on the mnist_ode shape exceeds the tf32x3 bound at least 10x."""
    assert _shape_id(SHAPES[MNIST_B128]) == "784x100tanh-100x784iden-td-B128"
    res, _ = _check(pkg, MNIST_B128, TIMES[0], "tf32", C_TF32X3)
    worst = max(r for r, _ in res.values())
    if os.environ.get("LRNDE_TEST_VERBOSE"):
        print("[bound] single-pass tf32 against the tf32x3 bound: " + " ".join(f"{k}={r:.3g}" for k, (r, _) in res.items()))
    assert worst >= 10, "\n".join(msg for _, msg in res.values())
