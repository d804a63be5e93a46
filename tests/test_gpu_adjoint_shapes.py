"""The hidden-space adjoint (csrc/lrnde_adjoint.cu) against the per-layer engines (LRNDE_NO_FUSED=1) at shapes where
its tiling branches: a single sample, a ragged last 64-sample tile, a second activation, with and without the time
column.  Same checks and bounds as test_gpu_parity.py::test_latent_space_engines_match_the_layer_engines."""
import os

import numpy as np
import pytest

import __graft_entry__ as entry

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    entry.build()
    return entry.load_package()


def rel(a, b):
    a = np.asarray(a, np.float64)
    b = np.asarray(b, np.float64)
    return float(np.abs(a - b).max() / (np.abs(b).max() + 1e-30))


# (D, H, activation, B, time column)
SHAPES = [(16, 12, "tanh", 1, True), (16, 12, "tanh", 65, True), (16, 12, "tanh", 65, False),
          (24, 20, "sigmoid", 33, True)]


@pytest.mark.parametrize("shape", SHAPES, ids=lambda s: f"{s[0]}x{s[1]}{s[2]}-B{s[3]}-{'td' if s[4] else 'notd'}")
def test_latent_adjoint_matches_the_layer_engines(pkg, shape):
    D, H, act, B, td = shape
    rng = np.random.default_rng(11)
    kw = dict(regularize="unbiased", abstol=1e-3, reltol=1e-3, save_start=False, precision="tf32x3")

    def node():
        c = pkg.Chain(pkg.Dense(D, H, act), pkg.Dense(H, D))
        return pkg.NeuralODE(pkg.TDChain(c) if td else c, **kw)

    ps = (node().initialparameters(rng) * (3 if D < 100 else 5)).astype(np.float32)
    x = (rng.standard_normal((D, B)) if D < 100 else rng.random((D, B))).astype(np.float32)
    cot = [(rng.standard_normal((D, B)) / B).astype(np.float32) for _ in range(2)]
    out = {}
    for mode in ("latent", "layers"):
        if mode == "layers":
            os.environ["LRNDE_NO_FUSED"] = "1"
        try:
            n = node()
            sol, st2 = n(x, ps, n.initialstates(np.random.default_rng(3)))
            d_x, d_ps = n.backward(sol, cot, 0.9)
            out[mode] = dict(u=[np.asarray(u).copy() for u in sol.u], reg=float(st2["reg_val"]), nfe=st2["nfe"],
                             log=sol.step_log(0), blog=sol.step_log(1), d_x=np.asarray(d_x).copy(),
                             d_ps=np.asarray(d_ps).copy(), nfb=sol.bwd_stats.nf_bwd)
            sol.free()
        finally:
            os.environ.pop("LRNDE_NO_FUSED", None)
    a, b = out["latent"], out["layers"]
    assert a["nfe"] == b["nfe"] and a["nfb"] == b["nfb"]
    assert np.array_equal(a["log"][3], b["log"][3]) and np.array_equal(a["blog"][3], b["blog"][3])
    np.testing.assert_allclose(a["log"][1], b["log"][1], rtol=2e-3)
    for ua, ub in zip(a["u"], b["u"]):
        assert rel(ua, ub) < 2e-5, rel(ua, ub)
    assert abs(a["reg"] - b["reg"]) <= 2e-3 * abs(b["reg"]), (a["reg"], b["reg"])
    assert rel(a["d_x"], b["d_x"]) < 3e-4 and rel(a["d_ps"], b["d_ps"]) < 3e-4, (rel(a["d_x"], b["d_x"]), rel(a["d_ps"], b["d_ps"]))
