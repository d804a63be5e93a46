"""Generates tests/golden/*.npz from the CPU oracle (oracle/lrnde_oracle.py).

The reference (Julia) cannot run in this image and holds no golden vectors of its own
(test/runtests.jl asserts only finiteness), so these fixtures pin the ORACLE: the CPU suite
checks the oracle still reproduces them, the GPU suite checks libLRNDE.so against them.

    python tests/golden/make_golden.py
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))
import oracle as orc  # noqa: E402

CASES = {
    # name: (layers [(in,out,act)...], td, input_act, B, kwargs, seed, d_reg)
    "tiny_td_gelu": ([(2, 4, "gelu"), (4, 2, "identity")], True, None, 3,
                     dict(regularize="unbiased"), 0, 2.5),
    "tiny_plain_biased": ([(2, 4, "gelu"), (4, 2, "identity")], False, None, 1,
                          dict(regularize="biased"), 1, 1.0),
    "mid_tanh_stiff": ([(16, 12, "tanh"), (12, 16, "identity")], True, None, 8,
                       dict(regularize="unbiased", regularize_type="stiffness_estimate",
                            abstol=1e-6, reltol=1e-6), 2, 0.7),
    "latent_saveat": ([(20, 40, "tanh"), (40, 20, "tanh"), (20, 40, "tanh"), (40, 20, "tanh")],
                      False, "tanh", 16,
                      dict(regularize="unbiased", abstol=1e-6, reltol=1e-6,
                           saveat=[0.0, 0.13, 0.37, 0.5, 0.81, 1.0]), 3, 0.3),
    "mnist_b16": ([(784, 100, "tanh"), (100, 784, "identity")], True, None, 16,
                  dict(regularize="unbiased", abstol=1e-6, reltol=1e-6, maxiters=10000,
                       save_start=False), 4, 2.5),
    "eval_mode": ([(5, 7, "sigmoid"), (7, 5, "relu")], True, None, 6,
                  dict(regularize="unbiased", abstol=1e-7, reltol=1e-5), 5, 0.0),
    # truncation-dominated regimes (weights x3: the Float32 and Float64 oracles agree on every
    # step to ~1e-5), where two Float32 implementations CAN be compared tightly
    "mid_x3_err": ([(16, 12, "tanh"), (12, 16, "identity")], True, None, 8,
                   dict(regularize="unbiased", abstol=1e-3, reltol=1e-3), 2, 0.7),
    "mid_x3_stiff": ([(16, 12, "tanh"), (12, 16, "identity")], True, None, 8,
                     dict(regularize="unbiased", regularize_type="stiffness_estimate",
                          abstol=1e-3, reltol=1e-3), 2, 0.7),
    "gelu3_x3_biased": ([(10, 24, "gelu"), (24, 24, "tanh"), (24, 10, "identity")], False, None, 33,
                        dict(regularize="biased", abstol=1e-3, reltol=1e-3), 6, 1.3),
}
SCALE = {"mid_x3_err": 3.0, "mid_x3_stiff": 3.0, "gelu3_x3_biased": 3.0}


def _run(model, kw, seed, name, x, ps, cots_in, d_reg, dtype, t1_index=None):
    node = orc.NeuralODE(model, dtype=dtype, pow_mode="fastpow_2023", **kw)
    st = node.initialstates(np.random.default_rng(seed + 100))
    if name == "eval_mode":
        st["training"] = False
    if t1_index is not None:       # :biased -- pin the sampled step index across dtypes
        class _R:
            def integers(self, lo, hi):
                return min(t1_index, hi - 1)
        st["rng"] = _R()
    sol, st2, aux = node.forward(x.astype(dtype), ps.astype(dtype), st)
    cots = cots_in(sol)
    d_x, d_ps = node.backward(aux, cots, d_reg, ps.astype(dtype))
    bsol = aux["bsol"]
    _, d_ps0 = node.backward(aux, cots, 0.0, ps.astype(dtype))     # adjoint part only
    aux["bsol"] = bsol
    aux["d_ps0"] = d_ps0
    return sol, st2, aux, cots, d_x, d_ps


def build(name):
    layers, td, input_act, B, kw, seed, d_reg = CASES[name]
    model = orc.MLP([orc.Dense(*l) for l in layers], time_dependent=td, input_act=input_act)
    rng = np.random.default_rng(seed)
    ps = orc.glorot_uniform_params(model, rng)
    if name in SCALE:
        ps = (ps * np.float32(SCALE[name]) + (0.1 * rng.standard_normal(ps.size))).astype(np.float32)
    elif layers[0][0] < 100:
        ps = ps + (0.1 * rng.standard_normal(ps.size)).astype(np.float32)   # non-zero biases
    else:
        # fresh Glorot weights give dynamics so slow that the Float32 error estimate is pure
        # rounding noise (EEst ~ 2e-3, the Float64 twin says 2e-4); x5 makes it truncation-
        # dominated so that step sequences of two Float32 implementations are comparable
        ps = (ps * np.float32(5.0)).astype(np.float32)
        ps[model.offsets[0][1]:model.offsets[0][1] + 100] = 0.1 * rng.standard_normal(100)
    D = layers[0][0]
    x = (rng.random((D, B), dtype=np.float32) if D == 784
         else rng.standard_normal((D, B)).astype(np.float32))
    crng = np.random.default_rng(seed + 7)
    cot_last = crng.standard_normal((D, B)).astype(np.float32)

    def cots_in(sol):
        r = np.random.default_rng(seed + 8)
        c = [r.standard_normal((D, B)).astype(np.float32) for _ in sol.u]
        c[-1] = cot_last
        if name in ("tiny_td_gelu", "mnist_b16") or kw.get("regularize") == "biased":
            c = [None] * (len(c) - 1) + [cot_last]     # the loss reads sol.u[end] only
        return c

    t1_index = 1 if kw.get("regularize") == "biased" else None
    sol, st2, aux, cots, d_x, d_ps = _run(model, kw, seed, name, x, ps, cots_in, d_reg, np.float32, t1_index)
    # Float64 twin: the size of the Float32 rounding noise in every compared quantity
    _, st64, aux64, _, d_x64, d_ps64 = _run(model, kw, seed, name, x, ps, cots_in, d_reg, np.float64, t1_index)
    s = aux["sol"]
    s64 = aux64["sol"]
    log64 = np.array([(t, dt, e, a) for (t, dt, e, a) in s64.step_log], dtype=np.float64)
    log = np.array([(t, dt, e, a) for (t, dt, e, a) in s.step_log], dtype=np.float64)
    blog = np.array([(t, dt, e, a) for (t, dt, e, a) in aux["bsol"].step_log], dtype=np.float64)
    out = dict(
        x=x, ps=ps, t=np.array(sol.t, np.float32), u=np.stack(sol.u, 0),
        cot=np.stack([np.zeros((D, B), np.float32) if c is None else c for c in cots], 0),
        cot_mask=np.array([c is not None for c in cots]),
        d_reg=np.float32(d_reg), d_x=d_x.astype(np.float32), nfe=np.int64(st2["nfe"]),
        reg_val=np.float32(st2["reg_val"]), naccept=np.int64(s.naccept), nreject=np.int64(s.nreject),
        step_log=log, bwd_step_log=blog, nf_bwd=np.int64(aux["bsol"].nf),
        t1=np.float32(aux.get("t1", 0.0)), dt_reg=np.float32(aux.get("dt_reg", 0.0)),
        step_log64=log64, reg_val64=np.float64(st64["reg_val"]),
        n_bwd64=np.int64(len(aux64["bsol"].step_log)),
        d_ps_rel64=np.float64(np.abs(d_ps64 - d_ps).max() / np.abs(d_ps64).max()),
        d_x_rel64=np.float64(np.abs(d_x64 - d_x).max() / (np.abs(d_x64).max() + 1e-300)),
    )
    stride = 53 if d_ps.size > 20000 else 1      # keep the fixture small: strided sample + norm
    d_ps0, d_ps0_64 = aux["d_ps0"], aux64["d_ps0"]
    out["d_ps_stride"] = np.int64(stride)
    out["d_ps"] = d_ps[::stride].astype(np.float32)
    out["d_ps_norm"] = np.float64(np.linalg.norm(d_ps.astype(np.float64)))
    out["d_ps0"] = d_ps0[::stride].astype(np.float32)
    out["d_ps0_norm"] = np.float64(np.linalg.norm(d_ps0.astype(np.float64)))
    out["d_ps0_rel64"] = np.float64(np.abs(d_ps0_64 - d_ps0).max() / np.abs(d_ps0_64).max())
    return out


if __name__ == "__main__":
    for name in CASES:
        out = build(name)
        np.savez_compressed(os.path.join(HERE, name + ".npz"), **out)
        n = min(len(out["step_log"]), len(out["step_log64"]))
        print(name, "nfe", out["nfe"], "reg32/64", out["reg_val"], out["reg_val64"], "steps", out["naccept"],
              out["nreject"], "f64 attempts", len(out["step_log64"]), "bwd attempts", len(out["bwd_step_log"]),
              "max|t32-t64|", np.abs(out["step_log"][:n, 0] - out["step_log64"][:n, 0]).max(),
              "dps rel32/64", out["d_ps_rel64"], "dps0", out["d_ps0_rel64"], "dx", out["d_x_rel64"])
