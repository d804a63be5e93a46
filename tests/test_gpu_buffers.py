"""Every C entry point that takes host_buffers gives the same bits from host arrays (numpy) as from device arrays
(torch CUDA tensors), and a device call leaves each of its input arrays unchanged.

Each case runs once per side on the same small inputs.  Device inputs are views whose wrapper conversion is a no-op,
so the library reads (and could write) the tensor the test holds; after the call every such tensor is compared with
a copy taken before it."""
import ctypes as C

import numpy as np
import pytest

import __graft_entry__ as entry

pytestmark = pytest.mark.gpu


@pytest.fixture(scope="module")
def pkg():
    return entry.load_package()


class Dev:
    """Device copies of host arrays, with a snapshot of each to check the call left it alone."""

    def __init__(self):
        import torch
        self.torch, self.kept = torch, []

    def __call__(self, a, layout="rev"):
        """A CUDA tensor equal to ``a`` whose storage the wrappers hand to the library as is: ``rev`` for the
        column-major wrappers (reversed axes), ``flat`` for arrays passed unchanged."""
        torch = self.torch
        a = np.asarray(a)
        if layout == "flat":
            t = torch.from_numpy(np.ascontiguousarray(a)).cuda()
            self.kept.append((t, t.clone()))
            return t
        rev = tuple(reversed(range(a.ndim)))
        base = torch.from_numpy(np.ascontiguousarray(a.transpose(rev))).cuda()
        self.kept.append((base, base.clone()))
        return base.permute(*rev)

    def check_unchanged(self):
        self.torch.cuda.synchronize()
        for t, snap in self.kept:
            assert self.torch.equal(t.view(self.torch.int32), snap.view(self.torch.int32))


def same(d, h):
    """Bit-identical (device result vs host result)."""
    d = d.detach().cpu().numpy() if hasattr(d, "detach") else np.asarray(d)
    h = np.asarray(h)
    assert d.shape == h.shape and d.dtype == h.dtype
    assert np.array_equal(np.ascontiguousarray(d).view(np.uint8), np.ascontiguousarray(h).view(np.uint8))


def ptr(a):
    if a is None:
        return None
    return C.c_void_p(a.data_ptr()) if hasattr(a, "data_ptr") else C.c_void_p(a.ctypes.data)


def rand(rng, *shape, scale=1.0):
    return (scale * rng.standard_normal(shape)).astype(np.float32)


@pytest.mark.parametrize("precision", ["fp32", "smem"])
def test_dynamics_eval_and_vjp(pkg, precision):
    rng = np.random.default_rng(1)
    chain = pkg.Chain(pkg.Dense(12, 16, "tanh"), pkg.Dense(16, 12))
    node = pkg.NeuralODE(chain, precision=precision)
    ps = node.initialparameters(rng)
    u, lam = rand(rng, 12, 37), rand(rng, 12, 37)
    dev = Dev()
    same(node.dynamics(dev(u), dev(ps, "flat"), 0.3), node.dynamics(u, ps, 0.3))
    ctx, L = node.ctx, pkg.lib()
    out = {}
    for host in (True, False):
        o, _ = node._opts("none", 0.0, 0.0, False, host)
        if host:
            args = [np.ascontiguousarray(u.T), ps, np.ascontiguousarray(lam.T)]
            a, dps = np.empty((37, 12), np.float32), np.empty(ps.size, np.float32)
        else:
            args = [dev(u.T, "flat"), dev(ps, "flat"), dev(lam.T, "flat")]
            a, dps = (dev.torch.empty((37, 12), device="cuda"), dev.torch.empty(ps.size, device="cuda"))
        pkg._lib.check(L.lrnde_dynamics_vjp(ctx._h, ctx.model_handle(chain), C.byref(o), ptr(args[1]), ptr(args[0]),
                                            0.3, ptr(args[2]), 37, ptr(a), ptr(dps)))
        out[host] = (a, dps)
    same(out[False][0], out[True][0])
    same(out[False][1], out[True][1])
    dev.check_unchanged()


def test_ode_forward_saved_states_backward_and_classifier_grad(pkg):
    rng = np.random.default_rng(2)
    chain = pkg.TDChain(pkg.Chain(pkg.Dense(16, 24, "tanh"), pkg.Dense(24, 16)))
    node = pkg.NeuralODE(chain, regularize="biased", abstol=1e-4, reltol=1e-4, precision="fp32")
    ps = node.initialparameters(rng)
    x = rand(rng, 16, 40)
    st = node.initialstates(np.random.default_rng(3))
    sol_h, st_h = node(x, ps, st)
    dev = Dev()
    sol_d, st_d = node(dev(x), dev(ps, "flat"), st)
    assert st_d["nfe"] == st_h["nfe"] and st_d["reg_val"] == st_h["reg_val"] and len(sol_d.u) == len(sol_h.u) > 3
    assert sol_d.t == sol_h.t
    for ud, uh in zip(sol_d.u, sol_h.u):
        same(ud, uh)
    cots = [rand(rng, 16, 40) for _ in sol_h.u]
    dx_h, dps_h = node.backward(sol_h, cots, 0.7)
    dx_d, dps_d = node.backward(sol_d, [dev(c) for c in cots], 0.7)
    same(dx_d, dx_h)
    same(dps_d, dps_h)
    for f in ("nf_bwd", "naccept_bwd", "nreject_bwd", "retcode_bwd"):
        assert getattr(sol_d.bwd_stats, f) == getattr(sol_h.bwd_stats, f)

    # the classifier's gradient: NeuralODE (u(t2) only) + Dense head + cross entropy
    cls = pkg.NeuralODE(chain, regularize="unbiased", abstol=1e-4, reltol=1e-4, precision="fp32")
    Cn, B = 5, 40
    wc, labels = rand(rng, Cn * 17, scale=0.3), rng.integers(0, Cn, B).astype(np.int32)
    L, ctx = pkg.lib(), cls.ctx
    out = {}
    for host in (True, False):
        o, _ = cls._opts("unbiased", 0.4, 0.0, True, host)
        if host:
            args = [ps, wc, np.ascontiguousarray(x.T), labels]
            loss, dps, dwc = C.c_float(), np.empty(ps.size, np.float32), np.empty(wc.size, np.float32)
        else:
            args = [dev(ps, "flat"), dev(wc, "flat"), dev(x.T, "flat"), dev(labels, "flat")]
            loss = C.c_float()
            dps, dwc = dev.torch.empty(ps.size, device="cuda"), dev.torch.empty(wc.size, device="cuda")
        stats = pkg._lib.Stats()
        pkg._lib.check(L.lrnde_classifier_grad(ctx._h, ctx.model_handle(chain), C.byref(o), *[ptr(a) for a in args],
                                               B, Cn, 0.1, 1.0, C.byref(loss), ptr(dps), ptr(dwc), C.byref(stats)))
        out[host] = (loss.value, dps, dwc, stats.nfe, stats.nf_bwd, stats.reg_val)
    assert out[False][0] == out[True][0] and out[False][3:] == out[True][3:]
    same(out[False][1], out[True][1])
    same(out[False][2], out[True][2])
    dev.check_unchanged()


@pytest.mark.parametrize("with_du", [True, False])
def test_head_ce(pkg, with_du):
    rng = np.random.default_rng(4)
    D, B, Cn = 20, 50, 7
    wc, u, labels = rand(rng, Cn * (D + 1)), rand(rng, B, D), rng.integers(0, Cn, B).astype(np.int32)
    L, ctx, dev = pkg.lib(), pkg.default_context(0), Dev()
    out = {}
    for host in (True, False):
        if host:
            args, mk = [wc, u, labels], (lambda n: np.empty(n, np.float32))
        else:
            args, mk = [dev(wc, "flat"), dev(u, "flat"), dev(labels, "flat")], (lambda n: dev.torch.empty(n, device="cuda"))
        loss, du, dwc = C.c_float(), (mk(D * B) if with_du else None), mk(wc.size)
        pkg._lib.check(L.lrnde_head_ce(ctx._h, *[ptr(a) for a in args], B, D, Cn, 1 if host else 0, C.byref(loss),
                                       ptr(du), ptr(dwc)))
        out[host] = (loss.value, du, dwc)
    assert out[False][0] == out[True][0]
    if with_du:
        same(out[False][1], out[True][1])
    same(out[False][2], out[True][2])
    dev.check_unchanged()


def _sde(pkg, **kw):
    drift = pkg.Chain(pkg.Dense(6, 10, "tanh"), pkg.Dense(10, 6))
    diffusion = pkg.Chain(pkg.Dense(6, 8, "tanh"), pkg.Dense(8, 6))
    return pkg.NeuralDSDE(drift, diffusion, **kw)


def test_sosri_step(pkg):
    rng = np.random.default_rng(5)
    sde = _sde(pkg)
    ps = sde.initialparameters(rng)
    nf = pkg.nparams(sde.drift)
    D, B = 6, 33
    uprev, dW, dZ = rand(rng, B, D), rand(rng, B, D, scale=0.1), rand(rng, B, D, scale=0.1)
    L, ctx, dev = pkg.lib(), sde.ctx, Dev()
    node = pkg.NeuralODE(sde.drift, precision="fp32")
    out = {}
    for host in (True, False):
        o, _ = node._opts("none", 0.0, 0.0, False, host)
        if host:
            args, u = [ps[:nf], ps[nf:], uprev, dW, dZ], np.empty((B, D), np.float32)
        else:
            args = [dev(ps[:nf], "flat"), dev(ps[nf:], "flat"), dev(uprev, "flat"), dev(dW, "flat"), dev(dZ, "flat")]
            u = dev.torch.empty((B, D), device="cuda")
        reg = C.c_float()
        pkg._lib.check(L.lrnde_sosri_step(ctx._h, ctx.model_handle(sde.drift), ctx.model_handle(sde.diffusion),
                                          C.byref(o), *[ptr(a) for a in args], 0.2, 0.05, 1.0 / 6.0, B, ptr(u),
                                          C.byref(reg)))
        out[host] = (u, reg.value)
    same(out[False][0], out[True][0])
    assert out[False][1] == out[True][1]
    dev.check_unchanged()


@pytest.mark.parametrize("kind", ["RKMilCommute", "LambaEulerHeun"])
def test_sde_aux_step(pkg, kind):
    rng = np.random.default_rng(6)
    sde = _sde(pkg)
    ps = sde.initialparameters(rng)
    uprev, dW = rand(rng, 6, 45), rand(rng, 6, 45, scale=0.1)
    dev = Dev()
    u_h, r_h = sde.perform_step(kind, ps, uprev, dW, 0.1, 0.05)
    u_d, r_d = sde.perform_step(kind, dev(ps, "flat"), dev(uprev), dev(dW), 0.1, 0.05)
    same(u_d, u_h)
    assert r_d == r_h
    dev.check_unchanged()


def test_sde_forward_states_backward(pkg):
    rng = np.random.default_rng(7)
    sde = _sde(pkg, regularize="biased", abstol=1e-2, reltol=1e-2)
    ps = sde.initialparameters(rng)
    x = rand(rng, 6, 40)
    st = sde.initialstates(np.random.default_rng(8))
    sol_h, st_h = sde(x, ps, st)
    dev = Dev()
    sol_d, st_d = sde(dev(x), dev(ps, "flat"), st)
    for k in ("nfe_drift", "nfe_diffusion", "reg_val"):
        assert st_d[k] == st_h[k]
    assert sol_d.t == sol_h.t and len(sol_d.u) == len(sol_h.u) > 2
    for ud, uh in zip(sol_d.u, sol_h.u):
        same(ud, uh)
    cots = [rand(rng, 6, 40) for _ in sol_h.u]
    dx_h, dps_h = sde.backward(sol_h, cots, 0.5)
    dx_d, dps_d = sde.backward(sol_d, [dev(c) for c in cots], 0.5)
    same(dx_d, dx_h)
    same(dps_d, dps_h)
    dev.check_unchanged()


def test_gru_forward_backward(pkg):
    rng = np.random.default_rng(9)
    cell = pkg.LatentGRUCell(3, 12, 4)
    rec = pkg.Recurrence(cell)
    ps = cell.initialparameters(rng)
    x = rand(rng, cell.features, 5, 21)
    d_y = rand(rng, 8, 21)
    dev = Dev()
    y_h, st_h = rec(x, ps)
    y_d, st_d = rec(dev(x), dev(ps, "flat"))
    same(y_d, y_h)
    same(rec.backward(st_d, dev(d_y)), rec.backward(st_h, d_y))
    rec.free(st_h)
    rec.free(st_d)
    dev.check_unchanged()


@pytest.mark.parametrize("with_dx", [True, False])
def test_mlp_forward_backward(pkg, with_dx):
    rng = np.random.default_rng(10)
    model = pkg.Chain(pkg.Dense(8, 14, "tanh"), pkg.Dense(14, 5))
    ps = pkg.glorot_uniform(model, rng)
    x, d_y = rand(rng, 8, 3, 11), rand(rng, 5, 3, 11)
    dev = Dev()
    same(pkg.mlp_forward(model, dev(ps, "flat"), dev(x)), pkg.mlp_forward(model, ps, x))
    L, ctx = pkg.lib(), pkg.default_context(0)
    descs = pkg.layers._layer_descs(model)
    out = {}
    for host in (True, False):
        if host:
            args = [ps, np.ascontiguousarray(x.T), np.ascontiguousarray(d_y.T)]
            mk = lambda *s: np.empty(s, np.float32)
        else:
            args = [dev(ps, "flat"), dev(x.T, "flat"), dev(d_y.T, "flat")]
            mk = lambda *s: dev.torch.empty(s, device="cuda")
        d_x, d_ps = (mk(33, 8) if with_dx else None), mk(ps.size)
        pkg._lib.check(L.lrnde_mlp_backward(ctx._h, descs, 2, *[ptr(a) for a in args], 33, 1 if host else 0,
                                            ptr(d_x), ptr(d_ps)))
        out[host] = (d_x, d_ps)
    if with_dx:
        same(out[False][0], out[True][0])
    same(out[False][1], out[True][1])
    dev.check_unchanged()


def test_reparameterize_and_latent_loss(pkg):
    rng = np.random.default_rng(11)
    Lz, B = 4, 19
    x = rand(rng, 2 * Lz, B)
    d_mu, d_ls = rand(rng, Lz, B), rand(rng, Lz, B)
    rep = pkg.ReparameterizeLayer(seed=3)
    dev = Dev()
    same(rep(dev(x))[0], rep(x)[0])
    same(rep.backward(dev(x), None, dev(d_mu), dev(d_ls)), rep.backward(x, None, d_mu, d_ls))
    F, T = 3, 6
    pred, data = rand(rng, F, T, B), rand(rng, F, T, B)
    mask = (rng.random((F, T, B)) < 0.7).astype(np.float32)
    mu, ls = rand(rng, Lz, B), rand(rng, Lz, B, scale=0.2)
    h = pkg.latent_loss(pred, data, mask, mu, ls, 0.3)
    d = pkg.latent_loss(dev(pred), dev(data), dev(mask), dev(mu), dev(ls), 0.3)
    assert d[:3] == h[:3]
    for a, b in zip(d[3:], h[3:]):
        same(a, b)
    dev.check_unchanged()
