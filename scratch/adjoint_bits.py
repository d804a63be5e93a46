"""Forward + backward of NeuralODE on the shapes the hidden-space adjoint routes on, written out for a bitwise
comparison of two builds (d_x, d_ps and the backward step log of every case).

    python scratch/adjoint_bits.py OUTDIR              # run this tree's build, write OUTDIR/<case>.npz
    python scratch/adjoint_bits.py --compare DIR1 DIR2  # numpy.array_equal on every array of every case
"""
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

# (D, H, activation, B)
SHAPES = [(16, 12, "tanh", 1), (16, 12, "tanh", 37), (16, 12, "tanh", 65), (33, 70, "gelu", 65),
          (784, 100, "tanh", 96), (784, 100, "tanh", 8192), (784, 100, "tanh", 9001),
          (24, 20, "sigmoid", 33), (24, 20, "relu", 33), (24, 20, "identity", 33)]
TOLS = (1e-3, 1.4e-8)


def cases():
    for (D, H, act, B) in SHAPES:
        for td in (True, False):
            for tol in TOLS:
                yield f"{D}x{H}{act}-B{B}-{'td' if td else 'notd'}-tol{tol:g}", (D, H, act, B, td, tol)


def run(outdir):
    sys.path.insert(0, ROOT)
    import __graft_entry__ as entry
    pkg = entry.load_package()
    os.makedirs(outdir, exist_ok=True)
    for name, (D, H, act, B, td, tol) in cases():
        c = pkg.Chain(pkg.Dense(D, H, act), pkg.Dense(H, D))
        node = pkg.NeuralODE(pkg.TDChain(c) if td else c, abstol=tol, reltol=tol, precision="tf32x3",
                             regularize="unbiased", save_start=False)
        rng = np.random.default_rng(7)
        ps = (node.initialparameters(rng) * 3.0).astype(np.float32)
        x = (rng.random((D, B)) if D >= 100 else rng.standard_normal((D, B))).astype(np.float32)
        cot = [(rng.standard_normal((D, B)) / B).astype(np.float32) for _ in range(2)]
        sol, st2 = node(x, ps, node.initialstates(np.random.default_rng(3)))
        d_x, d_ps = node.backward(sol, cot, 0.9)
        t, dt, eest, acc = sol.step_log(1)
        np.savez(os.path.join(outdir, name + ".npz"), d_x=np.asarray(d_x), d_ps=np.asarray(d_ps),
                 blog_t=np.asarray(t), blog_dt=np.asarray(dt), blog_eest=np.asarray(eest), blog_acc=np.asarray(acc),
                 nf_bwd=np.int64(sol.bwd_stats.nf_bwd))
        print(f"{name}: bwd steps {len(acc)} nf_bwd {sol.bwd_stats.nf_bwd}", flush=True)
        sol.free()


def compare(d1, d2):
    bad = 0
    for name, _ in cases():
        a, b = np.load(os.path.join(d1, name + ".npz")), np.load(os.path.join(d2, name + ".npz"))
        diff = [k for k in a.files if not np.array_equal(a[k], b[k])]
        bad += bool(diff)
        print(f"{name:40s} {'identical' if not diff else 'DIFFERENT: ' + ', '.join(diff)}")
    print(f"{bad} of {len(list(cases()))} cases differ")
    return bad


if __name__ == "__main__":
    if sys.argv[1] == "--compare":
        sys.exit(1 if compare(sys.argv[2], sys.argv[3]) else 0)
    run(sys.argv[1])
