"""In-kernel timeline of ladj::adj_chain_kernel (trace build: LRNDE_TRACE=1 python localregneuralde.jl_b200/build.py).
    python scratch/adj_trace.py [B]"""
import os, sys, ctypes as C, numpy as np, torch
sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
import __graft_entry__ as entry
pkg = entry.load_package(); L = C.CDLL(pkg.LIB_PATH)
dev = torch.device("cuda", 0)
ctx = pkg.Context(0, torch.cuda.current_stream(dev).cuda_stream)
chain = pkg.TDChain(pkg.Chain(pkg.Dense(784, 100, "tanh"), pkg.Dense(100, 784)))
B = int(sys.argv[1]) if len(sys.argv) > 1 else 8192
node = pkg.NeuralODE(chain, ctx=ctx, abstol=1.4e-8, reltol=1.4e-8, precision="tf32x3", regularize="unbiased")
ps = torch.from_numpy(node.initialparameters(np.random.default_rng(0))).to(dev)
x = torch.rand((B, 784), device=dev).t()
for it in range(2):
    sol, st2 = node(x, ps, node.initialstates(np.random.default_rng(1)))
    node.backward(sol, [(torch.randn((B, 784), device=dev) / B).t() for _ in sol.u], 0.0)
buf = (C.c_longlong * 1024)()
L.lrnde_debug_trace_adj(buf, 1024)
a = np.array(buf[:]).reshape(64, 16)
t0 = a[0, 0]
names = ["misc[start,A in TMEM,-,stages done,dbt done,end]", "stage top", "eps tile put", "prefetch done", "-", "-",
         "xi ready", "mma issue", "mma issued"]
for i, nm in enumerate(names):
    print(f"{nm:56s}", " ".join(f"{int(v - t0):7d}" if v else "      ." for v in a[i][:6]))
