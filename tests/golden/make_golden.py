"""Generate the golden vectors under tests/golden/ from the UNMODIFIED reference CPU path
(oracle/_ref/libenoki_ref.so = /root/reference headers + src/autodiff/autodiff.cpp built by
`make -C oracle ref`).  Run in the dev container (the reference does not travel to the GPU box);
the .npz files are committed.

    python tests/golden/make_golden.py

The tests import make_tape() and ref_math_inputs() from here to regenerate inputs, so the reference
library is only loaded when vectors are written.
"""
import ctypes
import hashlib
import os
import subprocess

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
R = None
P = lambda a: a.ctypes.data_as(ctypes.c_void_p)
SZ = ctypes.c_size_t


def load_ref():
    global R
    R = ctypes.CDLL(os.path.join(ROOT, "oracle", "_ref", "libenoki_ref.so"))


def unary(name, x):
    out = np.zeros_like(x)
    assert R.ref_unary_f32(name.encode(), P(x), P(out), SZ(len(x))) == 0
    return out


def main():
    load_ref()
    rng = np.random.default_rng(20260922)
    # --- C2: fused chain (SURVEY 8d) on 4099 elements
    n = 4099
    xs = [rng.uniform(-4, 4, n).astype(np.float32) for _ in range(4)]
    out = np.zeros(n, np.float32)
    R.ref_c2(*[P(x) for x in xs], P(out), SZ(n))
    np.savez_compressed(os.path.join(HERE, "c2.npz"), x0=xs[0], x1=xs[1], x2=xs[2], x3=xs[3], out=out)

    # --- C1: a*b + sin(c) (tests/dynamic.cpp path), linspace inputs of config #1 at reduced size
    n = 4096
    a = np.linspace(0, 1, n, dtype=np.float32); b = np.linspace(1, 2, n, dtype=np.float32); c = np.linspace(-3, 3, n, dtype=np.float32)
    out = np.zeros(n, np.float32)
    R.ref_c1(P(a), P(b), P(c), P(out), SZ(n))
    np.savez_compressed(os.path.join(HERE, "c1.npz"), a=a, b=b, c=c, out=out)

    # --- unary math on special + random values
    x = np.concatenate([np.array([0, -0.0, np.inf, -np.inf, np.nan, 1, -1, 1e-40, 88.5, -88.5, 8191.5, -8191.5], np.float32),
                        rng.uniform(-50, 50, 2000).astype(np.float32)])
    d = {"x": x}
    for name in ("sin", "cos", "exp", "log", "sqrt", "floor", "ceil", "round", "trunc", "tan", "asin", "acos", "atan",
                 "sinh", "cosh", "tanh", "erf"):
        d[name] = unary(name, x)
    np.savez_compressed(os.path.join(HERE, "unary.npz"), **d)

    # --- double-precision branches of sin/cos/exp/log
    x = np.concatenate([np.array([0, -0.0, np.inf, -np.inf, np.nan, 1, -1, 1e-310, 709.5, -709.5, 710, -710, 8191.5, -8191.5]),
                        rng.uniform(-700, 700, 1000), np.exp(rng.uniform(-700, 700, 1000))]).astype(np.float64)
    d = {"x": x}
    for name in ("sin", "cos", "exp", "log", "sqrt"):
        out = np.zeros_like(x)
        assert R.ref_unary_f64(name.encode(), P(x), P(out), SZ(len(x))) == 0
        d[name] = out
    np.savez_compressed(os.path.join(HERE, "unary_f64.npz"), **d)

    # --- C3 histogram: PCG32 samples -> erfinv -> 31 bins (tests/histogram.cpp:41-57), 2^16 samples
    n = 1 << 16
    u = np.zeros(n, np.float32)
    R.ref_pcg32_f32(ctypes.c_uint64(0), SZ(n), SZ(1), P(u))
    y = np.zeros(n, np.float32)
    R.ref_hist_samples(P(u), P(y), SZ(n))
    table = rng.uniform(0.5, 1.5, 31).astype(np.float32)
    idx = np.zeros(n, np.uint32); bins = np.zeros(31, np.uint32); hist = np.zeros(31, np.float32)
    R.ref_c3(P(y), SZ(n), P(table), P(idx), P(bins), P(hist))
    np.savez_compressed(os.path.join(HERE, "c3.npz"), u=u, y=y, table=table, idx=idx, bins=bins, hist=hist)

    # --- PCG32 raw draws
    m, draws = 257, 4
    pu = np.zeros(m * draws, np.uint32)
    R.ref_pcg32_u32(ctypes.c_uint64(0), SZ(m), SZ(draws), P(pu))
    np.savez_compressed(os.path.join(HERE, "pcg32.npz"), first=0, n=m, draws=draws, u32=pu)

    # --- tape: layered random graph (C4 shape, reduced): L levels x K nodes, width w, 2 in-edges per node
    for tag, (L, K, w) in {"small": (6, 8, 37), "wide": (4, 5, 1000)}.items():
        g = make_tape(rng, L, K, w)
        grads = np.zeros(len(g["want"]) * w, np.float32)
        rc = R.ref_tape_backward(len(g["node_size"]), P(g["node_size"]), len(g["src"]), P(g["src"]), P(g["dst"]),
                                 P(g["weights"]), P(g["woff"]), P(g["wsize"]), int(g["root"]), len(g["want"]), P(g["want"]),
                                 P(grads), 1)
        assert rc == 0
        np.savez_compressed(os.path.join(HERE, f"tape_{tag}.npz"), grads=grads, **g)

    # --- public-API autodiff expressions (tests/autodiff.cpp style)
    x = rng.uniform(0.2, 2.0, 513).astype(np.float32)
    d = {"x": x}
    for which in range(5):
        v = np.zeros_like(x); gr = np.zeros_like(x)
        assert R.ref_ad_expr(which, P(x), SZ(len(x)), P(v), P(gr)) == 0
        d[f"val{which}"] = v; d[f"grad{which}"] = gr
    np.savez_compressed(os.path.join(HERE, "ad_expr.npz"), **d)
    ref_compare()
    print("golden vectors written to", HERE)


MATH_SAMPLE = 2048


def ref_math_inputs():
    """[(name, oracle selector, float32 arguments)]: 2^18 arguments per function, special values first."""
    rng = np.random.default_rng(1)
    n = 1 << 18
    cases = []
    for name, which, gen in [("sin", 0, lambda: rng.uniform(-8192, 8192, n)), ("cos", 1, lambda: rng.uniform(-8192, 8192, n)),
                             ("exp", 2, lambda: rng.uniform(-100, 100, n)), ("log", 3, lambda: np.exp(rng.uniform(-80, 80, n))),
                             ("sqrt", 4, lambda: rng.uniform(0, 1e10, n))]:
        x = gen().astype(np.float32)
        x[:8] = [0, -0.0, np.inf, -np.inf, np.nan, 1, -1, 1e-40]
        cases.append((name, which, x))
    return cases


def ref_math_sample(n):
    """Indices of the stored sample: the special values and a seeded draw from the rest."""
    return np.unique(np.concatenate([np.arange(8), np.random.default_rng(2).integers(8, n, MATH_SAMPLE - 8)]))


def digest_f32(a):
    """SHA-256 of a float32 array with every NaN written as the one quiet NaN (NaN == NaN in the comparisons)."""
    a = np.array(a, np.float32)
    a[np.isnan(a)] = np.nan
    return hashlib.sha256(a.tobytes()).hexdigest()


def ref_compare():
    """What the oracle is compared with: the reference's float32 math on ref_math_inputs() (a sample of arguments and
    results, and the SHA-256 of every result), its rcp / rsqrt at a sample of the GPU test's arguments, the reference
    tape's gradients on make_tape(rng 5, 7, 12, 333), and the
    planner listings that tests/cpp/shim_plan (C++ code through include/enoki/cuda.h under the reference headers) prints."""
    d = {}
    for name, _, x in ref_math_inputs():
        out = unary(name, x)
        idx = ref_math_sample(len(x))
        d["idx"] = idx.astype(np.uint32)
        d[f"{name}_x"] = x[idx]; d[f"{name}_ref"] = out[idx]; d[f"{name}_sha256"] = np.array(digest_f32(out))
    np.savez_compressed(os.path.join(HERE, "ref_math.npz"), **d)

    # rcp / rsqrt of tests/test_gpu_eval.py::test_unary_f32 (rcpps / rsqrtps + one Newton step): a seeded sample
    d = {}
    for name, which, lo, hi in [("rcp", 5, -100, 100), ("rsqrt", 6, 1e-10, 1e10)]:
        x = np.random.default_rng(which).uniform(lo, hi, 1 << 18).astype(np.float32)
        idx = np.unique(np.random.default_rng(3).integers(0, len(x), 4096))
        d[f"{name}_idx"] = idx.astype(np.uint32); d[f"{name}_x"] = x[idx]; d[f"{name}_ref"] = unary(name, x)[idx]
    np.savez_compressed(os.path.join(HERE, "ref_rcp.npz"), **d)

    w = 333
    g = make_tape(np.random.default_rng(5), 7, 12, w)
    grads = np.zeros(len(g["want"]) * w, np.float32)
    assert R.ref_tape_backward(len(g["node_size"]), P(g["node_size"]), len(g["src"]), P(g["src"]), P(g["dst"]), P(g["weights"]),
                               P(g["woff"]), P(g["wsize"]), int(g["root"]), len(g["want"]), P(g["want"]), P(grads), 1) == 0
    np.savez_compressed(os.path.join(HERE, "ref_tape.npz"), grads=grads)

    out = subprocess.run([os.path.join(ROOT, "tests", "cpp", "shim_plan")], capture_output=True, text=True, check=True).stdout
    with open(os.path.join(HERE, "shim_plan.txt"), "w") as f:
        f.write(out)


def make_tape(rng, L, K, w, zero_frac=0.01):
    """SURVEY 8d C4 generator: L levels x K nodes of width w; every non-leaf node has 2 in-edges
    to random nodes of the previous level; weights U(0.5,1.5) with a few exact zeros; loss = size-1
    node with a weight-1 edge from every node of the last level."""
    node_size, src, dst, woff, wsize, ws = [], [], [], [], [], []
    off = 0
    for lvl in range(L):
        for k in range(K):
            node_size.append(w)
            nid = lvl * K + k + 1
            if lvl > 0:
                picks = rng.choice(K, 2, replace=False)
                for p in sorted(picks):
                    src.append((lvl - 1) * K + int(p) + 1); dst.append(nid)
                    wt = rng.uniform(0.5, 1.5, w).astype(np.float32)
                    wt[rng.uniform(0, 1, w) < zero_frac] = 0.0
                    ws.append(wt); woff.append(off); wsize.append(w); off += w
    node_size.append(1)
    loss = L * K + 1
    for k in range(K):
        src.append((L - 1) * K + k + 1); dst.append(loss)
        ws.append(np.ones(1, np.float32)); woff.append(off); wsize.append(1); off += 1
    return dict(node_size=np.array(node_size, np.uint32), src=np.array(src, np.uint32), dst=np.array(dst, np.uint32),
                weights=np.concatenate(ws), woff=np.array(woff, np.uint64), wsize=np.array(wsize, np.uint32),
                root=np.uint32(loss), want=np.arange(1, K + 1, dtype=np.uint32))


if __name__ == "__main__":
    main()
