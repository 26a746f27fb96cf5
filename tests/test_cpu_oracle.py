"""CPU suite: the oracle (plain-C restatement) against the committed golden vectors generated
from the unmodified reference and the reference's own known-answer values."""
import ctypes
import os

import numpy as np
import pytest

SZ = ctypes.c_size_t
GOLD = os.path.join(os.path.dirname(__file__), "golden")


def test_c2_golden(oracle, P):
    g = np.load(os.path.join(GOLD, "c2.npz"))
    out = np.zeros_like(g["out"])
    oracle.or_c2(P(g["x0"]), P(g["x1"]), P(g["x2"]), P(g["x3"]), P(out), SZ(len(out)))
    assert (out.view(np.uint32) == g["out"].view(np.uint32)).all()


def test_c1_golden(oracle, P):
    g = np.load(os.path.join(GOLD, "c1.npz"))
    out = np.zeros_like(g["out"])
    oracle.or_c1(P(g["a"]), P(g["b"]), P(g["c"]), P(out), SZ(len(out)))
    assert (out.view(np.uint32) == g["out"].view(np.uint32)).all()


@pytest.mark.parametrize("name,which", [("sin", 0), ("cos", 1), ("exp", 2), ("log", 3), ("sqrt", 4),
                                        ("floor", 9), ("ceil", 10), ("round", 11), ("trunc", 12)])
def test_unary_golden(oracle, P, name, which):
    g = np.load(os.path.join(GOLD, "unary.npz"))
    x = g["x"]; out = np.zeros_like(x)
    oracle.or_unary_f32(which, P(x), P(out), SZ(len(x)))
    want = g[name]
    same = (out.view(np.uint32) == want.view(np.uint32)) | (np.isnan(out) & np.isnan(want))
    assert same.all(), (name, x[~same][:5], out[~same][:5], want[~same][:5])


@pytest.mark.parametrize("name,which", [("sin", 0), ("cos", 1), ("exp", 2), ("log", 3), ("sqrt", 4)])
def test_unary_f64_golden(oracle, P, name, which):
    """Double branches of array_math.h sincos/exp/log against vectors from the unmodified reference."""
    g = np.load(os.path.join(GOLD, "unary_f64.npz"))
    x = g["x"]; out = np.zeros_like(x)
    oracle.or_unary_f64(which, P(x), P(out), SZ(len(x)))
    want = g[name]
    same = (out.view(np.uint64) == want.view(np.uint64)) | (np.isnan(out) & np.isnan(want))
    assert same.all(), (name, x[~same][:5], out[~same][:5], want[~same][:5])


def test_transcendental_ulp_bounds(oracle, P, ulp):
    """The reference's own accuracy pins: tests/explog.cpp:65-88 (exp <= 3 ulp on [-20,30], log <= 2 ulp)
    and tests/trig.cpp:3-22 (sin <= 19, cos <= 47 ulp on [-8192, 8192]) against libm in double."""
    rng = np.random.default_rng(0)
    n = 200_000
    def run(which, x):
        out = np.zeros_like(x); oracle.or_unary_f32(which, P(x), P(out), SZ(len(x))); return out
    x = rng.uniform(-20, 30, n).astype(np.float32)
    assert ulp(run(2, x), np.exp(x.astype(np.float64)).astype(np.float32)).max() <= 3
    x = rng.uniform(1e-20, 2e30, n).astype(np.float32)
    assert ulp(run(3, x), np.log(x.astype(np.float64)).astype(np.float32)).max() <= 2
    x = rng.uniform(-8192, 8192, n).astype(np.float32)
    assert ulp(run(0, x), np.sin(x.astype(np.float64)).astype(np.float32)).max() <= 19
    assert ulp(run(1, x), np.cos(x.astype(np.float64)).astype(np.float32)).max() <= 47


def test_pcg32_golden(oracle, P):
    g = np.load(os.path.join(GOLD, "pcg32.npz"))
    n, draws = int(g["n"]), int(g["draws"])
    out = np.zeros(n * draws, np.uint32)
    oracle.or_pcg32_u32(ctypes.c_uint64(int(g["first"])), SZ(n), SZ(draws), P(out))
    assert (out == g["u32"]).all()


def _pcg32_py(initstate, initseq, n):
    """Independent statement of PCG32 (O'Neill, pcg-c-basic) in pure Python."""
    M = (1 << 64) - 1
    st = {"s": 0}
    inc = ((initseq << 1) | 1) & M

    def nxt():
        old = st["s"]
        st["s"] = (old * 0x5851f42d4c957f2d + inc) & M
        xs = (((old >> 18) ^ old) >> 27) & 0xffffffff
        rot = old >> 59
        return ((xs >> rot) | (xs << ((-rot) & 31))) & 0xffffffff
    nxt(); st["s"] = (st["s"] + initstate) & M; nxt()
    return [nxt() for _ in range(n)]


def test_pcg32_known_answer(oracle, P):
    """Published pcg-c-basic demo vector: pcg32_srandom(42, 54) -> 0xa15c02b7 0x7b47f409 0xba1d3330 ...
    pins the pure-Python statement, which in turn pins the oracle for PCG32_DEFAULT_STATE and
    arbitrary streams (random.h:33-68)."""
    assert _pcg32_py(42, 54, 3) == [0xa15c02b7, 0x7b47f409, 0xba1d3330]
    for stream in (0, 1, 77, 0xda3e39cb94b95bdb):
        out = np.zeros(4, np.uint32)
        oracle.or_pcg32_u32(ctypes.c_uint64(stream), SZ(1), SZ(4), P(out))
        assert list(out) == _pcg32_py(0x853c49e6748fea9b, stream, 4)


def test_c3_golden(oracle, P):
    g = np.load(os.path.join(GOLD, "c3.npz"))
    n = len(g["y"])
    idx = np.zeros(n, np.uint32); bins = np.zeros(31, np.uint32); hist = np.zeros(31, np.float32)
    oracle.or_c3(P(g["y"]), SZ(n), P(g["table"]), P(idx), P(bins), P(hist))
    assert (idx == g["idx"]).all() and (bins == g["bins"]).all()
    assert (hist.view(np.uint32) == g["hist"].view(np.uint32)).all()
    u = np.zeros(n, np.float32)
    oracle.or_pcg32_f32(ctypes.c_uint64(0), SZ(n), SZ(1), P(u))
    assert (u == g["u"]).all()


@pytest.mark.parametrize("tag", ["small", "wide"])
def test_tape_golden(oracle, P, tag):
    g = dict(np.load(os.path.join(GOLD, f"tape_{tag}.npz")))
    want = g["grads"]
    got = np.zeros_like(want)
    rc = oracle.or_tape_backward(len(g["node_size"]), P(g["node_size"]), len(g["src"]), P(g["src"]), P(g["dst"]),
                                 P(g["weights"]), P(g["woff"]), P(g["wsize"]), int(g["root"]), len(g["want"]),
                                 P(g["want"]), P(got))
    assert rc == 0
    assert (got.view(np.uint32) == want.view(np.uint32)).all()


def test_morton_roundtrip(oracle, P):
    rng = np.random.default_rng(2)
    x = rng.integers(0, 1 << 16, 10000).astype(np.uint32); y = rng.integers(0, 1 << 16, 10000).astype(np.uint32)
    m = np.zeros_like(x); x2 = np.zeros_like(x); y2 = np.zeros_like(x)
    oracle.or_morton2_encode(P(x), P(y), P(m), SZ(len(x)))
    oracle.or_morton2_decode(P(m), P(x2), P(y2), SZ(len(x)))
    assert (x2 == x).all() and (y2 == y).all()
    assert m[0] == int("".join(b + a for a, b in zip(f"{x[0]:016b}", f"{y[0]:016b}")), 2)


# ---- against what the reference itself computed (golden/ref_*.npz, written by make_golden.ref_compare()) ----------
def _make_golden():
    import sys
    if GOLD not in sys.path:
        sys.path.insert(0, GOLD)
    import make_golden
    return make_golden


def test_oracle_vs_reference_math(oracle, P):
    """Bit for bit (NaN == NaN) on 2^18 arguments per function: at the stored sample value by value, everywhere through the
    SHA-256 of the reference's results."""
    mg = _make_golden()
    g = np.load(os.path.join(GOLD, "ref_math.npz"))
    idx = g["idx"]
    for name, which, x in mg.ref_math_inputs():
        n = len(x)
        assert (x[idx].view(np.uint32) == g[f"{name}_x"].view(np.uint32)).all(), f"{name}: the arguments are not the stored ones"
        b = np.zeros(n, np.float32)
        oracle.or_unary_f32(which, P(x), P(b), SZ(n))
        a = g[f"{name}_ref"]
        same = (a.view(np.uint32) == b[idx].view(np.uint32)) | (np.isnan(a) & np.isnan(b[idx]))
        assert same.all(), (name, x[idx][~same][:5], b[idx][~same][:5], a[~same][:5])
        assert mg.digest_f32(b) == str(g[f"{name}_sha256"]), name


def test_oracle_vs_reference_tape(oracle, P):
    g = _make_golden().make_tape(np.random.default_rng(5), 7, 12, 333)
    a = np.load(os.path.join(GOLD, "ref_tape.npz"))["grads"]
    b = np.zeros_like(a)
    args = (len(g["node_size"]), P(g["node_size"]), len(g["src"]), P(g["src"]), P(g["dst"]), P(g["weights"]), P(g["woff"]),
            P(g["wsize"]), int(g["root"]), len(g["want"]), P(g["want"]))
    assert oracle.or_tape_backward(*args, P(b)) == 0
    assert (a.view(np.uint32) == b.view(np.uint32)).all()


def test_histogram_known_answer(oracle, P):
    """tests/histogram.cpp:68-73: 16 Mi PCG32 samples -> erfinv -> 31 bins; bins[1]==2558, bins[2]==6380,
    743 +- 3 samples out of range.  erfinv is not restated in the oracle (it is traced op-by-op on the
    GPU); the committed golden samples come from the reference.  Here: check the binning rule on the
    2^16 golden samples sums to n minus the out-of-range count."""
    g = np.load(os.path.join(GOLD, "c3.npz"))
    assert int(g["bins"].sum()) + int((g["idx"] >= 31).sum()) == len(g["y"])
