"""CPU suite: the C-ABI library loads, exports every symbol include/enoki_b200.h declares, and the
host logic (trace recording, ref counting, scheduling, slot allocation) behaves like the reference's
jit.cu -- checked through the dry-run planner (no compute calls without a GPU)."""
import os
import re

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def test_library_exports_every_declared_symbol(ek):
    from enoki_b200 import _lib
    lib = ek.lib()
    hdr = open(os.path.join(ROOT, "include", "enoki_b200.h")).read()
    declared = set(re.findall(r"EK_API\s+[\w\s\*]+?\b(ek_\w+)\s*\(", hdr))
    assert len(declared) > 80
    for name in declared:
        assert hasattr(lib, name), f"{name} declared in include/enoki_b200.h but not exported"
    assert declared <= set(_lib.SIGNATURES) | {"ek_debug_plan"}


def test_no_cpu_fallback(ek):
    if ek.device_count() > 0:
        pytest.skip("GPU present")
    lib = ek.lib()
    assert lib.ek_init() == -1
    assert b"no CPU fallback" in lib.ek_last_error()
    x = ek.Float32(1.0) + ek.Float32(2.0)
    with pytest.raises(ek.EnokiError):
        x.eval()


def _fake(ek, n, k=1):
    """n-element 'evaluated' input backed by a fake device address (never dereferenced on CPU)."""
    return ek.Float32.map(0x7f0000000000 + 0x1000000 * k, n)


def test_plan_c2_program(ek):
    n = 1 << 20
    x = [_fake(ek, n, k) for k in range(4)]
    t = ek.fmadd(x[0], x[1], x[2])
    out = ek.fmadd(ek.sin(ek.fmadd(x[3], ek.exp(-(t * t)), x[0])), x[1], ek.sqrt(abs(t)))
    del t                                     # a live Python handle would be stored (jit.cu:1165-1169)
    plan = ek.debug_plan()
    assert "n=1048576 in=4" in plan and "out=1" in plan
    body = [l.split()[1] for l in plan.splitlines() if l.strip().startswith("body")]
    # two-address accumulator code with superinstructions: accumulator loads are fused (a=), -x / |x| are
    # input modifiers of exp / sqrt, the final fmadd takes the accumulator as its addend (FMAC) and stores
    # the result to global memory itself (stg): 9 DAG nodes -> 7 dispatched instructions
    assert body == ["FMA_F32", "MUL_F32", "EXP_F32", "FMA_F32", "SIN_F32", "SQRT_F32", "FMAC_F32"]
    assert " neg " in plan and " abs " in plan and " stg " in plan
    # single-use temporaries stay in the accumulator: only t and sin(...) need slots
    assert "tmp_slots=2" in plan
    del out


def test_plan_division_by_power_of_two_is_a_multiplication(ek):
    x = _fake(ek, 1000)
    a = x / 8.0
    b = x / 3.0
    c = x / -0.25
    plan = ek.debug_plan()
    body = [l.split()[1] for l in plan.splitlines() if l.strip().startswith("body")]
    assert body.count("DIV_F32") == 1 and body.count("MUL_F32") == 2, plan
    del a, b, c


def test_plan_many_inputs_64bit_and_sizes(ek):
    n = 100_000
    # (1) more input streams than staging units: the first 8 are staged (TMA), the rest are direct global loads
    xs = [ek.Float32.map(0x7f0000000000 + 0x1000000 * k, n) for k in range(12)]
    acc = xs[0]
    for x in xs[1:]:
        acc = acc + x
    plan = ek.debug_plan()
    assert "in=8" in plan and plan.count("LDG_32") == 4 and plan.count("ADD_F32") == 11
    del acc
    # (2) 64-bit values travel as two planes: unpack of the staged input, 64-bit ops, 64-bit store
    u = ek.UInt64.map(0x7e0000000000, n)
    v = (u * ek.UInt64(3)) >> ek.UInt64(5)
    plan = ek.debug_plan()
    body = [l.split()[1] for l in plan.splitlines() if l.strip().startswith("body")]
    assert body == ["LD_64", "MUL_I64", "SHR_U64", "ST_64"] and "tmp_slots=2" in plan
    del v
    # (3) one sweep per array size, larger first (jit.cu:1385-1508)
    a = ek.Float32.map(0x7d0000000000, 1000); b = ek.Float32.map(0x7c0000000000, 5000)
    r1 = a * 2.0; r2 = b + 1.0
    sweeps = [l for l in ek.debug_plan().splitlines() if l.startswith("sweep")]
    assert len(sweeps) == 2 and "n=5000" in sweeps[0] and "n=1000" in sweeps[1]
    del r1, r2


def test_plan_reduction_is_epilogue_and_phases(ek):
    n = 4096
    x = _fake(ek, n)
    y = (x * x) / ek.hsum(x * x)
    plan = ek.debug_plan()
    sweeps = [l for l in plan.splitlines() if l.startswith("sweep")]
    assert len(sweeps) == 2
    assert "phase=0" in sweeps[0] and "phase=1" in sweeps[1]
    assert "racc" in plan.lower() and "RFIN" in plan
    assert "scalars=1" in sweeps[1]           # the reduction result is read back as a uniform
    del y


def test_plan_unreferenced_temporaries_are_not_stored(ek):
    n = 1000
    x = _fake(ek, n)
    a = x + 1.0
    b = a * 2.0
    del a
    plan = ek.debug_plan()
    assert plan.count(" stg ") + plan.count("ST_32") == 1    # only b is externally referenced (jit.cu:1165-1169)
    del b
    assert ek.debug_plan() == ""              # nothing live any more


def test_size_mismatch_and_uninitialized_errors(ek):
    a, b = _fake(ek, 3), _fake(ek, 4, 2)
    with pytest.raises(ek.EnokiError, match="incompatible size"):
        _ = a + b
    with pytest.raises(ek.EnokiError, match="uninitialized"):
        _ = a + ek.Float32.from_index(0)


def test_privatised_histogram_plan(ek):
    n = 1 << 16
    y = _fake(ek, n)
    bins = ek.UInt32.map(0x7e0000000000, 31)
    idx = ek.UInt32((y + 4.0) * 31.0 / 8.0)
    mask = idx < ek.UInt32(31)
    lib = ek.lib()
    lib.ek_set_scatter_gather_operand(bins.index, 0)
    ptr = lib.ek_var_register_ptr(0x7e0000000000)
    one = ek.UInt32(1)
    h = lib.ek_trace_append(ek.EK_UINT32, ek.OP["SCATTER_ADD"], ptr, idx.index, mask.index, (4 << 32) | one.index)
    assert h != 0
    lib.ek_var_mark_side_effect(h)
    lib.ek_dec_ref_ext(ptr)
    lib.ek_set_scatter_gather_operand(0, 0)
    plan = ek.debug_plan()
    assert "SCATTER_ADD_I32_SMEM" in plan and "SMEM_ZERO" in plan and "SMEM_FLUSH_ADD_I32" in plan


def test_tape_bookkeeping_cpu(ek):
    """Node/edge ref counting without touching the GPU (autodiff.cpp:681-774)."""
    lib = ek.lib()
    F32 = ek.EK_FLOAT32
    a = lib.ek_tape_append_leaf(F32, 8)
    w = ek.Float32(2.0)
    import ctypes
    idx = (ctypes.c_uint32 * 1)(a); wh = (ctypes.c_uint32 * 1)(w.index)
    b = lib.ek_tape_append(F32, b"mul", 8, 1, idx, wh)
    assert a and b and lib.ek_tape_node_count(F32) == 2
    lib.ek_tape_dec_ref_ext(F32, a)            # still referenced by the edge
    assert lib.ek_tape_node_count(F32) == 2
    lib.ek_tape_dec_ref_ext(F32, b)            # frees b, which releases a
    assert lib.ek_tape_node_count(F32) == 0
    zero = (ctypes.c_uint32 * 1)(0)
    assert lib.ek_tape_append(F32, b"mul", 8, 1, zero, wh) == 0   # no differentiable input -> index 0


def test_simplify_graph_structure_cpu(ek):
    """Greedy vertex elimination (autodiff.cpp:990-1074) is host logic: interior nodes of a chain / a diamond are
    collapsed, their edge weights become traced products (mul_nz / fma_nz), nodes that are still referenced from
    outside stay.  No GPU needed: simplification only records trace nodes."""
    import ctypes
    lib = ek.lib()
    F32 = ek.EK_FLOAT32
    n = 64

    def weight(k):
        return ek.Float32.map(0x7b0000000000 + 0x100000 * k, n)

    def node(label, srcs, ws):
        idx = (ctypes.c_uint32 * len(srcs))(*srcs); wh = (ctypes.c_uint32 * len(ws))(*[w.index for w in ws])
        h = lib.ek_tape_append(F32, label, n, len(srcs), idx, wh)
        assert h
        return h
    assert lib.ek_tape_node_count(F32) == 0
    ws = [weight(k) for k in range(8)]
    leaf = lib.ek_tape_append_leaf(F32, n)
    a = node(b"a", [leaf], [ws[0]])
    b = node(b"b", [a], [ws[1]])
    c = node(b"c", [b], [ws[2]])
    # diamond on top of the chain: d = f(c, c') with c' = g(c)
    c2 = node(b"c2", [c], [ws[3]])
    d = node(b"d", [c, c2], [ws[4], ws[5]])
    for h in (a, b, c, c2):                     # interior nodes lose their external references
        lib.ek_tape_dec_ref_ext(F32, h)
    assert lib.ek_tape_node_count(F32) == 6
    assert lib.ek_tape_simplify(F32) == 0
    # only the leaf and the root survive, joined by one edge whose weight is an unevaluated product chain
    assert lib.ek_tape_node_count(F32) == 2
    plan = ek.debug_plan()
    assert plan.count("MULNZ_F32") + plan.count("FMANZ") >= 4, plan
    roots = (ctypes.c_uint32 * 1)(d)
    gv = lib.ek_tape_graphviz(F32, 1, roots)
    from enoki_b200 import _lib
    text = _lib.take_string(gv)
    assert text.count("->") == 1
    lib.ek_tape_dec_ref_ext(F32, d)
    lib.ek_tape_dec_ref_ext(F32, leaf)
    assert lib.ek_tape_node_count(F32) == 0


def test_cpp_header_shim_records_the_same_programs(ek):
    """The C++ drop-in header (include/enoki/cuda.h under the reference's router / array_math.h) must record what the
    Python mirror records: tests/cpp/shim_plan prints the planner's listing for expressions written as user C++ code.
    Its listing is stored in tests/golden/shim_plan.txt; where the program is built (it needs the reference headers at
    compile time) it must still print exactly that."""
    import subprocess
    listing = open(os.path.join(ROOT, "tests", "golden", "shim_plan.txt")).read()
    binp = os.path.join(ROOT, "tests", "cpp", "shim_plan")
    if os.path.exists(binp):
        out = subprocess.run([binp], capture_output=True, text=True, timeout=120)
        assert out.returncode == 0, out.stderr
        assert out.stdout == listing
    sections = dict((s.split("\n", 1)[0].strip(), s.split("\n", 1)[1]) for s in listing.split("== ")[1:])
    import gc
    gc.collect(); ek.lib().ek_debug_discard_side_effects(); gc.collect()      # scatters recorded by earlier tests
    assert ek.debug_plan() == ""
    # C2 through the Python mirror
    n = 1 << 20
    x = [_fake(ek, n, k) for k in range(4)]
    t = ek.fmadd(x[0], x[1], x[2])
    o = ek.fmadd(ek.sin(ek.fmadd(x[3], ek.exp(-(t * t)), x[0])), x[1], ek.sqrt(abs(t)))
    del t
    want = ek.debug_plan()
    del o
    strip = lambda s: "\n".join(re.sub(r"imm=0x[0-9a-f]+", "", l).rstrip() for l in s.strip().splitlines())
    assert strip(sections["c2"]) == strip(want)
    # reduction feeding a later phase, conversions, select: structure of the second listing
    ph = sections["phases"]
    sweeps = [l for l in ph.splitlines() if l.startswith("sweep")]
    assert len(sweeps) == 2 and "phase=0" in sweeps[0] and "phase=1" in sweeps[1] and "scalars=1" in sweeps[1]
    assert "RFIN" in ph and "CVT_F32_U32" in ph and "SEL_T_32" in ph


def test_resize_of_a_lazy_reduction_broadcasts(ek):
    """ADVICE r1 (medium): hsum() is a lazy size-1 variable here; resize() must give a broadcasting MOV node like it does
    for an evaluated scalar (jit.cu:357-364), not relabel the reduce node as wide (its sweep writes 8 bytes)."""
    import gc
    from enoki_b200 import Float32, hsum
    gc.collect(); ek.lib().ek_debug_discard_side_effects(); gc.collect()
    x = Float32.map(0x7f0000000000, 500)
    s = hsum(x * 2.0)
    red = s.index
    L = ek.lib()
    h = L.ek_var_set_size(red, 500, 1)
    assert h != 0 and h != red, "a new (MOV) variable is expected"
    assert L.ek_var_size(h) == 500
    s.index = h                                 # the call consumed the caller's reference on `red` (jit.cu:362)
    plan = ek.debug_plan()
    assert "n=500" in plan and "RFIN" in plan
    # without `copy` the reference refuses to resize an (evaluated) scalar: jit.cu:366-371
    s2 = hsum(x)
    assert L.ek_var_set_size(s2.index, 500, 0) == 0 and b"resize" in L.ek_last_error()
    del s, s2, x
    gc.collect(); ek.lib().ek_debug_discard_side_effects()


def test_qualification_battery_records_and_plans():
    """enoki_b200/ek_qualify --dry: every program of the kernel-qualification battery (csrc/ek_qualify.cpp) is recorded
    through the C ABI and planned in both modes (general kernels / fast kernel) on the host -- the battery itself must not be
    what fails on the GPU box."""
    import os
    import subprocess
    root = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
    exe = os.path.join(root, "enoki_b200", "ek_qualify")
    assert os.path.exists(exe), "enoki_b200/ek_qualify is not built (make -C enoki_b200/csrc)"
    r = subprocess.run([exe, "--dry"], capture_output=True, text=True, timeout=300)
    assert r.returncode == 0, r.stderr[-2000:]
    assert "recorded and planned in both modes" in r.stderr
