/*
 * ek_qualify.cpp -- kernel qualification battery (builds enoki_b200/ek_qualify; started by ek_init(), see the
 * comment in ek_runtime.cpp "kernel qualification").
 *
 * Every program below is recorded through the public C ABI and evaluated TWICE: with the 32-bit fast sweep kernel
 * switched off (general kernels: the path that passed the round-1 GPU test-suite) and switched on.  Both kernels run
 * the same device functions for every operation (ek_math.cuh), so all element-wise results and all integer results
 * must agree bit for bit; float reductions and float scatter_add totals are folded in a different order by the two
 * kernels and are compared against each other with the tolerance the parity tests use (1e-5 relative).
 * Exit status 0 = every comparison agreed, the fast kernel really executed the second pass, AND it is not slower than the
 * general kernel on C2 on this GPU (device time at 2^24 elements; timings written to the file named by argv[1]).
 *
 * Not a test of the backend against the reference (that is tests/ with oracle/): it only decides whether the fast
 * kernel may replace the general one on this machine.  Nothing here touches oracle/.
 */
#include "../../include/enoki_b200.h"
#include <cmath>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <functional>
#include <string>
#include <vector>

namespace {

struct H {                       /* scoped external reference */
    uint32_t h = 0;
    H() = default;
    explicit H(uint32_t v) : h(v) { if (!v) { fprintf(stderr, "ek_qualify: %s\n", ek_last_error()); exit(3); } }
    H(const H &o) : h(o.h) { if (h) ek_inc_ref_ext(h); }
    H(H &&o) noexcept : h(o.h) { o.h = 0; }
    H &operator=(H o) { std::swap(h, o.h); return *this; }
    ~H() { if (h) ek_dec_ref_ext(h); }
};

const ek_type F = EK_FLOAT32, U = EK_UINT32, I = EK_INT32, B = EK_BOOL;

uint32_t bits(float f) { uint32_t u; memcpy(&u, &f, 4); return u; }
H litf(float v) { return H(ek_trace_append(F, EK_OP_LITERAL, 0, 0, 0, bits(v))); }
H litu(uint32_t v, ek_type t = U) { return H(ek_trace_append(t, EK_OP_LITERAL, 0, 0, 0, v)); }
H op1(ek_type t, ek_op op, const H &a, uint64_t imm = 0) { return H(ek_trace_append(t, op, a.h, 0, 0, imm)); }
H op2(ek_type t, ek_op op, const H &a, const H &b) { return H(ek_trace_append(t, op, a.h, b.h, 0, 0)); }
H op3(ek_type t, ek_op op, const H &a, const H &b, const H &c) { return H(ek_trace_append(t, op, a.h, b.h, c.h, 0)); }
bool g_dry = false;                 /* --dry: record every program and plan it (host only, no GPU): checks the battery itself */
extern "C" char *ek_debug_plan(void);
extern "C" void ek_debug_discard_side_effects(void);
uintptr_t g_fake = 0x7f0000000000ull;
H upload(ek_type t, size_t n, const void *p) {
    if (g_dry) { g_fake += 0x100000000ull; return H(ek_var_register(t, n, (void *) g_fake, 0)); }
    return H(ek_var_copy_to_device(t, n, p));
}
int eval_all() {
    if (!g_dry) return ek_eval();
    char *plan = ek_debug_plan();
    if (!plan) return -1;
    free(plan);
    ek_debug_discard_side_effects();
    return 0;
}
H arange(size_t n) {
    H i(ek_trace_append(U, EK_OP_INDEX, 0, 0, 0, 0));
    if (!ek_var_set_size(i.h, n, 0)) { fprintf(stderr, "ek_qualify: %s\n", ek_last_error()); exit(3); }
    return i;
}
H gather(ek_type t, const H &src, const H &idx, const H &mask) {
    ek_set_scatter_gather_operand(src.h, 1);
    uint32_t p = ek_var_register_ptr(ek_var_ptr(src.h));
    H r(ek_trace_append(t, EK_OP_GATHER, p, idx.h, mask.h, 4));
    ek_dec_ref_ext(p);
    ek_set_scatter_gather_operand(0, 0);
    return r;
}
void scatter(ek_op op, ek_type vt, const H &dst, const H &val, const H &idx, const H &mask) {
    ek_set_scatter_gather_operand(dst.h, 0);
    uint32_t p = ek_var_register_ptr(ek_var_ptr(dst.h));
    uint32_t h = ek_trace_append(op == EK_OP_SCATTER_ADD ? vt : EK_UINT64, op, p, idx.h, mask.h, (4ull << 32) | val.h);
    if (!h) { fprintf(stderr, "ek_qualify: %s\n", ek_last_error()); exit(3); }
    ek_var_mark_side_effect(h);
    ek_dec_ref_ext(p);
    ek_var_mark_dirty(dst.h);
    ek_set_scatter_gather_operand(0, 0);
}

struct Result { std::string name; std::vector<uint8_t> bytes; int kind; double tol, scale; };
/* kind 0: exact; kind 1: f32 values, |a - b| <= tol * scale (scale 0: the largest finite |a| of the array) */
std::vector<Result> *g_out = nullptr;

void keep(const std::string &name, const H &v, int kind = 0, double tol = 1e-5, double scale = 0) {
    if (g_dry) { if (eval_all() != 0) { fprintf(stderr, "ek_qualify: %s: %s\n", name.c_str(), ek_last_error()); exit(3); } return; }
    if (ek_eval_var(v.h) != 0) { fprintf(stderr, "ek_qualify: %s: %s\n", name.c_str(), ek_last_error()); exit(3); }
    ek_sync();
    size_t n = ek_var_size(v.h);
    ek_type t = ek_var_type(v.h);
    size_t es = (t == EK_BOOL || t == EK_UINT8 || t == EK_INT8) ? 1 : (t == EK_INT64 || t == EK_UINT64 || t == EK_FLOAT64) ? 8 : 4;
    Result r; r.name = name; r.kind = kind; r.tol = tol; r.scale = scale; r.bytes.resize(n * es);
    ek_memcpy_from_device(r.bytes.data(), ek_var_ptr(v.h), n * es);
    g_out->push_back(std::move(r));
}

struct Rng {
    uint64_t s;
    explicit Rng(uint64_t seed) : s(seed * 0x9e3779b97f4a7c15ull + 0x1234567ull) {}
    uint32_t next() { s ^= s << 13; s ^= s >> 7; s ^= s << 17; return (uint32_t) (s >> 16); }
    uint32_t below(uint32_t n) { return next() % n; }
    float uniform(float lo, float hi) { return lo + (hi - lo) * (float) (next() & 0xffffff) / 16777216.f; }
};

/* random expression DAG over f32 / u32 values (the shape of tests/test_gpu_fuzz.py), a few outputs kept alive, the
   rest temporaries; reductions on top */
void random_dag(uint64_t seed, size_t n) {
    Rng rng(seed);
    std::vector<std::vector<float>> hf(3, std::vector<float>(n));
    std::vector<std::vector<uint32_t>> hu(2, std::vector<uint32_t>(n));
    for (auto &a : hf) for (auto &x : a) x = rng.uniform(-4.f, 4.f);
    for (auto &a : hu) for (auto &x : a) x = rng.next() ^ (rng.next() << 16);
    /* special values in the stream */
    hf[0][0] = 0.f; hf[0][1 % n] = -0.f; hf[1][2 % n] = INFINITY; hf[2][3 % n] = NAN; hf[1][4 % n] = 1e-41f;
    float sc = rng.uniform(-2.f, 2.f); uint32_t su = 1 + rng.below(99);
    std::vector<H> fl, it;
    for (auto &a : hf) fl.push_back(upload(F, n, a.data()));
    fl.push_back(upload(F, 1, &sc));                    /* evaluated scalar: uniform-pool operand */
    for (auto &a : hu) it.push_back(upload(U, n, a.data()));
    it.push_back(upload(U, 1, &su));
    int nodes = 8 + (int) rng.below(32);
    for (int k = 0; k < nodes; ++k) {
        uint32_t kind = rng.below(22);
        const H a = fl[rng.below((uint32_t) fl.size())], b = fl[rng.below((uint32_t) fl.size())], c = fl[rng.below((uint32_t) fl.size())];
        const H i = it[rng.below((uint32_t) it.size())], j = it[rng.below((uint32_t) it.size())];
        switch (kind) {
            case 0: fl.push_back(op2(F, EK_OP_ADD, a, b)); break;
            case 1: fl.push_back(op2(F, EK_OP_SUB, a, b)); break;
            case 2: fl.push_back(op2(F, EK_OP_MUL, a, b)); break;
            case 3: fl.push_back(op3(F, EK_OP_FMA, a, b, c)); break;
            case 4: fl.push_back(op2(F, rng.below(2) ? EK_OP_MAX : EK_OP_MIN, a, b)); break;
            case 5: fl.push_back(op1(F, EK_OP_ABS, a)); break;
            case 6: fl.push_back(op1(F, EK_OP_NEG, a)); break;
            case 7: fl.push_back(op1(F, EK_OP_SQRT, op1(F, EK_OP_ABS, a))); break;
            case 8: fl.push_back(op1(F, rng.below(2) ? EK_OP_FLOOR : EK_OP_CEIL, a)); break;
            case 9: { static const ek_op fn[4] = { EK_OP_SIN, EK_OP_EXP, EK_OP_COS, EK_OP_LOG }; fl.push_back(op1(F, fn[rng.below(4)], a)); } break;
            case 10: fl.push_back(op3(F, EK_OP_SELECT, op2(B, EK_OP_LT, a, b), a, c)); break;
            case 11: it.push_back(op2(U, EK_OP_ADD, i, j)); break;
            case 12: it.push_back(op2(U, EK_OP_MUL, i, j)); break;
            case 13: it.push_back(op2(U, EK_OP_OR, op2(U, EK_OP_XOR, i, j), op2(U, EK_OP_AND, i, j))); break;
            case 14: { uint32_t s = 1 + rng.below(30); it.push_back(op2(U, EK_OP_OR, op2(U, EK_OP_SHL, i, litu(s)), op2(U, EK_OP_SHR, j, litu(s)))); } break;
            case 15: it.push_back(op3(U, EK_OP_SELECT, op2(B, EK_OP_LT, i, j), i, j)); break;
            case 16: {
                H v = op2(F, EK_OP_MIN, op1(F, EK_OP_ABS, a), litf(1.0e6f));
                it.push_back(op1(U, EK_OP_CVT, v));
                fl.push_back(op1(F, EK_OP_CVT, op2(U, EK_OP_SHR, i, litu(8))));
            } break;
            /* literal operands in every position (the _U twins and the broadcast path) */
            case 17: fl.push_back(op3(F, EK_OP_FMA, a, litf(rng.uniform(-2, 2)), b)); break;
            case 18: fl.push_back(op3(F, EK_OP_FMA, a, b, litf(rng.uniform(-2, 2)))); break;
            case 19: fl.push_back(op2(F, rng.below(2) ? EK_OP_SUB : EK_OP_DIV, litf(rng.uniform(1, 3)), a)); break;
            case 20: fl.push_back(op3(F, EK_OP_SELECT, op2(B, EK_OP_GE, a, litf(0.25f)), litf(1.5f), b)); break;
            default: it.push_back(op2(U, EK_OP_SUB, op2(U, EK_OP_MAX, i, litu(1000u)), op2(U, EK_OP_MIN, j, litu(77u)))); break;
        }
    }
    char nm[64];
    std::vector<H> keep_f, keep_i;
    for (int k = 0; k < 4; ++k) keep_f.push_back(fl[rng.below((uint32_t) fl.size())]);
    for (int k = 0; k < 3; ++k) keep_i.push_back(it[rng.below((uint32_t) it.size())]);
    H red_i = op1(U, EK_OP_HSUM, keep_i[0]), red_f = op1(F, EK_OP_HSUM, keep_f[0]);
    /* (x86 max with a NaN operand returns the second operand, so a maximum over data with NaNs depends on the fold
       order, which differs between the kernels: take it over the NaN-free values) */
    H red_m = op1(F, EK_OP_HMAX, op3(F, EK_OP_SELECT, op2(B, EK_OP_EQ, keep_f[1], keep_f[1]), keep_f[1], litf(0.f)));
    fl.clear(); it.clear();
    if (eval_all() != 0) { fprintf(stderr, "ek_qualify: %s\n", ek_last_error()); exit(3); }
    for (size_t k = 0; k < keep_f.size(); ++k) { snprintf(nm, sizeof(nm), "dag%llu.f%zu", (unsigned long long) seed, k); keep(nm, keep_f[k]); }
    for (size_t k = 0; k < keep_i.size(); ++k) { snprintf(nm, sizeof(nm), "dag%llu.i%zu", (unsigned long long) seed, k); keep(nm, keep_i[k]); }
    snprintf(nm, sizeof(nm), "dag%llu.hsum_u32", (unsigned long long) seed); if (ek_var_size(keep_i[0].h) > 1) keep(nm, red_i);
    {   /* float sum: the two kernels fold in different orders -> compare relative to the sum of magnitudes */
        double mag = 0; if (!g_dry) { const Result &r0 = (*g_out)[g_out->size() - keep_f.size() - keep_i.size() - (ek_var_size(keep_i[0].h) > 1 ? 1 : 0)];
        const float *x = (const float *) r0.bytes.data();
        for (size_t k = 0; k < r0.bytes.size() / 4; ++k) if (std::isfinite(x[k])) mag += std::fabs((double) x[k]); }
        snprintf(nm, sizeof(nm), "dag%llu.hsum_f32", (unsigned long long) seed); if (ek_var_size(keep_f[0].h) > 1) keep(nm, red_f, 1, 4e-6, mag + 1e-30);
    }
    snprintf(nm, sizeof(nm), "dag%llu.hmax_f32", (unsigned long long) seed); if (ek_var_size(keep_f[1].h) > 1) keep(nm, red_m);
}

void directed(size_t n) {
    Rng rng(4242 + n);
    std::vector<float> h0(n), h1(n), h2(n), h3(n);
    for (size_t i = 0; i < n; ++i) { h0[i] = rng.uniform(-4, 4); h1[i] = rng.uniform(-4, 4); h2[i] = rng.uniform(-4, 4); h3[i] = rng.uniform(-4, 4); }
    H x0 = upload(F, n, h0.data()), x1 = upload(F, n, h1.data()), x2 = upload(F, n, h2.data()), x3 = upload(F, n, h3.data());
    {   /* C2 (bench.py): fused arith + exp / sin / sqrt chain, with the fused hsum */
        H t = op3(F, EK_OP_FMA, x0, x1, x2);
        H u = op1(F, EK_OP_EXP, op1(F, EK_OP_NEG, op2(F, EK_OP_MUL, t, t)));
        H v = op1(F, EK_OP_SIN, op3(F, EK_OP_FMA, x3, u, x0));
        H out = op3(F, EK_OP_FMA, v, x1, op1(F, EK_OP_SQRT, op1(F, EK_OP_ABS, t)));
        H s = op1(F, EK_OP_HSUM, out);
        t = H(); u = H(); v = H();
        keep("c2.out", out);
        double mag = 0; if (!g_dry) { const float *x = (const float *) g_out->back().bytes.data(); for (size_t k = 0; k < n; ++k) if (std::isfinite(x[k])) mag += std::fabs((double) x[k]); }
        keep("c2.hsum", s, 1, 4e-6, mag + 1e-30);
    }
    for (uint32_t bound : { 30u, 31u }) {   /* C3 (tests/histogram.cpp:41-57 shape): 31-entry table, 31 integer + 31 float bins;
                                               bound 31: the mask is implied by the bin count (assembler peephole), 30: it is not */
        std::vector<float> tab(31); for (int k = 0; k < 31; ++k) tab[k] = 0.5f + (float) k / 30.f;
        std::vector<uint32_t> zb(31, 0u); std::vector<float> zh(31, 0.f);
        H table = upload(F, 31, tab.data()), bins = upload(U, 31, zb.data()), hist = upload(F, 31, zh.data());
        H idx = op1(U, EK_OP_CVT, op2(F, EK_OP_DIV, op2(F, EK_OP_MUL, op2(F, EK_OP_SUB, x0, litf(-4.f)), litf(31.f)), litf(8.f)));
        H mask = op2(B, EK_OP_LT, idx, litu(bound));
        H w = gather(F, table, idx, mask);
        scatter(EK_OP_SCATTER_ADD, U, bins, litu(1u), idx, mask);
        scatter(EK_OP_SCATTER_ADD, F, hist, w, idx, mask);
        idx = H(); mask = H(); w = H();
        if (eval_all() != 0) { fprintf(stderr, "ek_qualify: %s\n", ek_last_error()); exit(3); }
        keep(bound == 31u ? "c3.bins" : "c3m.bins", bins); keep(bound == 31u ? "c3.hist" : "c3m.hist", hist, 1);
    }
    {   /* global gather / scatter / scatter_add (targets too large for shared memory), masked */
        const size_t m = 6000;
        std::vector<float> src(m); for (auto &v : src) v = rng.uniform(-1, 1);
        std::vector<uint32_t> hi(n); for (auto &v : hi) v = rng.below((uint32_t) m + 50);      /* some out of range: masked off */
        std::vector<uint32_t> zu(m, 0u); std::vector<float> zf(m, 0.f);
        H S = upload(F, m, src.data()), IDX = upload(U, n, hi.data()), TU = upload(U, m, zu.data()), TF = upload(F, m, zf.data());
        H ok = op2(B, EK_OP_LT, IDX, litu((uint32_t) m));
        H g = gather(F, S, IDX, ok);
        keep("gs.gather", op2(F, EK_OP_MUL, g, x1));
        scatter(EK_OP_SCATTER_ADD, U, TU, op2(U, EK_OP_AND, IDX, litu(7u)), IDX, ok);
        scatter(EK_OP_SCATTER_ADD, F, TF, x2, IDX, ok);
        if (eval_all() != 0) { fprintf(stderr, "ek_qualify: %s\n", ek_last_error()); exit(3); }
        keep("gs.add_u32", TU); keep("gs.add_f32", TF, 1);
        /* plain scatter of a permutation (no conflicts: order-independent) */
        std::vector<uint32_t> perm(n); for (size_t i = 0; i < n; ++i) perm[i] = (uint32_t) ((i * 7919u + 13u) % n);
        std::vector<uint8_t> seen(n, 0); bool is_perm = true; for (auto p : perm) { if (seen[p]) is_perm = false; seen[p] = 1; }
        if (is_perm) {
            std::vector<float> zz(n, 0.f);
            H P = upload(U, n, perm.data()), T2 = upload(F, n, zz.data());
            scatter(EK_OP_SCATTER, F, T2, op2(F, EK_OP_ADD, x0, x3), P, litu(1u, B));
            if (eval_all() != 0) { fprintf(stderr, "ek_qualify: %s\n", ek_last_error()); exit(3); }
            keep("gs.scatter", T2);
        }
    }
    {   /* mask arrays as outputs (8-bit stores) and as staged inputs (8-bit loads) of a later sweep; counts */
        H m1 = op2(B, EK_OP_GT, x0, x1), m2 = op2(B, EK_OP_LE, x2, litf(0.5f));
        H m = op2(B, EK_OP_OR, op2(B, EK_OP_AND, m1, m2), op1(B, EK_OP_NOT, m1));
        keep("mask.out", m);
        H sel = op3(F, EK_OP_SELECT, m, x0, op2(F, EK_OP_MUL, x1, litf(2.f)));      /* m now has storage: staged as bytes */
        keep("mask.select", sel);
        keep("mask.count", op1(U, EK_OP_COUNT, m)); keep("mask.any", op1(B, EK_OP_ANY, m2)); keep("mask.all", op1(B, EK_OP_ALL, m2));
    }
    {   /* index arithmetic with literals, signed ops, conversions with rounding modes */
        H i = arange(n);
        H h = op2(U, EK_OP_ADD, op2(U, EK_OP_MUL, i, litu(2654435761u)), litu(974711u));
        h = op2(U, EK_OP_MUL, op2(U, EK_OP_XOR, h, op2(U, EK_OP_SHR, h, litu(15u))), litu(2246822519u));
        keep("int.hash", h);
        H s = op1(I, EK_OP_CVT, op2(F, EK_OP_MUL, x0, litf(1000.f)));
        H s2 = op2(I, EK_OP_MAX, op2(I, EK_OP_SHR, s, litu(3u, I)), op1(I, EK_OP_NEG, op1(I, EK_OP_ABS, s)));
        keep("int.signed", s2);
        keep("int.floor2int", op1(I, EK_OP_FLOOR2INT, x1)); keep("int.ceil2int", op1(I, EK_OP_CEIL2INT, x1));
        keep("int.tofloat", op2(F, EK_OP_ADD, op1(F, EK_OP_CVT, s), op1(F, EK_OP_CVT, h)));
        keep("int.lt", op2(B, EK_OP_LT, s, litu(0u, I)));
        /* the remaining 32-bit operations of the fast kernel's set: integer multiply-add, signed / unsigned min, shifts by
           an array, every comparison, NOT, float rounding modes */
        H u2 = op2(U, EK_OP_AND, h, litu(31u));
        keep("int.mad", op3(U, EK_OP_FMA, h, u2, i));
        keep("int.minmax", op2(I, EK_OP_MIN, s, op2(I, EK_OP_SUB, litu(100u, I), s)));
        keep("int.shifts", op2(U, EK_OP_XOR, op2(U, EK_OP_SHL, h, u2), op2(I, EK_OP_SHR, s, op2(I, EK_OP_AND, s, litu(7u, I)))));
        keep("int.not", op1(U, EK_OP_NOT, h));
        H cmp = op2(B, EK_OP_OR, op2(B, EK_OP_OR, op2(B, EK_OP_NE, h, i), op2(B, EK_OP_GE, s, litu(5u, I))),
                    op2(B, EK_OP_AND, op2(B, EK_OP_LE, x0, x1), op2(B, EK_OP_NE, x2, x3)));
        keep("cmp.mix", op2(B, EK_OP_XOR, cmp, op2(B, EK_OP_GT, h, litu(0x80000000u))));
        keep("f32.round", op2(F, EK_OP_ADD, op1(F, EK_OP_ROUND, op2(F, EK_OP_MUL, x0, litf(3.3f))), op1(F, EK_OP_TRUNC, op2(F, EK_OP_MUL, x1, litf(2.7f)))));
        keep("f32.eq", op3(F, EK_OP_SELECT, op2(B, EK_OP_EQ, op1(F, EK_OP_FLOOR, x0), op1(F, EK_OP_FLOOR, x1)), x2, x3));
    }
    {   /* reductions: min / max / prod, integer sum, a reduction reused by a wide consumer (second phase) */
        keep("red.hmin", op1(F, EK_OP_HMIN, op2(F, EK_OP_MUL, x0, x1)));
        keep("red.hmax", op1(F, EK_OP_HMAX, op1(F, EK_OP_SIN, x2)));
        keep("red.hprod", op1(F, EK_OP_HPROD, op3(F, EK_OP_FMA, x3, litf(1e-4f), litf(1.f))), 1, 2e-3);
        H sq = op2(F, EK_OP_MUL, x0, x0);
        keep("red.normalised", op2(F, EK_OP_DIV, sq, op1(F, EK_OP_HSUM, sq)), 1);
        keep("red.mulnz", op3(F, EK_OP_FMA_NZ, x0, op1(F, EK_OP_FLOOR, x1), op2(F, EK_OP_MUL_NZ, x2, op1(F, EK_OP_FLOOR, x3))));
        keep("red.rcp", op2(F, EK_OP_ADD, op1(F, EK_OP_RCP, x0), op1(F, EK_OP_RSQRT, op1(F, EK_OP_ABS, x1))));
    }
}

void battery(std::vector<Result> &out) {
    g_out = &out;
    static const size_t sizes[] = { 4097, 100003, (1u << 20) + 5u };
    for (uint64_t seed = 0; seed < 18; ++seed) random_dag(seed, sizes[seed % 3]);
    directed(100003);
    directed((1u << 21) + 3u);
}

} // namespace

/* device time (per-launch CUDA events, ek_set_timing) of the C2 expression and of the C3 histogram in the current mode */
static void time_c2_c3(size_t n, double &c2_ms, double &c3_ms) {
    std::vector<float> h(n);
    Rng rng(99);
    H x[4];
    for (int k = 0; k < 4; ++k) { for (auto &v : h) v = rng.uniform(-4, 4); x[k] = upload(F, n, h.data()); }
    auto c2 = [&]() {
        H t = op3(F, EK_OP_FMA, x[0], x[1], x[2]);
        H u = op1(F, EK_OP_EXP, op1(F, EK_OP_NEG, op2(F, EK_OP_MUL, t, t)));
        H v = op1(F, EK_OP_SIN, op3(F, EK_OP_FMA, x[3], u, x[0]));
        H out = op3(F, EK_OP_FMA, v, x[1], op1(F, EK_OP_SQRT, op1(F, EK_OP_ABS, t)));
        t = H(); u = H(); v = H();
        if (eval_all() != 0) { fprintf(stderr, "ek_qualify: %s\n", ek_last_error()); exit(3); }
    };
    std::vector<float> tab(31); for (int k = 0; k < 31; ++k) tab[k] = 0.5f + (float) k / 30.f;
    H table = upload(F, 31, tab.data());
    auto c3 = [&]() {
        std::vector<uint32_t> zb(31, 0u); std::vector<float> zh(31, 0.f);
        H bins = upload(U, 31, zb.data()), hist = upload(F, 31, zh.data());
        H idx = op1(U, EK_OP_CVT, op2(F, EK_OP_DIV, op2(F, EK_OP_MUL, op2(F, EK_OP_SUB, x[0], litf(-4.f)), litf(31.f)), litf(8.f)));
        H mask = op2(B, EK_OP_LT, idx, litu(31u));
        H w = gather(F, table, idx, mask);
        scatter(EK_OP_SCATTER_ADD, U, bins, litu(1u), idx, mask);
        scatter(EK_OP_SCATTER_ADD, F, hist, w, idx, mask);
        idx = H(); mask = H(); w = H();
        if (eval_all() != 0) { fprintf(stderr, "ek_qualify: %s\n", ek_last_error()); exit(3); }
    };
    std::function<void()> fns[2] = { c2, c3 };
    for (int pass = 0; pass < 2; ++pass) {
        fns[pass](); fns[pass]();
        if (g_dry) continue;
        ek_sync();
        ek_set_timing(1); ek_stats_reset();
        for (int r = 0; r < 5; ++r) fns[pass]();
        ek_stats st; ek_stats_get(&st);
        ek_set_timing(0);
        (pass == 0 ? c2_ms : c3_ms) = st.sweep_launches ? st.total_kernel_ms / (double) st.sweep_launches : 0.0;
    }
}

int main(int argc, char **argv) {
    if (argc > 1 && strcmp(argv[1], "--dry") == 0) {
        g_dry = true;
        std::vector<Result> none;
        for (int mode = 0; mode < 2; ++mode) { ek_set_fast_mode(mode); battery(none); double a = 0, b = 0; time_c2_c3(100003, a, b); }
        fprintf(stderr, "ek_qualify --dry: every program of the battery was recorded and planned in both modes\n");
        return 0;
    }
    if (ek_device_count() == 0) { fprintf(stderr, "ek_qualify: no CUDA device\n"); return 2; }
    if (ek_init() != 0) { fprintf(stderr, "ek_qualify: %s\n", ek_last_error()); return 2; }
    std::vector<Result> ref, fast;
    ek_set_fast_mode(0);
    battery(ref);
    ek_stats st0; ek_stats_get(&st0);
    ek_set_fast_mode(1);
    ek_stats_reset();
    battery(fast);
    ek_stats st1; ek_stats_get(&st1);
    int bad = 0;
    if (st0.fast_launches != 0) { fprintf(stderr, "ek_qualify: the reference pass used the fast kernel\n"); bad++; }
    if (st1.fast_launches == 0) { fprintf(stderr, "ek_qualify: the fast kernel was never selected\n"); bad++; }
    if (ref.size() != fast.size()) { fprintf(stderr, "ek_qualify: result lists differ in length\n"); return 1; }
    for (size_t k = 0; k < ref.size(); ++k) {
        const Result &a = ref[k], &b = fast[k];
        if (a.bytes.size() != b.bytes.size()) { fprintf(stderr, "ek_qualify: %s: sizes differ\n", a.name.c_str()); bad++; continue; }
        if (a.kind == 0) {
            if (memcmp(a.bytes.data(), b.bytes.data(), a.bytes.size()) != 0) {
                size_t first = 0; while (first < a.bytes.size() && a.bytes[first] == b.bytes[first]) ++first;
                fprintf(stderr, "ek_qualify: %s: results differ (first at byte %zu of %zu)\n", a.name.c_str(), first, a.bytes.size());
                bad++;
            }
        } else {
            const float *x = (const float *) a.bytes.data(), *y = (const float *) b.bytes.data();
            size_t n = a.bytes.size() / 4, nb = 0; double scale = 0;
            for (size_t i = 0; i < n; ++i) if (std::isfinite(x[i])) scale = std::fmax(scale, std::fabs((double) x[i]));
            for (size_t i = 0; i < n; ++i) {
                if (std::isnan(x[i]) && std::isnan(y[i])) continue;
                if (x[i] == y[i]) continue;
                if (!(std::fabs((double) x[i] - (double) y[i]) <= a.tol * std::fmax(a.scale > 0 ? a.scale : scale, 1e-30))) ++nb;
            }
            if (nb) { fprintf(stderr, "ek_qualify: %s: %zu of %zu values differ by more than the tolerance\n", a.name.c_str(), nb, n); bad++; }
        }
    }
    fprintf(stderr, "ek_qualify: %zu results compared, %d disagreements, %llu sweeps on the fast kernel -> %s\n", ref.size(), bad,
            (unsigned long long) st1.fast_launches, bad ? "NOT qualified" : "results agree");
    if (bad) return 1;
    /* correct -- but is it faster here?  The fast kernel exists to beat the general one; if it does not on this GPU (C2, the
       headline workload, 2^24 elements, device time of the sweep launch), the general kernel stays in charge.  The numbers
       go into the small file named by argv[1] (ek_runtime.cpp: in the temporary directory) so that bench.py can report them. */
    double g2 = 0, g3 = 0, f2 = 0, f3 = 0;
    const size_t nt = (size_t) 1 << 24;
    ek_set_fast_mode(0); time_c2_c3(nt, g2, g3);
    ek_set_fast_mode(1); time_c2_c3(nt, f2, f3);
    const bool faster = f2 > 0 && f2 <= 1.03 * g2;
    fprintf(stderr, "ek_qualify: C2 at 2^24: general %.4f ms, fast %.4f ms; C3 at 2^24: general %.4f ms, fast %.4f ms -> %s\n", g2, f2, g3, f3,
            faster ? "qualified" : "NOT qualified (correct, but not faster than the general kernel on C2)");
    if (argc > 1) {
        FILE *f = fopen(argv[1], "w");
        if (f) {
            fprintf(f, "{\"elems\": %zu, \"c2_general_ms\": %.5f, \"c2_fast_ms\": %.5f, \"c3_general_ms\": %.5f, \"c3_fast_ms\": %.5f, \"fast_selected\": %s}\n",
                    nt, g2, f2, g3, f3, faster ? "true" : "false");
            fclose(f);
        }
    }
    return faster ? 0 : 4;
}
