/*
 * ek_runtime.cpp -- trace table, ref counting, allocator and C ABI glue.
 *
 * Behavioural spec = the reference's host runtime, src/cuda/jit.cu:
 *   Variable/Context :61-262, init :274-318, var lifecycle :329-495,
 *   ref counting :586-684, trace append :701-861, allocator :1636-1896.
 * Re-designed: dense handle table, opcodes instead of PTX text, one stream
 * (stream-ordered allocator, no free callbacks), scheduling in ek_eval.cpp.
 */
#include "ek_internal.h"
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <algorithm>
#include <sstream>
#include <string>
#include <vector>
#include <dlfcn.h>
#include <signal.h>
#include <spawn.h>
#include <sys/stat.h>
#include <sys/wait.h>
#include <unistd.h>
extern char **environ;

static EkContext *g_ctx = nullptr;
static thread_local std::string g_error;
static int g_device_request = -1;

EkContext &ek_ctx() {
    if (!g_ctx) {
        g_ctx = new EkContext();
        g_ctx->vars.resize(EK_REG_RESERVED);
    }
    return *g_ctx;
}

void ek_set_error(const std::string &msg) { g_error = msg; }

void ek_cuda_check_impl(cudaError_t err, const char *file, int line) {
    if (err != cudaSuccess) {
        /* common.cu:268-286: CUDA failures are fatal */
        fprintf(stderr, "enoki_b200: CUDA error %s (%s) at %s:%d\n", cudaGetErrorName(err),
                cudaGetErrorString(err), file, line);
        exit(EXIT_FAILURE);
    }
}

const char *ek_type_name(ek_type t) {
    static const char *names[] = { "invalid", "i8", "u8", "i16", "u16", "i32", "u32", "i64",
                                   "u64", "f16", "f32", "f64", "bool", "ptr" };
    return (unsigned) t <= EK_POINTER ? names[t] : "?";
}

const char *ek_op_name(ek_op op) {
    static const char *names[] = {
        "invalid", "literal", "index", "mov", "cvt", "bitcast", "neg", "abs", "sqrt", "rcp", "rsqrt",
        "exp", "log", "sin", "cos", "floor", "ceil", "round", "trunc", "floor2int", "ceil2int", "not",
        "popc", "clz", "ctz", "add", "sub", "mul", "mulhi", "div", "mod", "min", "max", "shl", "shr",
        "and", "or", "xor", "gt", "ge", "lt", "le", "eq", "ne", "mul_nz", "fma", "select", "fma_nz",
        "gather", "scatter", "scatter_add", "hsum", "hprod", "hmax", "hmin", "all", "any", "count" };
    return (unsigned) op < EK_OP__COUNT ? names[op] : "?";
}

extern "C" {

const char *ek_last_error(void) { return g_error.c_str(); }
const char *ek_version(void) { return "enoki_b200 0.1 (sm_100a)"; }

int ek_device_count(void) {
    int n = 0;
    if (cudaGetDeviceCount(&n) != cudaSuccess) { cudaGetLastError(); return 0; }
    return n;
}

int ek_set_device(int ordinal) {
    if (g_ctx && g_ctx->initialized) { ek_set_error("ek_set_device(): context already initialised"); return -1; }
    g_device_request = ordinal;
    return 0;
}

/* ---- kernel qualification ---------------------------------------------------------------------------------------
   The 32-bit fast sweep kernel (ek_sweep_fast.cu) was written in round 2 after this repository had lost its access to
   GPU hardware, so nothing in the tree has seen it run.  The runtime therefore does not trust it blindly: the first
   ek_init() on a machine runs `ek_qualify` (enoki_b200/ek_qualify, built from csrc/ek_qualify.cpp) in a CHILD PROCESS.
   The child evaluates a battery of programs twice -- through the general sweep kernels that passed the round-1 GPU
   test-suite, and through the fast kernel -- and compares the results bit for bit.  Only when every comparison agrees
   (exit status 0, within 150 s) is the fast kernel used; a wrong result, a CUDA error, a watchdog trap or a crash of the
   child all leave this process on the general kernels, with one line on stderr.  The verdict is remembered in a stamp
   file keyed on the library file and the GPU name, so the battery runs once per machine, not once per process.  The
   stamp and the helper's timings go to $TMPDIR (or /tmp), never next to the library: the installed tree may be
   read-only, and using it must not change it.
   EK_FAST=0 / EK_FAST=1 skip the qualification and force the answer (the child itself runs with EK_FAST=0 and switches
   modes through ek_set_fast_mode()). */
static std::string lib_path() {
    Dl_info info;
    if (dladdr((const void *) &ek_init, &info) && info.dli_fname) return info.dli_fname;
    return "";
}
static int decide_fast_mode(const char *gpu_name) {
    if (const char *e = getenv("EK_FAST")) return atoi(e) != 0 ? 1 : 0;
    const std::string lib = lib_path();
    if (lib.empty()) return 0;
    const std::string dir = lib.substr(0, lib.find_last_of('/'));
    const std::string helper = dir + "/ek_qualify";
    struct stat st_lib, st_helper;
    if (stat(lib.c_str(), &st_lib) != 0) return 0;
    if (stat(helper.c_str(), &st_helper) != 0) {
        fprintf(stderr, "enoki_b200: %s not found -- the fast sweep kernel stays off (general kernels are used)\n", helper.c_str());
        return 0;
    }
    char key[512];
    snprintf(key, sizeof(key), "lib %lld %lld gpu %s", (long long) st_lib.st_size, (long long) st_lib.st_mtime, gpu_name);
    const char *tmpdir = getenv("TMPDIR");
    const std::string state = std::string(tmpdir && *tmpdir ? tmpdir : "/tmp") + "/ek_b200_fast_";
    const std::string uid = std::to_string((long) getuid());
    const std::string stamp = state + "qualified_" + uid;
    if (FILE *f = fopen(stamp.c_str(), "r")) {
        char line[600] = { 0 }; int verdict = -1;
        if (fgets(line, sizeof(line), f)) { size_t l = strlen(line); while (l && (line[l - 1] == '\n' || line[l - 1] == '\r')) line[--l] = 0; }
        if (fscanf(f, "%d", &verdict) != 1) verdict = -1;
        fclose(f);
        if (verdict >= 0 && strcmp(line, key) == 0) return verdict ? 1 : 0;
    }
    /* run the battery in a child process (this process may already hold CUDA state: no fork-without-exec) */
    pid_t pid = 0;
    const std::string timing_file = state + "timing_" + uid + ".json";     /* read by bench.py */
    unlink(timing_file.c_str());          /* a failed battery writes none: never leave another library's timings there */
    char *argv[] = { const_cast<char *>(helper.c_str()), const_cast<char *>(timing_file.c_str()), nullptr };
    std::vector<std::string> envs;
    for (char **e = environ; e && *e; ++e) if (strncmp(*e, "EK_FAST=", 8) != 0) envs.push_back(*e);
    envs.push_back("EK_FAST=0");
    std::vector<char *> envp;
    for (auto &e : envs) envp.push_back(const_cast<char *>(e.c_str()));
    envp.push_back(nullptr);
    int verdict = 0;
    if (posix_spawn(&pid, helper.c_str(), nullptr, nullptr, argv, envp.data()) != 0) {
        fprintf(stderr, "enoki_b200: could not start %s -- the fast sweep kernel stays off\n", helper.c_str());
    } else {
        int status = 0; bool done = false;
        for (int waited_ms = 0; waited_ms < 150000; waited_ms += 50) {
            pid_t r = waitpid(pid, &status, WNOHANG);
            if (r == pid) { done = true; break; }
            if (r < 0) break;
            usleep(50000);
        }
        if (!done) { kill(pid, SIGKILL); waitpid(pid, &status, 0); }
        verdict = (done && WIFEXITED(status) && WEXITSTATUS(status) == 0) ? 1 : 0;
        if (!verdict)
            fprintf(stderr, "enoki_b200: the fast sweep kernel did NOT qualify on this machine (%s) -- general kernels are used\n",
                    !done ? "timeout" : WIFSIGNALED(status) ? "child crashed" :
                    (WIFEXITED(status) && WEXITSTATUS(status) == 4) ? "correct, but not faster than the general kernel here" : "results differ / CUDA error, see above");
    }
    const std::string tmp = stamp + "." + std::to_string((long) getpid());
    if (FILE *f = fopen(tmp.c_str(), "w")) {
        fprintf(f, "%s\n%d\n", key, verdict);
        fclose(f);
        if (rename(tmp.c_str(), stamp.c_str()) != 0) unlink(tmp.c_str());
    }
    return verdict;
}

int ek_init(void) {
    EkContext &ctx = ek_ctx();
    if (ctx.initialized) return 0;
    int n = ek_device_count();
    if (n == 0) {
        ek_set_error("ek_init(): no CUDA device available -- this backend has no CPU fallback");
        return -1;
    }
    ctx.device = g_device_request >= 0 ? g_device_request : 0;
    if (g_device_request < 0) {
        const char *lr = getenv("LOCAL_RANK");
        if (lr) ctx.device = atoi(lr) % n;
    }
    ek_cuda_check(cudaSetDevice(ctx.device));
    cudaDeviceProp prop;
    ek_cuda_check(cudaGetDeviceProperties(&prop, ctx.device));
    ctx.num_sms = prop.multiProcessorCount;
    ctx.smem_optin = prop.sharedMemPerBlockOptin;
    ek_cuda_check(cudaStreamCreateWithFlags(&ctx.stream, cudaStreamNonBlocking));
    ek_cuda_check(cudaEventCreate(&ctx.ev_start));
    ek_cuda_check(cudaEventCreate(&ctx.ev_stop));
    ek_cuda_check(cudaEventCreate(&ctx.tm_start));
    ek_cuda_check(cudaEventCreate(&ctx.tm_stop));
    ctx.max_grid = (uint32_t) ctx.num_sms * 32u;
    ek_cuda_check(cudaMalloc(&ctx.red_partials, sizeof(uint64_t) * EK_MAX_RED * ctx.max_grid));
    ek_cuda_check(cudaMalloc(&ctx.red_counters, sizeof(uint32_t) * EK_MAX_RED));
    ek_cuda_check(cudaMemset(ctx.red_counters, 0, sizeof(uint32_t) * EK_MAX_RED));
    ctx.initialized = true;
    ctx.fast_mode = decide_fast_mode(prop.name);
    static bool registered = false;
    if (!registered) { atexit(ek_shutdown); registered = true; }   /* jit.cu:315-318 */
    return 0;
}

void ek_set_fast_mode(int enable) { ek_ctx().fast_mode = enable ? 1 : 0; }
int ek_fast_mode(void) { return ek_ctx().fast_mode; }

void ek_shutdown(void) {
    if (!g_ctx) return;
    EkContext &ctx = *g_ctx;
    if (ctx.initialized) {
        cudaStreamSynchronize(ctx.stream);
        for (auto &v : ctx.vars) {
            if (v.used && v.data && v.free_data && !v.direct_pointer) cudaFree(v.data);
            delete v.label;
        }
        for (auto &kv : ctx.free_lists)
            for (void *p : kv.second) { if (kv.first.first == 2) cudaFreeHost(p); else cudaFree(p); }
        for (auto &kv : ctx.programs)
            for (auto &e : kv.second) { cudaFree(e.d_prog); cudaFree(e.d_lit); }
        cudaFree(ctx.red_partials); cudaFree(ctx.red_counters);
        if (ctx.flush_buf) cudaFree(ctx.flush_buf);
        cudaEventDestroy(ctx.ev_start); cudaEventDestroy(ctx.ev_stop);
        cudaEventDestroy(ctx.tm_start); cudaEventDestroy(ctx.tm_stop);
        cudaStreamDestroy(ctx.stream);
    }
    delete g_ctx;
    g_ctx = nullptr;
}

/* ------------------------------------------------------------------ allocator */
static void *alloc_impl(int kind, size_t size) {
    EkContext &ctx = ek_ctx();
    if (ek_init() != 0) { fprintf(stderr, "enoki_b200: %s\n", ek_last_error()); exit(EXIT_FAILURE); }
    if (size == 0) size = 1;
    size_t rounded = (size + 511) & ~(size_t) 511;
    auto key = std::make_pair(kind, rounded);
    auto it = ctx.free_lists.find(key);
    void *p = nullptr;
    if (it != ctx.free_lists.end() && !it->second.empty()) {
        p = it->second.back(); it->second.pop_back();
        ctx.cached -= rounded;
    } else {
        auto do_alloc = [&]() -> cudaError_t {
            switch (kind) {
                case 0: return cudaMalloc(&p, rounded);
                case 1: return cudaMallocManaged(&p, rounded);
                default: return cudaMallocHost(&p, rounded);
            }
        };
        cudaError_t err = do_alloc();
        if (err == cudaErrorMemoryAllocation) {       /* jit.cu:1715-1723: sync, trim, retry once */
            cudaGetLastError();
            if (ctx.pre_trim_hook) ctx.pre_trim_hook(ctx.pre_trim_arg);
            ek_sync(); ek_malloc_trim();
            err = do_alloc();
        }
        ek_cuda_check(err);
    }
    ctx.alloc_size[p] = rounded;
    ctx.alloc_kind[p] = kind;
    if (kind != 2) { ctx.used += rounded; ctx.watermark = std::max(ctx.watermark, ctx.used); }
    return p;
}

void *ek_malloc(size_t size) { return alloc_impl(0, size); }
void *ek_managed_malloc(size_t size) { return alloc_impl(1, size); }
void *ek_host_malloc(size_t size) { return alloc_impl(2, size); }

void ek_free(void *ptr) {
    if (!ptr || !g_ctx) return;
    EkContext &ctx = *g_ctx;
    auto it = ctx.alloc_size.find(ptr);
    if (it == ctx.alloc_size.end()) {
        /* not ours (e.g. user memory registered with dealloc=true): hand to the driver */
        cudaFree(ptr); cudaGetLastError();
        return;
    }
    size_t sz = it->second; int kind = ctx.alloc_kind[ptr];
    ctx.alloc_size.erase(it); ctx.alloc_kind.erase(ptr);
    if (kind != 2) ctx.used -= sz;
    ctx.cached += sz;
    /* all work is enqueued on one stream: the block may be reused by later launches at once */
    ctx.free_lists[std::make_pair(kind, sz)].push_back(ptr);
}
void ek_host_free(void *ptr) {
    if (!ptr || !g_ctx) return;
    EkContext &ctx = *g_ctx;
    /* host blocks may still be read by an in-flight async copy: drain first */
    if (ctx.initialized) cudaStreamSynchronize(ctx.stream);
    ek_free(ptr);
}

void ek_malloc_trim(void) {
    if (!g_ctx || !g_ctx->initialized) return;
    EkContext &ctx = *g_ctx;
    cudaStreamSynchronize(ctx.stream);
    for (auto &kv : ctx.free_lists) {
        for (void *p : kv.second) { if (kv.first.first == 2) cudaFreeHost(p); else cudaFree(p); }
        kv.second.clear();
    }
    ctx.cached = 0;
}

void ek_mem_get_info(size_t *free_bytes, size_t *total_bytes) {
    if (ek_init() != 0) { *free_bytes = *total_bytes = 0; return; }
    ek_cuda_check(cudaMemGetInfo(free_bytes, total_bytes));
}

void ek_memcpy_to_device(void *dst, const void *src, size_t size) {
    EkContext &ctx = ek_ctx(); ek_init();
    ek_cuda_check(cudaMemcpyAsync(dst, src, size, cudaMemcpyHostToDevice, ctx.stream));
    ek_cuda_check(cudaStreamSynchronize(ctx.stream));
}
void ek_memcpy_to_device_async(void *dst, const void *src, size_t size) {
    EkContext &ctx = ek_ctx(); ek_init();
    ek_cuda_check(cudaMemcpyAsync(dst, src, size, cudaMemcpyHostToDevice, ctx.stream));
}
void ek_memcpy_from_device(void *dst, const void *src, size_t size) {
    EkContext &ctx = ek_ctx(); ek_init();
    ek_cuda_check(cudaMemcpyAsync(dst, src, size, cudaMemcpyDeviceToHost, ctx.stream));
    ek_cuda_check(cudaStreamSynchronize(ctx.stream));
}
void ek_memcpy_from_device_async(void *dst, const void *src, size_t size) {
    EkContext &ctx = ek_ctx(); ek_init();
    ek_cuda_check(cudaMemcpyAsync(dst, src, size, cudaMemcpyDeviceToHost, ctx.stream));
}

/* Extension: device-to-device copy on the runtime's stream (interop with other frameworks' buffers) */
void ek_memcpy_device_async(void *dst, const void *src, size_t size) {
    EkContext &ctx = ek_ctx(); ek_init();
    ek_cuda_check(cudaMemcpyAsync(dst, src, size, cudaMemcpyDeviceToDevice, ctx.stream));
}

/* Extension (no reference counterpart): read-back on a second stream, so that it overlaps with host-to-device copies
   and kernels enqueued afterwards (PCIe is full duplex).  Ordered after everything enqueued so far; `src` must stay
   allocated until the next ek_sync(). */
void ek_memcpy_from_device_overlapped(void *dst, const void *src, size_t size) {
    EkContext &ctx = ek_ctx(); ek_init();
    if (!ctx.d2h_stream) {
        ek_cuda_check(cudaStreamCreateWithFlags(&ctx.d2h_stream, cudaStreamNonBlocking));
        ek_cuda_check(cudaEventCreateWithFlags(&ctx.d2h_event, cudaEventDisableTiming));
    }
    ek_cuda_check(cudaEventRecord(ctx.d2h_event, ctx.stream));
    ek_cuda_check(cudaStreamWaitEvent(ctx.d2h_stream, ctx.d2h_event, 0));
    ek_cuda_check(cudaMemcpyAsync(dst, src, size, cudaMemcpyDeviceToHost, ctx.d2h_stream));
}

void ek_sync(void) {
    if (!g_ctx || !g_ctx->initialized) return;
    ek_cuda_check(cudaStreamSynchronize(g_ctx->stream));
    if (g_ctx->d2h_stream) ek_cuda_check(cudaStreamSynchronize(g_ctx->d2h_stream));
}

void ek_fill(void *ptr, size_t elem_size, uint64_t value, size_t n) {
    EkContext &ctx = ek_ctx(); ek_init();
    if (n == 0) return;
    if (elem_size == 1 || value == 0) {
        ek_cuda_check(cudaMemsetAsync(ptr, (int) (value & 0xff), n * elem_size, ctx.stream));
        return;
    }
    ek_launch_fill(ptr, elem_size, value, n, ctx.stream);
    ctx.stats.launches++;
}
void ek_reverse(void *out, const void *in, size_t elem_size, size_t n) {
    EkContext &ctx = ek_ctx(); ek_init();
    if (n == 0) return;
    ek_launch_reverse(out, in, elem_size, n, ctx.stream);
    ctx.stats.launches++;
}

/* ------------------------------------------------------------------ variables */
static uint32_t var_new(ek_type type) {
    EkContext &ctx = ek_ctx();
    uint32_t idx;
    if (!ctx.free_handles.empty()) { idx = ctx.free_handles.back(); ctx.free_handles.pop_back(); }
    else { idx = (uint32_t) ctx.vars.size(); ctx.vars.emplace_back(); }
    EkVariable &v = ctx.vars[idx];
    v = EkVariable();
    v.type = type; v.used = true;
    v.seq = ctx.next_seq++;
    return idx;
}

static EkVariable *var_get(uint32_t index, const char *who) {
    EkContext &ctx = ek_ctx();
    if (index < EK_REG_RESERVED || index >= ctx.vars.size() || !ctx.vars[index].used) {
        ek_set_error(std::string(who) + ": unknown variable " + std::to_string(index));   /* jit.cu:207-212 */
        return nullptr;
    }
    return &ctx.vars[index];
}

static void inc_ref_int(uint32_t index) {
    if (index < EK_REG_RESERVED) return;
    ek_ctx().vars[index].ref_int++;
}

static void var_free(uint32_t first);

static void dec_ref_int(uint32_t index) {
    if (index < EK_REG_RESERVED) return;
    EkVariable &v = ek_ctx().vars[index];
    if (v.ref_int == 0) {
        fprintf(stderr, "ek_dec_ref_int(): Node %u has no internal references!\n", index);   /* jit.cu:646-649 */
        exit(EXIT_FAILURE);
    }
    if (--v.ref_int == 0 && v.ref_ext == 0) var_free(index);
}

void ek_inc_ref_ext(uint32_t index) {
    if (index < EK_REG_RESERVED) return;
    EkContext &ctx = ek_ctx();
    if (index >= ctx.vars.size() || !ctx.vars[index].used) return;
    ctx.vars[index].ref_ext++;
}

void ek_dec_ref_ext(uint32_t index) {
    if (index < EK_REG_RESERVED || !g_ctx) return;
    EkContext &ctx = *g_ctx;
    if (index >= ctx.vars.size() || !ctx.vars[index].used) return;
    EkVariable &v = ctx.vars[index];
    if (v.ref_ext == 0) {
        fprintf(stderr, "ek_dec_ref_ext(): Node %u has no external references!\n", index);   /* jit.cu:620-623 */
        exit(EXIT_FAILURE);
    }
    v.ref_ext--;
    if (v.ref_ext == 0 && !v.side_effect) ctx.live.erase(index);
    if (v.ref_ext == 0 && v.ref_int == 0) var_free(index);
}

/* jit.cu:437-453 cuda_var_free, iterative so that 10k-deep chains do not recurse */
static void var_free(uint32_t first) {
    EkContext &ctx = ek_ctx();
    std::vector<uint32_t> work { first };
    while (!work.empty()) {
        uint32_t idx = work.back(); work.pop_back();
        EkVariable &v = ctx.vars[idx];
        if (!v.used || v.ref_ext != 0 || v.ref_int != 0) continue;
        ctx.live.erase(idx);
        if (v.direct_pointer) ctx.ptr_map.erase(v.data);
        for (int i = 0; i < 4; ++i) {
            uint32_t d = v.dep[i];
            if (d >= EK_REG_RESERVED) {
                EkVariable &dv = ctx.vars[d];
                if (dv.ref_int == 0) { fprintf(stderr, "ek: internal refcount underflow on %u\n", d); exit(EXIT_FAILURE); }
                if (--dv.ref_int == 0 && dv.ref_ext == 0) work.push_back(d);
            }
        }
        if (v.extra_dep >= EK_REG_RESERVED) {
            EkVariable &dv = ctx.vars[v.extra_dep];
            if (dv.ref_ext == 0) { fprintf(stderr, "ek: external refcount underflow on %u\n", v.extra_dep); exit(EXIT_FAILURE); }
            dv.ref_ext--;
            if (dv.ref_ext == 0 && !dv.side_effect) ctx.live.erase(v.extra_dep);
            if (dv.ref_ext == 0 && dv.ref_int == 0) work.push_back(v.extra_dep);
        }
        if (v.data && v.free_data && !v.direct_pointer) ek_free(v.data);
        delete v.label;
        v = EkVariable();
        ctx.free_handles.push_back(idx);
    }
}

size_t ek_var_size(uint32_t index) { EkVariable *v = var_get(index, "ek_var_size()"); return v ? v->size : 0; }
void *ek_var_ptr(uint32_t index) { EkVariable *v = var_get(index, "ek_var_ptr()"); return v ? v->data : nullptr; }
ek_type ek_var_type(uint32_t index) { EkVariable *v = var_get(index, "ek_var_type()"); return v ? v->type : EK_INVALID; }

int ek_var_set_label(uint32_t index, const char *label) {
    EkVariable *v = var_get(index, "ek_var_set_label()"); if (!v) return -1;
    if (!v->label) v->label = new std::string();
    *v->label = label ? label : "";
    return 0;
}

int ek_var_mark_side_effect(uint32_t index) {
    EkVariable *v = var_get(index, "ek_var_mark_side_effect()"); if (!v) return -1;
    v->side_effect = true;
    return 0;
}

int ek_var_mark_dirty(uint32_t index) {
    EkVariable *v = var_get(index, "ek_var_mark_dirty()"); if (!v) return -1;
    v->dirty = true;
    ek_ctx().dirty.push_back(index);
    return 0;
}

int ek_set_scatter_gather_operand(uint32_t index, int gather) {
    EkContext &ctx = ek_ctx();
    if (index != 0) {
        EkVariable *v = var_get(index, "ek_set_scatter_gather_operand()"); if (!v) return -1;
        if (v->data == nullptr && v->op == EK_OP_LITERAL) { if (ek_eval_var(index) != 0) return -1; v = var_get(index, "ek_set_scatter_gather_operand()"); }
        if (v->data == nullptr || (gather && v->dirty)) { if (ek_eval() != 0) return -1; }   /* jit.cu:487-495 */
    }
    ctx.scatter_gather_operand = index;
    return 0;
}

uint32_t ek_var_register(ek_type type, size_t size, void *ptr, int dealloc) {
    if (size == 0) { ek_set_error("ek_var_register(): attempted to create a variable of size zero!"); return 0; }   /* jit.cu:386-388 */
    uint32_t idx = var_new(type);
    EkVariable &v = ek_ctx().vars[idx];
    v.data = ptr; v.size = size; v.free_data = dealloc != 0;
    v.ref_ext = 1;
    return idx;
}

uint32_t ek_var_register_ptr(const void *ptr) {
    EkContext &ctx = ek_ctx();
    auto it = ctx.ptr_map.find(ptr);
    if (it != ctx.ptr_map.end()) { ctx.vars[it->second].ref_ext++; return it->second; }   /* jit.cu:397-403 */
    uint32_t idx = var_new(EK_POINTER);
    EkVariable &v = ctx.vars[idx];
    v.data = (void *) ptr; v.size = 1; v.free_data = false; v.direct_pointer = true;
    v.ref_ext = 1;
    ctx.ptr_map[ptr] = idx;
    return idx;
}

uint32_t ek_var_copy_to_device(ek_type type, size_t size, const void *host) {
    if (size == 0) { ek_set_error("ek_var_copy_to_device(): size zero"); return 0; }
    size_t bytes = size * ek_type_size(type);
    void *dev = ek_malloc(bytes);
    void *tmp = ek_host_malloc(bytes);
    memcpy(tmp, host, bytes);
    ek_memcpy_to_device_async(dev, tmp, bytes);
    ek_host_free(tmp);
    return ek_var_register(type, size, dev, 1);
}

int ek_make_managed(uint32_t index) {
    if (index == 0) return 0;
    EkVariable *v = var_get(index, "ek_make_managed()"); if (!v) return -1;
    size_t bytes = v->size * ek_type_size(v->type);
    if (bytes == 0) return 0;
    if (v->data == nullptr || v->dirty) { if (ek_eval_var(index) != 0) return -1; v = var_get(index, "ek_make_managed()"); }
    cudaPointerAttributes attr;
    ek_cuda_check(cudaPointerGetAttributes(&attr, v->data));
    if (attr.type == cudaMemoryTypeManaged) return 0;
    void *p = ek_managed_malloc(bytes);
    ek_cuda_check(cudaMemcpyAsync(p, v->data, bytes, cudaMemcpyDeviceToDevice, ek_ctx().stream));
    if (v->free_data) ek_free(v->data);
    v->data = p; v->free_data = true;
    return 0;
}

int ek_fetch_element(void *dst, uint32_t index, size_t offset, size_t size) {
    EkVariable *v = var_get(index, "ek_fetch_element()"); if (!v) return -1;
    if (v->data == nullptr || v->dirty) { if (ek_eval_var(index) != 0) return -1; v = var_get(index, "ek_fetch_element()"); if (!v) return -1; }
    if (v->dirty) { ek_set_error("ek_fetch_element(): element is still marked as 'dirty' even after ek_eval()!"); return -1; }
    if (v->data == nullptr) { ek_set_error("ek_fetch_element(): tried to read from invalid/uninitialized CUDA array!"); return -1; }
    if (v->size == 1) offset = 0;
    if (offset >= v->size) { ek_set_error("ek_fetch_element(): out of bounds"); return -1; }
    ek_memcpy_from_device(dst, (uint8_t *) v->data + size * offset, size);
    return 0;
}

/* ------------------------------------------------------------------ trace append (jit.cu:701-861) */
static int op_arity(ek_op op) {
    if (op == EK_OP_LITERAL || op == EK_OP_INDEX) return 0;
    if (op >= EK_OP_MOV && op <= EK_OP_CTZ) return 1;
    if (op >= EK_OP_ADD && op <= EK_OP_MUL_NZ) return 2;
    if (op == EK_OP_FMA || op == EK_OP_SELECT || op == EK_OP_FMA_NZ) return 3;
    if (op == EK_OP_GATHER || op == EK_OP_SCATTER || op == EK_OP_SCATTER_ADD) return 3;
    if (op >= EK_OP_HSUM && op <= EK_OP_COUNT) return 1;
    return -1;
}

uint32_t ek_trace_append(ek_type type, ek_op op, uint32_t a, uint32_t b, uint32_t c, uint64_t imm) {
    EkContext &ctx = ek_ctx();
    int arity = op_arity(op);
    if (arity < 0 || ek_type_size(type) == 0) { ek_set_error("ek_trace_append(): invalid opcode/type"); return 0; }
    uint32_t deps[4] = { a, b, c, 0 };
    int ndeps = arity;
    if (op == EK_OP_SCATTER || op == EK_OP_SCATTER_ADD) { deps[3] = (uint32_t) (imm & 0xffffffffu); ndeps = 4; }
    for (int i = 0; i < ndeps; ++i) {
        if (deps[i] == 0) {
            ek_set_error("ek_trace_append(): arithmetic involving uninitialized variable!");   /* jit.cu:722-725 */
            return 0;
        }
        if (!var_get(deps[i], "ek_trace_append()")) return 0;
    }
    bool need_eval = false;
    for (int i = 0; i < ndeps; ++i) if (ctx.vars[deps[i]].dirty) need_eval = true;
    if (need_eval && ek_eval() != 0) return 0;                                                  /* jit.cu:729-730 */

    size_t size = 1; uint32_t subtree = 1;
    for (int i = 0; i < ndeps; ++i) size = std::max(size, ctx.vars[deps[i]].size);
    for (int i = 0; i < ndeps; ++i) {
        const EkVariable &d = ctx.vars[deps[i]];
        if (d.size != 1 && d.size != size) {                                                    /* jit.cu:776-782 */
            std::string msg = "ek_trace_append(): arithmetic involving arrays of incompatible size (";
            for (int j = 0; j < ndeps; ++j) msg += (j ? (j + 1 == ndeps ? " and " : ", ") : "") + std::to_string(ctx.vars[deps[j]].size);
            msg += std::string("). The instruction was \"") + ek_op_name(op) + "\".";
            ek_set_error(msg);
            return 0;
        }
        subtree += d.subtree_size;
    }
    if (op == EK_OP_GATHER && !ctx.vars[a].direct_pointer) {
        ek_set_error("ek_trace_append(): gather source must be a pointer registered with ek_var_register_ptr()");
        return 0;
    }
    if ((op == EK_OP_SCATTER || op == EK_OP_SCATTER_ADD) && !ctx.vars[a].direct_pointer) {
        ek_set_error("ek_trace_append(): scatter target must be a pointer registered with ek_var_register_ptr()");
        return 0;
    }
    /* x / (+-2^k) == x * (+-2^-k) bit for bit (an exact scaling rounds the same real number), and the multiply is one
       instruction where div.rn is a Newton iteration with a slow-path branch: rewrite divisions by power-of-two
       literals (C3's `* 31 / 8`) */
    if (op == EK_OP_DIV && (type == EK_FLOAT32 || type == EK_FLOAT64)) {
        const EkVariable &dv = ctx.vars[b];
        if (dv.op == EK_OP_LITERAL && dv.data == nullptr && dv.size == 1) {
            uint64_t rbits = 0; bool ok = false;
            if (type == EK_FLOAT32) {
                uint32_t bits = (uint32_t) dv.imm, e = (bits >> 23) & 0xffu;
                if ((bits & 0x7fffffu) == 0 && e >= 2 && e <= 252) { rbits = (bits & 0x80000000u) | ((254u - e) << 23); ok = true; }
            } else {
                uint64_t bits = dv.imm, e = (bits >> 52) & 0x7ffull;
                if ((bits & 0xfffffffffffffull) == 0 && e >= 2 && e <= 2044) { rbits = (bits & 0x8000000000000000ull) | ((2046ull - e) << 52); ok = true; }
            }
            if (ok) {
                uint32_t lit = ek_trace_append(type, EK_OP_LITERAL, 0, 0, 0, rbits);
                if (!lit) return 0;
                uint32_t r = ek_trace_append(type, EK_OP_MUL, a, lit, 0, 0);
                ek_dec_ref_ext(lit);
                return r;
            }
        }
    }
    bool is_reduce = op >= EK_OP_HSUM && op <= EK_OP_COUNT;
    uint32_t idx = var_new(type);
    EkVariable &v = ctx.vars[idx];
    v.op = op; v.imm = imm;
    v.size = is_reduce ? 1 : size;
    for (int i = 0; i < 4; ++i) v.dep[i] = deps[i];
    v.subtree_size = subtree;
    for (int i = 0; i < ndeps; ++i) inc_ref_int(deps[i]);
    v.ref_ext = 1;
    ctx.live.insert(idx);
    if (op == EK_OP_GATHER || op == EK_OP_SCATTER || op == EK_OP_SCATTER_ADD) {               /* jit.cu:794-799,852-858 */
        v.extra_dep = ctx.scatter_gather_operand;
        if (v.extra_dep >= EK_REG_RESERVED) ctx.vars[v.extra_dep].ref_ext++;
    }
    return idx;
}

uint32_t ek_var_set_size(uint32_t index, size_t size, int copy) {
    EkVariable *v = var_get(index, "ek_var_set_size()"); if (!v) return 0;
    if (v->size == size) return index;
    /* lazy reductions (hsum ... count) are size-1 results of a sweep over their operand: like an evaluated scalar they
       can only be widened through a broadcasting MOV, never in place (the reference evaluates them eagerly, so there
       the variable has data and takes this branch anyway) */
    const bool lazy_reduce = v->op >= EK_OP_HSUM && v->op <= EK_OP_COUNT;
    if (v->data != nullptr || v->ref_int > 0 || lazy_reduce) {
        if (v->size == 1 && copy) {                                                             /* jit.cu:357-364 */
            uint32_t nidx = ek_trace_append(v->type, EK_OP_MOV, index, 0, 0, 0);
            if (!nidx) return 0;
            ek_ctx().vars[nidx].size = size;
            ek_dec_ref_ext(index);
            return nidx;
        }
        ek_set_error("ek_var_set_size(): attempted to resize variable " + std::to_string(index) +
                     " which was already allocated (current size = " + std::to_string(v->size) +
                     ", requested size = " + std::to_string(size) + ")");                       /* jit.cu:366-371 */
        return 0;
    }
    v->size = size;
    return index;
}

int ek_register_callback(void (*cb)(void *), void *payload) {
    ek_ctx().callbacks.emplace_back(cb, payload);
    return 0;
}
int ek_unregister_callback(void (*cb)(void *), void *payload) {
    auto &cbs = ek_ctx().callbacks;
    auto it = std::find(cbs.begin(), cbs.end(), std::make_pair(cb, payload));
    if (it == cbs.end()) { ek_set_error("ek_unregister_callback(): entry not found!"); return -1; }
    cbs.erase(it);
    return 0;
}

void ek_set_log_level(uint32_t level) { ek_ctx().log_level = level; }
uint32_t ek_log_level(void) { return ek_ctx().log_level; }

char *ek_whos(void) {
    /* jit.cu:1564-1634 */
    EkContext &ctx = ek_ctx();
    std::ostringstream oss;
    oss << "\n  ID        Type   E/I Refs   Size        Memory     Ready    Label\n";
    oss << "  =================================================================\n";
    size_t mem_arith = 0, mem_alloc = 0;
    for (uint32_t i = EK_REG_RESERVED; i < ctx.vars.size(); ++i) {
        const EkVariable &v = ctx.vars[i];
        if (!v.used) continue;
        size_t bytes = v.size * ek_type_size(v.type);
        char line[256];
        snprintf(line, sizeof(line), "  %-9u %-6s %3u / %-5u %-11zu %-10zu %-8s %s\n", i, ek_type_name(v.type),
                 v.ref_ext, v.ref_int, v.size, bytes, v.data ? "[x]" : "[ ]", v.label ? v.label->c_str() : "");
        oss << line;
        if (v.data) mem_alloc += bytes; else mem_arith += bytes;
    }
    oss << "  =================================================================\n\n";
    oss << "  Memory usage (ready)       : " << mem_alloc << " bytes\n";
    oss << "  Memory usage (scheduled)   : " << mem_alloc << " + " << mem_arith << " bytes\n";
    oss << "  Memory savings             : " << mem_arith << " bytes (kept in registers/shared memory)\n";
    oss << "  Allocator                  : used " << ctx.used << ", cached " << ctx.cached << ", watermark " << ctx.watermark << "\n";
    return strdup(oss.str().c_str());
}

/* ------------------------------------------------------------------ instrumentation */
void ek_stats_reset(void) { ek_ctx().stats = ek_stats(); }
void ek_stats_get(ek_stats *out) { *out = ek_ctx().stats; }
void ek_set_timing(int enable) { ek_ctx().timing = enable != 0; }
void *ek_stream(void) { ek_init(); return (void *) ek_ctx().stream; }
void ek_timer_start(void) { EkContext &ctx = ek_ctx(); ek_init(); ek_cuda_check(cudaEventRecord(ctx.tm_start, ctx.stream)); }
float ek_timer_stop(void) {
    EkContext &ctx = ek_ctx();
    ek_cuda_check(cudaEventRecord(ctx.tm_stop, ctx.stream));
    ek_cuda_check(cudaEventSynchronize(ctx.tm_stop));
    float ms = 0; ek_cuda_check(cudaEventElapsedTime(&ms, ctx.tm_start, ctx.tm_stop));
    return ms;
}
void ek_flush_l2(void) {
    EkContext &ctx = ek_ctx(); ek_init();
    if (!ctx.flush_buf) { ctx.flush_bytes = (size_t) 256 << 20; ek_cuda_check(cudaMalloc(&ctx.flush_buf, ctx.flush_bytes)); }
    ek_launch_flush(ctx.flush_buf, ctx.flush_bytes, ctx.stream);
}

} /* extern "C" */
