// rb_jit.cu -- run-time specialisation: every uploaded chain gets kernels compiled FOR ITS OWN constants.
//
// The FR3 and chain32 families are this mechanism run ahead of time (rb_modelgen + nvcc at build time).  For any
// other chain of up to RB_JIT_MAX_N joints the same kernel templates (rb_dyn.cuh / rb_kernels.cuh, embedded in the
// library as text by the Makefile) are compiled with NVRTC against a table generated from the uploaded model, so
// the exact 0 / +-1 entries of its fixed rotations and offsets disappear from the instruction stream exactly as they
// do for the FR3.  The cubin is cached on disk (keyed by model + sources + compiler version), loaded with
// cudaLibraryLoadData and launched through cudaLaunchKernel; no driver-API linkage, no nvcc at run time.
// libnvrtc is dlopen'ed: if it is absent the engine falls back to the run-time-constant families.
#include <cuda_runtime.h>
#include <dlfcn.h>
#include <fcntl.h>
#include <sys/stat.h>
#include <unistd.h>

#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <fstream>
#include <mutex>
#include <string>
#include <vector>

#include "rb_host_model.h"
#include "rb_jit.h"
#include "rb_kernels.cuh"
#include "gen/jit_sources.h"      // rb_jit_src_names[], rb_jit_src_texts[], rb_jit_src_count

namespace {

// ---- the handful of NVRTC entry points, resolved at run time -----------------------------------------------------
typedef void* nvrtcProgram;
struct Nvrtc {
    void* so = nullptr;
    int (*CreateProgram)(nvrtcProgram*, const char*, const char*, int, const char* const*, const char* const*) = nullptr;
    int (*DestroyProgram)(nvrtcProgram*) = nullptr;
    int (*AddNameExpression)(nvrtcProgram, const char*) = nullptr;
    int (*CompileProgram)(nvrtcProgram, int, const char* const*) = nullptr;
    int (*GetLoweredName)(nvrtcProgram, const char*, const char**) = nullptr;
    int (*GetCUBINSize)(nvrtcProgram, size_t*) = nullptr;
    int (*GetCUBIN)(nvrtcProgram, char*) = nullptr;
    int (*GetProgramLogSize)(nvrtcProgram, size_t*) = nullptr;
    int (*GetProgramLog)(nvrtcProgram, char*) = nullptr;
    int (*Version)(int*, int*) = nullptr;
    std::string where;
};

const Nvrtc* load_nvrtc(std::string& err) {
    static Nvrtc nv;
    static std::string load_err;
    static std::once_flag once;
    std::call_once(once, [] {
        std::vector<std::string> cands;
        if (const char* e = getenv("RIGIDBODY_B200_NVRTC")) cands.push_back(e);
        cands.push_back("libnvrtc.so.12");
        cands.push_back("libnvrtc.so");
        const char* roots[3] = {getenv("CUDA_HOME"), getenv("CUDA_PATH"), "/usr/local/cuda"};
        for (const char* root : roots)
            if (root) { cands.push_back(std::string(root) + "/lib64/libnvrtc.so.12"); cands.push_back(std::string(root) + "/lib64/libnvrtc.so"); }
        for (const auto& c : cands) {
            nv.so = dlopen(c.c_str(), RTLD_NOW | RTLD_LOCAL);
            if (nv.so) { nv.where = c; break; }
        }
        if (!nv.so) { load_err = "libnvrtc not found (set RIGIDBODY_B200_NVRTC to its path)"; return; }
#define RB_SYM(field, name)                                                   \
    *(void**)(&nv.field) = dlsym(nv.so, name);                                \
    if (!nv.field) { load_err = std::string("libnvrtc lacks ") + name; return; }
        RB_SYM(CreateProgram, "nvrtcCreateProgram") RB_SYM(DestroyProgram, "nvrtcDestroyProgram")
        RB_SYM(AddNameExpression, "nvrtcAddNameExpression") RB_SYM(CompileProgram, "nvrtcCompileProgram")
        RB_SYM(GetLoweredName, "nvrtcGetLoweredName") RB_SYM(GetCUBINSize, "nvrtcGetCUBINSize")
        RB_SYM(GetCUBIN, "nvrtcGetCUBIN") RB_SYM(GetProgramLogSize, "nvrtcGetProgramLogSize")
        RB_SYM(GetProgramLog, "nvrtcGetProgramLog") RB_SYM(Version, "nvrtcVersion")
#undef RB_SYM
    });
    if (!load_err.empty() || !nv.so) { err = load_err.empty() ? "libnvrtc not loaded" : load_err; return nullptr; }
    return &nv;
}

const char* const kKernelExprs[RB_JIT_KERNELS] = {
    "rb_rnea_kernel<CtModel<TabJit>, false>", "rb_rnea_kernel<CtModel<TabJit>, true>",
    "rb_fd_kernel<CtModel<TabJit>, false>",   "rb_fd_kernel<CtModel<TabJit>, true>",
    "rb_crba_kernel<CtModel<TabJit>>",        "rb_fwd_kin_kernel<CtModel<TabJit>>",
    "rb_jac_kernel<CtModel<TabJit>>",         "rb_rollout_kernel<CtModel<TabJit>>",
    "rb_rnea_kernel<CtModel<TabJit, float>, false>", "rb_fd_kernel<CtModel<TabJit, float>, false>",
    "rb_rnea_fd_kernel<CtModel<TabJit>>",    "rb_rollout_kernel<CtModel<TabJit>, true>",
    "rb_rollout_kernel<CtModel<TabJit>, true, true>"};
// chains of RB_JIT_MAX_N+1 .. RB_JIT_LONG_MAX_N joints: the long-chain layouts of rb_kernels_long.cuh for rnea / crba
// (no n x n array in the thread), the plain kernels for fwd_kin / jac, nothing else
const char* const kLongExprs[RB_JIT_KERNELS] = {
    "rb_long_rnea_kernel<CtModel<TabJit>>", nullptr, nullptr, nullptr,
    "rb_long_crba_kernel<CtModel<TabJit>>", "rb_fwd_kin_kernel<CtModel<TabJit>>",
    "rb_jac_kernel<CtModel<TabJit>>",       nullptr, nullptr, nullptr, nullptr, nullptr, nullptr};
// the AoS variants stage 3 arrays of RB_BLOCK states through dynamic shared memory
size_t aos_smem(int n) { return (size_t)3 * RB_BLOCK * n * sizeof(double); }
const char* const kOptions[] = {"--gpu-architecture=sm_100a", "-std=c++17", "-lineinfo", "-default-device", "-DRB_DEVICE_ONLY=1"};

uint64_t fnv1a(uint64_t h, const void* data, size_t n) {
    const unsigned char* p = (const unsigned char*)data;
    for (size_t i = 0; i < n; ++i) { h ^= p[i]; h *= 0x100000001b3ULL; }
    return h;
}

// Where compiled kernels are cached: $RIGIDBODY_B200_CACHE, else $HOME/.cache/rigidbody_b200.  No HOME -> no cache (a
// predictable path under /tmp could be pre-planted by another user of the host).
std::string cache_dir() {
    if (const char* e = getenv("RIGIDBODY_B200_CACHE")) return e;
    const char* home = getenv("HOME");
    return home && *home ? std::string(home) + "/.cache/rigidbody_b200" : std::string();
}

// Creates the directory (0700) if needed and says whether it can be trusted: it must be a directory owned by this user
// that neither group nor others can write to -- anything they could write here we would later load and launch.
bool cache_dir_usable(const std::string& path) {
    if (path.empty()) return false;
    for (size_t i = 1; i <= path.size(); ++i)
        if (i == path.size() || path[i] == '/') mkdir(path.substr(0, i).c_str(), 0700);
    struct stat st;
    if (stat(path.c_str(), &st) != 0 || !S_ISDIR(st.st_mode)) return false;
    return st.st_uid == geteuid() && (st.st_mode & (S_IWGRP | S_IWOTH)) == 0;
}

// Cache file: "RBJ2" | key_len u64 | key bytes | n_names u32 | (len u32, bytes)* | cubin_len u64 | cubin | fnv1a64(cubin).
// `key` is the FULL key material (model table, options, kernel expressions, compiler version, a hash of the kernel
// sources): the file name is only a 64-bit hash of it, so a read compares every byte of the key and the checksum of
// the image and treats any mismatch (collision, stale file, bit rot, foreign file) as a miss.
bool cache_read(const std::string& file, const std::string& key, RbJitImage& img) {
    struct stat st;
    if (stat(file.c_str(), &st) != 0 || !S_ISREG(st.st_mode) || st.st_uid != geteuid() || (st.st_mode & (S_IWGRP | S_IWOTH))) return false;
    std::ifstream f(file, std::ios::binary);
    if (!f) return false;
    char magic[4]; uint64_t klen = 0; uint32_t cnt = 0;
    f.read(magic, 4); f.read((char*)&klen, 8);
    if (!f || memcmp(magic, "RBJ2", 4) != 0 || klen != key.size()) return false;
    std::string stored(klen, '\0'); f.read(&stored[0], (std::streamsize)klen);
    if (!f || stored != key) return false;
    f.read((char*)&cnt, 4);
    if (!f || cnt != RB_JIT_KERNELS) return false;
    img.lowered.clear();
    for (uint32_t k = 0; k < cnt; ++k) {
        uint32_t len = 0; f.read((char*)&len, 4);
        if (!f || len > 4096) return false;
        std::string s(len, '\0'); f.read(&s[0], len);
        img.lowered.push_back(s);
    }
    uint64_t clen = 0, sum = 0; f.read((char*)&clen, 8);
    if (!f || clen == 0 || clen > (64u << 20)) return false;
    img.cubin.resize(clen); f.read(img.cubin.data(), (std::streamsize)clen);
    f.read((char*)&sum, 8);
    if (!f) return false;
    return sum == fnv1a(0xcbf29ce484222325ULL, img.cubin.data(), img.cubin.size());
}

void cache_write(const std::string& file, const std::string& key, const RbJitImage& img) {
    const std::string tmp = file + ".tmp" + std::to_string((long)getpid());
    {
        const int fd = open(tmp.c_str(), O_WRONLY | O_CREAT | O_EXCL | O_NOFOLLOW, 0600);
        if (fd < 0) return;
        close(fd);
        std::ofstream f(tmp, std::ios::binary | std::ios::trunc);
        if (!f) { remove(tmp.c_str()); return; }
        uint64_t klen = key.size();
        uint32_t cnt = (uint32_t)img.lowered.size();
        f.write("RBJ2", 4); f.write((const char*)&klen, 8); f.write(key.data(), (std::streamsize)klen);
        f.write((const char*)&cnt, 4);
        for (const auto& s : img.lowered) { uint32_t len = (uint32_t)s.size(); f.write((const char*)&len, 4); f.write(s.data(), len); }
        uint64_t clen = img.cubin.size(); f.write((const char*)&clen, 8); f.write(img.cubin.data(), (std::streamsize)clen);
        const uint64_t sum = fnv1a(0xcbf29ce484222325ULL, img.cubin.data(), img.cubin.size());
        f.write((const char*)&sum, 8);
        if (!f) { remove(tmp.c_str()); return; }
    }
    rename(tmp.c_str(), file.c_str());      // atomic publish: concurrent processes never see a partial file
}

}  // namespace

int rb_jit_compile(const RbHostModel& m, RbJitImage& img, std::string& log) {
    if (m.n < 1 || m.n > RB_JIT_LONG_MAX_N) { log = "chain too long for unrolled kernels"; return RB_ERR_UNSUPPORTED; }
    // beyond RB_JIT_MAX_N joints the unrolled forward dynamics / rollout are no longer worth their compile time (nor
    // faster than the lane-per-joint kernel): compile the O(n) and output-bound kernels only
    const bool long_set = m.n > RB_JIT_MAX_N;
    if (long_set && !m.serial) { log = "trees beyond 18 joints run on the run-time-n family"; return RB_ERR_UNSUPPORTED; }
    const char* const* exprs = long_set ? kLongExprs : kKernelExprs;
    auto wanted = [&](int k) { return exprs[k] != nullptr; };
    std::string err;
    const Nvrtc* nv = load_nvrtc(err);
    if (!nv) { log = err; return RB_ERR_UNSUPPORTED; }
    const std::string main_src = std::string(long_set ? "#include \"rb_kernels_long.cuh\"\n" : "#include \"rb_kernels.cuh\"\n") +
                                 rb_model_emit_header(m, "TabJit");

    // cache key: everything that determines the cubin
    int vmaj = 0, vmin = 0;
    nv->Version(&vmaj, &vmin);
    // tuning knob: extra whitespace-separated compiler options (e.g. "-DRB_MINB_FD=2"), part of the cache key
    std::vector<std::string> extra;
    if (const char* e = getenv("RIGIDBODY_B200_JIT_FLAGS")) {
        std::string cur;
        for (const char* c = e;; ++c) {
            if (*c == ' ' || *c == '\0') { if (!cur.empty()) extra.push_back(cur); cur.clear(); if (!*c) break; }
            else cur += *c;
        }
    }
    uint64_t hs = 0xcbf29ce484222325ULL, hs2 = 0x84222325cbf29ce4ULL;       // the embedded kernel sources, two independent hashes
    for (int k = 0; k < rb_jit_src_count; ++k) {
        hs = fnv1a(hs, rb_jit_src_texts[k], strlen(rb_jit_src_texts[k]));
        hs2 = fnv1a(hs2 ^ (uint64_t)k, rb_jit_src_texts[k], strlen(rb_jit_src_texts[k]));
    }
    char num[96];
    snprintf(num, sizeof num, "nvrtc %d.%d kernels %d sources %016llx%016llx\n", vmaj, vmin, RB_JIT_KERNELS,
             (unsigned long long)hs, (unsigned long long)hs2);
    std::string key = num;
    for (const char* o : kOptions) { key += o; key += '\n'; }
    for (const std::string& o : extra) { key += o; key += '\n'; }
    for (int k = 0; k < RB_JIT_KERNELS; ++k) { key += exprs[k] ? exprs[k] : "-"; key += '\n'; }
    key += main_src;                                                        // includes the model table, digit for digit
    const uint64_t h = fnv1a(0xcbf29ce484222325ULL, key.data(), key.size());
    char keybuf[32]; snprintf(keybuf, sizeof keybuf, "%016llx", (unsigned long long)h);
    const std::string dir = cache_dir(), file = dir + "/" + keybuf + ".rbjit";
    const bool use_cache = cache_dir_usable(dir);      // empty $RIGIDBODY_B200_CACHE, no $HOME or an untrusted directory: no cache
    if (use_cache && cache_read(file, key, img)) { img.from_cache = true; log = "cache hit " + file; return RB_OK; }

    nvrtcProgram prog = nullptr;
    if (nv->CreateProgram(&prog, main_src.c_str(), "rb_jit_model.cu", rb_jit_src_count, rb_jit_src_texts, rb_jit_src_names) != 0) {
        log = "nvrtcCreateProgram failed"; return RB_ERR_CUDA;
    }
    for (int k = 0; k < RB_JIT_KERNELS; ++k) if (wanted(k)) nv->AddNameExpression(prog, exprs[k]);
    std::vector<const char*> opts(kOptions, kOptions + sizeof kOptions / sizeof kOptions[0]);
    for (const std::string& o : extra) opts.push_back(o.c_str());
    const int rc = nv->CompileProgram(prog, (int)opts.size(), opts.data());
    size_t ls = 0;
    nv->GetProgramLogSize(prog, &ls);
    if (ls > 1) { std::string l(ls, '\0'); nv->GetProgramLog(prog, &l[0]); log = l; }
    if (rc != 0) { nv->DestroyProgram(&prog); if (log.empty()) log = "nvrtcCompileProgram failed"; return RB_ERR_CUDA; }
    img.lowered.clear();
    for (int k = 0; k < RB_JIT_KERNELS; ++k) {
        const char* e = exprs[k];
        const char* low = nullptr;
        if (!wanted(k)) { img.lowered.push_back(std::string()); continue; }        // not part of this chain's kernel set
        if (nv->GetLoweredName(prog, e, &low) != 0 || !low) { nv->DestroyProgram(&prog); log = std::string("no lowered name for ") + e; return RB_ERR_CUDA; }
        img.lowered.push_back(low);
    }
    size_t cs = 0;
    nv->GetCUBINSize(prog, &cs);
    img.cubin.resize(cs);
    nv->GetCUBIN(prog, img.cubin.data());
    nv->DestroyProgram(&prog);
    img.from_cache = false;
    if (use_cache) cache_write(file, key, img);
    return RB_OK;
}

int rb_jit_load(const RbJitImage& img, int n, RbJitParam& out, std::string& err) {
    cudaLibrary_t lib = nullptr;
    cudaError_t e = cudaLibraryLoadData(&lib, img.cubin.data(), nullptr, nullptr, 0, nullptr, nullptr, 0);
    if (e != cudaSuccess) { err = std::string("cudaLibraryLoadData: ") + cudaGetErrorString(e); return RB_ERR_CUDA; }
    out.lib = lib;
    out.n = n;
    for (int k = 0; k < RB_JIT_KERNELS; ++k) {
        cudaKernel_t kern = nullptr;
        if (img.lowered[k].empty()) { out.k[k] = nullptr; continue; }
        e = cudaLibraryGetKernel(&kern, lib, img.lowered[k].c_str());
        if (e != cudaSuccess) { err = std::string("cudaLibraryGetKernel(") + img.lowered[k] + "): " + cudaGetErrorString(e); cudaLibraryUnload(lib); out.lib = nullptr; return RB_ERR_CUDA; }
        out.k[k] = kern;
    }
    if (aos_smem(n) > 48 * 1024)
        for (int k : {RB_JK_RNEA_AOS, RB_JK_FD_AOS})
            if (out.k[k]) cudaFuncSetAttribute((const void*)out.k[k], cudaFuncAttributeMaxDynamicSharedMemorySize, (int)aos_smem(n));
    return RB_OK;
}

void rb_jit_unload(RbJitParam& p) {
    if (p.lib) cudaLibraryUnload((cudaLibrary_t)p.lib);
    p.lib = nullptr;
}

// ---- launchers: same grids / blocks / shared memory as RbLaunch<M> in rb_kernels.cuh ---------------------------------
namespace {
// Launches kernel `k` of the chain's image over B states in blocks of `block` threads.  The kernel takes the (empty)
// model parameter, then `a` in order: each must have the exact type of its kernel parameter (size_t B and ld, not int).
template <class... A>
cudaError_t jlaunch(const void* param, int k, int block, size_t smem, size_t B, cudaStream_t st, A... a) {
    if (B == 0) return cudaSuccess;
    RbEmptyParam ep{0};
    void* args[] = {&ep, &a...};
    return cudaLaunchKernel((const void*)((const RbJitParam*)param)->k[k], dim3((unsigned)((B + block - 1) / block)), dim3(block),
                            args, smem, st);
}
cudaError_t j_rnea(const void* p, const double* q, const double* dq, const double* ddq, double* tau, size_t B, size_t ld, cudaStream_t st) {
    return jlaunch(p, RB_JK_RNEA, RB_BLOCK, 0, B, st, q, dq, ddq, tau, B, ld);
}
cudaError_t j_rnea_aos(const void* p, const double* q, const double* dq, const double* ddq, double* tau, size_t B, cudaStream_t st) {
    return jlaunch(p, RB_JK_RNEA_AOS, RB_BLOCK, aos_smem(((const RbJitParam*)p)->n), B, st, q, dq, ddq, tau, B, (size_t)0);
}
cudaError_t j_fd(const void* p, const double* q, const double* dq, const double* tau, double* qdd, size_t B, size_t ld, int* status, cudaStream_t st) {
    return jlaunch(p, RB_JK_FD, RB_BLOCK, 0, B, st, q, dq, tau, qdd, B, ld, status);
}
cudaError_t j_fd_aos(const void* p, const double* q, const double* dq, const double* tau, double* qdd, size_t B, int* status, cudaStream_t st) {
    return jlaunch(p, RB_JK_FD_AOS, RB_BLOCK, aos_smem(((const RbJitParam*)p)->n), B, st, q, dq, tau, qdd, B, (size_t)0, status);
}
cudaError_t j_crba(const void* p, const double* q, double* H, size_t B, size_t ld, cudaStream_t st) {
    return jlaunch(p, RB_JK_CRBA, RB_BLOCK, 0, B, st, q, H, B, ld);
}
cudaError_t j_fk(const void* p, const double* q, double* x, size_t B, size_t ld, cudaStream_t st) {
    return jlaunch(p, RB_JK_FK, RB_BLOCK, 0, B, st, q, x, B, ld);
}
cudaError_t j_jac(const void* p, const double* q, double* J, size_t B, size_t ld, cudaStream_t st) {
    return jlaunch(p, RB_JK_JAC, RB_BLOCK, 0, B, st, q, J, B, ld);
}
cudaError_t j_rollout(const void* p, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                      double* q_traj, double* dq_traj, double* q_fin, double* dq_fin, size_t B, size_t ld, int* status,
                      const double* cost_w, double* cost, cudaStream_t st) {
    return jlaunch(p, RB_JK_ROLLOUT, RB_RO_BLOCK, 0, B, st, q0, dq0, tau, dt, horizon, q_traj, dq_traj, q_fin, dq_fin, B, ld,
                   status, cost_w, cost);
}
cudaError_t j_rollout_tip(const void* p, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                          double* q_traj, double* dq_traj, double* q_fin, double* dq_fin, size_t B, size_t ld, int* status,
                          const double* cost_w, double* cost, cudaStream_t st) {
    return jlaunch(p, RB_JK_ROLLOUT_TIP, RB_RO_BLOCK, 0, B, st, q0, dq0, tau, dt, horizon, q_traj, dq_traj, q_fin, dq_fin, B, ld,
                   status, cost_w, cost);
}
cudaError_t j_rollout_col(const void* p, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                          double* q_traj, double* dq_traj, double* q_fin, double* dq_fin, size_t B, size_t ld, int* status,
                          const double* cost_w, double* cost, cudaStream_t st) {
    return jlaunch(p, RB_JK_ROLLOUT_COL, RB_RO_BLOCK, 0, B, st, q0, dq0, tau, dt, horizon, q_traj, dq_traj, q_fin, dq_fin, B, ld,
                   status, cost_w, cost);
}
cudaError_t j_rnea_f32(const void* p, const float* q, const float* dq, const float* ddq, float* tau, size_t B, size_t ld, cudaStream_t st) {
    return jlaunch(p, RB_JK_RNEA_F32, RB_BLOCK, 0, B, st, q, dq, ddq, tau, B, ld);
}
cudaError_t j_fd_f32(const void* p, const float* q, const float* dq, const float* tau, float* qdd, size_t B, size_t ld, int* status, cudaStream_t st) {
    return jlaunch(p, RB_JK_FD_F32, RB_BLOCK, 0, B, st, q, dq, tau, qdd, B, ld, status);
}
cudaError_t j_rnea_fd(const void* p, const double* q, const double* dq, const double* ddq, const double* tau_in, double* out,
                      size_t B, size_t ld, int* status, cudaStream_t st) {
    return jlaunch(p, RB_JK_RNEA_FD, RB_BLOCK, 0, B, st, q, dq, ddq, tau_in, out, B, ld, status);
}
}  // namespace

const RbOps* rb_ops_jit_long() {
    static const RbOps ops = [] {
        RbOps o{};
        o.name = "jit-long"; o.param_bytes = sizeof(RbJitParam);
        o.rnea = &j_rnea; o.crba = &j_crba; o.fwd_kin = &j_fk; o.jac = &j_jac;
        return o;
    }();
    return &ops;
}

const RbOps* rb_ops_jit() {
    static const RbOps ops = [] {
        RbOps o{};
        o.name = "jit-specialised"; o.param_bytes = sizeof(RbJitParam);
        o.rnea = &j_rnea; o.fd = &j_fd; o.rnea_aos = &j_rnea_aos; o.fd_aos = &j_fd_aos; o.crba = &j_crba; o.fwd_kin = &j_fk;
        o.jac = &j_jac; o.rollout = &j_rollout; o.rollout_tip = &j_rollout_tip; o.rollout_col = &j_rollout_col; o.rnea_f32 = &j_rnea_f32; o.fd_f32 = &j_fd_f32; o.rnea_fd = &j_rnea_fd;
        return o;
    }();
    return &ops;
}
