// rb_api.cu -- the C ABI declared in include/rigidbody.h.
//
// Host side of the engine: owns the flattened model, picks a kernel family, validates arguments, moves host
// batches through pinned/pipelined copies, and never lets an exception or a CUDA error escape as anything
// but an RbStatus + message.  There is no CPU implementation behind any entry point.
#include <cuda_runtime.h>

#include <algorithm>
#include <atomic>
#include <chrono>
#include <cmath>
#include <condition_variable>
#include <functional>
#include <thread>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <new>
#include <string>
#include <vector>

#include "../../include/rigidbody.h"
#include "rb_host_model.h"
#include "rb_jit.h"
#include "rb_kernels.cuh"
#include "rb_util.cuh"

namespace {

thread_local std::string g_err;

int fail(int code, const std::string& msg) { g_err = msg; return code; }
int fail_cuda(cudaError_t e, const char* what) {
    g_err = std::string(what) + ": " + cudaGetErrorName(e) + " (" + cudaGetErrorString(e) + ")";
    return RB_ERR_CUDA;
}
#define RB_CUDA(call)                                              \
    do {                                                           \
        cudaError_t e__ = (call);                                  \
        if (e__ != cudaSuccess) return fail_cuda(e__, #call);      \
    } while (0)

constexpr int kSlots = 3;       // depth of the host-batch pipeline

struct DevBuf {
    double* p = nullptr; size_t bytes = 0;
    int ensure(size_t need) {
        if (need <= bytes) return RB_OK;
        if (p) cudaFree(p);
        p = nullptr; bytes = 0;
        cudaError_t e = cudaMalloc((void**)&p, need);
        if (e != cudaSuccess) return fail_cuda(e, "cudaMalloc(staging)");
        bytes = need;
        return RB_OK;
    }
    void release() { if (p) cudaFree(p); p = nullptr; bytes = 0; }
};

// One entry point of an engine, bound when the engine is created: the launcher, its parameter block, and whether its
// kernels work in engine-owned scratch (RbOps::shared_scratch).
template <class Fn>
struct Bound { Fn fn = nullptr; const void* param = nullptr; bool shared = false; };

}  // namespace

// One host thread per device of a multi-device engine: runs the slice of a host batch that its device owns.
struct RbWorker {
    std::thread th;
    std::mutex m;
    std::condition_variable cv;
    std::function<int()> job;
    bool has_job = false, done = true, stop = false;
    int rc = RB_OK;
    std::string err;
    void run_loop() {
        std::unique_lock<std::mutex> lk(m);
        for (;;) {
            cv.wait(lk, [&] { return has_job || stop; });
            if (stop) return;
            std::function<int()> j = std::move(job);
            has_job = false;
            lk.unlock();
            int r = RB_ERR_ARG; std::string e;
            try { r = j(); if (r != RB_OK) e = g_err; }
            catch (const std::exception& ex) { r = RB_ERR_ARG; e = std::string("exception: ") + ex.what(); }
            lk.lock();
            rc = r; err = e; done = true;
            cv.notify_all();
        }
    }
    void start() { th = std::thread([this] { run_loop(); }); }
    void submit(std::function<int()> j) {
        std::lock_guard<std::mutex> lk(m);
        job = std::move(j); has_job = true; done = false;
        cv.notify_all();
    }
    int wait(std::string* e) {
        std::unique_lock<std::mutex> lk(m);
        cv.wait(lk, [&] { return done; });
        if (rc != RB_OK && e) *e = err;
        return rc;
    }
    void shutdown() {
        { std::lock_guard<std::mutex> lk(m); stop = true; cv.notify_all(); }
        if (th.joinable()) th.join();
    }
};

struct RbGpu {
    // A multi-device engine (multibody_gpu_new_multi) is a dispatcher: `peers` holds one ordinary single-device engine
    // per device and `workers` one host thread per peer; it owns no CUDA resources itself.  Host batches are cut into
    // contiguous slices, one per device (SURVEY.md 8e); empty for an ordinary engine.
    std::vector<RbGpu*> peers;
    std::vector<RbWorker*> workers;
    std::mutex mu_multi;                  // one multi-device call at a time (the workers hold one job each)
    int device = 0;
    int sm_count = 0;
    RbHostModel model;
    const RbOps* ops = nullptr;           // the primary family
    std::vector<unsigned char> param;     // host image of the kernel-parameter block `ops` expects
    std::vector<double> flat;             // the model rows as uploaded (rb_model.h layout)
    std::vector<unsigned char> param_n;   // parameter block of the fallback table (run-time-n family) if `ops` leaves entries null
    // bound by bind_entries; the optional entries (rnea_aos, fd_aos, rnea_fd, rnea_f32, fd_f32) are the primary family's alone
    Bound<decltype(RbOps::rnea)> rnea; Bound<decltype(RbOps::fd)> fd; Bound<decltype(RbOps::crba)> crba;
    Bound<decltype(RbOps::fwd_kin)> fwd_kin; Bound<decltype(RbOps::jac)> jac; Bound<decltype(RbOps::rollout)> rollout;
    size_t hpk_states = 0;
    RbJitParam jit{};                     // run-time compiled kernels (jit-specialised family); lib == nullptr if unused
    std::string family_note;              // why this family was chosen (e.g. the JIT fallback reason)
    bool split_rnea_fd = false;           // $RIGIDBODY_B200_FUSED=0: multibody_rnea_fd_batch issues the two launches instead of the fused kernel
    double* d_model = nullptr;            // model rows on the device (run-time-n family, tip pose, inverse kinematics)
    DevBuf scratch;                       // generic-n: per-thread strided scratch
    DevBuf hpk;                           // generic-n: packed H of one chunk of states (forward dynamics)
    DevBuf cost_w;                        // rollout cost weights (RB_CW_DOUBLES_COL doubles: rows, then the collision block), engine-owned: ordered like scratch
    DevBuf link_rot;                      // [n][9] Q_l^T of every link (RbHostModel::link_rot), for link poses in descriptor frames
    size_t scratch_threads = 0;
    cudaStream_t stream = nullptr, s_h2d = nullptr, s_d2h = nullptr;
    cudaEvent_t ev_h2d[kSlots] = {}, ev_comp[kSlots] = {}, ev_d2h[kSlots] = {};
    DevBuf in[kSlots], out[kSlots], tmp[kSlots];
    // Device status words (RB_STATUS_* bits set by kernels with atomicOr) and their pinned host mirrors:
    //   [0] accumulates over RB_MEM_DEVICE calls (any stream, any thread) until multibody_gpu_sync reads and clears it;
    //   [1] belongs to the ONE host-batch call holding `mu`: cleared when the call starts, read before `mu` is released,
    //       so a host call never reports (or swallows) a bit set by somebody else's states.
    int* d_status = nullptr;
    int* h_status = nullptr;              // pinned, 2 words
    std::mutex mu_status;                 // serialises readers of word [0]
    int sticky = RB_OK;
    std::atomic<uint64_t> launches{0};
    cudaEvent_t ev_scratch = nullptr;     // orders users of the engine-owned scratch (run-time-n / long-chain families) across streams
    std::mutex mu;                        // serialises host-batch calls that share the staging buffers
    std::mutex mu_scratch;                // guards ev_scratch
};

struct Multibody {
    RbHostModel model;
    RbGpu* gpu = nullptr;                 // created on first use
    std::mutex mu;
};

namespace {

// Kernel families that work in engine-owned scratch (RbOps::shared_scratch) must not overlap with each other
// across streams: every such launch waits for the previous one's event and records its own.
struct ScratchOrder {
    RbGpu* g; cudaStream_t st; bool on;
    ScratchOrder(RbGpu* g_, bool shared, cudaStream_t st_) : g(g_), st(st_), on(shared) {
        if (on) { g->mu_scratch.lock(); cudaStreamWaitEvent(st, g->ev_scratch, 0); }
    }
    ~ScratchOrder() {
        if (on) { cudaEventRecord(g->ev_scratch, st); g->mu_scratch.unlock(); }
    }
};

// Runs a bound entry on stream `st` (every RbOps launcher takes the stream last), ordered by ScratchOrder.
template <class Fn, class... A>
cudaError_t launch(RbGpu* g, const Bound<Fn>& e, cudaStream_t st, A... a) {
    ScratchOrder so(g, e.shared, st);
    return e.fn(e.param, a..., st);
}

struct DeviceGuard {
    int prev = -1; bool ok = true;
    explicit DeviceGuard(int dev) {
        if (cudaGetDevice(&prev) != cudaSuccess) { prev = -1; }
        if (prev != dev) ok = cudaSetDevice(dev) == cudaSuccess;
    }
    ~DeviceGuard() { if (prev >= 0) cudaSetDevice(prev); }
};

// Sets up the run-time-n family (model rows + scratch + H chunk on the device); `param` receives its parameter block.
int setup_generic_n(RbGpu* g, std::vector<unsigned char>* param) {
    const int n = g->model.n;
    const std::vector<double>& flat = g->flat;
    RB_CUDA(cudaMalloc((void**)&g->d_model, flat.size() * sizeof(double)));
    RB_CUDA(cudaMemcpy(g->d_model, flat.data(), flat.size() * sizeof(double), cudaMemcpyHostToDevice));
    // persistent grid: 8 blocks of RB_BLOCK threads per SM; scratch sized for the largest user (rollout)
    g->scratch_threads = (size_t)g->sm_count * 8 * RB_BLOCK;
    const bool tree = !g->model.serial;
    const size_t slots = (size_t)(tree ? 24 : 12) * n + (size_t)n * n;
    int rc = g->scratch.ensure(slots * g->scratch_threads * sizeof(double));
    if (rc != RB_OK) return rc;
    if (n > 32 || tree) {
        // forward dynamics of chains beyond a warp's width: H (packed upper triangle) of one chunk of states lives in
        // HBM between the kernel that builds it and the tile kernel that factorises it in shared memory (<= 1 GiB)
        const size_t np = (size_t)n * (n + 1) / 2;
        const size_t chunk = ((size_t)1024 << 20) / (np * sizeof(double));
        g->hpk_states = std::max<size_t>(1024, chunk / 1024 * 1024);
        rc = g->hpk.ensure(np * g->hpk_states * sizeof(double));
        if (rc != RB_OK) return rc;
    }
    RbNParam P{g->d_model, n, g->scratch.p, g->scratch_threads, slots, g->hpk.p, g->hpk_states, tree ? 1 : 0};
    param->assign(sizeof(P), 0);
    if (rb_ops_generic_n()->param_bytes != sizeof(P)) return fail(RB_ERR_ARG, "internal: RbNParam size mismatch");
    memcpy(param->data(), &P, sizeof(P));
    return RB_OK;
}

// Compiles (or reads from the disk cache) and loads the run-time specialised kernels of the chain and installs them as
// the primary family: rb_jit_compile builds the full set up to RB_JIT_MAX_N joints ("jit-specialised") and the long-chain
// set beyond ("jit-long").  On failure returns the status with the reason in `log`; the caller decides whether it is fatal.
int install_jit(RbGpu* g, std::string& log) {
    RbJitImage img;
    int rc = rb_jit_compile(g->model, img, log);
    if (rc == RB_OK) { std::string err; rc = rb_jit_load(img, g->model.n, g->jit, err); if (rc != RB_OK) log = err; }
    if (rc != RB_OK) return rc;
    g->ops = g->model.n > RB_JIT_MAX_N ? rb_ops_jit_long() : rb_ops_jit();
    g->param.assign(sizeof(RbJitParam), 0);
    memcpy(g->param.data(), &g->jit, sizeof(RbJitParam));
    g->family_note = std::string(g->model.serial ? "" : "kinematic tree: ") + (img.from_cache ? "kernels from the disk cache" : "kernels compiled with NVRTC");
    return RB_OK;
}

// Chooses the primary kernel family for the uploaded chain ($RIGIDBODY_B200_VARIANT forces one, $RIGIDBODY_B200_JIT=0
// keeps `auto` off the run-time compiler).  The families are tried top to bottom; the first that fits serves.
int pick_ops(RbGpu* g) {
    const char* force = getenv("RIGIDBODY_B200_VARIANT");
    const char* jit_env = getenv("RIGIDBODY_B200_JIT");
    const std::string want = force ? force : "auto";
    const bool any = want == "auto", jit_on = !(jit_env && std::string(jit_env) == "0");
    const int n = g->model.n;
    g->flat = rb_model_flat(g->model);
    const std::vector<double>& flat = g->flat;
    const std::string too_long = "RIGIDBODY_B200_VARIANT=jit-specialised needs a chain of at most " + std::to_string(RB_JIT_MAX_N) + " joints";
    std::string log;
    if (!g->model.serial) {
        // kinematic trees (parent[i] != i-1): run-time specialised kernels up to RB_JIT_MAX_N joints (the unrolled templates follow
        // the compile-time parent table, rb_dyn_tree.cuh), the run-time-n family otherwise
        if (!any && want != "generic-n" && want != "jit-specialised")
            return fail(RB_ERR_UNSUPPORTED, "RIGIDBODY_B200_VARIANT=" + want + " serves serial chains only; trees run on jit-specialised or generic-n");
        if ((want == "jit-specialised" || (any && jit_on)) && n <= RB_JIT_MAX_N) {
            const int rc = install_jit(g, log);
            if (rc == RB_OK) return RB_OK;
            if (want == "jit-specialised") return fail(rc, "run-time specialisation failed: " + log);
        } else if (want == "jit-specialised") {
            return fail(RB_ERR_UNSUPPORTED, too_long);
        }
        g->family_note = "kinematic tree: run-time-n kernels (rbn_tree_* recursions)";
        g->ops = rb_ops_generic_n();
        return setup_generic_n(g, &g->param);
    }
    const bool is_fr3 = n == 7 && memcmp(flat.data(), rb_fr3_table(), sizeof(double) * RB_MODEL_DOUBLES(7)) == 0;
    const bool is_c32 = n == 32 && memcmp(flat.data(), rb_chain32_table(), sizeof(double) * RB_MODEL_DOUBLES(32)) == 0;
    const bool jit_auto = any && jit_on && !is_c32;
    // the compiled-in FR3 model
    if ((any || want == "fr3-specialised") && is_fr3) {
        g->ops = rb_ops_fr3();
        g->param.assign(g->ops->param_bytes, 0);
        return RB_OK;
    }
    if (want == "fr3-specialised") return fail(RB_ERR_UNSUPPORTED, "RIGIDBODY_B200_VARIANT=fr3-specialised but the chain is not the compiled-in FR3 model");
    // any other short chain: the same templates compiled for ITS constants at run time (NVRTC, disk-cached)
    if ((want == "jit-specialised" || jit_auto) && n <= RB_JIT_MAX_N) {
        const int rc = install_jit(g, log);
        if (rc == RB_OK) return RB_OK;
        if (want == "jit-specialised") return fail(rc, "run-time specialisation failed: " + log);
        g->family_note = "run-time specialisation unavailable (" + log.substr(0, 200) + "); using run-time-constant kernels";
    } else if (want == "jit-specialised") {
        return fail(RB_ERR_UNSUPPORTED, too_long);
    }
    // chains of 19..32 joints: rnea / crba / fwd_kin / jac specialised at load time, forward dynamics and rollouts
    // through the fallback table (lane-per-joint kernels)
    if ((want == "jit-long" || jit_auto) && n > RB_JIT_MAX_N && n <= RB_JIT_LONG_MAX_N) {
        const int rc = install_jit(g, log);
        if (rc == RB_OK) return setup_generic_n(g, &g->param_n);
        if (want == "jit-long") return fail(rc, "run-time specialisation failed: " + log);
        g->family_note = "run-time specialisation unavailable (" + log.substr(0, 200) + "); using run-time-n kernels";
    } else if (want == "jit-long") {
        return fail(RB_ERR_UNSUPPORTED, "RIGIDBODY_B200_VARIANT=jit-long serves chains of 19..32 joints");
    }
    // any 7-joint chain, constants from the kernel-parameter bank
    if ((any || want == "generic-7") && n == 7) {
        g->ops = rb_ops_rt7();
        if (g->ops->param_bytes != flat.size() * sizeof(double)) return fail(RB_ERR_ARG, "internal: RbModelK<7> size mismatch");
        g->param.assign((const unsigned char*)flat.data(), (const unsigned char*)flat.data() + g->ops->param_bytes);
        return RB_OK;
    }
    if (want == "generic-7") return fail(RB_ERR_UNSUPPORTED, "RIGIDBODY_B200_VARIANT=generic-7 needs a 7-joint chain");
    if (!any && want != "generic-n" && want != "chain32-specialised" && want != "jit-specialised" && want != "jit-long")
        return fail(RB_ERR_ARG, "unknown RIGIDBODY_B200_VARIANT '" + want + "'");
    // the compiled-in 32-joint model: rnea / crba, the rest through the fallback table
    if ((any || want == "chain32-specialised") && is_c32) {
        g->ops = rb_ops_chain32();
        g->param.assign(g->ops->param_bytes, 0);
        return setup_generic_n(g, &g->param_n);
    }
    if (want == "chain32-specialised") return fail(RB_ERR_UNSUPPORTED, "RIGIDBODY_B200_VARIANT=chain32-specialised but the chain is not the compiled-in 32-joint model");
    g->ops = rb_ops_generic_n();
    return setup_generic_n(g, &g->param);
}

// Binds rnea, fd, crba, fwd_kin, jac and rollout once: to the primary family where it has the entry, otherwise to the
// fallback table, whose parameter block pick_ops set up for the families that need it.
int bind_entries(RbGpu* g) {
    bool ok = true;
    auto bind = [&](auto& e, auto RbOps::*fn) {
        const bool own = g->ops->*fn != nullptr;
        const RbOps* t = own ? g->ops : rb_ops_generic_n();
        e = {t->*fn, own ? g->param.data() : g->param_n.data(), t->shared_scratch};
        ok = ok && e.fn && (own || !g->param_n.empty());
    };
    bind(g->rnea, &RbOps::rnea); bind(g->fd, &RbOps::fd); bind(g->crba, &RbOps::crba);
    bind(g->fwd_kin, &RbOps::fwd_kin); bind(g->jac, &RbOps::jac); bind(g->rollout, &RbOps::rollout);
    return ok ? RB_OK : fail(RB_ERR_ARG, std::string("internal: kernel family '") + g->ops->name + "' leaves an entry point unbound");
}

int gpu_create(const RbHostModel& model, int device, RbGpu** out) {
    if (!out) return fail(RB_ERR_NULL, "out is NULL");
    *out = nullptr;
    int count = 0;
    cudaError_t e = cudaGetDeviceCount(&count);
    if (e != cudaSuccess || count == 0)
        return fail(RB_ERR_CUDA, std::string("no CUDA device available (") + cudaGetErrorString(e) +
                                     "); this engine has no CPU fallback");
    if (device < 0 || device >= count) return fail(RB_ERR_ARG, "device ordinal out of range");
    cudaDeviceProp prop;
    RB_CUDA(cudaGetDeviceProperties(&prop, device));
    // sm_100a code is architecture-specific: it runs on compute capability 10.0 and nothing else (not 10.3, not 12.x)
    if (prop.major != 10 || prop.minor != 0)
        return fail(RB_ERR_CUDA, std::string("device '") + prop.name + "' has compute capability " + std::to_string(prop.major) + "." +
                                     std::to_string(prop.minor) + "; the kernels are built (and run-time compiled) for sm_100a = 10.0 only");
    DeviceGuard dg(device);
    if (!dg.ok) return fail(RB_ERR_CUDA, "cudaSetDevice failed");
    RbGpu* g = new (std::nothrow) RbGpu();
    if (!g) return fail(RB_ERR_CUDA, "out of host memory");
    g->device = device;
    g->sm_count = prop.multiProcessorCount;
    g->model = model;
    auto bail = [&](int rc) { multibody_gpu_free(g); return rc; };
    if ((e = cudaStreamCreateWithFlags(&g->stream, cudaStreamNonBlocking)) != cudaSuccess) return bail(fail_cuda(e, "cudaStreamCreate"));
    if ((e = cudaStreamCreateWithFlags(&g->s_h2d, cudaStreamNonBlocking)) != cudaSuccess) return bail(fail_cuda(e, "cudaStreamCreate"));
    if ((e = cudaStreamCreateWithFlags(&g->s_d2h, cudaStreamNonBlocking)) != cudaSuccess) return bail(fail_cuda(e, "cudaStreamCreate"));
    for (int k = 0; k < kSlots; ++k) {
        if ((e = cudaEventCreateWithFlags(&g->ev_h2d[k], cudaEventDisableTiming)) != cudaSuccess) return bail(fail_cuda(e, "cudaEventCreate"));
        if ((e = cudaEventCreateWithFlags(&g->ev_comp[k], cudaEventDisableTiming)) != cudaSuccess) return bail(fail_cuda(e, "cudaEventCreate"));
        if ((e = cudaEventCreateWithFlags(&g->ev_d2h[k], cudaEventDisableTiming)) != cudaSuccess) return bail(fail_cuda(e, "cudaEventCreate"));
    }
    if ((e = cudaEventCreateWithFlags(&g->ev_scratch, cudaEventDisableTiming)) != cudaSuccess) return bail(fail_cuda(e, "cudaEventCreate"));
    if ((e = cudaMalloc((void**)&g->d_status, 2 * sizeof(int))) != cudaSuccess) return bail(fail_cuda(e, "cudaMalloc(status)"));
    if ((e = cudaMemset(g->d_status, 0, 2 * sizeof(int))) != cudaSuccess) return bail(fail_cuda(e, "cudaMemset(status)"));
    if ((e = cudaMallocHost((void**)&g->h_status, 2 * sizeof(int))) != cudaSuccess) return bail(fail_cuda(e, "cudaMallocHost(status)"));
    g->h_status[0] = g->h_status[1] = 0;
    // cost weights of multibody_rollout_cost: allocated once, here (a lazy first-call allocation would race)
    { int rcw = g->cost_w.ensure(sizeof(double) * RB_CW_DOUBLES_COL); if (rcw != RB_OK) return bail(rcw); }
    {
        const size_t bytes = sizeof(double) * g->model.link_rot.size();
        int rcl = g->link_rot.ensure(bytes);
        if (rcl != RB_OK) return bail(rcl);
        if ((e = cudaMemcpy(g->link_rot.p, g->model.link_rot.data(), bytes, cudaMemcpyHostToDevice)) != cudaSuccess)
            return bail(fail_cuda(e, "cudaMemcpy(link rotations)"));
    }
    int rc = pick_ops(g);
    if (rc == RB_OK) rc = bind_entries(g);
    if (rc != RB_OK) return bail(rc);
    // the tip-pose and inverse-kinematics kernels read the model rows from device memory whatever the family
    if (!g->d_model) {
        if ((e = cudaMalloc((void**)&g->d_model, g->flat.size() * sizeof(double))) != cudaSuccess) return bail(fail_cuda(e, "cudaMalloc(model)"));
        if ((e = cudaMemcpy(g->d_model, g->flat.data(), g->flat.size() * sizeof(double), cudaMemcpyHostToDevice)) != cudaSuccess)
            return bail(fail_cuda(e, "cudaMemcpy(model)"));
    }
    if (const char* f = getenv("RIGIDBODY_B200_FUSED")) g->split_rnea_fd = std::string(f) == "0";
    *out = g;
    return RB_OK;
}

// Reads and clears status word `which` (see RbGpu::d_status); maps it to an RbStatus.  Caller holds the lock that owns
// the word (mu for [1], mu_status for [0]) and g->stream has nothing of the caller's in flight but this.
int fetch_status(RbGpu* g, int which) {
    RB_CUDA(cudaMemcpyAsync(g->h_status + which, g->d_status + which, sizeof(int), cudaMemcpyDeviceToHost, g->stream));
    RB_CUDA(cudaMemsetAsync(g->d_status + which, 0, sizeof(int), g->stream));
    RB_CUDA(cudaStreamSynchronize(g->stream));
    const int bits = g->h_status[which];
    g->h_status[which] = 0;
    if (bits & RB_STATUS_NOT_SPD)
        return fail(RB_ERR_NOT_SPD, "forward dynamics: mass matrix not positive definite for at least one state (its qdd is NaN)");
    return RB_OK;
}

// A host-batch call that fails half-way must not return while copies it queued still read or write the caller's
// buffers, nor leave its staging slots and status word mid-flight for the next call.
void drain_host_pipeline(RbGpu* g) {
    cudaStreamSynchronize(g->s_h2d);
    cudaStreamSynchronize(g->stream);
    cudaStreamSynchronize(g->s_d2h);
    cudaMemsetAsync(g->d_status + 1, 0, sizeof(int), g->stream);
    cudaStreamSynchronize(g->stream);
    cudaGetLastError();
}

// ---- a batched op, described once, run from device or host memory ----
struct OpDesc {
    int n_in;                    // number of input state arrays
    const double* in[4];
    int in_per[4];               // doubles per state of each input
    double* out;
    int out_per;                 // doubles per state of the output
    // launch on SoA device buffers with leading dimension ld; `arg` is the op's own argument block (OpDesc::arg)
    cudaError_t (*launch)(RbGpu* g, const double* const* in, double* out, size_t B, size_t ld, cudaStream_t st, int* status,
                          const void* arg);
    // optional: launch directly on AoS device buffers (kernel stages through shared memory); null = transpose around `launch`
    cudaError_t (*launch_aos)(RbGpu* g, const double* const* in, double* out, size_t B, cudaStream_t st, int* status) = nullptr;
    bool (*has_aos)(RbGpu* g) = nullptr;
    const void* arg = nullptr;   // host block handed to `launch` unchanged (per-call options of the op)
};

int check_common(RbGpu* g, const OpDesc& op, size_t n_states, size_t& ld, RbLayout layout, RbMem mem) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    if (layout != RB_LAYOUT_SOA && layout != RB_LAYOUT_AOS) return fail(RB_ERR_ARG, "bad layout");
    if (mem != RB_MEM_HOST && mem != RB_MEM_DEVICE) return fail(RB_ERR_ARG, "bad mem");
    if (n_states == 0) return RB_OK;
    for (int k = 0; k < op.n_in; ++k) if (!op.in[k]) return fail(RB_ERR_NULL, "input pointer is NULL");
    if (!op.out) return fail(RB_ERR_NULL, "output pointer is NULL");
    if (layout == RB_LAYOUT_SOA) {
        if (ld == 0) ld = n_states;
        if (ld < n_states) return fail(RB_ERR_ARG, "ld < n_states");
    }
    return RB_OK;
}

int run_device(RbGpu* g, const OpDesc& op, size_t B, size_t ld, RbLayout layout, cudaStream_t st) {
    if (layout == RB_LAYOUT_SOA) {
        cudaError_t e = op.launch(g, op.in, op.out, B, ld, st, g->d_status, op.arg);
        g->launches += 1;
        if (e != cudaSuccess) return fail_cuda(e, "kernel launch");
        return RB_OK;
    }
    if (op.launch_aos && op.has_aos(g)) {
        cudaError_t e = op.launch_aos(g, op.in, op.out, B, st, g->d_status);
        g->launches += 1;
        if (e != cudaSuccess) return fail_cuda(e, "kernel launch");
        return RB_OK;
    }
    // AoS device pointers: transpose into per-call SoA scratch, compute, transpose back (stream-ordered).
    std::lock_guard<std::mutex> lk(g->mu);
    size_t in_d = 0;
    for (int k = 0; k < op.n_in; ++k) in_d += (size_t)op.in_per[k];
    int rc = g->in[0].ensure(in_d * B * sizeof(double)); if (rc) return rc;
    rc = g->out[0].ensure((size_t)op.out_per * B * sizeof(double)); if (rc) return rc;
    const double* soa_in[4]; size_t off = 0;
    for (int k = 0; k < op.n_in; ++k) {
        double* dst = g->in[0].p + off * B;
        cudaError_t e = rb_launch_aos_to_soa(op.in[k], dst, op.in_per[k], B, B, st);
        g->launches += 1;
        if (e != cudaSuccess) return fail_cuda(e, "aos_to_soa launch");
        soa_in[k] = dst; off += (size_t)op.in_per[k];
    }
    cudaError_t e = op.launch(g, soa_in, g->out[0].p, B, B, st, g->d_status, op.arg);
    g->launches += 1;
    if (e != cudaSuccess) return fail_cuda(e, "kernel launch");
    e = rb_launch_soa_to_aos(g->out[0].p, op.out, op.out_per, B, B, st);
    g->launches += 1;
    if (e != cudaSuccess) return fail_cuda(e, "soa_to_aos launch");
    // the transposes went through engine-owned staging: drain before another call may reuse it
    RB_CUDA(cudaStreamSynchronize(st));
    return RB_OK;
}

// Host batch: chunks flow H2D -> compute -> D2H on three streams through kSlots staging slots.  Caller holds g->mu.
int run_host_pipeline(RbGpu* g, const OpDesc& op, size_t B, size_t ld, RbLayout layout) {
    size_t in_d = 0;
    for (int k = 0; k < op.n_in; ++k) in_d += (size_t)op.in_per[k];
    const size_t per_state = (in_d + (size_t)op.out_per) * sizeof(double);
    size_t chunk = (size_t)(192u << 20) / per_state;                 // ~192 MiB of state per slot
    chunk = std::max<size_t>(1024, std::min<size_t>(chunk, (size_t)1 << 20));
    chunk = std::min(chunk, B);
    const bool aos = layout == RB_LAYOUT_AOS;
    const bool direct_aos = aos && op.launch_aos && op.has_aos(g);
    for (int s = 0; s < kSlots; ++s) {
        int rc = g->in[s].ensure(in_d * chunk * sizeof(double)); if (rc) return rc;
        rc = g->out[s].ensure((size_t)op.out_per * chunk * sizeof(double)); if (rc) return rc;
        if (aos) { rc = g->tmp[s].ensure(std::max(in_d, (size_t)op.out_per) * chunk * sizeof(double)); if (rc) return rc; }
    }
    size_t done = 0; int c = 0;
    for (; done < B; done += chunk, ++c) {
        const int s = c % kSlots;
        const size_t cnt = std::min(chunk, B - done);
        // inputs of this slot were last read by the compute of chunk c-kSlots
        if (c >= kSlots) RB_CUDA(cudaStreamWaitEvent(g->s_h2d, g->ev_comp[s], 0));
        // AoS: the landing zone tmp[s] also carried chunk c-kSlots' output to the host
        if (c >= kSlots && aos) RB_CUDA(cudaStreamWaitEvent(g->s_h2d, g->ev_d2h[s], 0));
        const double* soa_in[4]; size_t off = 0;
        for (int k = 0; k < op.n_in; ++k) {
            double* dst = g->in[s].p + off * chunk;
            if (!aos) {
                RB_CUDA(cudaMemcpy2DAsync(dst, cnt * sizeof(double), op.in[k] + done, ld * sizeof(double),
                                          cnt * sizeof(double), (size_t)op.in_per[k], cudaMemcpyHostToDevice, g->s_h2d));
            } else {
                // AoS chunk is one contiguous run; land it in tmp, transpose on the compute stream
                RB_CUDA(cudaMemcpyAsync(g->tmp[s].p + off * chunk, op.in[k] + done * (size_t)op.in_per[k],
                                        cnt * (size_t)op.in_per[k] * sizeof(double), cudaMemcpyHostToDevice, g->s_h2d));
            }
            soa_in[k] = dst; off += (size_t)op.in_per[k];
        }
        RB_CUDA(cudaEventRecord(g->ev_h2d[s], g->s_h2d));
        RB_CUDA(cudaStreamWaitEvent(g->stream, g->ev_h2d[s], 0));
        if (c >= kSlots) RB_CUDA(cudaStreamWaitEvent(g->stream, g->ev_d2h[s], 0));   // output slot drained
        if (aos && direct_aos) {
            // inputs landed in tmp[s] as AoS; the kernel reads them there and writes AoS output into out[s]
            const double* aos_in[4]; off = 0;
            for (int k = 0; k < op.n_in; ++k) { aos_in[k] = g->tmp[s].p + off * chunk; off += (size_t)op.in_per[k]; }
            cudaError_t e = op.launch_aos(g, aos_in, g->out[s].p, cnt, g->stream, g->d_status + 1);
            g->launches += 1;
            if (e != cudaSuccess) return fail_cuda(e, "kernel launch");
            RB_CUDA(cudaEventRecord(g->ev_comp[s], g->stream));
            RB_CUDA(cudaStreamWaitEvent(g->s_d2h, g->ev_comp[s], 0));
            RB_CUDA(cudaMemcpyAsync(op.out + done * (size_t)op.out_per, g->out[s].p, cnt * (size_t)op.out_per * sizeof(double),
                                    cudaMemcpyDeviceToHost, g->s_d2h));
            RB_CUDA(cudaEventRecord(g->ev_d2h[s], g->s_d2h));
            continue;
        }
        if (aos) {
            off = 0;
            for (int k = 0; k < op.n_in; ++k) {
                cudaError_t e = rb_launch_aos_to_soa(g->tmp[s].p + off * chunk, g->in[s].p + off * chunk, op.in_per[k], cnt, cnt, g->stream);
                g->launches += 1;
                if (e != cudaSuccess) return fail_cuda(e, "aos_to_soa launch");
                off += (size_t)op.in_per[k];
            }
            // SoA views inside the slot use ld = cnt
            off = 0;
            for (int k = 0; k < op.n_in; ++k) { soa_in[k] = g->in[s].p + off * chunk; off += (size_t)op.in_per[k]; }
        }
        cudaError_t e = op.launch(g, soa_in, g->out[s].p, cnt, cnt, g->stream, g->d_status + 1, op.arg);
        g->launches += 1;
        if (e != cudaSuccess) return fail_cuda(e, "kernel launch");
        if (aos) {
            e = rb_launch_soa_to_aos(g->out[s].p, g->tmp[s].p, op.out_per, cnt, cnt, g->stream);
            g->launches += 1;
            if (e != cudaSuccess) return fail_cuda(e, "soa_to_aos launch");
        }
        RB_CUDA(cudaEventRecord(g->ev_comp[s], g->stream));
        RB_CUDA(cudaStreamWaitEvent(g->s_d2h, g->ev_comp[s], 0));
        if (!aos) {
            RB_CUDA(cudaMemcpy2DAsync(op.out + done, ld * sizeof(double), g->out[s].p, cnt * sizeof(double),
                                      cnt * sizeof(double), (size_t)op.out_per, cudaMemcpyDeviceToHost, g->s_d2h));
        } else {
            RB_CUDA(cudaMemcpyAsync(op.out + done * (size_t)op.out_per, g->tmp[s].p, cnt * (size_t)op.out_per * sizeof(double),
                                    cudaMemcpyDeviceToHost, g->s_d2h));
        }
        RB_CUDA(cudaEventRecord(g->ev_d2h[s], g->s_d2h));
    }
    RB_CUDA(cudaStreamSynchronize(g->s_d2h));
    RB_CUDA(cudaStreamSynchronize(g->stream));
    return RB_OK;
}

int run_host(RbGpu* g, const OpDesc& op, size_t B, size_t ld, RbLayout layout, bool has_status) {
    std::lock_guard<std::mutex> lk(g->mu);
    int rc = RB_OK;
    if (has_status) {       // this call's own status word starts clean
        cudaError_t e = cudaMemsetAsync(g->d_status + 1, 0, sizeof(int), g->stream);
        if (e != cudaSuccess) return fail_cuda(e, "cudaMemsetAsync(status)");
    }
    rc = run_host_pipeline(g, op, B, ld, layout);
    if (rc != RB_OK) { const std::string keep = g_err; drain_host_pipeline(g); g_err = keep; return rc; }
    return has_status ? fetch_status(g, 1) : RB_OK;     // still under g->mu
}

// Contiguous slice of a batch owned by device `i` of `n`.
inline void slice_bounds(size_t B, size_t n, size_t i, size_t* lo, size_t* hi) { *lo = B * i / n; *hi = B * (i + 1) / n; }

const char* kMultiDeviceOnly = "a multi-device engine serves RB_MEM_HOST batches; for device pointers call the per-device engine (multibody_gpu_peer)";

// Runs job(i) for every peer on that peer's worker thread, waits for all of them; first hard error wins, otherwise
// RB_ERR_NOT_SPD if any slice reported it.
int run_on_peers(RbGpu* g, const std::function<int(size_t)>& job) {
    std::lock_guard<std::mutex> lk(g->mu_multi);
    const size_t n = g->peers.size();
    for (size_t i = 0; i < n; ++i) g->workers[i]->submit([&job, i] { return job(i); });
    int rc = RB_OK; std::string err;
    for (size_t i = 0; i < n; ++i) {
        std::string e;
        const int r = g->workers[i]->wait(&e);
        if (r != RB_OK && (rc == RB_OK || (rc == RB_ERR_NOT_SPD && r != RB_ERR_NOT_SPD))) { rc = r; err = "device " + std::to_string(g->peers[i]->device) + ": " + e; }
    }
    if (rc != RB_OK) g_err = err;
    return rc;
}

int run_host(RbGpu* g, const OpDesc& op, size_t B, size_t ld, RbLayout layout, bool has_status);

int run_op(RbGpu* g, OpDesc& op, size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream, bool has_status) {
    int rc = check_common(g, op, n_states, ld, layout, mem);
    if (rc != RB_OK || n_states == 0) return rc;
    if (!g->peers.empty()) {
        if (mem != RB_MEM_HOST) return fail(RB_ERR_UNSUPPORTED, kMultiDeviceOnly);
        const bool aos = layout == RB_LAYOUT_AOS;
        return run_on_peers(g, [&](size_t i) -> int {
            size_t lo, hi; slice_bounds(n_states, g->peers.size(), i, &lo, &hi);
            if (hi == lo) return RB_OK;
            RbGpu* pg = g->peers[i];
            OpDesc sub = op;            // same launchers, pointers advanced to the slice (SoA: column lo of every row)
            for (int k = 0; k < op.n_in; ++k) sub.in[k] = op.in[k] + lo * (aos ? (size_t)op.in_per[k] : 1);
            sub.out = op.out + lo * (aos ? (size_t)op.out_per : 1);
            DeviceGuard dg(pg->device);
            if (!dg.ok) return fail(RB_ERR_CUDA, "cudaSetDevice failed");
            return run_host(pg, sub, hi - lo, ld, layout, has_status);
        });
    }
    DeviceGuard dg(g->device);
    if (!dg.ok) return fail(RB_ERR_CUDA, "cudaSetDevice failed");
    if (mem == RB_MEM_DEVICE)
        return run_device(g, op, n_states, ld, layout, (cudaStream_t)stream);
    return run_host(g, op, n_states, ld, layout, has_status);
}

}  // namespace

// ===================================================================== construction
extern "C" int multibody_gpu_new(const RbChainDesc* desc, int device, RbGpu** out) {
    try {
        RbHostModel m; std::string err;
        int rc = rb_model_from_desc(desc, m, err);
        if (rc != RB_OK) { if (out) *out = nullptr; return fail(rc, err); }
        return gpu_create(m, device, out);
    } catch (const std::exception& e) { return fail(RB_ERR_ARG, std::string("exception: ") + e.what()); }
}

extern "C" int multibody_gpu_new_from_urdf(const char* urdf_path, int device, RbGpu** out) {
    try {
        RbHostModel m; std::string err;
        int rc = rb_model_from_urdf(urdf_path, m, err);
        if (rc != RB_OK) { if (out) *out = nullptr; return fail(rc, err); }
        return gpu_create(m, device, out);
    } catch (const std::exception& e) { return fail(RB_ERR_ARG, std::string("exception: ") + e.what()); }
}

namespace {
// n_dev single-device engines behind one dispatcher handle (n_dev == 1: just the engine).
int gpu_create_multi(const RbHostModel& model, const int* devices, int n_dev, RbGpu** out) {
    if (!out) return fail(RB_ERR_NULL, "out is NULL");
    *out = nullptr;
    if (!devices) return fail(RB_ERR_NULL, "devices is NULL");
    if (n_dev < 1 || n_dev > 64) return fail(RB_ERR_ARG, "n_dev must be 1..64");
    // test hook: RIGIDBODY_B200_ALLOW_DUPLICATE_DEVICES=1 lets a one-GPU box exercise the slicing / worker-thread path
    // (two engines on the same device); pointless in production, hence refused by default
    const char* dup = getenv("RIGIDBODY_B200_ALLOW_DUPLICATE_DEVICES");
    if (!(dup && dup[0] == '1'))
        for (int i = 0; i < n_dev; ++i)
            for (int k = 0; k < i; ++k)
                if (devices[i] == devices[k]) return fail(RB_ERR_ARG, "device listed twice");
    if (n_dev == 1) return gpu_create(model, devices[0], out);
    RbGpu* g = new (std::nothrow) RbGpu();
    if (!g) return fail(RB_ERR_CUDA, "out of host memory");
    g->device = devices[0];
    g->model = model;
    // the per-device engines are built concurrently (each may run the run-time compiler or read its disk cache)
    g->peers.assign((size_t)n_dev, nullptr);
    std::vector<int> rcs((size_t)n_dev, RB_OK);
    std::vector<std::string> errs((size_t)n_dev);
    {
        std::vector<std::thread> th;
        for (int i = 0; i < n_dev; ++i)
            th.emplace_back([&, i] {
                try { rcs[i] = gpu_create(model, devices[i], &g->peers[i]); if (rcs[i] != RB_OK) errs[i] = g_err; }
                catch (const std::exception& e) { rcs[i] = RB_ERR_ARG; errs[i] = std::string("exception: ") + e.what(); }
            });
        for (auto& t : th) t.join();
    }
    for (int i = 0; i < n_dev; ++i)
        if (rcs[i] != RB_OK) {
            const int rc = rcs[i]; const std::string msg = "device " + std::to_string(devices[i]) + ": " + errs[i];
            multibody_gpu_free(g);
            return fail(rc, msg);
        }
    g->ops = g->peers[0]->ops;            // kernel_variant and family_note only: the peers run the calls
    g->family_note = g->peers[0]->family_note;
    for (int i = 0; i < n_dev; ++i) {
        RbWorker* w = new (std::nothrow) RbWorker();
        if (!w) { multibody_gpu_free(g); return fail(RB_ERR_CUDA, "out of host memory"); }
        g->workers.push_back(w);
        w->start();
    }
    *out = g;
    return RB_OK;
}
}  // namespace

extern "C" int multibody_gpu_new_multi(const RbChainDesc* desc, const int* devices, int n_dev, RbGpu** out) {
    try {
        RbHostModel m; std::string err;
        int rc = rb_model_from_desc(desc, m, err);
        if (rc != RB_OK) { if (out) *out = nullptr; return fail(rc, err); }
        return gpu_create_multi(m, devices, n_dev, out);
    } catch (const std::exception& e) { return fail(RB_ERR_ARG, std::string("exception: ") + e.what()); }
}

extern "C" int multibody_gpu_new_multi_from_urdf(const char* urdf_path, const int* devices, int n_dev, RbGpu** out) {
    try {
        RbHostModel m; std::string err;
        int rc = rb_model_from_urdf(urdf_path, m, err);
        if (rc != RB_OK) { if (out) *out = nullptr; return fail(rc, err); }
        return gpu_create_multi(m, devices, n_dev, out);
    } catch (const std::exception& e) { return fail(RB_ERR_ARG, std::string("exception: ") + e.what()); }
}

extern "C" int multibody_gpu_n_devices(const RbGpu* g) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    return g->peers.empty() ? 1 : (int)g->peers.size();
}

extern "C" RbGpu* multibody_gpu_peer(RbGpu* g, int index) {
    if (!g) { fail(RB_ERR_NULL, "engine handle is NULL"); return nullptr; }
    if (g->peers.empty()) return index == 0 ? g : (fail(RB_ERR_ARG, "peer index out of range"), (RbGpu*)nullptr);
    if (index < 0 || index >= (int)g->peers.size()) { fail(RB_ERR_ARG, "peer index out of range"); return nullptr; }
    return g->peers[(size_t)index];
}

extern "C" int multibody_gpu_from_multibody(const Multibody* mb, int device, RbGpu** out) {
    if (!mb) return fail(RB_ERR_NULL, "Multibody handle is NULL");
    try { return gpu_create(mb->model, device, out); }
    catch (const std::exception& e) { return fail(RB_ERR_ARG, std::string("exception: ") + e.what()); }
}

extern "C" void multibody_gpu_free(RbGpu* g) {
    if (!g) return;
    if (!g->peers.empty() || !g->workers.empty()) {      // dispatcher of a multi-device engine: no CUDA resources of its own
        for (RbWorker* w : g->workers) { w->shutdown(); delete w; }
        for (RbGpu* pg : g->peers) multibody_gpu_free(pg);
        delete g;
        return;
    }
    DeviceGuard dg(g->device);
    cudaDeviceSynchronize();              // device calls may still be running on caller streams and use our scratch
    if (g->ev_scratch) cudaEventDestroy(g->ev_scratch);
    for (int k = 0; k < kSlots; ++k) {
        g->in[k].release(); g->out[k].release(); g->tmp[k].release();
        if (g->ev_h2d[k]) cudaEventDestroy(g->ev_h2d[k]);
        if (g->ev_comp[k]) cudaEventDestroy(g->ev_comp[k]);
        if (g->ev_d2h[k]) cudaEventDestroy(g->ev_d2h[k]);
    }
    g->scratch.release();
    g->hpk.release();
    g->cost_w.release();
    g->link_rot.release();
    rb_jit_unload(g->jit);
    if (g->d_model) cudaFree(g->d_model);
    if (g->d_status) cudaFree(g->d_status);
    if (g->h_status) cudaFreeHost(g->h_status);
    if (g->stream) cudaStreamDestroy(g->stream);
    if (g->s_h2d) cudaStreamDestroy(g->s_h2d);
    if (g->s_d2h) cudaStreamDestroy(g->s_d2h);
    delete g;
}

extern "C" int multibody_jit_precompile(const RbChainDesc* desc, const char* urdf_path, char* log, size_t log_len) {
    try {
        RbHostModel m; std::string err;
        int rc = desc ? rb_model_from_desc(desc, m, err) : rb_model_from_urdf(urdf_path, m, err);
        if (rc != RB_OK) return fail(rc, err);
        RbJitImage img; std::string l;
        rc = rb_jit_compile(m, img, l);
        if (log && log_len) { snprintf(log, log_len, "%s", l.c_str()); }
        if (rc != RB_OK) return fail(rc, "run-time specialisation failed: " + l);
        return RB_OK;
    } catch (const std::exception& e) { return fail(RB_ERR_ARG, std::string("exception: ") + e.what()); }
}

extern "C" const char* multibody_gpu_family_note(const RbGpu* g) { return g ? g->family_note.c_str() : ""; }

// ===================================================================== introspection
extern "C" int multibody_gpu_n_joints(const RbGpu* g) { return g ? g->model.n : fail(RB_ERR_NULL, "engine handle is NULL"); }
extern "C" int multibody_gpu_device(const RbGpu* g) { return g ? g->device : fail(RB_ERR_NULL, "engine handle is NULL"); }
extern "C" const char* multibody_gpu_kernel_variant(const RbGpu* g) { return g && g->ops ? g->ops->name : ""; }
extern "C" const char* multibody_last_error(void) { return g_err.c_str(); }
extern "C" uint64_t multibody_gpu_launch_count(const RbGpu* g) {
    if (!g) return 0;
    uint64_t total = g->launches.load();
    for (const RbGpu* pg : g->peers) total += pg->launches.load();
    return total;
}

static void copy_model(const RbHostModel& m, double* parent_rot, double* parent_trans, double* mass, double* h,
                       double* inertia_origin) {
    for (int i = 0; i < m.n; ++i) {
        const RbJointK& j = m.jt[i];
        if (parent_rot) memcpy(parent_rot + 9 * i, j.R, sizeof j.R);
        if (parent_trans) memcpy(parent_trans + 3 * i, j.t, sizeof j.t);
        if (mass) mass[i] = j.m;
        if (h) memcpy(h + 3 * i, j.h, sizeof j.h);
        if (inertia_origin) memcpy(inertia_origin + 6 * i, j.I, sizeof j.I);
    }
}

extern "C" int multibody_gpu_get_model(const RbGpu* g, double* parent_rot, double* parent_trans, double* mass,
                                       double* h, double* inertia_origin) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    copy_model(g->model, parent_rot, parent_trans, mass, h, inertia_origin);
    return RB_OK;
}

extern "C" int multibody_n_joints(const Multibody* mb) { return mb ? mb->model.n : fail(RB_ERR_NULL, "Multibody handle is NULL"); }

extern "C" int multibody_get_model(const Multibody* mb, double* parent_rot, double* parent_trans, double* mass,
                                   double* h, double* inertia_origin) {
    if (!mb) return fail(RB_ERR_NULL, "Multibody handle is NULL");
    copy_model(mb->model, parent_rot, parent_trans, mass, h, inertia_origin);
    return RB_OK;
}

extern "C" int multibody_get_chain(const Multibody* mb, int32_t* parent, double* axis, double* parent_rot, double* parent_trans,
                                   double* mass, double* com, double* inertia_com) {
    if (!mb) return fail(RB_ERR_NULL, "Multibody handle is NULL");
    for (int i = 0; i < mb->model.n; ++i) {
        const RbRawJoint& j = mb->model.raw[(size_t)i];
        if (parent) parent[i] = j.parent;
        if (axis) memcpy(axis + 3 * i, j.axis, sizeof j.axis);
        if (parent_rot) memcpy(parent_rot + 9 * i, j.R, sizeof j.R);
        if (parent_trans) memcpy(parent_trans + 3 * i, j.t, sizeof j.t);
        if (mass) mass[i] = j.mass;
        if (com) memcpy(com + 3 * i, j.com, sizeof j.com);
        if (inertia_com) memcpy(inertia_com + 9 * i, j.Ic, sizeof j.Ic);
    }
    return RB_OK;
}

extern "C" int multibody_gpu_get_limits(const RbGpu* g, RbJointLimits* out) {
    if (!g || !out) return fail(RB_ERR_NULL, "NULL argument");
    *out = g->model.lim;
    return RB_OK;
}

// ===================================================================== the batched hot path
extern "C" int multibody_rnea_batch(RbGpu* g, const double* q, const double* dq, const double* ddq, double* tau,
                                    size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    const int n = g->model.n;
    OpDesc op{3, {q, dq, ddq}, {n, n, n}, tau, n,
              [](RbGpu* g, const double* const* in, double* out, size_t B, size_t ld, cudaStream_t st, int* status, const void*) {
                  return launch(g, g->rnea, st, in[0], in[1], in[2], out, B, ld);
              },
              [](RbGpu* g, const double* const* in, double* out, size_t B, cudaStream_t st, int* status) {
                  return g->ops->rnea_aos(g->param.data(), in[0], in[1], in[2], out, B, st);
              },
              [](RbGpu* g) { return g->ops->rnea_aos != nullptr; }};
    return run_op(g, op, n_states, ld, layout, mem, stream, false);
}

extern "C" int multibody_forward_dynamics_batch(RbGpu* g, const double* q, const double* dq, const double* tau, double* qdd,
                                                size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    const int n = g->model.n;
    OpDesc op{3, {q, dq, tau}, {n, n, n}, qdd, n,
              [](RbGpu* g, const double* const* in, double* out, size_t B, size_t ld, cudaStream_t st, int* status, const void*) {
                  return launch(g, g->fd, st, in[0], in[1], in[2], out, B, ld, status);
              },
              [](RbGpu* g, const double* const* in, double* out, size_t B, cudaStream_t st, int* status) {
                  return g->ops->fd_aos(g->param.data(), in[0], in[1], in[2], out, B, status, st);
              },
              [](RbGpu* g) { return g->ops->fd_aos != nullptr; }};
    return run_op(g, op, n_states, ld, layout, mem, stream, true);
}

// ---- inverse and forward dynamics of the same states in one call: q and dq travel (and are staged) once ----
extern "C" int multibody_rnea_fd_batch(RbGpu* g, const double* q, const double* dq, const double* ddq, const double* tau_in,
                                       double* out, size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    const int n = g->model.n;
    OpDesc op{4, {q, dq, ddq, tau_in}, {n, n, n, n}, out, 2 * n,
              [](RbGpu* g, const double* const* in, double* out, size_t B, size_t ld, cudaStream_t st, int* status, const void*) {
                  const int n = g->model.n;
                  // one fused pass where the family has it (shared sin/cos, bias recursion and mass matrix)
                  if (g->ops->rnea_fd && !g->split_rnea_fd)
                      return g->ops->rnea_fd(g->param.data(), in[0], in[1], in[2], in[3], out, B, ld, status, st);
                  cudaError_t e = launch(g, g->rnea, st, in[0], in[1], in[2], out, B, ld);
                  if (e != cudaSuccess) return e;
                  g->launches += 1;
                  return launch(g, g->fd, st, in[0], in[1], in[3], out + (size_t)n * ld, B, ld, status);
              }};
    return run_op(g, op, n_states, ld, layout, mem, stream, true);
}

// ---- analytical derivatives (rb_deriv.cuh): the register-resident families only ----
extern "C" int multibody_rnea_derivatives_batch(RbGpu* g, const double* q, const double* dq, const double* ddq, double* out,
                                                size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    const int n = g->model.n;
    if (n > RB_RNEA_DERIV_MAX_N || !g->model.serial)
        return fail(RB_ERR_UNSUPPORTED, "inverse-dynamics derivative kernels serve serial chains of at most 32 joints");
    OpDesc op{3, {q, dq, ddq}, {n, n, n}, out, 2 * n * n,
              [](RbGpu* g, const double* const* in, double* out, size_t B, size_t ld, cudaStream_t st, int* status, const void*) {
                  return rb_launch_rnea_deriv(g->model.n, g->flat.data(), in[0], in[1], in[2], out, B, ld, st);
              }};
    return run_op(g, op, n_states, ld, layout, mem, stream, false);
}

extern "C" int multibody_fd_derivatives_batch(RbGpu* g, const double* q, const double* dq, const double* tau, double* out,
                                              size_t n_states, size_t ld, RbLayout layout, RbMem mem, void* stream) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    const int n = g->model.n;
    if (n > RB_DERIV_MAX_N || !g->model.serial)
        return fail(RB_ERR_UNSUPPORTED, "forward-dynamics derivative kernels serve serial chains of at most 12 joints");
    OpDesc op{3, {q, dq, tau}, {n, n, n}, out, 3 * n * n,
              [](RbGpu* g, const double* const* in, double* out, size_t B, size_t ld, cudaStream_t st, int* status, const void*) {
                  return rb_launch_fd_deriv(g->model.n, g->flat.data(), in[0], in[1], in[2], out, B, ld, status, st);
              }};
    return run_op(g, op, n_states, ld, layout, mem, stream, true);
}

// ---- optional fp32 mode: device-resident SoA batches only ----
namespace {
int f32_common(RbGpu* g, const void* a, const void* b, const void* c, const void* out, size_t n_states, size_t& ld) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    if (n_states == 0) return RB_OK;
    if (!a || !b || !c || !out) return fail(RB_ERR_NULL, "pointer is NULL");
    if (ld == 0) ld = n_states;
    if (ld < n_states) return fail(RB_ERR_ARG, "ld < n_states");
    return RB_OK;
}
}  // namespace

extern "C" int multibody_rnea_batch_f32(RbGpu* g, const float* q, const float* dq, const float* ddq, float* tau,
                                        size_t n_states, size_t ld, void* stream) {
    int rc = f32_common(g, q, dq, ddq, tau, n_states, ld);
    if (rc != RB_OK || n_states == 0) return rc;
    if (!g->peers.empty()) return fail(RB_ERR_UNSUPPORTED, kMultiDeviceOnly);
    if (!g->ops->rnea_f32) return fail(RB_ERR_UNSUPPORTED, std::string("kernel family '") + g->ops->name + "' has no fp32 kernels");
    DeviceGuard dg(g->device);
    cudaError_t e = g->ops->rnea_f32(g->param.data(), q, dq, ddq, tau, n_states, ld, (cudaStream_t)stream);
    g->launches += 1;
    if (e != cudaSuccess) return fail_cuda(e, "kernel launch");
    return RB_OK;
}

extern "C" int multibody_forward_dynamics_batch_f32(RbGpu* g, const float* q, const float* dq, const float* tau, float* qdd,
                                                    size_t n_states, size_t ld, void* stream) {
    int rc = f32_common(g, q, dq, tau, qdd, n_states, ld);
    if (rc != RB_OK || n_states == 0) return rc;
    if (!g->peers.empty()) return fail(RB_ERR_UNSUPPORTED, kMultiDeviceOnly);
    if (!g->ops->fd_f32) return fail(RB_ERR_UNSUPPORTED, std::string("kernel family '") + g->ops->name + "' has no fp32 kernels");
    DeviceGuard dg(g->device);
    cudaError_t e = g->ops->fd_f32(g->param.data(), q, dq, tau, qdd, n_states, ld, g->d_status, (cudaStream_t)stream);
    g->launches += 1;
    if (e != cudaSuccess) return fail_cuda(e, "kernel launch");
    return RB_OK;
}

extern "C" int multibody_crba_batch(RbGpu* g, const double* q, double* H, size_t n_states, size_t ld, RbLayout layout,
                                    RbMem mem, void* stream) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    const int n = g->model.n;
    OpDesc op{1, {q, nullptr, nullptr}, {n, 0, 0}, H, n * n,
              [](RbGpu* g, const double* const* in, double* out, size_t B, size_t ld, cudaStream_t st, int* status, const void*) {
                  return launch(g, g->crba, st, in[0], out, B, ld);
              }};
    return run_op(g, op, n_states, ld, layout, mem, stream, false);
}

extern "C" int multibody_fwd_kin_batch(RbGpu* g, const double* q, double* xyz, size_t n_states, size_t ld, RbLayout layout,
                                       RbMem mem, void* stream) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    const int n = g->model.n;
    OpDesc op{1, {q, nullptr, nullptr}, {n, 0, 0}, xyz, 3,
              [](RbGpu* g, const double* const* in, double* out, size_t B, size_t ld, cudaStream_t st, int* status, const void*) {
                  return launch(g, g->fwd_kin, st, in[0], out, B, ld);
              }};
    return run_op(g, op, n_states, ld, layout, mem, stream, false);
}

extern "C" int multibody_jac_batch(RbGpu* g, const double* q, double* J, size_t n_states, size_t ld, RbLayout layout,
                                   RbMem mem, void* stream) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    const int n = g->model.n;
    OpDesc op{1, {q, nullptr, nullptr}, {n, 0, 0}, J, 6 * n,
              [](RbGpu* g, const double* const* in, double* out, size_t B, size_t ld, cudaStream_t st, int* status, const void*) {
                  return launch(g, g->jac, st, in[0], out, B, ld);
              }};
    return run_op(g, op, n_states, ld, layout, mem, stream, false);
}

// ---- tip pose and inverse kinematics of the tip frame (rb_kernels_ik.cu): one kernel for every family ----
extern "C" int multibody_tip_pose_batch(RbGpu* g, const double* q, const double* offset, double* pose, size_t n_states, size_t ld,
                                        RbLayout layout, RbMem mem, void* stream) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    const int n = g->model.n;
    double off[3] = {0.0, 0.0, 0.0};
    if (offset)
        for (int k = 0; k < 3; ++k) {
            if (!std::isfinite(offset[k])) return fail(RB_ERR_ARG, "offset must be finite");
            off[k] = offset[k];
        }
    OpDesc op{1, {q, nullptr, nullptr}, {n, 0, 0}, pose, 12,
              [](RbGpu* g, const double* const* in, double* out, size_t B, size_t ld, cudaStream_t st, int* status, const void* arg) {
                  return rb_launch_tip_pose(g->d_model, g->model.n, (const double*)arg, in[0], out, B, ld, st);
              }};
    op.arg = off;
    return run_op(g, op, n_states, ld, layout, mem, stream, false);
}

namespace {
static_assert(RB_CL_MAX_SPHERES == RB_MAX_SPHERES && RB_CL_MAX_OBSTACLES == RB_MAX_OBSTACLES, "collision block caps");

// Checks an RbCollisionCost and packs it into the collision block (RB_CL_* entries): sphere centres rotated into the
// engines' re-based link frames (c -> Q_l^T c) and stably grouped by link, sphere obstacles before half-spaces, normals
// normalised.  `on` = the terms can add something (some sphere, some obstacle, some weight not zero).
int pack_collision(const RbHostModel& m, const RbCollisionCost* c, double* blk, bool* on) {
    *on = false;
    if (!c) return RB_OK;
    if (c->n_spheres < 0 || c->n_spheres > RB_MAX_SPHERES) return fail(RB_ERR_ARG, "n_spheres must lie in [0, RB_MAX_SPHERES]");
    if (c->n_obstacles < 0 || c->n_obstacles > RB_MAX_OBSTACLES) return fail(RB_ERR_ARG, "n_obstacles must lie in [0, RB_MAX_OBSTACLES]");
    const int S = c->n_spheres, O = c->n_obstacles, n = m.n;
    if (S > 0 && (!c->link || !c->center || !c->radius)) return fail(RB_ERR_NULL, "collision sphere arrays are NULL");
    if (O > 0 && (!c->kind || !c->obstacle)) return fail(RB_ERR_NULL, "collision obstacle arrays are NULL");
    for (double v : {c->margin, c->w, c->w_final})
        if (!std::isfinite(v) || v < 0.0) return fail(RB_ERR_ARG, "collision margin and weights must be finite and non-negative");
    memset(blk, 0, sizeof(double) * RB_CL_COUNT);
    blk[RB_CL_MARGIN] = c->margin; blk[RB_CL_W] = c->w; blk[RB_CL_WF] = c->w_final;
    int count[RB_MAX_N + 1] = {};
    for (int k = 0; k < S; ++k) {
        if (c->link[k] < 0 || c->link[k] >= n) return fail(RB_ERR_ARG, "collision sphere link outside [0, n)");
        for (int a = 0; a < 3; ++a) if (!std::isfinite(c->center[3 * k + a])) return fail(RB_ERR_ARG, "collision sphere centres must be finite");
        if (!std::isfinite(c->radius[k]) || c->radius[k] < 0.0) return fail(RB_ERR_ARG, "collision sphere radii must be finite and non-negative");
        count[c->link[k] + 1] += 1;
    }
    for (int l = 0; l < n; ++l) count[l + 1] += count[l];
    for (int l = 0; l <= n; ++l) blk[RB_CL_TAB + l] = count[l];
    for (int k = 0; k < S; ++k) {                             // stable: spheres of one link keep their order
        const int l = c->link[k];
        double* sp = blk + RB_CL_SPH + 4 * count[l]++;
        const double* Qt = &m.link_rot[9 * (size_t)l];
        for (int a = 0; a < 3; ++a)
            sp[a] = Qt[3 * a] * c->center[3 * k] + Qt[3 * a + 1] * c->center[3 * k + 1] + Qt[3 * a + 2] * c->center[3 * k + 2];
        sp[3] = c->radius[k];
    }
    int nos = 0, noh = 0;
    for (int o = 0; o < O; ++o) {
        const double* ob = c->obstacle + 4 * o;
        for (int a = 0; a < 4; ++a) if (!std::isfinite(ob[a])) return fail(RB_ERR_ARG, "collision obstacles must be finite");
        if (c->kind[o] == RB_OBSTACLE_SPHERE) {
            if (ob[3] < 0.0) return fail(RB_ERR_ARG, "collision obstacle radii must be non-negative");
            nos += 1;
        } else if (c->kind[o] == RB_OBSTACLE_HALFSPACE) {
            if (!(std::sqrt(ob[0] * ob[0] + ob[1] * ob[1] + ob[2] * ob[2]) > 0.0)) return fail(RB_ERR_ARG, "half-space normals must not be zero");
            noh += 1;
        } else {
            return fail(RB_ERR_ARG, "unknown collision obstacle kind");
        }
    }
    int at_s = 0, at_h = nos;
    for (int o = 0; o < O; ++o) {
        const double* ob = c->obstacle + 4 * o;
        double* d = blk + RB_CL_OBS + 4 * (c->kind[o] == RB_OBSTACLE_SPHERE ? at_s++ : at_h++);
        if (c->kind[o] == RB_OBSTACLE_SPHERE) {
            for (int a = 0; a < 4; ++a) d[a] = ob[a];
        } else {
            const double len = std::sqrt(ob[0] * ob[0] + ob[1] * ob[1] + ob[2] * ob[2]);
            for (int a = 0; a < 3; ++a) d[a] = ob[a] / len;
            d[3] = ob[3];
        }
    }
    blk[RB_CL_NOS] = nos; blk[RB_CL_NOH] = noh;
    *on = S > 0 && O > 0 && (c->w > 0.0 || c->w_final > 0.0);
    return RB_OK;
}
}  // namespace

extern "C" int multibody_link_poses_batch(RbGpu* g, const double* q, double* pose, size_t n_states, size_t ld, RbLayout layout,
                                          RbMem mem, void* stream) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    const int n = g->model.n;
    OpDesc op{1, {q, nullptr, nullptr}, {n, 0, 0}, pose, 12 * n,
              [](RbGpu* g, const double* const* in, double* out, size_t B, size_t ld, cudaStream_t st, int* status, const void*) {
                  return rb_launch_link_poses(g->d_model, (const double*)g->link_rot.p, g->model.n, in[0], out, B, ld, st);
              }};
    return run_op(g, op, n_states, ld, layout, mem, stream, false);
}

extern "C" int multibody_sphere_distance_batch(RbGpu* g, const double* q, const RbCollisionCost* col, double* out, size_t n_states,
                                               size_t ld, RbLayout layout, RbMem mem, void* stream) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    if (!col) return fail(RB_ERR_NULL, "collision terms are NULL");
    const int n = g->model.n;
    std::vector<double> blk(RB_CL_COUNT);
    bool on;
    const int rc = pack_collision(g->model, col, blk.data(), &on);
    if (rc != RB_OK) return rc;
    if (col->n_spheres == 0 || col->n_obstacles == 0) return fail(RB_ERR_ARG, "sphere distances need at least one sphere and one obstacle");
    // the block goes to the engine's cost-weight buffer, shared by every cost call: ordered like scratch
    OpDesc op{1, {q, nullptr, nullptr}, {n, 0, 0}, out, 2,
              [](RbGpu* g, const double* const* in, double* out, size_t B, size_t ld, cudaStream_t st, int* status, const void* arg) {
                  ScratchOrder so(g, true, st);
                  double* d = (double*)g->cost_w.p + RB_CW_COL;
                  cudaError_t e = cudaMemcpyAsync(d, arg, sizeof(double) * RB_CL_COUNT, cudaMemcpyHostToDevice, st);
                  if (e != cudaSuccess) return e;
                  return rb_launch_sphere_distance(g->d_model, g->model.n, d, in[0], out, B, ld, st);
              }};
    op.arg = blk.data();
    return run_op(g, op, n_states, ld, layout, mem, stream, false);
}

namespace {
// Checks an RbIkOptions and packs it into the kernel's parameter block.
int pack_ik(const RbHostModel& m, const RbIkOptions* o, const double* R_target, RbIkParam& P) {
    if (!o) return fail(RB_ERR_NULL, "IK options are NULL");
    memset(&P, 0, sizeof(P));
    const int n = m.n;
    for (int k = 0; k < 3; ++k) {
        P.offset[k] = o->offset ? o->offset[k] : 0.0;
        P.w_p[k] = o->w_p ? o->w_p[k] : 1.0;
        if (!std::isfinite(P.offset[k])) return fail(RB_ERR_ARG, "IK offset must be finite");
        if (!std::isfinite(P.w_p[k]) || P.w_p[k] < 0.0) return fail(RB_ERR_ARG, "IK weights must be finite and non-negative");
    }
    if (!std::isfinite(o->w_R) || o->w_R < 0.0) return fail(RB_ERR_ARG, "IK weights must be finite and non-negative");
    if (o->max_iters < 0) return fail(RB_ERR_ARG, "IK max_iters < 0");
    if (!(o->tol_p >= 0.0) || !(o->tol_R >= 0.0)) return fail(RB_ERR_ARG, "IK tolerances must be non-negative");
    if (!(o->damping >= 1e-12 && o->damping <= 1e12)) return fail(RB_ERR_ARG, "IK damping must lie in [1e-12, 1e12]");
    if (o->w_R > 0.0 && !R_target) return fail(RB_ERR_NULL, "R_target is NULL but w_R > 0");
    for (int i = 0; i < n; ++i) {
        P.lower[i] = o->lower ? o->lower[i] : -INFINITY;
        P.upper[i] = o->upper ? o->upper[i] : INFINITY;
        if (std::isnan(P.lower[i]) || std::isnan(P.upper[i]) || P.lower[i] > P.upper[i])
            return fail(RB_ERR_ARG, "IK bounds must not be NaN and lower <= upper");
    }
    P.w_R = o->w_R;
    for (int k = 0; k < 3; ++k) { P.sw[k] = std::sqrt(P.w_p[k]); P.sw[3 + k] = std::sqrt(2.0 * P.w_R); }
    P.tol_p = o->tol_p; P.tol_R = o->tol_R; P.damping = o->damping; P.max_iters = o->max_iters;
    P.tree = m.serial ? 0 : 1;
    return RB_OK;
}
}  // namespace

extern "C" int multibody_ik_batch(RbGpu* g, const double* q_init, const double* p_target, const double* R_target,
                                  const RbIkOptions* opt, double* out, size_t n_problems, size_t ld, RbLayout layout,
                                  RbMem mem, void* stream) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    const int n = g->model.n;
    RbIkParam P;
    const int rc = pack_ik(g->model, opt, R_target, P);
    if (rc != RB_OK) return rc;
    // w_R == 0: position only, R_target is neither read nor staged
    OpDesc op{P.w_R > 0.0 ? 3 : 2, {q_init, p_target, R_target}, {n, 3, 9}, out, n + 3,
              [](RbGpu* g, const double* const* in, double* out, size_t B, size_t ld, cudaStream_t st, int* status, const void* arg) {
                  const RbIkParam& P = *(const RbIkParam*)arg;
                  return rb_launch_ik(g->d_model, g->model.n, P, in[0], in[1], P.w_R > 0.0 ? in[2] : nullptr, out, B, ld, g->sm_count, st);
              }};
    op.arg = &P;
    return run_op(g, op, n_problems, ld, layout, mem, stream, false);
}

namespace {
// Host and/or AoS arguments of the rollout entries, moved through the engine's staging buffers as SoA with ld = n_traj.
// An input or output is `arrays` consecutive state arrays (n doubles per trajectory each: q0 is one, tau `horizon`),
// or, `plain`, one vector of n_traj doubles (the cost).  A NULL pointer is neither copied nor handed on.
struct StagedIn { const double* p; size_t arrays; };
struct StagedOut { double* p; size_t arrays; bool plain; };
using StagedRun = std::function<int(const double* const* d_in, double* const* d_out, int* d_stat)>;

// Brings `ins` in, calls run() on the staged copies (SoA, ld = n_traj; NULL where the caller passed NULL), brings `outs`
// back, and drains the stream.  `aos_stride`: elements between consecutive steps of the caller's AoS arrays (0 = n_traj * n,
// a dense [H][n_traj][n] array; a multi-device engine passes the stride of the whole batch when it hands out slices).
// Takes g->mu; a host call owns status word 1 and reports it.
int run_staged(RbGpu* g, const std::vector<StagedIn>& ins, const std::vector<StagedOut>& outs, size_t n_traj, size_t ld,
               RbLayout layout, RbMem mem, size_t aos_stride, cudaStream_t st, const StagedRun& run) {
    std::lock_guard<std::mutex> lk(g->mu);
    int* const d_stat = g->d_status + (mem == RB_MEM_HOST ? 1 : 0);
    if (mem == RB_MEM_HOST) RB_CUDA(cudaMemsetAsync(d_stat, 0, sizeof(int), st));
    auto staged = [&]() -> int {
    const int n = g->model.n;
    const size_t B = n_traj, one = (size_t)n * B;
    const bool aos = layout == RB_LAYOUT_AOS, host = mem == RB_MEM_HOST;
    const size_t src_step = aos ? (aos_stride ? aos_stride : one) : (size_t)n * ld;    // caller's distance between steps
    size_t in_arrays = 0, out_arrays = 0, out_plain = 0;
    for (const StagedIn& a : ins) in_arrays += a.arrays;
    for (const StagedOut& a : outs) (a.plain ? out_plain : out_arrays) += a.arrays;
    // in[0]: the inputs in order      out[0]: the outputs in order      tmp[0]: AoS landing zone
    int rc = g->in[0].ensure(in_arrays * one * sizeof(double)); if (rc) return rc;
    rc = g->out[0].ensure((out_arrays * one + out_plain * B) * sizeof(double)); if (rc) return rc;
    if (aos) { rc = g->tmp[0].ensure(std::max(in_arrays, out_arrays) * one * sizeof(double)); if (rc) return rc; }
    double* d_tmp = g->tmp[0].p;
    auto bring_in = [&](const double* src, double* dst, size_t arrays) -> int {
        // `arrays` consecutive state arrays
        for (size_t a = 0; a < arrays; ++a) {
            const double* s_a = src + a * src_step;
            double* d_a = dst + a * one;
            if (!aos) {
                RB_CUDA(cudaMemcpy2DAsync(d_a, B * sizeof(double), s_a, ld * sizeof(double), B * sizeof(double), (size_t)n,
                                          host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, st));
            } else {
                const double* a_src = s_a;
                if (host) {
                    double* land = d_tmp + a * one;
                    RB_CUDA(cudaMemcpyAsync(land, s_a, one * sizeof(double), cudaMemcpyHostToDevice, st));
                    a_src = land;
                }
                cudaError_t e = rb_launch_aos_to_soa(a_src, d_a, n, B, B, st);
                g->launches += 1;
                if (e != cudaSuccess) return fail_cuda(e, "aos_to_soa launch");
            }
        }
        return RB_OK;
    };
    std::vector<const double*> d_in(ins.size());
    double* d = g->in[0].p;
    for (size_t k = 0; k < ins.size(); ++k) {
        d_in[k] = ins[k].p ? d : nullptr;
        if (ins[k].p) { rc = bring_in(ins[k].p, d, ins[k].arrays); if (rc) return rc; }
        d += ins[k].arrays * one;
    }
    std::vector<double*> d_out(outs.size());
    d = g->out[0].p;
    for (size_t k = 0; k < outs.size(); ++k) {
        d_out[k] = outs[k].p ? d : nullptr;
        d += outs[k].arrays * (outs[k].plain ? B : one);
    }
    rc = run(d_in.data(), d_out.data(), d_stat); if (rc) return rc;
    auto bring_out = [&](const double* src, double* dst, size_t arrays) -> int {
        if (!dst) return RB_OK;
        for (size_t a = 0; a < arrays; ++a) {
            const double* s_a = src + a * one;
            double* d_a = dst + a * src_step;
            if (!aos) {
                RB_CUDA(cudaMemcpy2DAsync(d_a, ld * sizeof(double), s_a, B * sizeof(double), B * sizeof(double), (size_t)n,
                                          host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, st));
            } else {
                double* a_dst = host ? d_tmp + a * one : d_a;
                cudaError_t e2 = rb_launch_soa_to_aos(s_a, a_dst, n, B, B, st);
                g->launches += 1;
                if (e2 != cudaSuccess) return fail_cuda(e2, "soa_to_aos launch");
                if (host) RB_CUDA(cudaMemcpyAsync(d_a, a_dst, one * sizeof(double), cudaMemcpyDeviceToHost, st));
            }
        }
        return RB_OK;
    };
    d = g->out[0].p;
    bool first = true;
    for (size_t k = 0; k < outs.size(); ++k) {
        const StagedOut& o = outs[k];
        if (o.plain) {
            if (o.p) RB_CUDA(cudaMemcpyAsync(o.p, d, B * sizeof(double), host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, st));
            d += o.arrays * B;
            continue;
        }
        // the AoS landing zone is reused per output array group, so drain between groups
        if (!first && aos && host) RB_CUDA(cudaStreamSynchronize(st));
        first = false;
        rc = bring_out(d, o.p, o.arrays); if (rc) return rc;
        d += o.arrays * one;
    }
    // everything above went through engine-owned staging: drain before another call may reuse it
    RB_CUDA(cudaStreamSynchronize(st));
    return RB_OK;
    };
    const int rc_staged = staged();
    if (rc_staged != RB_OK) {       // copies already queued must not outlive the call
        const std::string keep = g_err;
        cudaStreamSynchronize(st);
        if (mem == RB_MEM_HOST) drain_host_pipeline(g);
        g_err = keep;
        return rc_staged;
    }
    return mem == RB_MEM_HOST ? fetch_status(g, 1) : RB_OK;     // still under g->mu
}

// Checks the weights of an RbQuadCost and packs them into the layout of the engine's cost-weight block (RB_CW_* rows).
int pack_cost_weights(int n, const RbQuadCost* w, double* cw) {
    memset(cw, 0, sizeof(double) * RB_CW_ROWS * RB_MAX_N);
    const double* rows[RB_CW_ROWS] = {w->q_ref, w->w_q, w->w_dq, w->w_tau, w->w_q_final, w->w_dq_final};
    for (int r = 0; r < RB_CW_ROWS; ++r)
        if (rows[r]) for (int i = 0; i < n; ++i) {
            if (!std::isfinite(rows[r][i]) || (r != RB_CW_QREF && rows[r][i] < 0.0)) return fail(RB_ERR_ARG, "cost weights must be finite and non-negative");
            cw[r * RB_MAX_N + i] = rows[r][i];
        }
    return RB_OK;
}

// The whole cost-weight block of a cost call and the terms it carries: the RB_CW_* rows, the RB_CW_TIP row with tip
// terms, and the collision block (at RB_CW_COL) with collision terms.  bytes() = the part a call uploads.
struct CostBlock {
    double w[RB_CW_DOUBLES_COL];
    RbCostTerms terms = RB_COST_QUAD;
    size_t bytes() const {
        const size_t doubles = terms == RB_COST_TIP_COL ? (size_t)RB_CW_DOUBLES_COL
                             : terms == RB_COST_TIP     ? (size_t)RB_CW_ROWS_TIP * RB_MAX_N
                                                        : (size_t)RB_CW_ROWS * RB_MAX_N;
        return sizeof(double) * doubles;
    }
};

// Checks the terms of an RbTipCost and packs them into row RB_CW_TIP (RB_TW_* entries).  `on` = some weight is not
// zero; a tip cost whose weights are all zero adds nothing, and the call runs as one without tip terms.
int pack_tip_weights(const RbTipCost* t, double* row, bool* on) {
    memset(row, 0, sizeof(double) * RB_MAX_N);
    *on = false;
    if (!t) return RB_OK;
    const struct { const double* v; int at, len; bool weight; } parts[] = {
        {t->offset, RB_TW_OFFSET, 3, false}, {t->p_ref, RB_TW_PREF, 3, false}, {t->w_p, RB_TW_WP, 3, true},
        {t->w_p_final, RB_TW_WPF, 3, true}, {t->R_ref, RB_TW_RREF, 9, false}, {&t->w_R, RB_TW_WR, 1, true},
        {&t->w_R_final, RB_TW_WRF, 1, true}};
    for (const auto& pt : parts) {
        if (!pt.v) continue;
        for (int k = 0; k < pt.len; ++k) {
            const double v = pt.v[k];
            if (!std::isfinite(v) || (pt.weight && v < 0.0)) return fail(RB_ERR_ARG, "tip cost terms must be finite and its weights non-negative");
            row[pt.at + k] = v;
            if (pt.weight && v != 0.0) *on = true;
        }
    }
    if (!t->R_ref) row[RB_TW_RREF] = row[RB_TW_RREF + 4] = row[RB_TW_RREF + 8] = 1.0;
    return RB_OK;
}

// Checks and packs every part of a cost call's weights, and picks its terms from those that are on.  Collision terms run
// in the kernels that carry the tip terms too: with collision terms on, the tip row is uploaded whatever its weights.
int pack_cost_block(const RbHostModel& m, const RbQuadCost* w, const RbTipCost* tip, const RbCollisionCost* col, CostBlock& cb) {
    bool tip_on = false, col_on = false;
    int rc = pack_cost_weights(m.n, w, cb.w);
    if (rc == RB_OK) rc = pack_tip_weights(tip, cb.w + RB_CW_TIP * RB_MAX_N, &tip_on);
    if (rc == RB_OK) rc = pack_collision(m, col, cb.w + RB_CW_COL, &col_on);
    cb.terms = col_on ? RB_COST_TIP_COL : tip_on ? RB_COST_TIP : RB_COST_QUAD;
    return rc;
}

int rollout_impl(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                 double* q_traj, double* dq_traj, double* q_final, double* dq_final, const RbQuadCost* w, const RbTipCost* tip,
                 const RbCollisionCost* col, double* cost, size_t n_traj, size_t ld, RbLayout layout, RbMem mem, void* stream,
                 size_t aos_stride = 0) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    if (!g->peers.empty()) {
        if (layout != RB_LAYOUT_SOA && layout != RB_LAYOUT_AOS) return fail(RB_ERR_ARG, "bad layout");
        if (mem != RB_MEM_HOST) return fail(mem == RB_MEM_DEVICE ? RB_ERR_UNSUPPORTED : RB_ERR_ARG, mem == RB_MEM_DEVICE ? kMultiDeviceOnly : "bad mem");
        if (n_traj == 0) return RB_OK;
        const bool aos = layout == RB_LAYOUT_AOS;
        const size_t n = (size_t)g->model.n;
        if (!aos) { if (ld == 0) ld = n_traj; if (ld < n_traj) return fail(RB_ERR_ARG, "ld < n_traj"); }
        return run_on_peers(g, [&](size_t i) -> int {
            size_t lo, hi; slice_bounds(n_traj, g->peers.size(), i, &lo, &hi);
            if (hi == lo) return RB_OK;
            const size_t o = lo * (aos ? n : 1);              // offset of trajectory lo inside one state array
            auto at = [&](const double* p) { return p ? p + o : nullptr; };
            auto atw = [&](double* p) { return p ? p + o : nullptr; };
            return rollout_impl(g->peers[i], at(q0), at(dq0), at(tau), dt, horizon, atw(q_traj), atw(dq_traj), atw(q_final), atw(dq_final),
                                w, tip, col, cost ? cost + lo : nullptr, hi - lo, ld, layout, mem, nullptr, aos ? n_traj * n : 0);
        });
    }
    if (layout != RB_LAYOUT_SOA && layout != RB_LAYOUT_AOS) return fail(RB_ERR_ARG, "bad layout");
    if (mem != RB_MEM_HOST && mem != RB_MEM_DEVICE) return fail(RB_ERR_ARG, "bad mem");
    if (horizon < 0) return fail(RB_ERR_ARG, "horizon < 0");
    if (!std::isfinite(dt)) return fail(RB_ERR_ARG, "dt must be finite");
    if (n_traj == 0) return RB_OK;
    // horizon == 0 is a rollout of no steps: q_final = q0, dq_final = dq0, cost = the terminal cost; tau is not read
    if (horizon == 0 && !q_final && !dq_final && !cost) return RB_OK;
    if (!q0 || !dq0 || (!tau && horizon > 0)) return fail(RB_ERR_NULL, "input pointer is NULL");
    if (layout == RB_LAYOUT_SOA) { if (ld == 0) ld = n_traj; if (ld < n_traj) return fail(RB_ERR_ARG, "ld < n_traj"); }
    if (cost && !w) return fail(RB_ERR_NULL, "cost weights are NULL");
    DeviceGuard dg(g->device);
    if (!dg.ok) return fail(RB_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t st = mem == RB_MEM_DEVICE ? (cudaStream_t)stream : g->stream;
    CostBlock cb;
    if (cost) { const int rc = pack_cost_block(g->model, w, tip, col, cb); if (rc != RB_OK) return rc; }
    // One rollout over device SoA arrays: in = (q0, dq0, tau), out = (q_traj, dq_traj, q_final, dq_final, cost).  The cost
    // weights go to the engine's device block, shared by all cost rollouts and hence ordered like scratch.
    auto run = [&](const double* const* in, double* const* out, size_t ldr, int* d_stat) -> int {
        const auto& ro = g->rollout;
        cudaError_t e;
        {
            ScratchOrder so(g, cost != nullptr || ro.shared, st);
            if (cost) RB_CUDA(cudaMemcpyAsync(g->cost_w.p, cb.w, cb.bytes(), cudaMemcpyHostToDevice, st));
            e = ro.fn(ro.param, in[0], in[1], in[2], dt, horizon, out[0], out[1], out[2], out[3], n_traj, ldr, d_stat,
                      cost ? g->cost_w.p : nullptr, out[4], cb.terms, st);
        }
        g->launches += 1;
        if (e != cudaSuccess) return fail_cuda(e, "rollout launch");
        return RB_OK;
    };
    if (mem == RB_MEM_DEVICE && layout == RB_LAYOUT_SOA) {
        const double* const in[] = {q0, dq0, tau};
        double* const out[] = {q_traj, dq_traj, q_final, dq_final, cost};
        return run(in, out, ld, g->d_status);
    }
    // Host pointers and/or AoS: stage everything on the device as SoA with ld = n_traj, run once, bring results back.
    const size_t H = (size_t)horizon;
    return run_staged(g, {{q0, 1}, {dq0, 1}, {tau, H}}, {{q_traj, H, false}, {dq_traj, H, false}, {q_final, 1, false}, {dq_final, 1, false}, {cost, 1, true}},
                      n_traj, ld, layout, mem, aos_stride, st,
                      [&](const double* const* in, double* const* out, int* d_stat) { return run(in, out, n_traj, d_stat); });
}
// Arguments of multibody_rollout_vjp (q_traj .. g_dqf) and multibody_rollout_cost_grad (w, cost).
struct GradArgs {
    const double *q0, *dq0, *tau; double dt; int horizon;
    const double *q_traj, *dq_traj, *g_q, *g_dq, *g_qf, *g_dqf;
    const RbQuadCost* w; double* cost;
    double *grad_tau, *grad_q0, *grad_dq0;
    const RbTipCost* tip = nullptr;       // multibody_rollout_tip_cost_grad
    const RbCollisionCost* col = nullptr; // multibody_rollout_collision_cost_grad
};

// The trajectory workspace of one chunk of a cost-gradient call, 2 H n doubles per trajectory, stays within this.
constexpr size_t kGradWorkspace = (size_t)1 << 30;

// Both gradient entries on device SoA arrays with leading dimension ld, asynchronous on st.  The cost gradient runs the
// engine's rollout launcher (so that its cost is multibody_rollout_cost's, bit for bit) into a stream-ordered workspace,
// then the adjoint over the stored trajectory, chunk by chunk; the weight upload and every launch sit in one ScratchOrder
// region because the weight block is shared by all cost rollouts on the engine.
int grad_device(RbGpu* g, const GradArgs& a, const CostBlock& cb, size_t B, size_t ld, cudaStream_t st, int* d_stat) {
    const int n = g->model.n;
    RbAdjointArgs ad{a.q0, a.dq0, a.tau, a.q_traj, a.dq_traj, ld, a.g_q, a.g_dq, a.g_qf, a.g_dqf, nullptr,
                     a.grad_tau, a.grad_q0, a.grad_dq0, a.dt, a.horizon};
    if (!a.cost) {
        cudaError_t e = rb_launch_rollout_adjoint(n, g->flat.data(), ad, B, ld, d_stat, st);
        g->launches += 1;
        return e == cudaSuccess ? RB_OK : fail_cuda(e, "rollout adjoint launch");
    }
    ScratchOrder so(g, true, st);
    RB_CUDA(cudaMemcpyAsync(g->cost_w.p, cb.w, cb.bytes(), cudaMemcpyHostToDevice, st));
    ad.cost_w = g->cost_w.p;
    ad.terms = cb.terms;
    const auto& ro = g->rollout;
    const size_t H = (size_t)a.horizon, nn = (size_t)n;
    // A rollout writes its trajectory with the leading dimension of its inputs: a chunk whose inputs are not already a
    // dense [n][chunk] block (a cut batch, a padded ld) gets a dense copy of them next to its trajectory.
    const bool whole = H == 0 || (ld == B && 2 * H * nn * B * sizeof(double) <= kGradWorkspace);
    const size_t per_traj = (whole ? 2 * H : 3 * H + 2) * nn * sizeof(double);
    size_t chunk = whole ? B : kGradWorkspace / per_traj;
    if (!whole) chunk = std::max<size_t>(1, std::min(B, chunk >= 32 ? chunk / 32 * 32 : chunk));
    double* ws = nullptr;
    if (H > 0) RB_CUDA(cudaMallocAsync((void**)&ws, per_traj * chunk, st));
    int rc = RB_OK;
    for (size_t lo = 0; lo < B && rc == RB_OK; lo += chunk) {
        const size_t cnt = std::min(chunk, B - lo);
        const size_t lw = whole ? ld : cnt;                   // leading dimension of the rollout (and of the trajectory)
        double* qt = ws; double* dqt = ws ? ws + H * nn * cnt : nullptr;
        const double *rq0 = a.q0 + lo, *rdq0 = a.dq0 + lo, *rtau = a.tau ? a.tau + lo : nullptr;
        cudaError_t e = cudaSuccess;
        if (!whole) {
            double* in = ws + 2 * H * nn * cnt;
            e = cudaMemcpy2DAsync(in, cnt * sizeof(double), rq0, ld * sizeof(double), cnt * sizeof(double), nn, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess)
                e = cudaMemcpy2DAsync(in + nn * cnt, cnt * sizeof(double), rdq0, ld * sizeof(double), cnt * sizeof(double), nn, cudaMemcpyDeviceToDevice, st);
            if (e == cudaSuccess)
                e = cudaMemcpy2DAsync(in + 2 * nn * cnt, cnt * sizeof(double), rtau, ld * sizeof(double), cnt * sizeof(double), H * nn, cudaMemcpyDeviceToDevice, st);
            if (e != cudaSuccess) { rc = fail_cuda(e, "cudaMemcpy2DAsync(gradient workspace)"); break; }
            rq0 = in; rdq0 = in + nn * cnt; rtau = in + 2 * nn * cnt;
        }
        e = ro.fn(ro.param, rq0, rdq0, rtau, a.dt, a.horizon, qt, dqt, nullptr, nullptr, cnt, lw, d_stat, g->cost_w.p, a.cost + lo, cb.terms, st);
        g->launches += 1;
        if (e != cudaSuccess) { rc = fail_cuda(e, "rollout launch"); break; }
        RbAdjointArgs c = ad;
        c.q0 = a.q0 + lo; c.dq0 = a.dq0 + lo; c.tau = a.tau ? a.tau + lo : nullptr;
        c.q_traj = qt; c.dq_traj = dqt; c.ld_traj = lw;
        c.grad_tau = a.grad_tau ? a.grad_tau + lo : nullptr;
        c.grad_q0 = a.grad_q0 ? a.grad_q0 + lo : nullptr;
        c.grad_dq0 = a.grad_dq0 ? a.grad_dq0 + lo : nullptr;
        e = rb_launch_rollout_adjoint(n, g->flat.data(), c, cnt, ld, d_stat, st);
        g->launches += 1;
        if (e != cudaSuccess) rc = fail_cuda(e, "rollout adjoint launch");
    }
    if (ws) { cudaError_t e = cudaFreeAsync(ws, st); if (e != cudaSuccess && rc == RB_OK) rc = fail_cuda(e, "cudaFreeAsync(gradient workspace)"); }
    return rc;
}

int grad_impl(RbGpu* g, const GradArgs& a, size_t n_traj, size_t ld, RbLayout layout, RbMem mem, void* stream, size_t aos_stride = 0) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    if (g->model.n > RB_DERIV_MAX_N || !g->model.serial)
        return fail(RB_ERR_UNSUPPORTED, "rollout gradients use the forward-dynamics derivative kernels, which serve serial chains of at most 12 joints");
    if (layout != RB_LAYOUT_SOA && layout != RB_LAYOUT_AOS) return fail(RB_ERR_ARG, "bad layout");
    if (!g->peers.empty()) {
        if (mem != RB_MEM_HOST) return fail(mem == RB_MEM_DEVICE ? RB_ERR_UNSUPPORTED : RB_ERR_ARG, mem == RB_MEM_DEVICE ? kMultiDeviceOnly : "bad mem");
        if (n_traj == 0) return RB_OK;
        const bool aos = layout == RB_LAYOUT_AOS;
        const size_t n = (size_t)g->model.n;
        if (!aos) { if (ld == 0) ld = n_traj; if (ld < n_traj) return fail(RB_ERR_ARG, "ld < n_traj"); }
        return run_on_peers(g, [&](size_t i) -> int {
            size_t lo, hi; slice_bounds(n_traj, g->peers.size(), i, &lo, &hi);
            if (hi == lo) return RB_OK;
            const size_t o = lo * (aos ? n : 1);              // offset of trajectory lo inside one state array
            auto at = [&](const double* p) { return p ? p + o : nullptr; };
            auto atw = [&](double* p) { return p ? p + o : nullptr; };
            GradArgs s = a;
            s.q0 = at(a.q0); s.dq0 = at(a.dq0); s.tau = at(a.tau); s.q_traj = at(a.q_traj); s.dq_traj = at(a.dq_traj);
            s.g_q = at(a.g_q); s.g_dq = at(a.g_dq); s.g_qf = at(a.g_qf); s.g_dqf = at(a.g_dqf);
            s.cost = a.cost ? a.cost + lo : nullptr;
            s.grad_tau = atw(a.grad_tau); s.grad_q0 = atw(a.grad_q0); s.grad_dq0 = atw(a.grad_dq0);
            return grad_impl(g->peers[i], s, hi - lo, ld, layout, mem, nullptr, aos ? n_traj * n : 0);
        });
    }
    if (mem != RB_MEM_HOST && mem != RB_MEM_DEVICE) return fail(RB_ERR_ARG, "bad mem");
    if (a.horizon < 0) return fail(RB_ERR_ARG, "horizon < 0");
    if (!std::isfinite(a.dt)) return fail(RB_ERR_ARG, "dt must be finite");
    if (n_traj == 0) return RB_OK;
    const bool cost = a.w != nullptr;
    const size_t H = (size_t)a.horizon;
    if (!a.q0 || !a.dq0 || (H > 0 && (!a.tau || (!cost && (!a.q_traj || !a.dq_traj))))) return fail(RB_ERR_NULL, "input pointer is NULL");
    if (layout == RB_LAYOUT_SOA) { if (ld == 0) ld = n_traj; if (ld < n_traj) return fail(RB_ERR_ARG, "ld < n_traj"); }
    CostBlock cb;
    if (cost) { const int rc = pack_cost_block(g->model, a.w, a.tip, a.col, cb); if (rc != RB_OK) return rc; }
    if (!cost && !a.grad_tau && !a.grad_q0 && !a.grad_dq0) return RB_OK;
    DeviceGuard dg(g->device);
    if (!dg.ok) return fail(RB_ERR_CUDA, "cudaSetDevice failed");
    cudaStream_t st = mem == RB_MEM_DEVICE ? (cudaStream_t)stream : g->stream;
    if (mem == RB_MEM_DEVICE && layout == RB_LAYOUT_SOA) return grad_device(g, a, cb, n_traj, ld, st, g->d_status);
    // Host pointers and/or AoS: staged like the rollout; the staged call then runs as a device SoA call with ld = n_traj.
    return run_staged(g, {{a.q0, 1}, {a.dq0, 1}, {a.tau, H}, {a.q_traj, H}, {a.dq_traj, H}, {a.g_q, H}, {a.g_dq, H}, {a.g_qf, 1}, {a.g_dqf, 1}},
                      {{a.grad_tau, H, false}, {a.grad_q0, 1, false}, {a.grad_dq0, 1, false}, {a.cost, 1, true}},
                      n_traj, ld, layout, mem, aos_stride, st, [&](const double* const* in, double* const* out, int* d_stat) -> int {
        const GradArgs s{in[0], in[1], in[2], a.dt, a.horizon, in[3], in[4], in[5], in[6], in[7], in[8], a.w, out[3], out[0], out[1], out[2], a.tip, a.col};
        return grad_device(g, s, cb, n_traj, n_traj, st, d_stat);
    });
}
}  // namespace

extern "C" int multibody_rollout(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                                 double* q_traj, double* dq_traj, double* q_final, double* dq_final,
                                 size_t n_traj, size_t ld, RbLayout layout, RbMem mem, void* stream) {
    return rollout_impl(g, q0, dq0, tau, dt, horizon, q_traj, dq_traj, q_final, dq_final, nullptr, nullptr, nullptr, nullptr, n_traj, ld,
                        layout, mem, stream);
}

extern "C" int multibody_rollout_cost(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                                      const RbQuadCost* weights, double* cost, double* q_final, double* dq_final,
                                      size_t n_traj, size_t ld, RbLayout layout, RbMem mem, void* stream) {
    if (!cost) return fail(RB_ERR_NULL, "cost output pointer is NULL");
    return rollout_impl(g, q0, dq0, tau, dt, horizon, nullptr, nullptr, q_final, dq_final, weights, nullptr, nullptr, cost, n_traj, ld,
                        layout, mem, stream);
}

extern "C" int multibody_rollout_tip_cost(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                                          const RbQuadCost* weights, const RbTipCost* tip, double* cost, double* q_final, double* dq_final,
                                          size_t n_traj, size_t ld, RbLayout layout, RbMem mem, void* stream) {
    if (!cost) return fail(RB_ERR_NULL, "cost output pointer is NULL");
    const RbQuadCost none{};
    return rollout_impl(g, q0, dq0, tau, dt, horizon, nullptr, nullptr, q_final, dq_final, weights ? weights : &none, tip, nullptr, cost,
                        n_traj, ld, layout, mem, stream);
}

extern "C" int multibody_rollout_collision_cost(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                                                const RbQuadCost* weights, const RbTipCost* tip, const RbCollisionCost* col, double* cost,
                                                double* q_final, double* dq_final, size_t n_traj, size_t ld, RbLayout layout, RbMem mem,
                                                void* stream) {
    if (!cost) return fail(RB_ERR_NULL, "cost output pointer is NULL");
    const RbQuadCost none{};
    return rollout_impl(g, q0, dq0, tau, dt, horizon, nullptr, nullptr, q_final, dq_final, weights ? weights : &none, tip, col, cost,
                        n_traj, ld, layout, mem, stream);
}

extern "C" int multibody_rollout_vjp(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                                     const double* q_traj, const double* dq_traj,
                                     const double* g_q_traj, const double* g_dq_traj, const double* g_q_final, const double* g_dq_final,
                                     double* grad_tau, double* grad_q0, double* grad_dq0,
                                     size_t n_traj, size_t ld, RbLayout layout, RbMem mem, void* stream) {
    const GradArgs a{q0, dq0, tau, dt, horizon, q_traj, dq_traj, g_q_traj, g_dq_traj, g_q_final, g_dq_final, nullptr, nullptr,
                     grad_tau, grad_q0, grad_dq0};
    return grad_impl(g, a, n_traj, ld, layout, mem, stream);
}

extern "C" int multibody_rollout_cost_grad(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                                           const RbQuadCost* weights, double* cost, double* grad_tau, double* grad_q0, double* grad_dq0,
                                           size_t n_traj, size_t ld, RbLayout layout, RbMem mem, void* stream) {
    if (!weights) return fail(RB_ERR_NULL, "cost weights are NULL");
    if (!cost) return fail(RB_ERR_NULL, "cost output pointer is NULL");
    const GradArgs a{q0, dq0, tau, dt, horizon, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, weights, cost,
                     grad_tau, grad_q0, grad_dq0};
    return grad_impl(g, a, n_traj, ld, layout, mem, stream);
}

extern "C" int multibody_rollout_tip_cost_grad(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt, int horizon,
                                               const RbQuadCost* weights, const RbTipCost* tip, double* cost, double* grad_tau,
                                               double* grad_q0, double* grad_dq0, size_t n_traj, size_t ld, RbLayout layout, RbMem mem,
                                               void* stream) {
    if (!cost) return fail(RB_ERR_NULL, "cost output pointer is NULL");
    const RbQuadCost none{};
    const GradArgs a{q0, dq0, tau, dt, horizon, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, weights ? weights : &none, cost,
                     grad_tau, grad_q0, grad_dq0, tip};
    return grad_impl(g, a, n_traj, ld, layout, mem, stream);
}

extern "C" int multibody_rollout_collision_cost_grad(RbGpu* g, const double* q0, const double* dq0, const double* tau, double dt,
                                                     int horizon, const RbQuadCost* weights, const RbTipCost* tip,
                                                     const RbCollisionCost* col, double* cost, double* grad_tau, double* grad_q0,
                                                     double* grad_dq0, size_t n_traj, size_t ld, RbLayout layout, RbMem mem,
                                                     void* stream) {
    if (!cost) return fail(RB_ERR_NULL, "cost output pointer is NULL");
    const RbQuadCost none{};
    const GradArgs a{q0, dq0, tau, dt, horizon, nullptr, nullptr, nullptr, nullptr, nullptr, nullptr, weights ? weights : &none, cost,
                     grad_tau, grad_q0, grad_dq0, tip, col};
    return grad_impl(g, a, n_traj, ld, layout, mem, stream);
}

// ===================================================================== helpers
extern "C" int multibody_gpu_fill(RbGpu* g, double* dev_out, uint64_t seed, uint32_t field, const double* lo, const double* hi,
                                  size_t first_index, size_t count, size_t ld, void* stream) {
    if (!g || !dev_out || !lo || !hi) return fail(RB_ERR_NULL, "NULL argument");
    if (!g->peers.empty()) return fail(RB_ERR_UNSUPPORTED, kMultiDeviceOnly);
    if (ld == 0) ld = count;
    if (ld < count) return fail(RB_ERR_ARG, "ld < count");
    if (field >= 64) return fail(RB_ERR_ARG, "field must be < 64");
    DeviceGuard dg(g->device);
    RbFillRange rg;
    for (int i = 0; i < g->model.n; ++i) { rg.lo[i] = lo[i]; rg.hi[i] = hi[i]; }
    cudaError_t e = rb_launch_fill(dev_out, seed, field, g->model.n, rg, first_index, count, ld, (cudaStream_t)stream);
    g->launches += 1;
    if (e != cudaSuccess) return fail_cuda(e, "fill launch");
    return RB_OK;
}

extern "C" int multibody_gpu_sync(RbGpu* g) {
    if (!g) return fail(RB_ERR_NULL, "engine handle is NULL");
    if (!g->peers.empty()) {
        int rc = RB_OK; std::string err;
        for (RbGpu* pg : g->peers) {
            const int r = multibody_gpu_sync(pg);
            if (r != RB_OK && (rc == RB_OK || rc == RB_ERR_NOT_SPD)) { rc = r; err = g_err; }
        }
        if (rc != RB_OK) g_err = err;
        return rc;
    }
    DeviceGuard dg(g->device);
    std::lock_guard<std::mutex> lk(g->mu_status);
    RB_CUDA(cudaDeviceSynchronize());      // device calls run on caller streams: wait for all of them
    return fetch_status(g, 0);
}

extern "C" int multibody_gpu_status(RbGpu* g) { return multibody_gpu_sync(g); }

extern "C" int multibody_host_alloc(void** out, size_t bytes) {
    if (!out) return fail(RB_ERR_NULL, "out is NULL");
    *out = nullptr;
    RB_CUDA(cudaMallocHost(out, bytes ? bytes : 1));
    return RB_OK;
}
extern "C" void multibody_host_free(void* p) { if (p) cudaFreeHost(p); }

// Bare transfer ceiling of the path RB_MEM_HOST calls use (include/rigidbody.h).
extern "C" int multibody_gpu_measure_copy_peak(RbGpu* g, size_t h2d_bytes, size_t d2h_bytes, int reps,
                                               double* h2d_gbs, double* d2h_gbs) {
    if (!g || !h2d_gbs || !d2h_gbs) return fail(RB_ERR_NULL, "NULL argument");
    if (reps < 1) return fail(RB_ERR_ARG, "reps < 1");
    std::vector<RbGpu*> devs = g->peers.empty() ? std::vector<RbGpu*>{g} : g->peers;
    const size_t nd = devs.size();
    // Streamed through host buffers of up to 2 GiB per direction and device, walked front to back: a small buffer copied
    // over and over would be served from the host's last-level cache (hundreds of MB on current server CPUs) and promise a
    // rate that a real batch, which streams from DRAM, never sees (measured: 98 vs 73 GB/s for two GPUs).
    const size_t cap = (size_t)2048 << 20;
    struct Side { void* h = nullptr; void* d = nullptr; size_t buf = 0; };
    std::vector<Side> up(nd), down(nd);
    std::vector<int> rcs(nd, RB_OK); std::vector<std::string> errs(nd);
    auto cleanup = [&] {
        for (size_t i = 0; i < nd; ++i) {
            DeviceGuard dg(devs[i]->device);
            for (Side* sd : {&up[i], &down[i]}) { if (sd->h) cudaFreeHost(sd->h); if (sd->d) cudaFree(sd->d); }
        }
    };
    for (size_t i = 0; i < nd; ++i) {
        DeviceGuard dg(devs[i]->device);
        const size_t per_up = h2d_bytes / nd, per_down = d2h_bytes / nd;
        up[i].buf = std::max<size_t>(1, std::min(cap, per_up)); down[i].buf = std::max<size_t>(1, std::min(cap, per_down));
        cudaError_t e = cudaMallocHost(&up[i].h, up[i].buf);
        if (e == cudaSuccess) e = cudaMalloc(&up[i].d, up[i].buf);
        if (e == cudaSuccess) e = cudaMallocHost(&down[i].h, down[i].buf);
        if (e == cudaSuccess) e = cudaMalloc(&down[i].d, down[i].buf);
        if (e != cudaSuccess) { cleanup(); return fail_cuda(e, "copy probe allocation"); }
        memset(up[i].h, 1, up[i].buf);
    }
    auto pass = [&](size_t i) -> int {           // one device: both directions at once, as the pipeline runs them
        RbGpu* pg = devs[i];
        DeviceGuard dg(pg->device);
        const size_t per_up = h2d_bytes / nd, per_down = d2h_bytes / nd;
        // pieces of 64 MiB, like the chunks of the real pipeline; the host side advances through its whole buffer
        const size_t piece = (size_t)64 << 20;
        for (size_t off = 0; off < per_up; off += piece) {
            const size_t len = std::min(piece, per_up - off), ho = off % up[i].buf;
            const size_t l2 = std::min(len, up[i].buf - ho);
            RB_CUDA(cudaMemcpyAsync((char*)up[i].d + ho, (char*)up[i].h + ho, l2, cudaMemcpyHostToDevice, pg->s_h2d));
        }
        for (size_t off = 0; off < per_down; off += piece) {
            const size_t len = std::min(piece, per_down - off), ho = off % down[i].buf;
            const size_t l2 = std::min(len, down[i].buf - ho);
            RB_CUDA(cudaMemcpyAsync((char*)down[i].h + ho, (char*)down[i].d + ho, l2, cudaMemcpyDeviceToHost, pg->s_d2h));
        }
        RB_CUDA(cudaStreamSynchronize(pg->s_h2d));
        RB_CUDA(cudaStreamSynchronize(pg->s_d2h));
        return RB_OK;
    };
    auto all = [&]() -> int {
        std::vector<std::thread> th;
        for (size_t i = 0; i < nd; ++i) th.emplace_back([&, i] { rcs[i] = pass(i); if (rcs[i] != RB_OK) errs[i] = g_err; });
        for (auto& t : th) t.join();
        for (size_t i = 0; i < nd; ++i) if (rcs[i] != RB_OK) return fail(rcs[i], errs[i]);
        return RB_OK;
    };
    int rc = all();                               // warm-up
    // MEAN over the timed passes, not the best one: when several processes probe at the same time (bench.py under
    // torchrun) their passes drift apart, and a process's fastest pass is the one the others were not competing in
    double total = 0.0; int done = 0;
    for (int r = 0; r < reps && rc == RB_OK; ++r) {
        const auto t0 = std::chrono::steady_clock::now();
        rc = all();
        total += std::chrono::duration<double>(std::chrono::steady_clock::now() - t0).count();
        ++done;
    }
    cleanup();
    if (rc != RB_OK) return rc;
    const double sec = total / done;
    *h2d_gbs = (double)(h2d_bytes / nd * nd) / sec / 1e9;
    *d2h_gbs = (double)(d2h_bytes / nd * nd) / sec / 1e9;
    return RB_OK;
}

extern "C" int multibody_gpu_measure_fp64_peak(RbGpu* g, int millis, double* tflops) {
    if (!g || !tflops) return fail(RB_ERR_NULL, "NULL argument");
    if (!g->peers.empty()) g = g->peers[0];
    DeviceGuard dg(g->device);
    double* d_out = nullptr;
    RB_CUDA(cudaMalloc((void**)&d_out, sizeof(double)));
    cudaEvent_t a, b;
    RB_CUDA(cudaEventCreate(&a)); RB_CUDA(cudaEventCreate(&b));
    // The roofline denominator must be the best DFMA rate the chip sustains for `millis`, so two occupancies are tried
    // (16 and 32 resident warps per SM, 8 independent chains each: 64 warps per SM measured 6 % lower) and the better
    // one is reported; tools/ubench_fp64_peak.cu cross-checks it by wall clock (profiles/r2_ubench_fp64_peak.txt).
    int rc = RB_OK;
    double best = 0.0;
    for (int threads : {128, 256}) {
        const int blocks = g->sm_count * 4;
        auto run = [&](int iters, float* ms) -> int {
            RB_CUDA(cudaEventRecord(a, g->stream));
            RB_CUDA(rb_launch_fp64_peak(d_out, blocks, threads, iters, g->stream));
            g->launches += 1;
            RB_CUDA(cudaEventRecord(b, g->stream));
            RB_CUDA(cudaEventSynchronize(b));
            RB_CUDA(cudaEventElapsedTime(ms, a, b));
            return RB_OK;
        };
        float ms = 0.f;
        rc = run(200, &ms);                                  // warm-up + calibration
        if (rc == RB_OK) rc = run(200, &ms);
        if (rc != RB_OK) break;
        const int iters = (int)std::max(200.0, 200.0 * (millis > 0 ? millis : 50) / std::max(ms, 1e-3f));
        rc = run(iters, &ms);
        if (rc != RB_OK) break;
        const double flops = (double)blocks * threads * 8.0 * RB_PEAK_INNER * (double)iters * 2.0;
        best = std::max(best, flops / (ms * 1e-3) / 1e12);
    }
    if (rc == RB_OK) *tflops = best;
    cudaEventDestroy(a); cudaEventDestroy(b); cudaFree(d_out);
    return rc;
}

// ===================================================================== Part 1: the reference's six symbols
// When this library is linked next to the Rust cdylib `rigidbody_bindings` (which already exports these names,
// rigidbody_bindings/src/lib.rs:8-78), build with -DRB_NO_REFERENCE_SYMBOLS and let
// rust/rigidbody_gpu_bindings bridge its `Multibody` to multibody_gpu_new (see INTEGRATION.md).
#ifndef RB_NO_REFERENCE_SYMBOLS
static Multibody* mb_load(const char* path) {
    try {
        Multibody* mb = new (std::nothrow) Multibody();
        if (!mb) { fail(RB_ERR_CUDA, "out of host memory"); return nullptr; }
        std::string err;
        int rc = rb_model_from_urdf(path, mb->model, err);
        if (rc != RB_OK) { fail(rc, err); delete mb; return nullptr; }
        return mb;
    } catch (const std::exception& e) { fail(RB_ERR_ARG, std::string("exception: ") + e.what()); return nullptr; }
}

extern "C" Multibody* multibody_new(void) {
    const char* p = getenv("RIGIDBODY_URDF");
    return mb_load(p ? p : "assets/fr3.urdf");
}
extern "C" Multibody* multibody_new_from_urdf(const char* urdf_path) { return mb_load(urdf_path); }

extern "C" void multibody_free(Multibody* mb) {
    if (!mb) return;
    if (mb->gpu) multibody_gpu_free(mb->gpu);
    delete mb;
}
extern "C" void multibody_free_result(double* p) { free(p); }

static RbGpu* mb_engine(const Multibody* cmb) {
    Multibody* mb = const_cast<Multibody*>(cmb);
    std::lock_guard<std::mutex> lk(mb->mu);
    if (!mb->gpu) {
        const char* d = getenv("RIGIDBODY_DEVICE");
        if (gpu_create(mb->model, d ? atoi(d) : 0, &mb->gpu) != RB_OK) return nullptr;
    }
    return mb->gpu;
}

template <class F>
static double* mb_single(const Multibody* mb, size_t out_count, F&& call) {
    if (!mb) { fail(RB_ERR_NULL, "Multibody handle is NULL"); return nullptr; }
    RbGpu* g = mb_engine(mb);
    if (!g) return nullptr;
    double* out = (double*)malloc(out_count * sizeof(double));
    if (!out) { fail(RB_ERR_CUDA, "out of host memory"); return nullptr; }
    if (call(g, out) != RB_OK) { free(out); return nullptr; }
    return out;
}

extern "C" double* multibody_rnea(const Multibody* mb, const double* q, const double* dq, const double* ddq) {
    return mb_single(mb, mb ? mb->model.n : 0, [&](RbGpu* g, double* out) {
        return multibody_rnea_batch(g, q, dq, ddq, out, 1, 0, RB_LAYOUT_AOS, RB_MEM_HOST, nullptr);
    });
}
extern "C" double* multibody_crba(const Multibody* mb, const double* q) {
    return mb_single(mb, mb ? (size_t)mb->model.n * mb->model.n : 0, [&](RbGpu* g, double* out) {
        return multibody_crba_batch(g, q, out, 1, 0, RB_LAYOUT_AOS, RB_MEM_HOST, nullptr);
    });
}
extern "C" double* multibody_fwd_kin(const Multibody* mb, const double* q) {
    return mb_single(mb, 3, [&](RbGpu* g, double* out) {
        return multibody_fwd_kin_batch(g, q, out, 1, 0, RB_LAYOUT_AOS, RB_MEM_HOST, nullptr);
    });
}
extern "C" double* multibody_jac(const Multibody* mb, const double* q) {
    return mb_single(mb, mb ? (size_t)6 * mb->model.n : 0, [&](RbGpu* g, double* out) {
        return multibody_jac_batch(g, q, out, 1, 0, RB_LAYOUT_AOS, RB_MEM_HOST, nullptr);
    });
}
#endif  // RB_NO_REFERENCE_SYMBOLS
