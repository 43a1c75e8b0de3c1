// rb_jit.h -- run-time specialised kernels (see rb_jit.cu).
#pragma once
#include <string>
#include <vector>
#include "rb_host_model.h"

#define RB_JIT_MAX_N 18        // longest chain the register-resident unrolled kernels are compiled for (FD falls off a cliff at 20)
#define RB_JIT_LONG_MAX_N 32   // 19..32 joints: only rnea / crba / fwd_kin / jac are compiled ("jit-long"); the rest falls through
#define RB_JIT_KERNELS 12
enum : int { RB_JK_RNEA = 0, RB_JK_RNEA_AOS, RB_JK_FD, RB_JK_FD_AOS, RB_JK_CRBA, RB_JK_FK, RB_JK_JAC, RB_JK_ROLLOUT,
             RB_JK_RNEA_F32, RB_JK_FD_F32, RB_JK_RNEA_FD, RB_JK_ROLLOUT_TIP };

struct RbJitImage {             // what the compiler produces / the disk cache holds
    std::vector<char> cubin;
    std::vector<std::string> lowered;   // mangled kernel names, RB_JK_* order
    bool from_cache = false;
};

struct RbJitParam {             // parameter block of the "jit-specialised" RbOps table
    void* lib;                  // cudaLibrary_t
    void* k[RB_JIT_KERNELS];    // cudaKernel_t
    int n;
};

// Compile (or fetch from the disk cache) the kernels for one chain.  Needs libnvrtc, not a GPU.
int rb_jit_compile(const RbHostModel& m, RbJitImage& img, std::string& log);
// Load a compiled image into the current device's context.
int rb_jit_load(const RbJitImage& img, int n, RbJitParam& out, std::string& err);
void rb_jit_unload(RbJitParam& p);

struct RbOps;
const RbOps* rb_ops_jit();
const RbOps* rb_ops_jit_long();   // the partial table of chains of RB_JIT_MAX_N+1 .. RB_JIT_LONG_MAX_N joints
