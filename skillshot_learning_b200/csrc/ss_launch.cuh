// ss_launch.cuh -- programmatic dependent launch (PDL) for the kernels of one DDPG update.
//
// A 65,536-row update is nine dependent launches of 10-60 us each; between two of them the stream pays the drain of the
// first grid (the SMs that ran three tiles idle while the others run their fourth), the launch latency of the second and
// its prologue (barrier set-up, tensor-memory allocation, shared-memory clearing, weight staging).  Launched with
// programmatic stream serialization, the CTAs of the next grid are placed as soon as an SM has room for them -- for the
// tensor-core kernels, which take an SM's whole shared memory: as soon as that SM's CTA of the previous grid exits -- and
// run their prologue there; griddepcontrol.wait then holds them until the previous grid has completed and its writes are
// visible.
//
// Rules every kernel of such a chain follows (ss_ddpg_update is the only caller that switches the mode on):
//   * before griddep_wait(): no global write, and no global read of anything the chain writes -- EXCEPT, when the caller
//     says so (kPdlEarlyWeights), the network parameters the kernel stages into shared memory
//   * griddep_launch() comes AFTER griddep_wait(): when the next grid's CTAs start, this grid has passed its wait, so
//     every grid before the previous one is complete.  A kernel may therefore stage, ahead of its wait, parameters that
//     its immediate predecessor does not write; ss_ddpg_update sets kPdlEarlyWeights exactly for those launches
//   * every CTA executes the wait (a grid whose CTAs all skipped it could complete before its predecessor)
// Both instructions are no-ops in a grid launched the ordinary way, which is how every other caller launches these kernels.
#pragma once
#include <cuda_runtime.h>

namespace sslaunch {

// kPdlEarlyAfterFirst: the next tensor-core launch stages its parameters behind the wait (its predecessor writes them), the
// ones after it ahead of it
// kPdlPairCriticLate: in an actor -> critic pair launch only the actor role stages ahead of the wait
// kPdlSampleEarly: replay_sample_kernel gathers BEFORE its wait (and waits before it exits, so that its completion still
// implies its predecessor's): the caller guarantees that its predecessor on the stream neither writes the ring nor reads
// or writes the minibatch buffers of this call
enum : int { kPdlOff = 0, kPdlOn = 1, kPdlEarlyWeights = 2, kPdlEarlyAfterFirst = 4, kPdlPairCriticLate = 8, kPdlSampleEarly = 16 };

// the launch mode of the calling host thread; set by ss_ddpg_update around each entry point it calls
int &pdl_mode();
// whether ss_ddpg_update / ss_selfplay_rollout chain their launches at all: yes unless ss_set_dependent_launch(0)
bool chain_enabled();

struct PdlScope {                     // sets the mode for the lifetime of the object
    int saved;
    explicit PdlScope(int mode) : saved(pdl_mode()) { pdl_mode() = mode; }
    ~PdlScope() { pdl_mode() = saved; }
};

// whether the tensor-core launch about to be made may stage its parameters ahead of griddepcontrol.wait
inline int take_early_weights() {
    int &m = pdl_mode();
    if (!(m & kPdlOn)) return 0;
    if (m & kPdlEarlyAfterFirst) { m = (m & ~kPdlEarlyAfterFirst) | kPdlEarlyWeights; return 0; }
    return (m & kPdlEarlyWeights) ? 1 : 0;
}

template <class... KArgs, class... Args>
inline cudaError_t launch(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st, Args &&...args) {
    cudaLaunchConfig_t cfg = {};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    if (pdl_mode() & kPdlOn) { cfg.attrs = attr; cfg.numAttrs = 1; }
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}

#ifdef __CUDACC__
__device__ __forceinline__ void griddep_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void griddep_launch() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
#endif

}  // namespace sslaunch
