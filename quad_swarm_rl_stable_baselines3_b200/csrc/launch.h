// launch.h -- per-lane-group launchers.  The kernels are templates on KG (lanes per env) and, for the upstream step kernel,
// on the compile-time feature set; every KG is compiled in its own translation unit (kernels_kg.cu with -DQS_KG=n) so that
// the library builds in parallel.  quadsim.cu only sees these plain functions.  (A persistent, TMA-prefetched form of the
// step kernel was measured slower than this one-warp-tile-per-warp form and removed: profiles/README.md.)
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include "quadsim_kernels.cuh"
#include "fork_kernels.cuh"

namespace qs {

struct LaunchShape { int grid, block; size_t smem; };

// one table entry per KG in {1, 2, 4, 8, 16, 32}
struct KgLaunchers {
    // set the shared-memory attributes of the handle's kernels
    void (*prepare)(int feat, size_t smem, int block, bool fork);
    void (*step)(int feat, LaunchShape s, cudaStream_t st, const DevConst &c, const DevPtrs &P, const float4 *actions,
                 float *obs, float *rew, uint8_t *done, float *term_obs, uint8_t *reset_success);
    void (*reset)(int feat, LaunchShape s, cudaStream_t st, const DevConst &c, const DevPtrs &P, const uint8_t *mask, float *obs);
    void (*fork_step)(LaunchShape s, cudaStream_t st, const DevConst &c, const ForkConst &f, const DevPtrs &P, const ForkPtrs &F,
                      const float2 *actions, float *obs, float *rew, uint8_t *done, float *term_obs, uint8_t *reset_success);
    void (*fork_reset)(LaunchShape s, cudaStream_t st, const DevConst &c, const ForkConst &f, const DevPtrs &P, const ForkPtrs &F,
                       const uint8_t *mask, float *obs);
};

const KgLaunchers &launchers_kg1();
const KgLaunchers &launchers_kg2();
const KgLaunchers &launchers_kg4();
const KgLaunchers &launchers_kg8();
const KgLaunchers &launchers_kg16();
const KgLaunchers &launchers_kg32();

}  // namespace qs
