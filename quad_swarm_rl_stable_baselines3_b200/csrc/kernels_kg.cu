// kernels_kg.cu -- instantiates every kernel for ONE lane-group width (compile with -DQS_KG=1|2|4|8|16|32).
#include <cstdlib>
#include <map>
#include <mutex>
#include <utility>

#include "launch.h"

#ifndef QS_KG
#error "compile with -DQS_KG=<lanes per env>"
#endif

namespace qs {
namespace {

constexpr int KG = QS_KG;

// Shared-memory attributes of one kernel.  `block` > 0: size the shared-memory carve-out to what the resident blocks need
// (+1 KB per block of driver reservation) and leave the rest of the unified array to L1.  The step kernels stream their state
// (no L1 reuse) but spill a few registers at the 128-register cap; with the maximum carve-out L1 shrinks to ~28 KB, the 16
// resident warps' stack frames do not fit and every spill reload becomes an L2 round trip (profiles/README.md, v5: 89.3 ->
// 86.3 us).  `block` == 0 (the reset kernels): maximum carve-out.
// The attributes belong to the kernel instantiation on a device, not to a handle: several handles (train env + eval env, as
// sb_train.py runs them) share them, so both the dynamic shared-memory limit and the carve-out are only ever RAISED -- a later,
// smaller handle must not pull the limit below what an earlier one launches with (cudaErrorInvalidValue on its next step).
struct AttrState { int max_bytes = 0; int carve = -1; };
inline AttrState &attr_state(const void *kernel)
{
    static std::mutex mu;
    static std::map<std::pair<int, const void *>, AttrState> table;
    int dev = 0;
    cudaGetDevice(&dev);
    std::lock_guard<std::mutex> lock(mu);
    return table[std::make_pair(dev, kernel)];
}

template <typename... Args>
void set_attr(size_t bytes, void (*kernel)(Args...), int block = 0)
{
    AttrState &st = attr_state(reinterpret_cast<const void *>(kernel));
    if (bytes > 48 * 1024 && (int)bytes > st.max_bytes) {
        cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)bytes);
        st.max_bytes = (int)bytes;
    }
    int carve = cudaSharedmemCarveoutMaxShared;
    if (block > 0) {
        int nblk = 0, dev = 0, smem_sm = 233472;
        cudaGetDevice(&dev);
        cudaDeviceGetAttribute(&smem_sm, cudaDevAttrMaxSharedMemoryPerMultiprocessor, dev);
        if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&nblk, kernel, block, bytes) == cudaSuccess && nblk > 0) {
            const long long need = (long long)nblk * ((long long)bytes + 1024);
            carve = (int)((need * 100 + smem_sm - 1) / smem_sm) + 2;
            if (carve > 100) carve = 100;
        }
    }
    if (const char *e = getenv("QS_CARVEOUT")) { int v = atoi(e); if (v >= 0 && v <= 100) carve = v; }   // tuning knob (percent of max shared)
    if (carve == cudaSharedmemCarveoutMaxShared) carve = 100;
    if (carve > st.carve) {
        cudaFuncSetAttribute(kernel, cudaFuncAttributePreferredSharedMemoryCarveout, carve);
        st.carve = carve;
    }
}

// feature sets of the upstream step kernel: bit 0 obstacles, bit 1 downwash, bit 2 formation scenarios (never with obstacles)
#define QS_FEAT_SWITCH(FEATv, CALL)                       \
    switch (FEATv) {                                      \
        case 0: { constexpr int FEAT = 0; CALL; } break;  \
        case 1: { constexpr int FEAT = 1; CALL; } break;  \
        case 2: { constexpr int FEAT = 2; CALL; } break;  \
        case 3: { constexpr int FEAT = 3; CALL; } break;  \
        case 4: { constexpr int FEAT = 4; CALL; } break;  \
        default: { constexpr int FEAT = 6; CALL; } break; \
    }
void prepare(int feat, size_t smem, int block, bool fork)
{
    if (fork) {
        set_attr(smem, fork_step_kernel<KG>, block);
        set_attr(smem, fork_reset_kernel<KG>);
        return;
    }
    QS_FEAT_SWITCH(feat, set_attr(smem, step_kernel<KG, FEAT>, block));
    set_attr(smem, reset_kernel<KG, false, false>);
    set_attr(smem, reset_kernel<KG, true, false>);
    set_attr(smem, reset_kernel<KG, false, true>);
}

void step(int feat, LaunchShape s, cudaStream_t st, const DevConst &c, const DevPtrs &P, const float4 *actions, float *obs,
          float *rew, uint8_t *done, float *term_obs, uint8_t *reset_success)
{
    QS_FEAT_SWITCH(feat, (step_kernel<KG, FEAT><<<s.grid, s.block, s.smem, st>>>(c, P, actions, obs, rew, done, term_obs, reset_success)));
}

void reset(int feat, LaunchShape s, cudaStream_t st, const DevConst &c, const DevPtrs &P, const uint8_t *mask, float *obs)
{
    if (feat & 1) reset_kernel<KG, true, false><<<s.grid, s.block, s.smem, st>>>(c, P, mask, obs);
    else if (feat & 4) reset_kernel<KG, false, true><<<s.grid, s.block, s.smem, st>>>(c, P, mask, obs);
    else reset_kernel<KG, false, false><<<s.grid, s.block, s.smem, st>>>(c, P, mask, obs);
}

void fork_step(LaunchShape s, cudaStream_t st, const DevConst &c, const ForkConst &f, const DevPtrs &P, const ForkPtrs &F,
               const float2 *actions, float *obs, float *rew, uint8_t *done, float *term_obs, uint8_t *reset_success)
{
    fork_step_kernel<KG><<<s.grid, s.block, s.smem, st>>>(c, f, P, F, actions, obs, rew, done, term_obs, reset_success);
}

void fork_reset(LaunchShape s, cudaStream_t st, const DevConst &c, const ForkConst &f, const DevPtrs &P, const ForkPtrs &F,
                const uint8_t *mask, float *obs)
{
    fork_reset_kernel<KG><<<s.grid, s.block, s.smem, st>>>(c, f, P, F, mask, obs);
}

const KgLaunchers table = { prepare, step, reset, fork_step, fork_reset };

}  // namespace

#define QS_CAT2(a, b) a##b
#define QS_CAT(a, b) QS_CAT2(a, b)
const KgLaunchers &QS_CAT(launchers_kg, QS_KG)() { return table; }

}  // namespace qs
