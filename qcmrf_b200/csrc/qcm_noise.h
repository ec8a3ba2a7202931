// Host-side pieces shared by the batched small-circuit launchers (qcm_small.cu) and the noisy-shot launcher
// (qcm_noise.cu).  Internal: nothing here is exported from the library.
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <mutex>

namespace qcm {

constexpr int kSmallMaxQubits = 13;        // qcm_small_max_qubits: one state in shared memory

// Per-device, grow-only work space of the batched path: ONE device buffer, ONE pinned host buffer for the
// inputs (a single H2D copy), one stream and two events -- created once, reused by every call (the first
// version paid ~15 cudaMalloc + cudaFree per batch, 10-25 ms next to a 0.07 ms kernel).  Guarded by a mutex:
// calls on the same device serialise.
struct SmallArena {
    std::mutex mu;
    void *dev = nullptr;
    size_t dev_cap = 0;
    void *pin = nullptr;
    size_t pin_cap = 0;
    cudaStream_t st = nullptr;
    cudaEvent_t e0 = nullptr, e1 = nullptr;
};
extern SmallArena g_arena[64];

inline size_t up256(size_t x) { return (x + 255) & ~size_t(255); }

cudaError_t arena_reserve(SmallArena &A, size_t dev_bytes, size_t pin_bytes);

// Enqueue k_readout_keys on `st`: flips the measured clbits of keys[c * shots + s] (device arrays; stream_ids may
// be null: circuit index) by the per-clbit tables readout[c][64][2].
cudaError_t launch_readout_keys(cudaStream_t st, int n_circuits, uint64_t shots, uint64_t seed, const uint64_t *stream_ids,
                                const int32_t *n_clbits, const double *readout, uint64_t *keys);

}  // namespace qcm
