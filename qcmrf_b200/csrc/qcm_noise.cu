// Noisy shots of small circuits: every shot is a trajectory -- the unfused gate list with Pauli errors drawn after
// the gates that carry a channel -- simulated in shared memory, then measured once and read out through per-clbit
// assignment errors.  Fusion cannot apply: every shot runs a different circuit.
//
// k_traj<R, CTA>: grid (trajectory groups, circuits).  Up to kWarpMaxQubits qubits one warp runs one trajectory
// (2^10 amplitudes: 8 KiB complex64, 16 KiB complex128) and a gate needs only __syncwarp; above that a CTA runs one
// trajectory.  The CTA's trajectories share the gate stream, staged cooperatively kChunk gates at a time in shared
// memory together with each trajectory's Pauli draws for those gates.  A Pauli is an index permutation and a phase,
// never a 2x2 product; a 2-qubit Pauli is two 1-qubit ones.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "qcm_kernels.cuh"
#include "qcm_noise.h"
#include "qcmrf_b200.h"

using namespace qcm;

namespace {

constexpr int kWarpMaxQubits = 10;         // one warp per trajectory up to here, one CTA above
constexpr int kTrajWarps = 4;              // trajectories per CTA in warp mode
constexpr int kChunk = 32;                 // gates staged per step (one Pauli draw per lane)
// Philox keys of the error and readout draws: distinct from the sampler's (seed), the product sampler's and the
// released-qubit keys, so that no two kinds of draw ever share a (key, stream, counter).
constexpr uint64_t kNoiseKey = 0x165667B19E3779F9ull;
constexpr uint64_t kReadoutKey = 0x27D4EB2F165667C5ull;

// The measured clbits of `key` flipped by their assignment errors: ro[2b + v] = P(flip | clbit b read as v).  Four
// clbits share one Philox call, counter shot * 16 + b / 4; a group of four whose flip probabilities are all 0
// draws nothing (it cannot flip).
__device__ __forceinline__ uint64_t readout_flip(uint64_t key, const double *ro, int ncl, uint64_t seed, uint64_t stream,
                                                 uint64_t shot) {
    for (int b0 = 0; b0 < ncl; b0 += 4) {
        bool any = false;
#pragma unroll
        for (int j = 0; j < 4; ++j)
            if (b0 + j < ncl) any |= (ro[2 * (b0 + j)] > 0.0) | (ro[2 * (b0 + j) + 1] > 0.0);
        if (!any) continue;
        uint32_t r[4];
        philox4(seed ^ kReadoutKey, stream, shot * 16ull + (uint64_t)(b0 >> 2), r);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int b = b0 + j;
            if (b < ncl) {
                const uint32_t v = (uint32_t)(key >> b) & 1u;
                if ((double)r[j] * (1.0 / 4294967296.0) < ro[2 * b + v]) key ^= 1ull << b;
            }
        }
    }
    return key;
}

__global__ void __launch_bounds__(kThreads) k_readout_keys(int n_circuits, uint64_t shots, uint64_t seed,
                                                           const uint64_t *stream_ids, const int32_t *n_clbits,
                                                           const double *readout, uint64_t *keys) {
    const uint64_t n = (uint64_t)n_circuits * shots;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (uint64_t)gridDim.x * blockDim.x) {
        const uint64_t c = i / shots, s = i - c * shots;
        keys[i] = readout_flip(keys[i], readout + 128 * c, n_clbits[c], seed, stream_ids ? stream_ids[c] : c, s);
    }
}

template <typename R> struct Amp { R x, y; };

template <typename R> struct StagedGate {
    R m[8];
    int32_t target;
    uint32_t ctrl_mask, ctrl_value;
};

struct TrajArgs {
    const int32_t *n_qubits;
    const int64_t *gate_begin;
    const qcm_gate *gates;
    const qcm_channel *channels;
    const int32_t *clbit_qubit;   // [n_circuits][64]
    const int32_t *n_clbits;
    const double *readout;        // [n_circuits][64][2] or null
    const uint64_t *stream_ids;   // or null: circuit index
    const int32_t *circ;          // circuits of this launch: blockIdx.y -> circuit
    uint64_t shots, seed;
    uint64_t *keys_out;           // [n_circuits][shots]
    int32_t *status_out;          // per circuit: 1 when a trajectory's norm was not finite and positive
};

// Pauli `code` (1 X, 2 Y, 3 Z) on qubit q, by thread t of a group of G.
template <typename R, int G>
__device__ __forceinline__ void apply_pauli(Amp<R> *psi, uint32_t half, int code, int q, int t) {
    for (uint32_t p = t; p < half; p += G) {
        const uint32_t i0 = (uint32_t)insert_zero(p, q), i1 = i0 | (1u << q);
        const Amp<R> a0 = psi[i0], a1 = psi[i1];
        if (code == 1) {
            psi[i0] = a1; psi[i1] = a0;
        } else if (code == 2) {                         // Y = [[0, -i], [i, 0]]
            psi[i0] = Amp<R>{a1.y, -a1.x}; psi[i1] = Amp<R>{-a0.y, a0.x};
        } else {
            psi[i1] = Amp<R>{-a1.x, -a1.y};
        }
    }
}

template <typename R, bool CTA>
__global__ void __launch_bounds__(CTA ? kThreads : 32 * kTrajWarps) k_traj(const TrajArgs a) {
    constexpr int G = CTA ? kThreads : 32;          // threads per trajectory
    constexpr int W = CTA ? 1 : kTrajWarps;         // trajectories per CTA
    extern __shared__ __align__(16) unsigned char smem_raw[];
    __shared__ StagedGate<R> sg[kChunk];
    __shared__ int32_t pk[W][kChunk];                // per trajectory and staged gate: packed Pauli, 0 = none
    __shared__ double part[W][G];
    const int c = a.circ[blockIdx.y];
    const int N = a.n_qubits[c];
    const uint32_t dim = 1u << N, half = dim >> 1;
    const int w = CTA ? 0 : (int)(threadIdx.x >> 5);
    const int t = CTA ? (int)threadIdx.x : (int)(threadIdx.x & 31);
    Amp<R> *psi = reinterpret_cast<Amp<R> *>(smem_raw) + (size_t)w * dim;
    const qcm_gate *gates = a.gates + a.gate_begin[c];
    const int64_t ng = a.gate_begin[c + 1] - a.gate_begin[c];
    const uint64_t stream = a.stream_ids ? a.stream_ids[c] : (uint64_t)c;
    const uint64_t groups = (a.shots + W - 1) / W;
    auto gsync = [] { if constexpr (CTA) __syncthreads(); else __syncwarp(); };

    for (uint64_t grp = blockIdx.x; grp < groups; grp += gridDim.x) {
        const uint64_t s = grp * W + w;
        const bool live = s < a.shots;               // uniform over the trajectory's threads
        __syncthreads();                             // the previous trajectory's outcome has been read
        for (uint32_t i = t; i < dim; i += G) psi[i] = Amp<R>{i == 0 ? R(1) : R(0), R(0)};
        for (int64_t cb = 0; cb < ng; cb += kChunk) {
            const int cn = ng - cb < kChunk ? (int)(ng - cb) : kChunk;
            __syncthreads();                         // the previous chunk has been applied by every trajectory
            for (int i = threadIdx.x; i < cn; i += blockDim.x) {
                const qcm_gate &g = gates[cb + i];
#pragma unroll
                for (int k = 0; k < 8; ++k) sg[i].m[k] = (R)g.m[k];
                sg[i].target = g.target;
                sg[i].ctrl_mask = g.ctrl_mask;
                sg[i].ctrl_value = g.ctrl_value;
            }
            if (t < cn) {                            // lane t draws gate cb + t's error for this trajectory
                int32_t code = 0;
                const int ch = gates[cb + t].channel;
                if (live && ch >= 0) {
                    const qcm_channel &C = a.channels[ch];
                    const double u = philox_uniform(a.seed ^ kNoiseKey, stream, s * (uint64_t)ng + (uint64_t)(cb + t));
                    if (!(u < C.cum[0])) {
                        int k = 1;
                        while (k < C.n_paulis - 1 && !(u < C.cum[k])) ++k;
                        code = (k & 3) | (C.qubit[0] << 2) | (((k >> 2) & 3) << 8) | ((C.qubit[1] & 63) << 10);
                    }
                }
                pk[w][t] = code;
            }
            __syncthreads();
            if (!live) continue;
            for (int j = 0; j < cn; ++j) {
                const StagedGate<R> &g = sg[j];
                const int tq = g.target;
                const uint32_t cm = g.ctrl_mask, cv = g.ctrl_value;
                const R m0 = g.m[0], m1 = g.m[1], m2 = g.m[2], m3 = g.m[3], m4 = g.m[4], m5 = g.m[5], m6 = g.m[6], m7 = g.m[7];
                for (uint32_t p = t; p < half; p += G) {
                    const uint32_t i0 = (uint32_t)insert_zero(p, tq), i1 = i0 | (1u << tq);
                    if ((i0 & cm) != cv) continue;
                    const R x0 = psi[i0].x, y0 = psi[i0].y, x1 = psi[i1].x, y1 = psi[i1].y;
                    psi[i0].x = m0 * x0 - m1 * y0 + m2 * x1 - m3 * y1;
                    psi[i0].y = m0 * y0 + m1 * x0 + m2 * y1 + m3 * x1;
                    psi[i1].x = m4 * x0 - m5 * y0 + m6 * x1 - m7 * y1;
                    psi[i1].y = m4 * y0 + m5 * x0 + m6 * y1 + m7 * x1;
                }
                gsync();
                const int32_t code = pk[w][j];
                if (code & 3) { apply_pauli<R, G>(psi, half, code & 3, (code >> 2) & 63, t); gsync(); }
                if ((code >> 8) & 3) { apply_pauli<R, G>(psi, half, (code >> 8) & 3, (code >> 10) & 63, t); gsync(); }
            }
        }
        gsync();
        // ---- outcome: inverse CDF over |psi|^2 in a fixed order (contiguous segment per thread) ------------------
        const uint32_t per = (dim + G - 1) / G;
        const uint32_t s0 = min(dim, (uint32_t)t * per), s1 = min(dim, s0 + per);
        double acc = 0.0;
        for (uint32_t i = s0; i < s1; ++i) acc += (double)psi[i].x * (double)psi[i].x + (double)psi[i].y * (double)psi[i].y;
        part[w][t] = acc;
        gsync();
        if (t == 0 && live) {
            double total = 0.0;
            for (int k = 0; k < G; ++k) total += part[w][k];
            uint32_t idx = 0;
            if (!(total > 0.0) || !isfinite(total)) {
                a.status_out[c] = 1;
            } else {
                const double u = philox_uniform(a.seed, stream, s) * total;
                double run = 0.0, run_last = 0.0;
                int sel = -1, last = -1;
                for (int k = 0; k < G; ++k) {
                    const double pkk = part[w][k];
                    if (pkk > 0.0) {
                        last = k; run_last = run;
                        if (run + pkk > u) { sel = k; break; }
                    }
                    run += pkk;
                }
                if (sel < 0) { sel = last; run = run_last; }       // rounding pushed u past the total
                const uint32_t b0 = (uint32_t)sel * per, b1 = min(dim, b0 + per);
                int64_t hit = -1, nz = -1;                       // never return a zero-probability state
                for (uint32_t i = b0; i < b1; ++i) {
                    const double wi = (double)psi[i].x * (double)psi[i].x + (double)psi[i].y * (double)psi[i].y;
                    if (wi > 0.0) {
                        nz = i;
                        run += wi;
                        if (run > u) { hit = i; break; }
                    }
                }
                idx = (uint32_t)(hit >= 0 ? hit : nz);
            }
            const int ncl = a.n_clbits[c];
            uint64_t key = idx;
            if (ncl > 0) {
                const int32_t *cq = a.clbit_qubit + 64 * c;
                key = 0;
                for (int b = 0; b < ncl; ++b)
                    if (cq[b] >= 0) key |= (uint64_t)((idx >> cq[b]) & 1u) << b;
                if (a.readout) key = readout_flip(key, a.readout + 128 * c, ncl, a.seed, stream, s);
            }
            a.keys_out[(uint64_t)c * a.shots + s] = key;
        }
    }
}

thread_local std::string g_noise_error;

bool bad_prob(double p) { return !(p >= 0.0 && p <= 1.0); }

}  // namespace

namespace qcm {

cudaError_t launch_readout_keys(cudaStream_t st, int n_circuits, uint64_t shots, uint64_t seed, const uint64_t *stream_ids,
                                const int32_t *n_clbits, const double *readout, uint64_t *keys) {
    const uint64_t n = (uint64_t)n_circuits * shots;
    const unsigned blocks = (unsigned)std::min<uint64_t>((n + kThreads - 1) / kThreads, 1u << 16);
    k_readout_keys<<<std::max(1u, blocks), kThreads, 0, st>>>(n_circuits, shots, seed, stream_ids, n_clbits, readout, keys);
    return cudaGetLastError();
}

}  // namespace qcm

extern "C" {

int qcm_run_noisy_small(int device, int precision, int n_circuits, const int32_t *n_qubits, const int64_t *gate_begin,
                        const qcm_gate *gates, const qcm_channel *channels, int n_channels, const int32_t *clbit_qubit,
                        const int32_t *n_clbits, const double *readout, const uint64_t *stream_ids, uint64_t shots,
                        uint64_t seed, uint64_t *keys_out, double *device_ms_out) {
    if (n_circuits <= 0 || !n_qubits || !gate_begin || n_channels < 0 || (n_channels && !channels)) return QCM_ERR_INVALID;
    if (precision != QCM_C64 && precision != QCM_C128) return QCM_ERR_INVALID;
    if (shots && (!keys_out || !clbit_qubit || !n_clbits)) return QCM_ERR_INVALID;
    if (gate_begin[0] != 0) return QCM_ERR_INVALID;
    for (int c = 0; c < n_circuits; ++c) {
        if (n_qubits[c] < 0) return QCM_ERR_INVALID;
        if (n_qubits[c] > kSmallMaxQubits) return QCM_ERR_UNSUPPORTED;
        if (gate_begin[c + 1] < gate_begin[c]) return QCM_ERR_INVALID;
    }
    const int64_t n_gates = gate_begin[n_circuits];
    if (n_gates && !gates) return QCM_ERR_INVALID;
    for (int k = 0; k < n_channels; ++k) {
        const qcm_channel &ch = channels[k];
        if (ch.n_paulis != 4 && ch.n_paulis != 16) return QCM_ERR_INVALID;
        if (ch.qubit[0] < 0 || (ch.n_paulis == 4 ? ch.qubit[1] != -1 : (ch.qubit[1] < 0 || ch.qubit[1] == ch.qubit[0])))
            return QCM_ERR_INVALID;
        double prev = 0.0;
        for (int j = 0; j < ch.n_paulis; ++j) {
            if (!(ch.cum[j] >= prev)) return QCM_ERR_INVALID;
            prev = ch.cum[j];
        }
        if (ch.cum[ch.n_paulis - 1] != 1.0) return QCM_ERR_INVALID;
    }
    int maxq_warp = -1, maxq_cta = -1;
    std::vector<int32_t> circ_warp, circ_cta;
    for (int c = 0; c < n_circuits; ++c) {
        const int N = n_qubits[c];
        const uint32_t full = (1u << N) - 1u;
        for (int64_t i = gate_begin[c]; i < gate_begin[c + 1]; ++i) {
            const qcm_gate &g = gates[i];
            if (g.target < 0 || g.target >= N || (g.ctrl_mask & ~full) || ((g.ctrl_mask >> g.target) & 1u) ||
                (g.ctrl_value & ~g.ctrl_mask) || g.channel < -1 || g.channel >= n_channels)
                return QCM_ERR_INVALID;
            for (int k = 0; k < 8; ++k)
                if (!std::isfinite(g.m[k])) return QCM_ERR_INVALID;
            if (g.channel >= 0) {
                const qcm_channel &ch = channels[g.channel];
                if (ch.qubit[0] >= N || ch.qubit[1] >= N) return QCM_ERR_INVALID;
            }
        }
        if (shots) {
            if (n_clbits[c] < 0 || n_clbits[c] > 64) return QCM_ERR_INVALID;
            for (int b = 0; b < n_clbits[c]; ++b) {
                if (clbit_qubit[64 * c + b] < -1 || clbit_qubit[64 * c + b] >= N) return QCM_ERR_INVALID;
                if (readout && (bad_prob(readout[128 * c + 2 * b]) || bad_prob(readout[128 * c + 2 * b + 1])))
                    return QCM_ERR_INVALID;
            }
        }
        if (N <= kWarpMaxQubits) { circ_warp.push_back(c); maxq_warp = std::max(maxq_warp, N); }
        else { circ_cta.push_back(c); maxq_cta = std::max(maxq_cta, N); }
    }
    if (!shots) {
        if (device_ms_out) *device_ms_out = 0.0;
        return QCM_OK;
    }
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return QCM_ERR_NO_DEVICE;
    if (device < 0 || device >= ndev || device >= 64) return QCM_ERR_INVALID;
#define NZ_CUDA(call)                                                                  \
    do {                                                                                \
        cudaError_t e_ = (call);                                                        \
        if (e_ != cudaSuccess) {                                                        \
            g_noise_error = std::string(#call) + ": " + cudaGetErrorString(e_);         \
            rc = (e_ == cudaErrorMemoryAllocation) ? QCM_ERR_NOMEM : QCM_ERR_CUDA;      \
            goto done;                                                                  \
        }                                                                               \
    } while (0)
    int rc = QCM_OK;
    TrajArgs a{};
    SmallArena &A = g_arena[device];
    std::lock_guard<std::mutex> lock(A.mu);
    std::vector<int32_t> status(n_circuits, 0);
    const size_t amp = precision == QCM_C64 ? 8 : 16;
    const size_t nc = (size_t)n_circuits;
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += up256(std::max<size_t>(bytes, 1)); return o; };
    const size_t o_nq = take(nc * 4), o_gb = take((nc + 1) * 8), o_g = take((size_t)n_gates * sizeof(qcm_gate)),
                 o_ch = take((size_t)n_channels * sizeof(qcm_channel)), o_cq = take(64 * nc * 4), o_ncl = take(nc * 4),
                 o_ro = take(readout ? nc * 128 * 8 : 0), o_sid = take(stream_ids ? nc * 8 : 0),
                 o_cw = take(circ_warp.size() * 4), o_cc = take(circ_cta.size() * 4);
    const size_t in_bytes = off;
    const size_t o_keys = take(shots * nc * 8), o_status = take(nc * 4);
    char *hp, *dp;
    NZ_CUDA(cudaSetDevice(device));
    NZ_CUDA(arena_reserve(A, off, in_bytes));
    hp = (char *)A.pin;
    dp = (char *)A.dev;
    memcpy(hp + o_nq, n_qubits, nc * 4);
    memcpy(hp + o_gb, gate_begin, (nc + 1) * 8);
    if (n_gates) memcpy(hp + o_g, gates, (size_t)n_gates * sizeof(qcm_gate));
    if (n_channels) memcpy(hp + o_ch, channels, (size_t)n_channels * sizeof(qcm_channel));
    memcpy(hp + o_cq, clbit_qubit, 64 * nc * 4);
    memcpy(hp + o_ncl, n_clbits, nc * 4);
    if (readout) memcpy(hp + o_ro, readout, nc * 128 * 8);
    if (stream_ids) memcpy(hp + o_sid, stream_ids, nc * 8);
    if (!circ_warp.empty()) memcpy(hp + o_cw, circ_warp.data(), circ_warp.size() * 4);
    if (!circ_cta.empty()) memcpy(hp + o_cc, circ_cta.data(), circ_cta.size() * 4);
    NZ_CUDA(cudaMemcpyAsync(dp, hp, in_bytes, cudaMemcpyHostToDevice, A.st));
    NZ_CUDA(cudaMemsetAsync(dp + o_status, 0, nc * 4, A.st));
    a.n_qubits = (const int32_t *)(dp + o_nq);
    a.gate_begin = (const int64_t *)(dp + o_gb);
    a.gates = (const qcm_gate *)(dp + o_g);
    a.channels = (const qcm_channel *)(dp + o_ch);
    a.clbit_qubit = (const int32_t *)(dp + o_cq);
    a.n_clbits = (const int32_t *)(dp + o_ncl);
    a.readout = readout ? (const double *)(dp + o_ro) : nullptr;
    a.stream_ids = stream_ids ? (const uint64_t *)(dp + o_sid) : nullptr;
    a.shots = shots;
    a.seed = seed;
    a.keys_out = (uint64_t *)(dp + o_keys);
    a.status_out = (int32_t *)(dp + o_status);
    NZ_CUDA(cudaEventRecord(A.e0, A.st));
    for (int mode = 0; mode < 2; ++mode) {
        const std::vector<int32_t> &list = mode ? circ_cta : circ_warp;
        if (list.empty()) continue;
        const int W = mode ? 1 : kTrajWarps;
        const size_t smem = (size_t)W * (amp << (mode ? maxq_cta : maxq_warp));
        const uint64_t groups = (shots + W - 1) / W;
        const unsigned gx = (unsigned)std::min<uint64_t>(groups, 1u << 20);
        for (size_t first = 0; first < list.size(); first += 65535) {
            TrajArgs b = a;
            b.circ = (const int32_t *)(dp + (mode ? o_cc : o_cw)) + first;
            const dim3 grid(gx, (unsigned)std::min<size_t>(65535, list.size() - first));
            if (mode == 0 && precision == QCM_C64) {
                NZ_CUDA(cudaFuncSetAttribute(k_traj<float, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                k_traj<float, false><<<grid, 32 * kTrajWarps, smem, A.st>>>(b);
            } else if (mode == 0) {
                NZ_CUDA(cudaFuncSetAttribute(k_traj<double, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                k_traj<double, false><<<grid, 32 * kTrajWarps, smem, A.st>>>(b);
            } else if (precision == QCM_C64) {
                NZ_CUDA(cudaFuncSetAttribute(k_traj<float, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                k_traj<float, true><<<grid, kThreads, smem, A.st>>>(b);
            } else {
                NZ_CUDA(cudaFuncSetAttribute(k_traj<double, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                k_traj<double, true><<<grid, kThreads, smem, A.st>>>(b);
            }
            NZ_CUDA(cudaGetLastError());
        }
    }
    NZ_CUDA(cudaEventRecord(A.e1, A.st));
    NZ_CUDA(cudaMemcpyAsync(status.data(), dp + o_status, nc * 4, cudaMemcpyDeviceToHost, A.st));
    NZ_CUDA(cudaMemcpyAsync(keys_out, dp + o_keys, shots * nc * 8, cudaMemcpyDeviceToHost, A.st));
    NZ_CUDA(cudaStreamSynchronize(A.st));
    if (device_ms_out) {
        float ms = 0.f;
        NZ_CUDA(cudaEventElapsedTime(&ms, A.e0, A.e1));
        *device_ms_out = ms;
    }
    for (int c = 0; c < n_circuits; ++c)
        if (status[c]) { g_noise_error = "circuit " + std::to_string(c) + ": a trajectory's norm is not finite and positive"; rc = QCM_ERR_INVALID; }
done:
    return rc;
#undef NZ_CUDA
}

}  // extern "C"
