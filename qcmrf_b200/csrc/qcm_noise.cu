// Noisy shots of small circuits: every shot is a trajectory -- the unfused gate list with Pauli errors drawn after
// the gates that carry a channel -- simulated in shared memory, then measured once and read out through per-clbit
// assignment errors.  Fusion cannot apply: every shot runs a different circuit.
//
// k_traj<R, CTA, KRAUS>: grid (trajectory groups, circuits).  Up to kWarpMaxQubits qubits one warp runs one
// trajectory (2^10 amplitudes: 8 KiB complex64, 16 KiB complex128) and a gate needs only __syncwarp; above that a CTA
// runs one trajectory.  The CTA's trajectories share the gate stream, staged cooperatively kChunk gates at a time in
// shared memory together with each trajectory's error draws for those gates.  A Pauli is an index permutation and a
// phase, never a 2x2 product; a 2-qubit Pauli is two 1-qubit ones.
//
// KRAUS = false (qcm_run_noisy_small): a gate's error is one Pauli channel, drawn as a packed Pauli code.  KRAUS =
// true (qcm_run_noisy_small_kraus): a gate's error is up to kMaxStages stages, each a Pauli channel or a 1-qubit
// Kraus channel.  Every stage's uniform is state-independent, so it is still drawn ahead of the apply loop by one
// lane per staged gate; a Pauli stage is resolved to its code right there.  A Kraus stage needs the state: the
// trajectory reduces the stage qubit's 1-qubit density matrix in fp64 (an xor butterfly per warp, so every lane
// holds bit-identical sums; in CTA mode the 8 warp partials then add in a fixed order through shared memory),
// picks K_i with probability tr(K_i^dagger K_i rho_q) and applies K_i / sqrt(p_i) as an uncontrolled 2x2.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstring>
#include <mutex>
#include <string>
#include <type_traits>
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
constexpr uint64_t kKrausKey = 0x85EBCA77C2B2AE63ull;     // the stage draws of qcm_run_noisy_small_kraus
constexpr int kMaxStages = 4;                            // stages of one gate error (qcm_gate_error)

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

// KRAUS mode's arguments.  A struct of its own: the Pauli-only kernels keep their parameter block, and with it
// their code, instruction for instruction.
struct KrausTrajArgs : TrajArgs {
    const qcm_gate_error *errors; // qcm_gate.channel indexes these
    const qcm_kraus *krauses;
};

// KRAUS mode, in dynamic shared memory after the W states: per staged gate its stages' Kraus records (-1: a Pauli
// stage) and, per trajectory, staged gate and stage, the draw: a packed Pauli code or the Kraus stage's uniform.
struct StagedError {
    int32_t n;
    int32_t kraus[kMaxStages];
};
union StageDraw {
    double u;
    int32_t code;
};

// Packed code of the Pauli channel C for uniform u: code & 3 on qubit (code >> 2) & 63, (code >> 8) & 3 on qubit
// (code >> 10) & 63; 0 = identity.
__device__ __forceinline__ int32_t pauli_code(const qcm_channel &C, double u) {
    int32_t code = 0;
    if (!(u < C.cum[0])) {
        int k = 1;
        while (k < C.n_paulis - 1 && !(u < C.cum[k])) ++k;
        code = (k & 3) | (C.qubit[0] << 2) | (((k >> 2) & 3) << 8) | ((C.qubit[1] & 63) << 10);
    }
    return code;
}

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

// Kraus stage K on the trajectory psi (G threads, thread t; `red`: 4 doubles per warp of shared memory in CTA mode).
// Returns false, with psi unchanged, when sum_i p_i is not finite and positive.  Every thread takes the same branch
// and the same operator: the fp64 sums are bit-identical on all threads.
template <typename R, bool CTA>
__device__ __forceinline__ bool apply_kraus(Amp<R> *psi, uint32_t half, const qcm_kraus &K, double u, int t, double *red) {
    constexpr int G = CTA ? kThreads : 32;
    const int q = K.qubit;
    double r00 = 0.0, r11 = 0.0, rx = 0.0, ry = 0.0;        // rho_00, rho_11, rho_10 = sum a1 conj(a0)
#pragma unroll 1
    for (uint32_t p = t; p < half; p += G) {
        const uint32_t i0 = (uint32_t)insert_zero(p, q), i1 = i0 | (1u << q);
        const double x0 = psi[i0].x, y0 = psi[i0].y, x1 = psi[i1].x, y1 = psi[i1].y;
        r00 += x0 * x0 + y0 * y0;
        r11 += x1 * x1 + y1 * y1;
        rx += x1 * x0 + y1 * y0;
        ry += y1 * x0 - x1 * y0;
    }
#pragma unroll
    for (int m = 16; m; m >>= 1) {
        r00 += __shfl_xor_sync(0xffffffffu, r00, m);
        r11 += __shfl_xor_sync(0xffffffffu, r11, m);
        rx += __shfl_xor_sync(0xffffffffu, rx, m);
        ry += __shfl_xor_sync(0xffffffffu, ry, m);
    }
    if constexpr (CTA) {
        if ((t & 31) == 0) {
            double *r = red + 4 * (t >> 5);
            r[0] = r00; r[1] = r11; r[2] = rx; r[3] = ry;
        }
        __syncthreads();
        r00 = r11 = rx = ry = 0.0;
#pragma unroll
        for (int k = 0; k < G / 32; ++k) {
            r00 += red[4 * k]; r11 += red[4 * k + 1]; rx += red[4 * k + 2]; ry += red[4 * k + 3];
        }
    }
    // p_i = tr(K_i^dagger K_i rho) = M00 rho_00 + M11 rho_11 + 2 Re(M01 rho_10), M = K_i^dagger K_i
    double pr[kMaxStages], tot = 0.0;
#pragma unroll
    for (int i = 0; i < 4; ++i) {
        pr[i] = 0.0;
        if (i < K.n_ops) {
            const double *k = K.k[i];
            const double m00 = k[0] * k[0] + k[1] * k[1] + k[4] * k[4] + k[5] * k[5];
            const double m11 = k[2] * k[2] + k[3] * k[3] + k[6] * k[6] + k[7] * k[7];
            const double mx = k[0] * k[2] + k[1] * k[3] + k[4] * k[6] + k[5] * k[7];      // conj(k0) k1 + conj(k2) k3
            const double my = k[0] * k[3] - k[1] * k[2] + k[4] * k[7] - k[5] * k[6];
            const double p = m00 * r00 + m11 * r11 + 2.0 * (mx * rx - my * ry);
            pr[i] = p > 0.0 ? p : 0.0;                           // rounding below an exact 0: never chosen
        }
        tot += pr[i];
    }
    if (!(tot > 0.0) || !isfinite(tot)) return false;
    const double x = u * tot;
    double run = 0.0, psel = 0.0;
    int sel = 0;
    bool hit = false;                // until an operator is hit, sel is the last one with p > 0: it catches rounding
#pragma unroll                       // that pushed x past the total
    for (int i = 0; i < 4; ++i) {
        if (!hit && pr[i] > 0.0) {
            sel = i;
            psel = pr[i];
            hit = run + pr[i] > x;
            run += pr[i];
        }
    }
    const double sc = 1.0 / sqrt(psel);
    const double *k = K.k[sel];
    const R m0 = (R)(k[0] * sc), m1 = (R)(k[1] * sc), m2 = (R)(k[2] * sc), m3 = (R)(k[3] * sc), m4 = (R)(k[4] * sc),
            m5 = (R)(k[5] * sc), m6 = (R)(k[6] * sc), m7 = (R)(k[7] * sc);
#pragma unroll 1
    for (uint32_t p = t; p < half; p += G) {
        const uint32_t i0 = (uint32_t)insert_zero(p, q), i1 = i0 | (1u << q);
        const R x0 = psi[i0].x, y0 = psi[i0].y, x1 = psi[i1].x, y1 = psi[i1].y;
        psi[i0].x = m0 * x0 - m1 * y0 + m2 * x1 - m3 * y1;
        psi[i0].y = m0 * y0 + m1 * x0 + m2 * y1 + m3 * x1;
        psi[i1].x = m4 * x0 - m5 * y0 + m6 * x1 - m7 * y1;
        psi[i1].y = m4 * y0 + m5 * x0 + m6 * y1 + m7 * x1;
    }
    return true;
}

template <typename R, bool CTA, bool KRAUS>
__global__ void __launch_bounds__(CTA ? kThreads : 32 * kTrajWarps) k_traj(const std::conditional_t<KRAUS, KrausTrajArgs, TrajArgs> a) {
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
    // KRAUS: sd[w * kChunk + j][st], se[j] after the W states of this circuit's size
    StageDraw(*sd)[kMaxStages] = reinterpret_cast<StageDraw(*)[kMaxStages]>(smem_raw + (size_t)W * dim * sizeof(Amp<R>));
    StagedError *se = reinterpret_cast<StagedError *>(sd + W * kChunk);

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
                if constexpr (KRAUS) {
                    const int e = g.channel;
                    const int n = e >= 0 ? a.errors[e].n_stages : 0;
                    se[i].n = n;
#pragma unroll
                    for (int j = 0; j < kMaxStages; ++j)
                        se[i].kraus[j] = (j < n && a.errors[e].kind[j] == 1) ? a.errors[e].index[j] : -1;
                }
            }
            if constexpr (KRAUS) {
                if (t < cn) {                        // lane t draws the stages of gate cb + t for this trajectory
                    const int e = gates[cb + t].channel;
                    if (live && e >= 0) {
                        const qcm_gate_error &E = a.errors[e];
                        const uint64_t ctr = (s * (uint64_t)ng + (uint64_t)(cb + t)) * (uint64_t)kMaxStages;
                        for (int j = 0; j < E.n_stages; ++j) {
                            const double u = philox_uniform(a.seed ^ kKrausKey, stream, ctr + (uint64_t)j);
                            if (E.kind[j] == 0) sd[w * kChunk + t][j].code = pauli_code(a.channels[E.index[j]], u);
                            else sd[w * kChunk + t][j].u = u;
                        }
                    }
                }
            } else if (t < cn) {                     // lane t draws gate cb + t's error for this trajectory
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
                if constexpr (KRAUS) {
                    for (int st = 0; st < se[j].n; ++st) {
                        const int kr = se[j].kraus[st];
                        if (kr < 0) {
                            const int32_t code = sd[w * kChunk + j][st].code;
                            if (code & 3) { apply_pauli<R, G>(psi, half, code & 3, (code >> 2) & 63, t); gsync(); }
                            if ((code >> 8) & 3) { apply_pauli<R, G>(psi, half, (code >> 8) & 3, (code >> 10) & 63, t); gsync(); }
                        } else {
                            if (!apply_kraus<R, CTA>(psi, half, a.krauses[kr], sd[w * kChunk + j][st].u, t, part[0]) && t == 0)
                                a.status_out[c] = 1;
                            gsync();
                        }
                    }
                } else {
                    const int32_t code = pk[w][j];
                    if (code & 3) { apply_pauli<R, G>(psi, half, code & 3, (code >> 2) & 63, t); gsync(); }
                    if ((code >> 8) & 3) { apply_pauli<R, G>(psi, half, (code >> 8) & 3, (code >> 10) & 63, t); gsync(); }
                }
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

namespace {

thread_local std::string g_noise_error;

bool bad_prob(double p) { return !(p >= 0.0 && p <= 1.0); }

bool bad_kraus(const qcm_kraus &K) {
    if (K.n_ops < 1 || K.n_ops > kMaxStages || K.qubit < 0) return true;
    double m00 = 0.0, m11 = 0.0, mx = 0.0, my = 0.0;                // sum_i K_i^dagger K_i
    for (int i = 0; i < K.n_ops; ++i) {
        const double *k = K.k[i];
        for (int j = 0; j < 8; ++j)
            if (!std::isfinite(k[j])) return true;
        m00 += k[0] * k[0] + k[1] * k[1] + k[4] * k[4] + k[5] * k[5];
        m11 += k[2] * k[2] + k[3] * k[3] + k[6] * k[6] + k[7] * k[7];
        mx += k[0] * k[2] + k[1] * k[3] + k[4] * k[6] + k[5] * k[7];
        my += k[0] * k[3] - k[1] * k[2] + k[4] * k[7] - k[5] * k[6];
    }
    return !(std::fabs(m00 - 1.0) <= 1e-10 && std::fabs(m11 - 1.0) <= 1e-10 && std::hypot(mx, my) <= 1e-10);
}

template <typename R, bool CTA, bool KRAUS>
cudaError_t launch_traj(const dim3 &grid, size_t smem, cudaStream_t st, const KrausTrajArgs &b) {
    const cudaError_t e = cudaFuncSetAttribute(k_traj<R, CTA, KRAUS>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem);
    if (e != cudaSuccess) return e;
    k_traj<R, CTA, KRAUS><<<grid, CTA ? kThreads : 32 * kTrajWarps, smem, st>>>(b);
    return cudaGetLastError();
}

template <bool CTA, bool KRAUS>
cudaError_t launch_traj(int precision, const dim3 &grid, size_t smem, cudaStream_t st, const KrausTrajArgs &b) {
    return precision == QCM_C64 ? launch_traj<float, CTA, KRAUS>(grid, smem, st, b)
                                : launch_traj<double, CTA, KRAUS>(grid, smem, st, b);
}

// Both entry points: validation (before any device query), the arena and the launches.  errors == nullptr: gate
// channels index `channels` (k_traj<R, CTA, false>); otherwise they index `errors` (k_traj<R, CTA, true>).
int run_noisy(int device, int precision, int n_circuits, const int32_t *n_qubits, const int64_t *gate_begin,
              const qcm_gate *gates, const qcm_gate_error *errors, int n_errors, const qcm_channel *channels,
              int n_channels, const qcm_kraus *krauses, int n_kraus, const int32_t *clbit_qubit, const int32_t *n_clbits,
              const double *readout, const uint64_t *stream_ids, uint64_t shots, uint64_t seed, uint64_t *keys_out,
              double *device_ms_out) {
    const bool kraus = errors != nullptr;
    const int n_records = kraus ? n_errors : n_channels;      // what qcm_gate.channel indexes
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
    if (kraus && (n_errors < 0 || n_kraus < 0 || (n_kraus && !krauses))) return QCM_ERR_INVALID;
    for (int k = 0; kraus && k < n_errors; ++k) {
        const qcm_gate_error &E = errors[k];
        if (E.n_stages < 1 || E.n_stages > kMaxStages) return QCM_ERR_INVALID;
        for (int j = 0; j < E.n_stages; ++j)
            if (E.kind[j] < 0 || E.kind[j] > 1 || E.index[j] < 0 || E.index[j] >= (E.kind[j] ? n_kraus : n_channels))
                return QCM_ERR_INVALID;
    }
    for (int k = 0; kraus && k < n_kraus; ++k)
        if (bad_kraus(krauses[k])) return QCM_ERR_INVALID;
    int maxq_warp = -1, maxq_cta = -1;
    std::vector<int32_t> circ_warp, circ_cta;
    for (int c = 0; c < n_circuits; ++c) {
        const int N = n_qubits[c];
        const uint32_t full = (1u << N) - 1u;
        for (int64_t i = gate_begin[c]; i < gate_begin[c + 1]; ++i) {
            const qcm_gate &g = gates[i];
            if (g.target < 0 || g.target >= N || (g.ctrl_mask & ~full) || ((g.ctrl_mask >> g.target) & 1u) ||
                (g.ctrl_value & ~g.ctrl_mask) || g.channel < -1 || g.channel >= n_records)
                return QCM_ERR_INVALID;
            for (int k = 0; k < 8; ++k)
                if (!std::isfinite(g.m[k])) return QCM_ERR_INVALID;
            if (g.channel >= 0 && !kraus) {
                const qcm_channel &ch = channels[g.channel];
                if (ch.qubit[0] >= N || ch.qubit[1] >= N) return QCM_ERR_INVALID;
            } else if (g.channel >= 0) {
                const qcm_gate_error &E = errors[g.channel];
                const uint32_t on = g.ctrl_mask | (1u << g.target);      // the gate's qubits
                for (int j = 0; j < E.n_stages; ++j) {
                    if (E.kind[j] == 0) {
                        const qcm_channel &ch = channels[E.index[j]];
                        if (ch.qubit[0] >= N || ch.qubit[1] >= N) return QCM_ERR_INVALID;
                    } else if (krauses[E.index[j]].qubit >= N || !((on >> krauses[E.index[j]].qubit) & 1u)) {
                        return QCM_ERR_INVALID;
                    }
                }
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
    KrausTrajArgs a{};
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
                 o_cw = take(circ_warp.size() * 4), o_cc = take(circ_cta.size() * 4),
                 o_err = take(kraus ? (size_t)n_errors * sizeof(qcm_gate_error) : 0),
                 o_kr = take(kraus ? (size_t)n_kraus * sizeof(qcm_kraus) : 0);
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
    if (kraus && n_errors) memcpy(hp + o_err, errors, (size_t)n_errors * sizeof(qcm_gate_error));
    if (kraus && n_kraus) memcpy(hp + o_kr, krauses, (size_t)n_kraus * sizeof(qcm_kraus));
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
    a.errors = kraus ? (const qcm_gate_error *)(dp + o_err) : nullptr;
    a.krauses = kraus ? (const qcm_kraus *)(dp + o_kr) : nullptr;
    NZ_CUDA(cudaEventRecord(A.e0, A.st));
    for (int mode = 0; mode < 2; ++mode) {
        const std::vector<int32_t> &list = mode ? circ_cta : circ_warp;
        if (list.empty()) continue;
        const int W = mode ? 1 : kTrajWarps;
        const size_t smem = (size_t)W * (amp << (mode ? maxq_cta : maxq_warp)) +
                            (kraus ? W * kChunk * sizeof(StageDraw[kMaxStages]) + kChunk * sizeof(StagedError) : 0);
        const uint64_t groups = (shots + W - 1) / W;
        const unsigned gx = (unsigned)std::min<uint64_t>(groups, 1u << 20);
        for (size_t first = 0; first < list.size(); first += 65535) {
            KrausTrajArgs b = a;
            b.circ = (const int32_t *)(dp + (mode ? o_cc : o_cw)) + first;
            const dim3 grid(gx, (unsigned)std::min<size_t>(65535, list.size() - first));
            if (mode == 0 && !kraus) NZ_CUDA((launch_traj<false, false>(precision, grid, smem, A.st, b)));
            else if (mode == 0) NZ_CUDA((launch_traj<false, true>(precision, grid, smem, A.st, b)));
            else if (!kraus) NZ_CUDA((launch_traj<true, false>(precision, grid, smem, A.st, b)));
            else NZ_CUDA((launch_traj<true, true>(precision, grid, smem, A.st, b)));
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

}  // namespace

extern "C" {

int qcm_run_noisy_small(int device, int precision, int n_circuits, const int32_t *n_qubits, const int64_t *gate_begin,
                        const qcm_gate *gates, const qcm_channel *channels, int n_channels, const int32_t *clbit_qubit,
                        const int32_t *n_clbits, const double *readout, const uint64_t *stream_ids, uint64_t shots,
                        uint64_t seed, uint64_t *keys_out, double *device_ms_out) {
    return run_noisy(device, precision, n_circuits, n_qubits, gate_begin, gates, nullptr, 0, channels, n_channels,
                     nullptr, 0, clbit_qubit, n_clbits, readout, stream_ids, shots, seed, keys_out, device_ms_out);
}

int qcm_run_noisy_small_kraus(int device, int precision, int n_circuits, const int32_t *n_qubits,
                              const int64_t *gate_begin, const qcm_gate *gates, const qcm_gate_error *errors,
                              int n_errors, const qcm_channel *channels, int n_channels, const qcm_kraus *krauses,
                              int n_kraus, const int32_t *clbit_qubit, const int32_t *n_clbits, const double *readout,
                              const uint64_t *stream_ids, uint64_t shots, uint64_t seed, uint64_t *keys_out,
                              double *device_ms_out) {
    if (!errors) return QCM_ERR_INVALID;
    return run_noisy(device, precision, n_circuits, n_qubits, gate_begin, gates, errors, n_errors, channels, n_channels,
                     krauses, n_kraus, clbit_qubit, n_clbits, readout, stream_ids, shots, seed, keys_out, device_ms_out);
}

}  // extern "C"
