// Device kernels of the qcmrf_b200 statevector engine (sm_100a).
//
// Everything here is HBM-bound amplitude streaming: 128-bit vector loads/stores,
// coefficient tables staged in shared memory, enough independent loads in flight per
// thread to cover DRAM latency, grids sized as a multiple of the SM count.  There is
// no GEMM-shaped work on this path, so no tensor-core code (DESIGN.md, "Kernels").
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>

#include <type_traits>

#include "qcmrf_b200.h"

namespace qcm {

constexpr int kThreads = 256;

// Batch axis (theta / beta sweeps over one graph, BASELINE config 3): a handle may hold `batch` states of
// 2^n_local amplitudes in ONE allocation, all running the same program with per-point coefficient tables.
// Every kernel then runs with the sweep point as blockIdx.y: state, tables and per-point outputs are offset by
// blockIdx.y times the strides in its argument block (all zero-cost for a plain handle: gridDim.y == 1).
template <typename T> __device__ __forceinline__ T *batch_ptr(T *p, uint64_t stride_bytes) {
    return reinterpret_cast<T *>(reinterpret_cast<unsigned char *>(const_cast<typename std::remove_const<T>::type *>(p)) +
                                 (uint64_t)blockIdx.y * stride_bytes);
}

__host__ __device__ __forceinline__ uint64_t insert_zero(uint64_t x, int pos) {
    const uint64_t lo = x & ((1ull << pos) - 1ull);
    return ((x >> pos) << (pos + 1)) | lo;
}

// ----------------------------------------------------------------------------------
// 128-bit (or 64-bit) amplitude vector IO.  V = complex numbers per vector.
// ----------------------------------------------------------------------------------
template <typename R, int V> struct VecIO;

template <> struct VecIO<float, 2> {
    using T = float4;
    static __device__ __forceinline__ void load(const void *st, uint64_t amp, float (&re)[2], float (&im)[2]) {
        const float4 t = __ldcs(reinterpret_cast<const float4 *>(st) + (amp >> 1));
        re[0] = t.x; im[0] = t.y; re[1] = t.z; im[1] = t.w;
    }
    static __device__ __forceinline__ void store(void *st, uint64_t amp, const float (&re)[2], const float (&im)[2]) {
        __stcs(reinterpret_cast<float4 *>(st) + (amp >> 1), make_float4(re[0], im[0], re[1], im[1]));
    }
    static __device__ __forceinline__ void load_nc(const void *st, uint64_t amp, float (&re)[2], float (&im)[2]) {
        const float4 t = __ldg(reinterpret_cast<const float4 *>(st) + (amp >> 1));
        re[0] = t.x; im[0] = t.y; re[1] = t.z; im[1] = t.w;
    }
};
template <> struct VecIO<float, 1> {
    using T = float2;
    static __device__ __forceinline__ void load(const void *st, uint64_t amp, float (&re)[1], float (&im)[1]) {
        const float2 t = __ldcs(reinterpret_cast<const float2 *>(st) + amp);
        re[0] = t.x; im[0] = t.y;
    }
    static __device__ __forceinline__ void store(void *st, uint64_t amp, const float (&re)[1], const float (&im)[1]) {
        __stcs(reinterpret_cast<float2 *>(st) + amp, make_float2(re[0], im[0]));
    }
    static __device__ __forceinline__ void load_nc(const void *st, uint64_t amp, float (&re)[1], float (&im)[1]) {
        const float2 t = __ldg(reinterpret_cast<const float2 *>(st) + amp);
        re[0] = t.x; im[0] = t.y;
    }
};
template <> struct VecIO<double, 1> {
    using T = double2;
    static __device__ __forceinline__ void load(const void *st, uint64_t amp, double (&re)[1], double (&im)[1]) {
        const double2 t = __ldcs(reinterpret_cast<const double2 *>(st) + amp);
        re[0] = t.x; im[0] = t.y;
    }
    static __device__ __forceinline__ void store(void *st, uint64_t amp, const double (&re)[1], const double (&im)[1]) {
        __stcs(reinterpret_cast<double2 *>(st) + amp, make_double2(re[0], im[0]));
    }
    static __device__ __forceinline__ void load_nc(const void *st, uint64_t amp, double (&re)[1], double (&im)[1]) {
        const double2 t = __ldg(reinterpret_cast<const double2 *>(st) + amp);
        re[0] = t.x; im[0] = t.y;
    }
};

// ----------------------------------------------------------------------------------
// Blocked multiplexer pass.
//
// One sweep applies a list of uniformly-controlled single-qubit gates ("members")
// whose targets all lie in a set of M block qubits.  A thread owns, for one
// assignment of the non-block bits, the 2^M amplitudes (x V consecutive ones) that
// differ in the block bits: they sit in registers, every member is 2^(M-1)
// register-to-register butterflies with ONE table lookup, and each amplitude crosses
// HBM once per pass instead of once per gate.  M = 1 is the plain in-place gate pass.
//
// Lazy materialisation: block qubits >= n_in are known |0> on input; their upper
// halves are not read (zero registers) and butterflies on all-zero pairs are skipped
// (`nz` tracks which registers can be non-zero; it is uniform across the grid).
// ----------------------------------------------------------------------------------
struct MemberDesc {
    int8_t pos;                     // position of the member's target inside tq[]; -1: diagonal member
                                    // (amp *= table[idx], 2 reals per entry) applied to every register
    int8_t n_ctrl;
    int8_t ctrl[QCM_MAX_CTRL];      // qubit feeding table-index bit j (may be global)
    uint16_t low_bit;               // 1 << j for the j with ctrl[j] == 0, else 0
    int32_t tab_off;                // offset, in reals, of this member's table in shared memory
    int32_t src_off;                // offset, in reals, of the table in `tables` (global)
};

struct BlockArgs {
    void *state;
    const void *tables;             // device, already in the state's real type
    int32_t n_in, n_out;
    int32_t tq[QCM_MAX_BLOCK];      // block qubits, ascending
    int32_t n_members;
    int32_t ctrl_below_32;          // every index qubit of every member is below 32
    uint64_t rank_bits;             // rank << n_local
    uint64_t bstate, btab;          // batch strides in BYTES: state, tables (real type)
    MemberDesc mem[QCM_MAX_MEMBERS];
};

template <typename R, int V, int NR, int P, bool LAZY>
__device__ __forceinline__ void butterfly(R (&ar)[NR][V], R (&ai)[NR][V], const R (&m)[8], int v,
                                          uint32_t nz) {
    if constexpr ((1 << P) < NR) {
#pragma unroll
        for (int r = 0; r < NR; ++r) {
            if (r & (1 << P)) continue;
            const int r1 = r | (1 << P);
            if constexpr (LAZY)
                if (!(((nz >> r) | (nz >> r1)) & 1u)) continue;   // uniform branch
            const R x0 = ar[r][v], y0 = ai[r][v], x1 = ar[r1][v], y1 = ai[r1][v];
            ar[r][v] = m[0] * x0 - m[1] * y0 + m[2] * x1 - m[3] * y1;
            ai[r][v] = m[0] * y0 + m[1] * x0 + m[2] * y1 + m[3] * x1;
            ar[r1][v] = m[4] * x0 - m[5] * y0 + m[6] * x1 - m[7] * y1;
            ai[r1][v] = m[4] * y0 + m[5] * x0 + m[6] * y1 + m[7] * x1;
        }
    }
}

template <typename R>
__device__ __forceinline__ void load_m8(const R *p, R (&m)[8]) {
    if constexpr (sizeof(R) == 4) {
        const float4 m0 = *reinterpret_cast<const float4 *>(p);
        const float4 m1 = *reinterpret_cast<const float4 *>(p + 4);
        m[0] = m0.x; m[1] = m0.y; m[2] = m0.z; m[3] = m0.w;
        m[4] = m1.x; m[5] = m1.y; m[6] = m1.z; m[7] = m1.w;
    } else {
#pragma unroll
        for (int q = 0; q < 4; ++q) {
            const double2 t = *reinterpret_cast<const double2 *>(p + 2 * q);
            m[2 * q] = t.x; m[2 * q + 1] = t.y;
        }
    }
}

// LAZY = false: every block qubit is materialised on input (n_in == n_out): no zero tracking.
template <typename R, int V, int M, int U, bool LAZY>
__global__ void __launch_bounds__(kThreads) k_block(const __grid_constant__ BlockArgs a) {
    constexpr int NR = 1 << M;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    R *tab = reinterpret_cast<R *>(smem_raw);
    void *const state = batch_ptr(a.state, a.bstate);
    for (int g = 0; g < a.n_members; ++g) {
        const R *src = reinterpret_cast<const R *>(batch_ptr(a.tables, a.btab)) + a.mem[g].src_off;
        R *dst = tab + a.mem[g].tab_off;
        const int cnt = (a.mem[g].pos < 0 ? 2 : 8) << a.mem[g].n_ctrl;
        for (int i = threadIdx.x; i < cnt; i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    using IO = VecIO<R, V>;

    uint64_t toff[M];
    uint32_t zmask = 0;
#pragma unroll
    for (int j = 0; j < M; ++j) {
        toff[j] = 1ull << a.tq[j];
        if (LAZY && a.tq[j] >= a.n_in) zmask |= 1u << j;
    }
    uint32_t nz0 = 0;
#pragma unroll
    for (int r = 0; r < NR; ++r)
        if ((r & zmask) == 0) nz0 |= 1u << r;

    const uint64_t nvec = (1ull << (a.n_out - M)) / V;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x * U;
    for (uint64_t bv0 = (uint64_t)blockIdx.x * blockDim.x * U + threadIdx.x; bv0 < nvec; bv0 += stride) {
        R ar[U][NR][V], ai[U][NR][V];
        uint64_t base[U];
        bool ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t bv = bv0 + (uint64_t)u * blockDim.x;
            ok[u] = bv < nvec;
            uint64_t b = bv * V;
#pragma unroll
            for (int j = 0; j < M; ++j) b = insert_zero(b, a.tq[j]);
            base[u] = b;
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                if (ok[u] && (!LAZY || ((nz0 >> r) & 1u))) {
                    uint64_t off = b;
#pragma unroll
                    for (int j = 0; j < M; ++j)
                        if ((r >> j) & 1) off += toff[j];
                    IO::load(state, off, ar[u][r], ai[u][r]);
                } else {
#pragma unroll
                    for (int v = 0; v < V; ++v) { ar[u][r][v] = R(0); ai[u][r][v] = R(0); }
                }
            }
        }
        uint32_t nz = nz0;
        for (int g = 0; g < a.n_members; ++g) {
            const int pos = a.mem[g].pos;
            const int nc = a.mem[g].n_ctrl;
            const R *mt = tab + a.mem[g].tab_off;
            const uint32_t low_bit = a.mem[g].low_bit;      // table-index bit fed by qubit 0 (V == 2 only)
#pragma unroll
            for (int u = 0; u < U; ++u) {
                // table index of the vector's first amplitude; its second one differs in qubit 0 only
                const uint64_t gi = base[u] | a.rank_bits;
                uint32_t idx0 = 0;
                if (a.ctrl_below_32) {
                    const uint32_t lo = (uint32_t)gi;
                    for (int j = 0; j < nc; ++j) idx0 |= ((lo >> a.mem[g].ctrl[j]) & 1u) << j;
                } else {
                    for (int j = 0; j < nc; ++j) idx0 |= (uint32_t)((gi >> a.mem[g].ctrl[j]) & 1ull) << j;
                }
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    const uint32_t idx = v ? (idx0 | low_bit) : idx0;
                    if (pos < 0) {                                  // diagonal member
                        const R c = mt[2 * idx], sn = mt[2 * idx + 1];
#pragma unroll
                        for (int r = 0; r < NR; ++r) {
                            const R x = ar[u][r][v], y = ai[u][r][v];
                            ar[u][r][v] = c * x - sn * y;
                            ai[u][r][v] = c * y + sn * x;
                        }
                        continue;
                    }
                    R m[8];
                    load_m8<R>(mt + 8 * idx, m);
                    switch (pos) {
                        case 0: butterfly<R, V, NR, 0, LAZY>(ar[u], ai[u], m, v, nz); break;
                        case 1: butterfly<R, V, NR, 1, LAZY>(ar[u], ai[u], m, v, nz); break;
                        case 2: butterfly<R, V, NR, 2, LAZY>(ar[u], ai[u], m, v, nz); break;
                        case 3: butterfly<R, V, NR, 3, LAZY>(ar[u], ai[u], m, v, nz); break;
                        default: butterfly<R, V, NR, 4, LAZY>(ar[u], ai[u], m, v, nz); break;
                    }
                }
            }
            if (LAZY && pos >= 0) {
                // registers that can be non-zero after a butterfly on bit `pos`
                const uint32_t sh = 1u << pos;
                uint32_t lowsel = 0;
#pragma unroll
                for (int r = 0; r < NR; ++r)
                    if (!(r & sh)) lowsel |= 1u << r;
                nz = nz | ((nz & lowsel) << sh) | ((nz & ~lowsel) >> sh);
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (!ok[u]) continue;
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                uint64_t off = base[u];
#pragma unroll
                for (int j = 0; j < M; ++j)
                    if ((r >> j) & 1) off += toff[j];
                IO::store(state, off, ar[u][r], ai[u][r]);
            }
        }
    }
}

// ----------------------------------------------------------------------------------
// Low-order-target pass (north star (ii); SURVEY.md 2, K4).
//
// k_block pairs amplitudes 2^t apart with one 128-bit access per lane: for a target below the
// width of a warp's access (t = 0: 64-bit loads; t = 1..4: 16-byte pieces at a 2^(t+4)-byte stride)
// the pairs of a butterfly sit INSIDE the vectors and lanes of one coalesced warp access.  Here a
// warp owns a contiguous row of 2^LB amplitudes (LB = log2(V * 32 * 2^UB): 512 complex64 = 4 KiB)
// and every lane holds 2^UB vectors of it, each load/store a full 512-byte warp access:
//     row bit 0          (V == 2)  the two amplitudes of a lane's 128-bit vector   -> in registers
//     row bits VB..VB+4            the lane                                        -> __shfl_xor_sync
//     row bits VB+5..LB-1          the lane's 2^UB vectors                         -> in registers
// so a gate on ANY of the LB low qubits is a butterfly on data the warp already holds: no strided
// access, no shared-memory staging of amplitudes (shared memory only holds the coefficient tables).
// Up to two further targets above the row (MH of them; UB shrinks to keep 32 data registers) ride
// along as a register dimension, their row copies 2^th amplitudes apart, so a blocked pass that mixes
// low and high targets stays one sweep.  Members are applied in order, as in k_block.
// ----------------------------------------------------------------------------------
constexpr int kLowqMaxHigh = 2;
constexpr int kLowqRegBits = 4;             // register-index bits that can feed a table index (v + u bits)

struct LowqMember {
    int8_t pos;                     // target: row bit 0..LB-1; LB + k: high target k; -1: diagonal member
    int8_t n_ctrl;
    int8_t ctrl[QCM_MAX_CTRL];      // qubit feeding table-index bit j (any qubit but the pass's targets)
    uint16_t rbit[kLowqRegBits];    // table-index bit fed by register-index bit b (v, then the u bits), else 0
    uint16_t rany;                  // OR of rbit[]: 0 => one table entry serves all of a thread's registers
    int32_t tab_off, src_off;       // reals: shared-memory / global offsets of the member's table
};

struct LowqArgs {
    void *state;
    const void *tables;             // device, state's real type
    int32_t n;                      // materialised qubits (the pass is in place: n_in == n_out)
    int32_t n_members;
    int32_t th[kLowqMaxHigh];       // high targets, ascending (>= LB)
    uint64_t rank_bits;
    uint64_t bstate, btab;          // batch strides in bytes
    LowqMember mem[QCM_MAX_MEMBERS];
};

template <typename R, int V, int UB, int MH>
__global__ void __launch_bounds__(kThreads) k_lowq(const __grid_constant__ LowqArgs a) {
    constexpr int VB = V == 2 ? 1 : 0;
    constexpr int LB = VB + 5 + UB;             // row bits
    constexpr int NU = 1 << UB, NH = 1 << MH;
    constexpr int NR = V * NU * NH;             // amplitudes per thread; register index r = v | u << VB | h << (VB + UB)
    constexpr int kWarps = kThreads / 32;
    using IO = VecIO<R, V>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    R *tab = reinterpret_cast<R *>(smem_raw);
    void *const state = batch_ptr(a.state, a.bstate);
    for (int g = 0; g < a.n_members; ++g) {
        const R *src = reinterpret_cast<const R *>(batch_ptr(a.tables, a.btab)) + a.mem[g].src_off;
        R *dst = tab + a.mem[g].tab_off;
        const int cnt = (a.mem[g].pos < 0 ? 2 : 8) << a.mem[g].n_ctrl;
        for (int i = threadIdx.x; i < cnt; i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t nrows = 1ull << (a.n - LB - MH);
    // one row per warp, a CTA's 8 rows adjacent, CTAs in launch (= address) order
    for (uint64_t row = (uint64_t)blockIdx.x * kWarps + warp; row < nrows; row += (uint64_t)gridDim.x * kWarps) {
        uint64_t base = row << LB;
#pragma unroll
        for (int k = 0; k < MH; ++k) base = insert_zero(base, a.th[k]);
        R xr[NR], xi[NR];
#pragma unroll
        for (int h = 0; h < NH; ++h) {
            uint64_t hb = base;
#pragma unroll
            for (int k = 0; k < MH; ++k)
                if ((h >> k) & 1) hb += 1ull << a.th[k];
#pragma unroll
            for (int u = 0; u < NU; ++u) {
                R tr[V], ti[V];
                IO::load(state, hb + ((uint64_t)u * 32 + lane) * V, tr, ti);
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    xr[v | (u << VB) | (h << (VB + UB))] = tr[v];
                    xi[v | (u << VB) | (h << (VB + UB))] = ti[v];
                }
            }
        }
        // the part of the global index that is the same for all of this thread's registers
        const uint64_t gi = (base + (uint64_t)lane * V) | a.rank_bits;
        for (int g = 0; g < a.n_members; ++g) {
            const LowqMember &m = a.mem[g];
            const R *mt = tab + m.tab_off;
            uint32_t idx0 = 0;
            for (int j = 0; j < m.n_ctrl; ++j) idx0 |= (uint32_t)((gi >> m.ctrl[j]) & 1ull) << j;
            auto ridx = [&](int r) -> uint32_t {           // r is a compile-time constant after unrolling
                uint32_t i = idx0;
#pragma unroll
                for (int b = 0; b < VB + UB; ++b)
                    if ((r >> b) & 1) i |= m.rbit[b];
                return i;
            };
            const int pos = m.pos;
            // UNI: no register-index bit feeds the table index -> one entry serves all of the thread's registers
            auto apply = [&](auto UNIc) {
                constexpr bool UNI = decltype(UNIc)::value;
                if (pos < 0) {                              // diagonal member
                    R c0 = R(0), s0 = R(0);
                    if constexpr (UNI) { c0 = mt[2 * idx0]; s0 = mt[2 * idx0 + 1]; }
#pragma unroll
                    for (int r = 0; r < NR; ++r) {
                        R c = c0, sn = s0;
                        if constexpr (!UNI) { const uint32_t idx = ridx(r); c = mt[2 * idx]; sn = mt[2 * idx + 1]; }
                        const R x = xr[r], y = xi[r];
                        xr[r] = c * x - sn * y;
                        xi[r] = c * y + sn * x;
                    }
                    return;
                }
                R q[8];
                if constexpr (UNI) load_m8<R>(mt + 8 * idx0, q);
                if (pos >= VB && pos < VB + 5) {
                    // ---- target = a lane bit: the partner amplitude lives in lane ^ (1 << j)
                    const int j = pos - VB;
                    const bool up = (lane >> j) & 1;
#pragma unroll
                    for (int r = 0; r < NR; ++r) {
                        if constexpr (!UNI) load_m8<R>(mt + 8 * ridx(r), q);
                        // own coefficient / partner coefficient: row `up` of the 2x2
                        const R ar = up ? q[6] : q[0], ai = up ? q[7] : q[1];
                        const R br = up ? q[4] : q[2], bi = up ? q[5] : q[3];
                        const R pr = __shfl_xor_sync(0xffffffffu, xr[r], 1 << j);
                        const R pi = __shfl_xor_sync(0xffffffffu, xi[r], 1 << j);
                        const R x = xr[r], y = xi[r];
                        xr[r] = ar * x - ai * y + br * pr - bi * pi;
                        xi[r] = ar * y + ai * x + br * pi + bi * pr;
                    }
                    return;
                }
                // ---- target = a register bit (vector slot, one of the lane's vectors, or a high target)
                const int rb = pos < VB ? 0 : (pos < LB ? pos - 5 : VB + UB + (pos - LB));
                auto in_regs = [&](auto RBc) {
                    constexpr int RB = decltype(RBc)::value;
                    if constexpr (RB < VB + UB + MH) {
#pragma unroll
                        for (int r = 0; r < NR; ++r) {
                            if (r & (1 << RB)) continue;
                            const int r1 = r | (1 << RB);
                            if constexpr (!UNI) load_m8<R>(mt + 8 * ridx(r), q);
                            const R x0 = xr[r], y0 = xi[r], x1 = xr[r1], y1 = xi[r1];
                            xr[r] = q[0] * x0 - q[1] * y0 + q[2] * x1 - q[3] * y1;
                            xi[r] = q[0] * y0 + q[1] * x0 + q[2] * y1 + q[3] * x1;
                            xr[r1] = q[4] * x0 - q[5] * y0 + q[6] * x1 - q[7] * y1;
                            xi[r1] = q[4] * y0 + q[5] * x0 + q[6] * y1 + q[7] * x1;
                        }
                    }
                };
                switch (rb) {
                    case 0: in_regs(std::integral_constant<int, 0>{}); break;
                    case 1: in_regs(std::integral_constant<int, 1>{}); break;
                    case 2: in_regs(std::integral_constant<int, 2>{}); break;
                    default: in_regs(std::integral_constant<int, 3>{}); break;
                }
            };
            if (m.rany == 0) apply(std::true_type{});
            else apply(std::false_type{});
        }
#pragma unroll
        for (int h = 0; h < NH; ++h) {
            uint64_t hb = base;
#pragma unroll
            for (int k = 0; k < MH; ++k)
                if ((h >> k) & 1) hb += 1ull << a.th[k];
#pragma unroll
            for (int u = 0; u < NU; ++u) {
                R tr[V], ti[V];
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    tr[v] = xr[v | (u << VB) | (h << (VB + UB))];
                    ti[v] = xi[v | (u << VB) | (h << (VB + UB))];
                }
                IO::store(state, hb + ((uint64_t)u * 32 + lane) * V, tr, ti);
            }
        }
    }
}

// ----------------------------------------------------------------------------------
// Fused qubit-swap + gate pass over NVLink peer memory (sharded states).
//
// A qubit-swap all-to-all brings the s global qubits on-GPU as the s highest local qubits, and the
// sweeps that wanted them as targets follow.  Fused: for every rest-index i the 2^s amplitudes a
// blocked pass over those qubits needs are exactly  peer_r.state[(c_me << (n_local - s)) | i],
// r = 0 .. 2^s-1  (c_me: this rank's coordinate, peer_r: the rank with coordinate r; r == c_me is
// local).  The kernel loads its 2^s register vectors straight from the peers' shards (mapped
// through CUDA IPC, plain 128-bit loads over NVLink), applies the members in registers and
// stores to an out-of-place local buffer: one kernel instead of an all-to-all plus s passes, and
// the transfer overlaps the arithmetic tile by tile.  No flags, no spinning: the host brackets
// the launch with barriers (peers must have finished writing the state that is read here, and
// must have finished reading before the old buffer is reused).
// ----------------------------------------------------------------------------------
struct GatherArgs {
    const void *src[1 << QCM_MAX_GATHER];   // src[r]: peer r's slab c_me (device pointers, peer-mapped)
    void *dst;                              // local output state (2^n_local amplitudes)
    const void *tables;
    int32_t n_local, s;
    int32_t n_members;
    int32_t ctrl_below_32;
    uint64_t rank_bits;                     // NEW rank bits (after the swap), rank << n_local
    MemberDesc mem[QCM_MAX_MEMBERS];        // pos = index among the s swapped-in qubits
};

template <typename R, int V, int M, int U>
__global__ void __launch_bounds__(kThreads) k_block_gather(const __grid_constant__ GatherArgs a) {
    constexpr int NR = 1 << M;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    R *tab = reinterpret_cast<R *>(smem_raw);
    for (int g = 0; g < a.n_members; ++g) {
        const R *src = reinterpret_cast<const R *>(a.tables) + a.mem[g].src_off;
        R *dst = tab + a.mem[g].tab_off;
        const int cnt = (a.mem[g].pos < 0 ? 2 : 8) << a.mem[g].n_ctrl;
        for (int i = threadIdx.x; i < cnt; i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    using IO = VecIO<R, V>;
    const uint64_t slab = 1ull << (a.n_local - M);
    const uint64_t nvec = slab / V;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x * U;
    for (uint64_t bv0 = (uint64_t)blockIdx.x * blockDim.x * U + threadIdx.x; bv0 < nvec; bv0 += stride) {
        R ar[U][NR][V], ai[U][NR][V];
        bool ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t bv = bv0 + (uint64_t)u * blockDim.x;
            ok[u] = bv < nvec;
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                if (ok[u]) IO::load(a.src[r], bv * V, ar[u][r], ai[u][r]);
                else {
#pragma unroll
                    for (int v = 0; v < V; ++v) { ar[u][r][v] = R(0); ai[u][r][v] = R(0); }
                }
            }
        }
        for (int g = 0; g < a.n_members; ++g) {
            const int pos = a.mem[g].pos;
            const int nc = a.mem[g].n_ctrl;
            const R *mt = tab + a.mem[g].tab_off;
            const uint32_t low_bit = a.mem[g].low_bit;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint64_t gi = ((bv0 + (uint64_t)u * blockDim.x) * V) | a.rank_bits;
                uint32_t idx0 = 0;
                if (a.ctrl_below_32) {
                    const uint32_t lo = (uint32_t)gi;
                    for (int j = 0; j < nc; ++j) idx0 |= ((lo >> a.mem[g].ctrl[j]) & 1u) << j;
                } else {
                    for (int j = 0; j < nc; ++j) idx0 |= (uint32_t)((gi >> a.mem[g].ctrl[j]) & 1ull) << j;
                }
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    const uint32_t idx = v ? (idx0 | low_bit) : idx0;
                    if (pos < 0) {
                        const R c = mt[2 * idx], sn = mt[2 * idx + 1];
#pragma unroll
                        for (int r = 0; r < NR; ++r) {
                            const R x = ar[u][r][v], y = ai[u][r][v];
                            ar[u][r][v] = c * x - sn * y;
                            ai[u][r][v] = c * y + sn * x;
                        }
                        continue;
                    }
                    R m[8];
                    load_m8<R>(mt + 8 * idx, m);
                    switch (pos) {
                        case 0: butterfly<R, V, NR, 0, false>(ar[u], ai[u], m, v, 0u); break;
                        case 1: butterfly<R, V, NR, 1, false>(ar[u], ai[u], m, v, 0u); break;
                        default: butterfly<R, V, NR, 2, false>(ar[u], ai[u], m, v, 0u); break;
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (!ok[u]) continue;
            const uint64_t bv = bv0 + (uint64_t)u * blockDim.x;
#pragma unroll
            for (int r = 0; r < NR; ++r) IO::store(a.dst, (uint64_t)r * slab + bv * V, ar[u][r], ai[u][r]);
        }
    }
}

// ----------------------------------------------------------------------------------
// The same fused pass with the peers' slabs streamed by the TMA engine (cp.async.bulk) through a
// shared-memory ring: one producer thread keeps STAGES x 2^M bulk copies of kGatherTileBytes x U
// in flight per CTA (NVLink reads need far more bytes in flight than a few LDG.128 per thread),
// completion is counted on an mbarrier per stage (expect_tx), the 256 consumer threads take their
// 2^M register vectors from shared memory, apply the members, store to the local output buffer and
// release the stage (one arrive per warp).  A CTA handles K consecutive tiles, CTAs are
// launched in address order.
// ----------------------------------------------------------------------------------
constexpr int kGatherTileBytes = kThreads * 16;         // one 16-byte vector per consumer thread

__device__ __forceinline__ uint32_t smem_u32(const void *p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
    uint32_t done;
    do {
        asm volatile("{\n.reg .pred p;\nmbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\nselp.u32 %0, 1, 0, p;\n}"
                     : "=r"(done) : "r"(bar), "r"(parity) : "memory");
    } while (!done);
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes, uint32_t bar) {
    asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];"
                 ::"r"(dst), "l"(src), "r"(bytes), "r"(bar) : "memory");
}

template <typename R, int V, int M, int U, int STAGES>
__global__ void __launch_bounds__(kThreads + 32) k_block_gather_tma(const __grid_constant__ GatherArgs a, const int tiles_per_cta) {
    constexpr int NR = 1 << M;
    constexpr uint32_t kTile = kGatherTileBytes * U;             // bytes per source per stage
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw);     // full[STAGES], empty[STAGES]
    unsigned char *ring = smem_raw + 256;
    R *tab = reinterpret_cast<R *>(ring + (size_t)STAGES * NR * kTile);
    static_assert(2 * STAGES * 8 <= 256, "barrier block");
    for (int g = 0; g < a.n_members; ++g) {
        const R *src = reinterpret_cast<const R *>(a.tables) + a.mem[g].src_off;
        R *dst = tab + a.mem[g].tab_off;
        const int cnt = (a.mem[g].pos < 0 ? 2 : 8) << a.mem[g].n_ctrl;
        for (int i = threadIdx.x; i < cnt; i += blockDim.x) dst[i] = src[i];
    }
    if (threadIdx.x == 0) {
        for (int st = 0; st < STAGES; ++st) {
            mbar_init(smem_u32(bars + st), 1);                       // producer's arrive.expect_tx
            mbar_init(smem_u32(bars + STAGES + st), kThreads / 32);  // one arrive per consumer warp
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    const uint64_t slab = 1ull << (a.n_local - M);
    const uint64_t tile0 = (uint64_t)blockIdx.x * tiles_per_cta;     // tile = kThreads * U vectors of V amplitudes
    if (threadIdx.x >= kThreads) {
        if (threadIdx.x == kThreads) {
            for (int k = 0; k < tiles_per_cta; ++k) {
                const int st = k % STAGES;
                if (k >= STAGES) mbar_wait(smem_u32(bars + STAGES + st), ((k / STAGES) - 1) & 1);
                const uint32_t full = smem_u32(bars + st);
                mbar_expect_tx(full, NR * kTile);
#pragma unroll
                for (int r = 0; r < NR; ++r)
                    bulk_g2s(smem_u32(ring + ((size_t)st * NR + r) * kTile),
                             reinterpret_cast<const unsigned char *>(a.src[r]) + (tile0 + k) * kTile, kTile, full);
            }
        }
        return;
    }
    using IO = VecIO<R, V>;
    for (int k = 0; k < tiles_per_cta; ++k) {
        const int st = k % STAGES;
        mbar_wait(smem_u32(bars + st), (k / STAGES) & 1);
        R ar[U][NR][V], ai[U][NR][V];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                const unsigned char *sp = ring + ((size_t)st * NR + r) * kTile + ((size_t)u * kThreads + threadIdx.x) * 16;
                if constexpr (V == 2) {
                    const float4 t = *reinterpret_cast<const float4 *>(sp);
                    ar[u][r][0] = t.x; ai[u][r][0] = t.y; ar[u][r][1] = t.z; ai[u][r][1] = t.w;
                } else {
                    const double2 d = *reinterpret_cast<const double2 *>(sp);
                    ar[u][r][0] = d.x; ai[u][r][0] = d.y;
                }
            }
        const uint64_t bv0 = (tile0 + k) * ((uint64_t)kThreads * U) + threadIdx.x;   // vector index of u = 0
        for (int g = 0; g < a.n_members; ++g) {
            const int pos = a.mem[g].pos;
            const int nc = a.mem[g].n_ctrl;
            const R *mt = tab + a.mem[g].tab_off;
            const uint32_t low_bit = a.mem[g].low_bit;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint64_t gi = ((bv0 + (uint64_t)u * kThreads) * V) | a.rank_bits;
                uint32_t idx0 = 0;
                if (a.ctrl_below_32) {
                    const uint32_t lo = (uint32_t)gi;
                    for (int j = 0; j < nc; ++j) idx0 |= ((lo >> a.mem[g].ctrl[j]) & 1u) << j;
                } else {
                    for (int j = 0; j < nc; ++j) idx0 |= (uint32_t)((gi >> a.mem[g].ctrl[j]) & 1ull) << j;
                }
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    const uint32_t idx = v ? (idx0 | low_bit) : idx0;
                    if (pos < 0) {
                        const R c = mt[2 * idx], sn = mt[2 * idx + 1];
#pragma unroll
                        for (int r = 0; r < NR; ++r) {
                            const R x = ar[u][r][v], y = ai[u][r][v];
                            ar[u][r][v] = c * x - sn * y;
                            ai[u][r][v] = c * y + sn * x;
                        }
                        continue;
                    }
                    R m[8];
                    load_m8<R>(mt + 8 * idx, m);
                    switch (pos) {
                        case 0: butterfly<R, V, NR, 0, false>(ar[u], ai[u], m, v, 0u); break;
                        case 1: butterfly<R, V, NR, 1, false>(ar[u], ai[u], m, v, 0u); break;
                        default: butterfly<R, V, NR, 2, false>(ar[u], ai[u], m, v, 0u); break;
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int r = 0; r < NR; ++r)
                IO::store(a.dst, (uint64_t)r * slab + (bv0 + (uint64_t)u * kThreads) * V, ar[u][r], ai[u][r]);
        // Release the stage only here, after the stores: they depend on the shared-memory loads above, so
        // those have completed.  An arrive issued right behind the LDS can overtake them (LDS queue behind
        // this SM's global stores, SYNCS does not): the producer's next bulk copy then lands in the stage
        // while a warp is still reading it -- measured as rare 128-512 B stale chunks (tools/gather_check.py).
        __syncwarp();
        if ((threadIdx.x & 31) == 0) mbar_arrive(smem_u32(bars + STAGES + st));
    }
}

// ----------------------------------------------------------------------------------
// The fused qubit swap + gate pass IN PLACE: no second state buffer, so it also serves shards that fill the GPU
// (37 qubits on 8 GPUs: 128 GiB per rank).  Same data flow as k_block_gather_tma -- rank c reads slab c of every
// peer r and its own, applies the members, and writes the 2^s results over ITS OWN slabs r -- plus one flag per
// (tile, peer) that orders the two accesses to the same memory:
//     peer r reads  my.state[slab r][tile t]      (it needs it as its input)
//     I overwrite   my.state[slab r][tile t]      (with my output)
// Once my bulk copy of peer r's tile t has landed in shared memory a dedicated signalling warp stores `epoch` to peer
// r's flag [t][c] over NVLink -- as soon as the ring stage fills, i.e. up to STAGES-1 tiles before the consumers get to
// that tile; before the consumers overwrite my slab r of tile t they wait until MY flag [t][r] shows the epoch.  The
// stores are also delayed by one tile (results wait in registers), so the flag has had several tile times to arrive
// and the wait almost never spins.  Everybody reads before waiting and CTAs are
// dispatched in tile order on every rank, so there is no circular wait; a spin that exceeds `spin_limit` clocks
// gives up and raises *err (the host reports it) instead of hanging the GPU.
// ----------------------------------------------------------------------------------
struct GatherFlags {
    uint32_t *flags[1 << QCM_MAX_GATHER];   // flags[r]: rank (coordinate) r's array [tiles][2^s], peer-mapped; [c_me]: local
    uint32_t epoch;
    int32_t c_me;
    int32_t *err;
    long long spin_limit;
};

// The signal only says "my read of your tile has completed" (the data already sits in my shared memory, observed
// through the mbarrier): it orders nothing of mine, so a relaxed system-scope store is enough -- a release would fence
// this thread's own earlier global stores at system scope, microseconds per tile.
__device__ __forceinline__ void st_relaxed_sys(uint32_t *p, uint32_t v) {
    asm volatile("st.relaxed.sys.global.u32 [%0], %1;" ::"l"(p), "r"(v) : "memory");
}
__device__ __forceinline__ uint32_t ld_relaxed_sys(const uint32_t *p) {
    uint32_t v;
    asm volatile("ld.relaxed.sys.global.u32 %0, [%1];" : "=r"(v) : "l"(p) : "memory");
    return v;
}

template <typename R, int V, int M, int U, int STAGES>
__global__ void __launch_bounds__(kThreads + 96) k_block_gather_inplace(const __grid_constant__ GatherArgs a, const __grid_constant__ GatherFlags f,
                                                                        const int tiles_per_cta) {
    constexpr int NR = 1 << M;
    constexpr uint32_t kTile = kGatherTileBytes * U;             // bytes per source per stage
    extern __shared__ __align__(16) unsigned char smem_raw[];
    uint64_t *bars = reinterpret_cast<uint64_t *>(smem_raw);     // full[STAGES], empty[STAGES]
    volatile int *ready = reinterpret_cast<volatile int *>(smem_raw + 240);   // tiles whose peers have all signalled
    unsigned char *ring = smem_raw + 256;
    R *tab = reinterpret_cast<R *>(ring + (size_t)STAGES * NR * kTile);
    static_assert(2 * STAGES * 8 <= 240, "barrier block");
    for (int g = 0; g < a.n_members; ++g) {
        const R *src = reinterpret_cast<const R *>(a.tables) + a.mem[g].src_off;
        R *dst = tab + a.mem[g].tab_off;
        const int cnt = (a.mem[g].pos < 0 ? 2 : 8) << a.mem[g].n_ctrl;
        for (int i = threadIdx.x; i < cnt; i += blockDim.x) dst[i] = src[i];
    }
    if (threadIdx.x == 0) {
        for (int st = 0; st < STAGES; ++st) {
            mbar_init(smem_u32(bars + st), 1);
            mbar_init(smem_u32(bars + STAGES + st), kThreads / 32);
        }
        *ready = 0;
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    const uint64_t slab = 1ull << (a.n_local - M);
    const uint64_t tile0 = (uint64_t)blockIdx.x * tiles_per_cta;
    if (threadIdx.x >= kThreads + 64) {
        // polling warp: watches the peers' flags for this CTA's tiles, ahead of the consumers, and publishes in shared
        // memory how many tiles may be overwritten -- the consumers never pay the L2 round trip of a system-scope load
        const int r = (int)threadIdx.x - (kThreads + 64);
        for (int k = 0; k < tiles_per_cta; ++k) {
            if (r < NR && r != f.c_me) {
                const uint32_t *p = f.flags[f.c_me] + (tile0 + k) * NR + r;
                if ((int32_t)(ld_relaxed_sys(p) - f.epoch) < 0) {
                    const long long t0 = clock64();
                    while ((int32_t)(ld_relaxed_sys(p) - f.epoch) < 0) {
                        __nanosleep(32);
                        if (clock64() - t0 > f.spin_limit) { *f.err = 1; break; }
                    }
                }
            }
            __syncwarp();
            if (r == 0) {
                __threadfence_block();
                *ready = k + 1;
            }
        }
        return;
    }
    if (threadIdx.x >= kThreads) {
        if (threadIdx.x == kThreads) {
            for (int k = 0; k < tiles_per_cta; ++k) {
                const int st = k % STAGES;
                if (k >= STAGES) mbar_wait(smem_u32(bars + STAGES + st), ((k / STAGES) - 1) & 1);
                const uint32_t full = smem_u32(bars + st);
                mbar_expect_tx(full, NR * kTile);
#pragma unroll
                for (int r = 0; r < NR; ++r)
                    bulk_g2s(smem_u32(ring + ((size_t)st * NR + r) * kTile),
                             reinterpret_cast<const unsigned char *>(a.src[r]) + (tile0 + k) * kTile, kTile, full);
            }
        } else if (threadIdx.x >= kThreads + 32 && threadIdx.x < kThreads + 64) {
            // signalling warp: lane r tells peer r, as soon as tile k has landed here, that it may overwrite what was read
            const int r = (int)threadIdx.x - (kThreads + 32);
            for (int k = 0; k < tiles_per_cta; ++k) {
                mbar_wait(smem_u32(bars + (k % STAGES)), (k / STAGES) & 1);
                if (r < NR && r != f.c_me) st_relaxed_sys(f.flags[r] + (tile0 + k) * NR + f.c_me, f.epoch);
            }
        }
        return;
    }
    using IO = VecIO<R, V>;
    R pr[U][NR][V], pi[U][NR][V];                                // the previous tile's results, waiting for their flags
    auto flush = [&](uint64_t tile) {
        // every peer has read the slabs of `tile` that are about to be overwritten: the polling warp says so in shared
        // memory; each thread's stores below are control-dependent on its own look at that counter
        const int need = (int)(tile - tile0) + 1;
        while (*ready < need) {
            if (*reinterpret_cast<volatile int32_t *>(f.err)) break;       // the polling warp gave up
        }
        const uint64_t bv0 = tile * ((uint64_t)kThreads * U) + threadIdx.x;
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int r = 0; r < NR; ++r)
                IO::store(a.dst, (uint64_t)r * slab + (bv0 + (uint64_t)u * kThreads) * V, pr[u][r], pi[u][r]);
    };
    for (int k = 0; k < tiles_per_cta; ++k) {
        const int st = k % STAGES;
        mbar_wait(smem_u32(bars + st), (k / STAGES) & 1);
        R ar[U][NR][V], ai[U][NR][V];
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                const unsigned char *sp = ring + ((size_t)st * NR + r) * kTile + ((size_t)u * kThreads + threadIdx.x) * 16;
                if constexpr (V == 2) {
                    const float4 t = *reinterpret_cast<const float4 *>(sp);
                    ar[u][r][0] = t.x; ai[u][r][0] = t.y; ar[u][r][1] = t.z; ai[u][r][1] = t.w;
                } else {
                    const double2 d = *reinterpret_cast<const double2 *>(sp);
                    ar[u][r][0] = d.x; ai[u][r][0] = d.y;
                }
            }
        if (k > 0) flush(tile0 + k - 1);
        const uint64_t bv0 = (tile0 + k) * ((uint64_t)kThreads * U) + threadIdx.x;
        for (int g = 0; g < a.n_members; ++g) {
            const int pos = a.mem[g].pos;
            const int nc = a.mem[g].n_ctrl;
            const R *mt = tab + a.mem[g].tab_off;
            const uint32_t low_bit = a.mem[g].low_bit;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint64_t gi = ((bv0 + (uint64_t)u * kThreads) * V) | a.rank_bits;
                uint32_t idx0 = 0;
                for (int j = 0; j < nc; ++j) idx0 |= (uint32_t)((gi >> a.mem[g].ctrl[j]) & 1ull) << j;
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    const uint32_t idx = v ? (idx0 | low_bit) : idx0;
                    if (pos < 0) {
                        const R c = mt[2 * idx], sn = mt[2 * idx + 1];
#pragma unroll
                        for (int r = 0; r < NR; ++r) {
                            const R x = ar[u][r][v], y = ai[u][r][v];
                            ar[u][r][v] = c * x - sn * y;
                            ai[u][r][v] = c * y + sn * x;
                        }
                        continue;
                    }
                    R m[8];
                    load_m8<R>(mt + 8 * idx, m);
                    switch (pos) {
                        case 0: butterfly<R, V, NR, 0, false>(ar[u], ai[u], m, v, 0u); break;
                        case 1: butterfly<R, V, NR, 1, false>(ar[u], ai[u], m, v, 0u); break;
                        default: butterfly<R, V, NR, 2, false>(ar[u], ai[u], m, v, 0u); break;
                    }
                }
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u)
#pragma unroll
            for (int r = 0; r < NR; ++r)
#pragma unroll
                for (int v = 0; v < V; ++v) { pr[u][r][v] = ar[u][r][v]; pi[u][r][v] = ai[u][r][v]; }
        // release the stage behind the arithmetic that consumed every register loaded from it (see k_block_gather_tma)
        __syncwarp();
        if ((threadIdx.x & 31) == 0) mbar_arrive(smem_u32(bars + STAGES + st));
    }
    flush(tile0 + tiles_per_cta - 1);
}

// ----------------------------------------------------------------------------------
// Expansion pass (lazy materialisation fast path).
//
// All M block qubits are the new qubits n_in .. n_in+M-1, each the target of exactly
// one member, all known |0> on input.  Then
//     out[x | a << n_in] = in[x] * prod_j table_j[idx_j(x)][a_j][0] * prod_d diag_d[idx_d(x)]
// -- one complex multiply per output amplitude.  The products are precombined by
// k_expand_table over the union of the members' index qubits (nu bits) into
// ctab[a][cidx]; the pass stages ctab in shared memory, reads each input amplitude
// once and writes its 2^M images: read 2^n_in, write 2^(n_in+M), nothing else.
// ----------------------------------------------------------------------------------
constexpr int kChunkBits = 10;                  // 1024 amplitudes per leaf chunk of the sampler's sum tree
constexpr int kFanBits = 5;                     // 32 children per tree node: one per lane, a level costs one 256-byte load

__device__ __forceinline__ double warp_sum(double x) {
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) x += __shfl_xor_sync(0xffffffffu, x, o);
    return x;
}

constexpr int kExpandThreadsMax = 1024;
constexpr int kExpandMaxBits = 12;          // nu + M: 4096 entries (32 KB c64, 64 KB c128)

struct ExpandArgs {
    void *state;
    const void *ctab;               // device, [2^M][2^nu] complex in the state's real type
    int32_t n_in, nu;
    int32_t cu_below_32;            // every index qubit is below 32: 32-bit index arithmetic
    int8_t cu[kExpandMaxBits];      // union of index qubits: cidx bit j <-> qubit cu[j]
    uint64_t rank_bits;
    unsigned long long *tile_counter;   // non-null: persistent CTAs fetch tiles in order from this counter
    double *tree_out;                   // non-null: also emit sum |in|^2 per 2^kChunkBits input amplitudes (the
                                        // sampler's level-0 sums); requires blockDim.x * V == 2^kChunkBits
    double *sub_out;                    // with tree_out: the per-warp sums (32*V amplitudes each), a finer level the
                                        // sampler uses to avoid scanning a whole chunk times 2^M branches
    uint64_t bstate, bctab;             // batch strides in bytes: state, combined table (tree_out is not batched)
};

struct ExpandTableArgs {
    const double *tables;           // fp64 tables of the program
    void *ctab;
    int32_t M, nu, n_members, is_double;
    int8_t mpos[QCM_MAX_MEMBERS];   // target position 0..M-1, or -1 for a diagonal member
    int8_t mnc[QCM_MAX_MEMBERS];
    int8_t mbit[QCM_MAX_MEMBERS][QCM_MAX_CTRL];     // member index bit j <-> cidx bit mbit[g][j]
    int64_t moff[QCM_MAX_MEMBERS];
    unsigned long long *tile_counter;   // reset to 0 here for the pass that follows
    uint64_t btab64, bctab;             // batch strides in bytes: fp64 tables, combined table
};

static __global__ void k_expand_table(const __grid_constant__ ExpandTableArgs a) {
    const uint32_t n = 1u << (a.M + a.nu);
    const uint32_t e = blockIdx.x * blockDim.x + threadIdx.x;
    if (e == 0 && a.tile_counter) *a.tile_counter = 0ull;
    if (e >= n) return;
    const double *const tables = batch_ptr(a.tables, a.btab64);
    void *const ctab = batch_ptr(a.ctab, a.bctab);
    const uint32_t cidx = e & ((1u << a.nu) - 1u), r = e >> a.nu;
    double re = 1.0, im = 0.0;
    for (int g = 0; g < a.n_members; ++g) {
        uint32_t idx = 0;
        for (int j = 0; j < a.mnc[g]; ++j) idx |= ((cidx >> a.mbit[g][j]) & 1u) << j;
        double fr, fi;
        if (a.mpos[g] < 0) {
            fr = tables[a.moff[g] + 2 * idx];
            fi = tables[a.moff[g] + 2 * idx + 1];
        } else {
            const int bit = (r >> a.mpos[g]) & 1u;                  // column 0 of the 2x2: m00 / m10
            fr = tables[a.moff[g] + 8 * idx + 4 * bit];
            fi = tables[a.moff[g] + 8 * idx + 4 * bit + 1];
        }
        const double nr = re * fr - im * fi;
        im = re * fi + im * fr;
        re = nr;
    }
    if (a.is_double) reinterpret_cast<double2 *>(ctab)[e] = make_double2(re, im);
    else reinterpret_cast<float2 *>(ctab)[e] = make_float2((float)re, (float)im);
}

// Q0: qubit 0 is an index qubit; the host puts it at cidx bit 0, so the coefficients of the two
// amplitudes of a 128-bit vector are adjacent table entries (one 128-bit shared load for c64).
template <typename R, int V, int M, int U, bool Q0>
__global__ void __launch_bounds__(kExpandThreadsMax) k_expand(const __grid_constant__ ExpandArgs a) {
    constexpr int NR = 1 << M;
    using IO = VecIO<R, V>;
    using C2 = typename std::conditional<sizeof(R) == 4, float2, double2>::type;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    C2 *tab = reinterpret_cast<C2 *>(smem_raw);
    void *const state = batch_ptr(a.state, a.bstate);
    {
        const C2 *src = reinterpret_cast<const C2 *>(batch_ptr(a.ctab, a.bctab));
        for (int i = threadIdx.x; i < (NR << a.nu); i += blockDim.x) tab[i] = src[i];
    }
    __syncthreads();
    const int nu = a.nu;
    const uint64_t nvec = (1ull << a.n_in) / V;
    const uint64_t ostride = 1ull << a.n_in;
    // Tiles (blockDim * U vectors) are taken in address order: either one per CTA in launch order, or by
    // persistent CTAs from a global counter.  CTAs that are resident together then work on one compact
    // window of the state, which is what keeps the 2^M write streams on open DRAM pages; a grid-stride
    // loop lets the CTAs drift apart and costs ~20 % of the bandwidth (profiles/r01_notes.md).
    const uint64_t tile_vecs = (uint64_t)blockDim.x * U;
    const uint64_t ntiles = (nvec + tile_vecs - 1) / tile_vecs;
    __shared__ unsigned long long s_tile[2];
    int parity = 0;
    for (uint64_t tile = blockIdx.x;; tile += gridDim.x) {
        if (a.tile_counter) {
            if (threadIdx.x == 0) s_tile[parity] = atomicAdd(a.tile_counter, 1ull);
            __syncthreads();
            tile = s_tile[parity];
            parity ^= 1;
        }
        if (tile >= ntiles) break;
        const uint64_t bv0 = tile * tile_vecs + threadIdx.x;
        R xr[U][V], xi[U][V];
        bool ok[U];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t bv = bv0 + (uint64_t)u * blockDim.x;
            ok[u] = bv < nvec;
            if (ok[u]) IO::load(state, bv * V, xr[u], xi[u]);
        }
        if (a.tree_out) {
            // level-0 sums of the sampler's tree over the INPUT (sum_a |out[x,a]|^2 = |in[x]|^2): sub-tile
            // u of this tile is exactly one chunk.  Fixed association: xor-shuffle tree, then warps in order.
            __shared__ double s_w[U][32];
#pragma unroll
            for (int u = 0; u < U; ++u) {
                double w = 0.0;
                if (ok[u]) {
#pragma unroll
                    for (int v = 0; v < V; ++v) w += (double)xr[u][v] * (double)xr[u][v] + (double)xi[u][v] * (double)xi[u][v];
                }
                w = warp_sum(w);
                if ((threadIdx.x & 31) == 0) {
                    s_w[u][threadIdx.x >> 5] = w;
                    if (ok[u]) a.sub_out[(tile * U + u) * (blockDim.x >> 5) + (threadIdx.x >> 5)] = w;
                }
            }
            __syncthreads();
            if (threadIdx.x < U && tile * U + threadIdx.x < (nvec * V) >> kChunkBits) {
                double t = 0.0;
                for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += s_w[threadIdx.x][i];
                a.tree_out[tile * U + threadIdx.x] = t;
            }
            __syncthreads();
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            if (!ok[u]) continue;
            const uint64_t b = (bv0 + (uint64_t)u * blockDim.x) * V;
            const uint64_t gi = b | a.rank_bits;
            uint32_t cidx = 0;
            if (a.cu_below_32) {
                const uint32_t lo = (uint32_t)gi;
                for (int j = 0; j < nu; ++j) cidx |= ((lo >> a.cu[j]) & 1u) << j;
            } else {
                for (int j = 0; j < nu; ++j) cidx |= (uint32_t)((gi >> a.cu[j]) & 1ull) << j;
            }
            const C2 *t0 = tab + cidx;          // V == 2: b is even, so cidx bit 0 is clear when Q0
#pragma unroll
            for (int r = 0; r < NR; ++r) {
                R orr[V], oi[V];
                C2 c0, c1;
                if constexpr (V == 2 && Q0 && sizeof(R) == 4) {
                    const float4 cc = *reinterpret_cast<const float4 *>(t0 + (r << nu));
                    c0 = make_float2(cc.x, cc.y);
                    c1 = make_float2(cc.z, cc.w);
                } else {
                    c0 = t0[r << nu];
                    c1 = c0;
                }
                orr[0] = c0.x * xr[u][0] - c0.y * xi[u][0];
                oi[0] = c0.x * xi[u][0] + c0.y * xr[u][0];
                if constexpr (V == 2) {
                    orr[1] = c1.x * xr[u][1] - c1.y * xi[u][1];
                    oi[1] = c1.x * xi[u][1] + c1.y * xr[u][1];
                }
                IO::store(state, b + (uint64_t)r * ostride, orr, oi);
            }
        }
    }
}

// ----------------------------------------------------------------------------------
// Wide expansion pass (5..QCM_MAX_EXPAND new qubits): product tree instead of a precombined table.
//
//     out[x | a << n_in] = in[x] * prod_d diag_d[idx_d(x)] * prod_j f_j[a_j],   f_j[a] = table_j[idx_j(x)][a][0]
//
// A thread reads one vector of V input amplitudes, looks up the 2M factors once (the member tables
// are tiny and live in shared memory) and walks the 2^M outputs as a product tree: the low ML levels
// are unrolled (one complex multiply per tree node, stores in ascending address order), the high
// M-ML levels are a loop with a short multiply chain per iteration.  ~2 complex multiplies per
// output instead of 1, but no 2^(M+nu)-entry table, so M is only limited by the register file; a
// 16-ancilla circuit becomes two passes and the intermediate levels all but vanish from the byte
// count (34 qubits: 77.9 GB -> 69.5 GB per circuit).  2^M write streams per thread are fine as long
// as tiles are handed out in address order (tools/membench3.cu: 6.3-6.7 TB/s for 16..256 streams).
// ----------------------------------------------------------------------------------
constexpr int kTreeLow = 4;                     // unrolled levels

struct TreeMember {
    int8_t n_ctrl;
    int8_t ctrl[QCM_MAX_CTRL];
    uint16_t low_bit;               // table-index bit fed by qubit 0
    int32_t tab_off;                // reals, in shared memory: per index 4 reals (f0.re f0.im f1.re f1.im); diag: 2
    int32_t src_off;                // reals, in the program's tables (8 per index; diag: 2)
};

struct ExpandTreeArgs {
    void *state;
    const void *tables;             // device, state's real type
    int32_t n_in, M, n_diag;
    int32_t ctrl_below_32;
    uint64_t rank_bits;
    double *tree_out;               // see ExpandArgs
    double *sub_out;                // per-vector |in|^2 sums (the sampler's finest level)
    uint64_t bstate, btab;          // batch strides in bytes (k_expand_tree; the rotated pass is never batched)
    TreeMember mem[QCM_MAX_EXPAND]; // member j targets qubit n_in + j
    TreeMember diag[4];
};

template <typename R> struct CplxOf { using T = float2; };
template <> struct CplxOf<double> { using T = double2; };

template <typename R, int V, int L>
struct TreeEmit {
    using C2 = typename CplxOf<R>::T;
    // p: partial product for the levels above L; f[l][a][v]: factor of level l; r: output index bits above level L
    static __device__ __forceinline__ void run(void *state, uint64_t base, uint64_t ostride, const R (&pr)[V], const R (&pi)[V],
                                               const R (&fr)[kTreeLow][2][V], const R (&fi)[kTreeLow][2][V], uint32_t r) {
#pragma unroll
        for (int a = 0; a < 2; ++a) {
            R qr[V], qi[V];
#pragma unroll
            for (int v = 0; v < V; ++v) {
                qr[v] = pr[v] * fr[L - 1][a][v] - pi[v] * fi[L - 1][a][v];
                qi[v] = pr[v] * fi[L - 1][a][v] + pi[v] * fr[L - 1][a][v];
            }
            TreeEmit<R, V, L - 1>::run(state, base, ostride, qr, qi, fr, fi, r | ((uint32_t)a << (L - 1)));
        }
    }
};
template <typename R, int V>
struct TreeEmit<R, V, 0> {
    static __device__ __forceinline__ void run(void *state, uint64_t base, uint64_t ostride, const R (&pr)[V], const R (&pi)[V],
                                               const R (&)[kTreeLow][2][V], const R (&)[kTreeLow][2][V], uint32_t r) {
        VecIO<R, V>::store(state, base + (uint64_t)r * ostride, pr, pi);
    }
};

template <typename R, int V>
__global__ void __launch_bounds__(kExpandThreadsMax) k_expand_tree(const __grid_constant__ ExpandTreeArgs a) {
    using IO = VecIO<R, V>;
    extern __shared__ __align__(16) unsigned char smem_raw[];
    R *tab = reinterpret_cast<R *>(smem_raw);
    void *const state = batch_ptr(a.state, a.bstate);
    const R *gt = reinterpret_cast<const R *>(batch_ptr(a.tables, a.btab));
    for (int j = 0; j < a.M; ++j) {                       // column 0 of every 2x2: (m00, m10)
        const int n = 1 << a.mem[j].n_ctrl;
        for (int i = threadIdx.x; i < n; i += blockDim.x) {
            const R *src = gt + a.mem[j].src_off + 8 * i;
            R *dst = tab + a.mem[j].tab_off + 4 * i;
            dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[4]; dst[3] = src[5];
        }
    }
    for (int d = 0; d < a.n_diag; ++d) {
        const int n = 2 << a.diag[d].n_ctrl;
        for (int i = threadIdx.x; i < n; i += blockDim.x) tab[a.diag[d].tab_off + i] = gt[a.diag[d].src_off + i];
    }
    __syncthreads();

    const uint64_t nvec = (1ull << a.n_in) / V;
    const uint64_t ostride = 1ull << a.n_in;
    const int MH = a.M - kTreeLow;                        // >= 1
    auto index_of = [&](const TreeMember &m, uint64_t gi) -> uint32_t {
        uint32_t idx = 0;
        if (a.ctrl_below_32) {
            const uint32_t lo = (uint32_t)gi;
            for (int j = 0; j < m.n_ctrl; ++j) idx |= ((lo >> m.ctrl[j]) & 1u) << j;
        } else {
            for (int j = 0; j < m.n_ctrl; ++j) idx |= (uint32_t)((gi >> m.ctrl[j]) & 1ull) << j;
        }
        return idx;
    };
    // one tile (blockDim vectors) per CTA, in launch = address order
    for (uint64_t tile = blockIdx.x; tile * blockDim.x < nvec; tile += gridDim.x) {
        const uint64_t bv = tile * blockDim.x + threadIdx.x;
        const bool ok = bv < nvec;
        const uint64_t b = bv * V;
        const uint64_t gi = b | a.rank_bits;
        R xr[V], xi[V];
#pragma unroll
        for (int v = 0; v < V; ++v) { xr[v] = R(0); xi[v] = R(0); }
        if (ok) IO::load(state, b, xr, xi);
        if (a.tree_out) {
            __shared__ double s_w[32];
            double w = 0.0;
#pragma unroll
            for (int v = 0; v < V; ++v) w += (double)xr[v] * (double)xr[v] + (double)xi[v] * (double)xi[v];
            if (ok) a.sub_out[bv] = w;
            w = warp_sum(w);
            if ((threadIdx.x & 31) == 0) s_w[threadIdx.x >> 5] = w;
            __syncthreads();
            if (threadIdx.x == 0 && tile < (nvec * V) >> kChunkBits) {
                double t = 0.0;
                for (int i = 0; i < (int)(blockDim.x >> 5); ++i) t += s_w[i];
                a.tree_out[tile] = t;
            }
            __syncthreads();
        }
        if (!ok) continue;
        for (int d = 0; d < a.n_diag; ++d) {
            const uint32_t i0 = index_of(a.diag[d], gi);
#pragma unroll
            for (int v = 0; v < V; ++v) {
                const uint32_t idx = v ? (i0 | a.diag[d].low_bit) : i0;
                const R c = tab[a.diag[d].tab_off + 2 * idx], sn = tab[a.diag[d].tab_off + 2 * idx + 1];
                const R x = xr[v], y = xi[v];
                xr[v] = c * x - sn * y;
                xi[v] = c * y + sn * x;
            }
        }
        // factors of the unrolled low levels
        R fr[kTreeLow][2][V], fi[kTreeLow][2][V];
#pragma unroll
        for (int l = 0; l < kTreeLow; ++l) {
            const uint32_t i0 = index_of(a.mem[l], gi);
#pragma unroll
            for (int v = 0; v < V; ++v) {
                const uint32_t idx = v ? (i0 | a.mem[l].low_bit) : i0;
                const R *f = tab + a.mem[l].tab_off + 4 * idx;
                fr[l][0][v] = f[0]; fi[l][0][v] = f[1]; fr[l][1][v] = f[2]; fi[l][1][v] = f[3];
            }
        }
        // table entries of the high levels (at most QCM_MAX_EXPAND - kTreeLow of them)
        uint32_t hidx[QCM_MAX_EXPAND - kTreeLow][V];
#pragma unroll
        for (int l = 0; l < QCM_MAX_EXPAND - kTreeLow; ++l) {
            if (l < MH) {
                const uint32_t i0 = index_of(a.mem[kTreeLow + l], gi);
#pragma unroll
                for (int v = 0; v < V; ++v) hidx[l][v] = v ? (i0 | a.mem[kTreeLow + l].low_bit) : i0;
            }
        }
        for (uint32_t rh = 0; rh < (1u << MH); ++rh) {
            R pr[V], pi[V];
#pragma unroll
            for (int v = 0; v < V; ++v) { pr[v] = xr[v]; pi[v] = xi[v]; }
#pragma unroll
            for (int l = 0; l < QCM_MAX_EXPAND - kTreeLow; ++l) {
                if (l < MH) {
                    const int bit = (rh >> l) & 1u;
#pragma unroll
                    for (int v = 0; v < V; ++v) {
                        const R *f = tab + a.mem[kTreeLow + l].tab_off + 4 * hidx[l][v] + 2 * bit;
                        const R c = f[0], sn = f[1];
                        const R x = pr[v], y = pi[v];
                        pr[v] = c * x - sn * y;
                        pi[v] = c * y + sn * x;
                    }
                }
            }
            TreeEmit<R, V, kTreeLow>::run(state, b + ((uint64_t)rh << (a.n_in + kTreeLow)), ostride, pr, pi, fr, fi, 0u);
        }
    }
}

// ----------------------------------------------------------------------------------
// Wide expansion pass, ROTATED output (the last pass of a program; QCM_FLAG_ROTATED_OUTPUT_OK).
//
// Same maths as k_expand_tree, but the result is stored with the M new qubits as the LOW address
// bits:   out_phys[(x << M) | a] = in[x] * prod_d diag_d[idx_d(x)] * prod_j f_j[a_j].
// The 2^M images of an input amplitude are then one contiguous run and the whole pass is a single
// sequential write stream (the layout k_init and memset reach 7.4-7.6 TB/s on) instead of 2^M
// streams 2^n_in amplitudes apart (6.3-6.9 TB/s, tools/membench3.cu).  The engine undoes the
// rotation in every reader (post-selection, sampler, qcm_get_amplitudes): callers keep seeing
// logical indices x | a << n_in.
//
// A warp owns 32 inputs per batch (pairs, interleaved with the CTA's other warps).  Phase A (lane i
// owns one input): one load, the sampler's sums, every table index of x, and the part of the product that does not depend
// on the lane's image bits -- U[s][v] = in[x] * diag * f_0[v] * prod_{j >= LB} f_j[s_j] (LB = 5 + log2 V
// image bits are covered by one warp store: vector slot v and the lane) -- parked in shared memory
// together with the table offsets of the lane-indexed members.  Phase B (all lanes, one input at a
// time, everything about x is a shared-memory broadcast): L = prod of the lane-indexed members'
// factors at the lane's bits (LB - 1 - (V == 2) complex multiplies... 4), then out[s] = L * U[s] -- one
// complex multiply per output amplitude, one 512-byte warp store per s, addresses ascending.
// The input comes from a scratch copy (the output overwrites it).  A CTA covers 2^kChunkBits
// inputs, so the sampler's level-0 sum is one value per CTA.
// ----------------------------------------------------------------------------------
// shared memory per warp: U[NS][32] 16-byte vectors, A[32][4] + B[32][8] complex
constexpr int kLowRow = 33;                              // padded row of the lane-indexed product tables (bank spread)

// shared memory per warp: U[NS][32] 16-byte vectors, A[4][33] + B[8][33] complex
template <typename R, int MH> __host__ __device__ constexpr size_t low_warp_bytes() {
    return (size_t)(1 << MH) * 32 * 16 + (size_t)12 * kLowRow * 2 * sizeof(R);
}
// small CTAs (8 / 4 warps): five or more resident per SM, so one CTA's start-up (table staging) overlaps the others' stores
template <typename R> __host__ __device__ constexpr int low_threads() { return sizeof(R) == 4 ? 256 : 128; }

// ---- the image arithmetic of the rotated pass, shared by k_expand_low and by the readers of an unwritten (virtual)
// result, which compute the images they need from the pass's input instead of loading them (DESIGN.md 3).  Every
// complex multiply is written with explicit roundings, so the FMA contraction cannot differ between the kernel and a
// reader: a computed image is bit-identical to the stored one.  fac(member, bit, fr, fi) yields f_member[bit] at the
// input's table index.
__device__ __forceinline__ void low_cmul(float ar, float ai, float br, float bi, float &cr, float &ci) {
    const float t = __fmul_rn(ai, bi), u = __fmul_rn(ai, br);
    cr = __fmaf_rn(ar, br, -t);
    ci = __fmaf_rn(ar, bi, u);
}
__device__ __forceinline__ void low_cmul(double ar, double ai, double br, double bi, double &cr, double &ci) {
    const double t = __dmul_rn(ai, bi), u = __dmul_rn(ai, br);
    cr = __fma_rn(ar, br, -t);
    ci = __fma_rn(ar, bi, u);
}
// table index of member m at global index gi
__device__ __forceinline__ uint32_t low_index(const TreeMember &m, uint64_t gi) {
    uint32_t idx = 0;
#pragma unroll 1
    for (int j = 0; j < m.n_ctrl; ++j) idx |= (uint32_t)((gi >> m.ctrl[j]) & 1ull) << j;
    return idx;
}
// p = in[x] * prod_d diag_d[idx_d(x)]; diag(d, idx) points at the real part of entry idx of diagonal d
template <typename R, typename D>
__device__ __forceinline__ void low_diag(const ExpandTreeArgs &a, uint64_t gi, D diag, R &pr, R &pi) {
#pragma unroll 1
    for (int d = 0; d < a.n_diag; ++d) {
        const R *c = diag(d, low_index(a.diag[d], gi));
        low_cmul(pr, pi, c[0], c[1], pr, pi);
    }
}
// q[v] = p * f_0[v] (complex64: member 0 is the vector slot), or p itself
template <typename R, int V, typename F>
__device__ __forceinline__ void low_q(F fac, R pr, R pi, int v, R &qr, R &qi) {
    if constexpr (V == 2) {
        R fr, fi;
        fac(0, v, fr, fi);
        low_cmul(pr, pi, fr, fi, qr, qi);
    } else {
        qr = pr; qi = pi;
    }
}
// g[s] = prod_{l < mh} f_{lb + l}[s_l], from 1
template <typename R, typename F>
__device__ __forceinline__ void low_g(F fac, int lb, int mh, uint32_t s, R &gr, R &gi) {
    gr = R(1); gi = R(0);
#pragma unroll
    for (int l = 0; l < mh; ++l) {
        R fr, fi;
        fac(lb + l, (s >> l) & 1, fr, fi);
        low_cmul(gr, gi, fr, fi, gr, gi);
    }
}
// A[t] = f_{j0}[t_0] f_{j0+1}[t_1],  B[t] = f_{j0+2}[t_0] f_{j0+3}[t_1] f_{j0+4}[t_2]
template <typename R, typename F>
__device__ __forceinline__ void low_a(F fac, int j0, int t, R &cr, R &ci) {
    R xr, xi, yr, yi;
    fac(j0, t & 1, xr, xi);
    fac(j0 + 1, t >> 1, yr, yi);
    low_cmul(xr, xi, yr, yi, cr, ci);
}
template <typename R, typename F>
__device__ __forceinline__ void low_b(F fac, int j0, int t, R &cr, R &ci) {
    R xr, xi, yr, yi, zr, zi;
    fac(j0 + 2, t & 1, xr, xi);
    fac(j0 + 3, (t >> 1) & 1, yr, yi);
    fac(j0 + 4, t >> 2, zr, zi);
    low_cmul(xr, xi, yr, yi, xr, xi);
    low_cmul(xr, xi, zr, zi, cr, ci);
}
// image im (0 <= im < 2^M) of the input with diagonal product p: the amplitude k_expand_low stores at (x << M) | im,
// L * U[s][v] with im = v | lane << (V - 1) | s << LB and lane = ta | tb << 2, L = A[ta] B[tb]
template <typename R, int V, typename F>
__device__ __forceinline__ void low_image(F fac, int M, R pr, R pi, uint32_t im, R &outr, R &outi) {
    constexpr int LB = V == 2 ? 6 : 5, J0 = V == 2 ? 1 : 0;
    const uint32_t lane = (im >> (V - 1)) & 31u;
    R qr, qi, gr, gi, ur, ui, ar, ai, br, bi, lr, li;
    low_q<R, V>(fac, pr, pi, (int)(im & 1u), qr, qi);
    low_g<R>(fac, LB, M - LB, im >> LB, gr, gi);
    low_cmul(qr, qi, gr, gi, ur, ui);
    low_a<R>(fac, J0, (int)(lane & 3u), ar, ai);
    low_b<R>(fac, J0, (int)(lane >> 2), br, bi);
    low_cmul(ar, ai, br, bi, lr, li);
    low_cmul(lr, li, ur, ui, outr, outi);
}
// f_member[bit] read from the program's tables (8 reals per index, column 0 of each 2x2: m00 at 0, m10 at 4)
template <typename R>
__device__ __forceinline__ void low_fac_global(const ExpandTreeArgs &a, int member, uint64_t gi, int bit, R &fr, R &fi) {
    const R *f = reinterpret_cast<const R *>(a.tables) + a.mem[member].src_off + 8 * low_index(a.mem[member], gi) + 4 * bit;
    fr = f[0]; fi = f[1];
}
template <typename R>
__device__ __forceinline__ const R *low_diag_global(const ExpandTreeArgs &a, int d, uint32_t idx) {
    return reinterpret_cast<const R *>(a.tables) + a.diag[d].src_off + 2 * idx;
}

// out[j] = sum of the 2^gbits consecutive values in[j << gbits ...], in index order (deterministic)
static __global__ void __launch_bounds__(kThreads) k_group_sum(const double *in, int gbits, uint64_t n_out, double *out) {
    const uint64_t j = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (j >= n_out) return;
    double t = 0.0;
    for (uint64_t i = j << gbits; i < ((j + 1) << gbits); ++i) t += in[i];
    out[j] = t;
}

// TB: log2 of the inputs one CTA covers (its tile is 2^(TB + M) output amplitudes, contiguous).  a.tree_out
// receives one partial sum per WARP (index blockIdx * warps + warp); k_group_sum folds them into the
// sampler's level-0 sums.
// NW: warps per CTA.  The size of the region a CTA writes decides how compact the window of concurrently written addresses
// is (tools/membench4.cu, profiles/r02_notes.md: a bare sequential writer loses 5 % going from 32 KiB to 512 KiB per CTA),
// so small CTAs -- few warps, one batch of 32 inputs each -- are the default shape.
// EMIT = false: the sums only (input load, sub_out, level 0) -- the result is left unwritten and its readers compute the
// images they need (the virtual last pass, DESIGN.md 3); same TB / NW as the materialising launch, so the same tree.
template <typename R, int V, int MH, int TB, int NW = low_threads<R>() / 32, bool EMIT = true>
__global__ void __launch_bounds__(NW * 32) k_expand_low(const __grid_constant__ ExpandTreeArgs a, const void *__restrict__ in) {
    constexpr int LB = V == 2 ? 6 : 5;                   // image bits covered by one warp store
    constexpr int J0 = V == 2 ? 1 : 0;                   // first lane-indexed member (member 0 is the vector slot for V == 2)
    constexpr int NS = 1 << MH;                          // warp stores per input
    constexpr int M = LB + MH;
    constexpr int kWarps = NW;
    using C2 = typename CplxOf<R>::T;
    using V16 = typename VecIO<R, V>::T;                  // float4 (two complex64) or double2 (one complex128)
    extern __shared__ __align__(16) unsigned char smem_raw[];
    R *tab = reinterpret_cast<R *>(smem_raw + low_warp_bytes<R, MH>() * kWarps);
    const R *gt = reinterpret_cast<const R *>(a.tables);
    const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
    const uint64_t tile = blockIdx.x;                                   // grid = 2^(n_in - TB), launch = address order
    constexpr int kPerWarp = (1 << TB) / kWarps;                        // inputs per warp per tile
    static_assert(kPerWarp >= 32 && kPerWarp % 32 == 0, "a warp takes whole batches of 32 inputs");
    // The warps of a CTA interleave at a granularity of two inputs (a pair shares the sampler's finest
    // sum): at step i of phase B the warps write runs 2 * 2^M amplitudes apart, so the CTA's stores
    // stay inside one moving window instead of one stream per warp (DRAM row locality).
    auto x_first = [&](int batch) -> uint64_t { return (tile << TB) + (uint64_t)batch * (32 * kWarps) + 2u * warp; };
    auto in_at = [&](uint64_t x0, uint32_t pstride) -> C2 {
        return reinterpret_cast<const C2 *>(in)[x0 + (uint64_t)(lane >> 1) * pstride + (lane & 1)];
    };
    // the first input amplitude is requested before anything else (its DRAM latency then overlaps the table staging)
    C2 next_in = in_at(x_first(0), 2 * kWarps);
    if constexpr (EMIT) {
        for (int j = 0; j < M; ++j) {                     // column 0 of every 2x2: (m00, m10)
            const int n = 1 << a.mem[j].n_ctrl;
            for (int i = threadIdx.x; i < n; i += blockDim.x) {
                const R *src = gt + a.mem[j].src_off + 8 * i;
                R *dst = tab + a.mem[j].tab_off + 4 * i;
                dst[0] = src[0]; dst[1] = src[1]; dst[2] = src[4]; dst[3] = src[5];
            }
        }
        for (int d = 0; d < a.n_diag; ++d) {
            const int n = 2 << a.diag[d].n_ctrl;
            for (int i = threadIdx.x; i < n; i += blockDim.x) tab[a.diag[d].tab_off + i] = gt[a.diag[d].src_off + i];
        }
        __syncthreads();                                  // the only block-level barrier: member tables staged
    }
    unsigned char *wbase = smem_raw + low_warp_bytes<R, MH>() * warp;
    V16 *Us = reinterpret_cast<V16 *>(wbase);                                      // [NS][32]
    C2 *As = reinterpret_cast<C2 *>(wbase + (size_t)NS * 32 * 16);                 // [4][kLowRow]: a lane reads row lane & 3
    C2 *Bs = As + 4 * kLowRow;                                                     // [8][kLowRow]: a lane reads row lane >> 2
    const C2 *my_a = As + (lane & 3) * kLowRow, *my_b = Bs + (lane >> 2) * kLowRow;

    // one batch of 32 inputs x0 + (i >> 1) * pstride + (i & 1), i = 0..31; `mine` is lane's input amplitude
    auto do_batch = [&](const uint64_t x0, const uint32_t pstride, const C2 mine, double &wacc) {
        auto x_of = [&](int i) -> uint64_t { return x0 + (uint64_t)(i >> 1) * pstride + (i & 1); };
        // ---- phase A: lane i prepares input x_of(i)
        {
            const uint64_t x = x_of(lane);
            const uint64_t gi = x | a.rank_bits;
            if (a.tree_out) {
                const double w = (double)mine.x * (double)mine.x + (double)mine.y * (double)mine.y;
                if constexpr (V == 2) {
                    const double w2 = w + __shfl_xor_sync(0xffffffffu, w, 1);
                    if (!(lane & 1)) a.sub_out[x >> 1] = w2;
                } else {
                    a.sub_out[x] = w;
                }
                wacc += w;
            }
            if constexpr (!EMIT) return;
            R pr = mine.x, pi = mine.y;
            low_diag(a, gi, [&](int d, uint32_t idx) { return tab + a.diag[d].tab_off + 2 * idx; }, pr, pi);
            __syncwarp();                                 // the previous batch's phase B is done with the tables
            uint32_t off[M];                              // table offset (reals) of member j at this input's index
#pragma unroll
            for (int j = 0; j < M; ++j) off[j] = (uint32_t)a.mem[j].tab_off + 4u * low_index(a.mem[j], gi);
            auto fac = [&](int member, int bit, R &fr, R &fi) {          // f_member[bit] at this input's table index
                const C2 f = *reinterpret_cast<const C2 *>(tab + off[member] + 2 * bit);
                fr = f.x; fi = f.y;
            };
            // U[s][v] = in * diag * f_0[v] * prod_{l < MH} f_{LB+l}[s_l]
            R qr[V], qi[V];
#pragma unroll
            for (int v = 0; v < V; ++v) low_q<R, V>(fac, pr, pi, v, qr[v], qi[v]);
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                R gr, gim;
                low_g<R>(fac, LB, MH, s, gr, gim);
                R ur[V], ui[V];
#pragma unroll
                for (int v = 0; v < V; ++v) low_cmul(qr[v], qi[v], gr, gim, ur[v], ui[v]);
                if constexpr (V == 2) Us[s * 32 + lane] = make_float4(ur[0], ui[0], ur[1], ui[1]);
                else Us[s * 32 + lane] = make_double2(ur[0], ui[0]);
            }
            // A[a] = f_{J0}[a_0] f_{J0+1}[a_1],  B[b] = f_{J0+2}[b_0] f_{J0+3}[b_1] f_{J0+4}[b_2]  (lane = a | b << 2)
#pragma unroll
            for (int t = 0; t < 4; ++t) {
                C2 o;
                low_a<R>(fac, J0, t, o.x, o.y);
                As[t * kLowRow + lane] = o;
            }
#pragma unroll
            for (int t = 0; t < 8; ++t) {
                C2 o;
                low_b<R>(fac, J0, t, o.x, o.y);
                Bs[t * kLowRow + lane] = o;
            }
            __syncwarp();
        }
        // ---- phase B: all lanes, one input at a time
#pragma unroll 2
        for (int i = 0; i < 32; ++i) {
            const C2 fa = my_a[i], fb = my_b[i];
            R lr, li;
            low_cmul(fa.x, fa.y, fb.x, fb.y, lr, li);
            const uint64_t obase = (x_of(i) << M) + (uint64_t)lane * V;
#pragma unroll
            for (int s = 0; s < NS; ++s) {
                const V16 u = Us[s * 32 + i];
                R orr[V], oi[V];
                if constexpr (V == 2) {
                    low_cmul(lr, li, u.x, u.y, orr[0], oi[0]);
                    low_cmul(lr, li, u.z, u.w, orr[1], oi[1]);
                } else {
                    low_cmul(lr, li, u.x, u.y, orr[0], oi[0]);
                }
                VecIO<R, V>::store(a.state, obase + ((uint64_t)s << LB), orr, oi);
            }
        }
    };

    {
        double wacc = 0.0;
#pragma unroll 1
        for (int batch = 0; batch < kPerWarp / 32; ++batch) {
            const C2 mine = next_in;
            // the next batch's input amplitude is fetched while this batch's stores drain (a CTA with several batches
            // per warp then never waits on the input read between batches)
            if (batch + 1 < kPerWarp / 32) next_in = in_at(x_first(batch + 1), 2 * kWarps);
            do_batch(x_first(batch), 2 * kWarps, mine, wacc);
        }
        if (a.tree_out) {
            wacc = warp_sum(wacc);
            if (lane == 0) a.tree_out[tile * kWarps + warp] = wacc;
        }
    }
}

// ----------------------------------------------------------------------------------
// Diagonal pass: amp *= table[index bits]
// ----------------------------------------------------------------------------------
struct DiagArgs {
    void *state;
    const void *table;              // device, 2 reals per entry
    int32_t n_ctrl;
    int32_t n_active;
    int8_t ctrl[QCM_MAX_CTRL];
    uint64_t rank_bits;
    uint64_t bstate, btab;          // batch strides in bytes
};

template <typename R, int V, int U>
__global__ void __launch_bounds__(kThreads) k_diag(const __grid_constant__ DiagArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    R *tab = reinterpret_cast<R *>(smem_raw);
    void *const state = batch_ptr(a.state, a.bstate);
    {
        const R *g = reinterpret_cast<const R *>(batch_ptr(a.table, a.btab));
        for (int i = threadIdx.x; i < (2 << a.n_ctrl); i += blockDim.x) tab[i] = g[i];
    }
    __syncthreads();
    using IO = VecIO<R, V>;
    const uint64_t nvec = (1ull << a.n_active) / V;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x * U;
    for (uint64_t v0 = (uint64_t)blockIdx.x * blockDim.x * U + threadIdx.x; v0 < nvec; v0 += stride) {
        R re[U][V], im[U][V];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t vi = v0 + (uint64_t)u * blockDim.x;
            if (vi < nvec) IO::load(state, vi * V, re[u], im[u]);
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t vi = v0 + (uint64_t)u * blockDim.x;
            if (vi >= nvec) continue;
#pragma unroll
            for (int v = 0; v < V; ++v) {
                const uint64_t gi = (vi * V + v) | a.rank_bits;
                uint32_t idx = 0;
                for (int j = 0; j < a.n_ctrl; ++j) idx |= (uint32_t)((gi >> a.ctrl[j]) & 1ull) << j;
                const R c = tab[2 * idx], s = tab[2 * idx + 1];
                const R x = re[u][v], y = im[u][v];
                re[u][v] = c * x - s * y;
                im[u][v] = c * y + s * x;
            }
            IO::store(state, vi * V, re[u], im[u]);
        }
    }
}

// Several diagonal passes in ONE sweep (a BLOCK header with zero targets whose members are all DIAG): the
// projections of a release-width circuit's ancillas (DESIGN.md 2a) are 2-3 diagonal tables of <= 10 index bits
// each; applied together every amplitude crosses HBM once instead of once per table.
// Table index from runs of consecutive index qubits: idx = sum_r ((gi >> start_r) & (2^len_r - 1)) << pos_r.  The
// planner sorts a diagonal table's index qubits, so 10 of them are usually 1-3 runs (a dozen instructions instead
// of one shift/mask/or per qubit with a constant-bank load each: the 3-table projection pass of the chain-20 sweep
// went from instruction-bound 2.3 TB/s to the HBM roofline).
struct IndexRuns {
    int32_t n_runs;
    int32_t below_32;                // every index qubit is below 32: 32-bit shifts
    // run r contributes  (gi >> shift[r]) & mask[r]  (mask already sits at the run's table-index position; the host
    // guarantees start >= position, which holds for ascending index qubits)
    uint32_t mask[QCM_MAX_CTRL];
    int32_t shift[QCM_MAX_CTRL];
};
struct DiagMultiRuns { IndexRuns m[QCM_MAX_MEMBERS]; };

template <typename R, int V, int U>
__global__ void __launch_bounds__(kThreads) k_diag_multi(const __grid_constant__ BlockArgs a, const __grid_constant__ DiagMultiRuns runs) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    R *tab = reinterpret_cast<R *>(smem_raw);
    void *const state = batch_ptr(a.state, a.bstate);
    for (int g = 0; g < a.n_members; ++g) {
        const R *src = reinterpret_cast<const R *>(batch_ptr(a.tables, a.btab)) + a.mem[g].src_off;
        R *dst = tab + a.mem[g].tab_off;
        for (int i = threadIdx.x; i < (2 << a.mem[g].n_ctrl); i += blockDim.x) dst[i] = src[i];
    }
    __syncthreads();
    using IO = VecIO<R, V>;
    const uint64_t nvec = (1ull << a.n_out) / V;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x * U;
    for (uint64_t v0 = (uint64_t)blockIdx.x * blockDim.x * U + threadIdx.x; v0 < nvec; v0 += stride) {
        R re[U][V], im[U][V];
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t vi = v0 + (uint64_t)u * blockDim.x;
            if (vi < nvec) IO::load(state, vi * V, re[u], im[u]);
        }
        for (int g = 0; g < a.n_members; ++g) {
            const R *mt = tab + a.mem[g].tab_off;
            const IndexRuns &rn = runs.m[g];
            const uint32_t low_bit = a.mem[g].low_bit;
#pragma unroll
            for (int u = 0; u < U; ++u) {
                const uint64_t gi = ((v0 + (uint64_t)u * blockDim.x) * V) | a.rank_bits;
                uint32_t idx0 = 0;
                if (rn.below_32) {
                    const uint32_t lo = (uint32_t)gi;
                    for (int r = 0; r < rn.n_runs; ++r) idx0 |= (lo >> rn.shift[r]) & rn.mask[r];
                } else {
                    for (int r = 0; r < rn.n_runs; ++r) idx0 |= (uint32_t)(gi >> rn.shift[r]) & rn.mask[r];
                }
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    const uint32_t idx = v ? (idx0 | low_bit) : idx0;
                    const R c = mt[2 * idx], sn = mt[2 * idx + 1];
                    const R x = re[u][v], y = im[u][v];
                    re[u][v] = c * x - sn * y;
                    im[u][v] = c * y + sn * x;
                }
            }
        }
#pragma unroll
        for (int u = 0; u < U; ++u) {
            const uint64_t vi = v0 + (uint64_t)u * blockDim.x;
            if (vi < nvec) IO::store(state, vi * V, re[u], im[u]);
        }
    }
}

// ----------------------------------------------------------------------------------
// Product-state initialisation (write-only).  amp[i] = lo[i & (2^L-1)] * hi[i >> L],
// the two factor tables are built by k_init_tables from the per-qubit 2-vectors.
// ----------------------------------------------------------------------------------
// lo is stored in the state's real type (a lane's vector of V amplitudes is then ONE 128-bit load of
// V adjacent lo entries, so the factor tables cost no more L2 traffic than the state costs HBM traffic);
// hi stays fp64: it is warp-uniform and read once per thread.
static __global__ void k_init_tables(const double *qv /* n*4 */, int n, int L, void *lo, double2 *hi, int lo_is_float,
                                     uint64_t bqv, uint64_t blo, uint64_t bhi /* batch strides, bytes */) {
    qv = batch_ptr(qv, bqv);
    lo = batch_ptr(lo, blo);
    hi = batch_ptr(hi, bhi);
    const uint64_t nlo = 1ull << L, nhi = 1ull << (n - L);
    const uint64_t t = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (t >= nlo + nhi) return;
    const bool is_hi = t >= nlo;
    const uint64_t bits = is_hi ? t - nlo : t;
    const int q0 = is_hi ? L : 0, q1 = is_hi ? n : L;
    double re = 1.0, im = 0.0;
    for (int q = q0; q < q1; ++q) {
        const int b = (int)((bits >> (q - q0)) & 1ull);
        const double fr = qv[4 * q + 2 * b], fi = qv[4 * q + 2 * b + 1];
        const double nr = re * fr - im * fi;
        im = re * fi + im * fr;
        re = nr;
    }
    if (is_hi) hi[bits] = make_double2(re, im);
    else if (lo_is_float) reinterpret_cast<float2 *>(lo)[bits] = make_float2((float)re, (float)im);
    else reinterpret_cast<double2 *>(lo)[bits] = make_double2(re, im);
}

constexpr int kInitU = 8;                       // vectors per thread: a CTA writes 32 KiB (c64), in address order

template <typename R, int V>
__global__ void __launch_bounds__(kThreads) k_init(void *state, const void *lo, const double2 *hi, int n, int L,
                                                   uint64_t bstate, uint64_t blo, uint64_t bhi) {
    using IO = VecIO<R, V>;
    state = batch_ptr(state, bstate);
    lo = batch_ptr(lo, blo);
    hi = batch_ptr(hi, bhi);
    const uint64_t nvec = (1ull << n) / V;
    const uint64_t lmask = (1ull << L) - 1ull;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x * kInitU;
    for (uint64_t v0 = (uint64_t)blockIdx.x * blockDim.x * kInitU + threadIdx.x; v0 < nvec; v0 += stride) {
#pragma unroll
        for (int u = 0; u < kInitU; ++u) {
            const uint64_t vi = v0 + (uint64_t)u * blockDim.x;
            if (vi >= nvec) break;
            const uint64_t i = vi * V;
            const double2 h = __ldg(hi + (i >> L));
            R re[V], im[V];
            if (h.x == 0.0 && h.y == 0.0) {
#pragma unroll
                for (int v = 0; v < V; ++v) { re[v] = R(0); im[v] = R(0); }
            } else {
                R lr[V], li[V];
                IO::load_nc(lo, i & lmask, lr, li);      // V adjacent entries (i is a multiple of V, L >= 1 when V == 2)
#pragma unroll
                for (int v = 0; v < V; ++v) {
                    re[v] = (R)((double)lr[v] * h.x - (double)li[v] * h.y);
                    im[v] = (R)((double)lr[v] * h.y + (double)li[v] * h.x);
                }
            }
            IO::store(state, i, re, im);
        }
    }
}

// zero-fill amplitudes [first, first+count)
template <typename R>
__global__ void __launch_bounds__(kThreads) k_zero(void *state, uint64_t first, uint64_t count, uint64_t bstate) {
    state = batch_ptr(state, bstate);
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x * kInitU;
    for (uint64_t i0 = (uint64_t)blockIdx.x * blockDim.x * kInitU + threadIdx.x; i0 < count; i0 += stride) {
#pragma unroll
        for (int u = 0; u < kInitU; ++u) {
            const uint64_t i = i0 + (uint64_t)u * blockDim.x;
            if (i >= count) break;
            R re[1] = {R(0)}, im[1] = {R(0)};
            VecIO<R, 1>::store(state, first + i, re, im);
        }
    }
}

// ----------------------------------------------------------------------------------
// Qubit exchange (local): amplitudes with (bit a, bit b) = (1,0) <-> (0,1), a < b.
// ----------------------------------------------------------------------------------
template <typename R, int V>
__global__ void __launch_bounds__(kThreads) k_swap(void *state, int qa, int qb, int n_active, uint64_t bstate) {
    using IO = VecIO<R, V>;
    state = batch_ptr(state, bstate);
    const uint64_t nvec = (1ull << (n_active - 2)) / V;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t vi = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; vi < nvec; vi += stride) {
        uint64_t b = insert_zero(insert_zero(vi * V, qa), qb);
        const uint64_t i10 = b | (1ull << qa), i01 = b | (1ull << qb);
        R r0[V], m0[V], r1[V], m1[V];
        IO::load(state, i10, r0, m0);
        IO::load(state, i01, r1, m1);
        IO::store(state, i10, r1, m1);
        IO::store(state, i01, r0, m0);
    }
}

// ----------------------------------------------------------------------------------
// Reductions.  All sums are fp64 and use a fixed association (lane-strided partials,
// shuffle tree) so that results do not depend on the grid or on the GPU count.
// ----------------------------------------------------------------------------------

constexpr int kSubCluster = 4;                  // adjacent 16-byte vectors per lane per cluster
// i-th vector (of 16 or 32) that lane `lane` owns inside a chunk
__device__ __forceinline__ uint32_t sub_vec(uint32_t lane, uint32_t i) {
    return kSubCluster * lane + (i % kSubCluster) + 32u * kSubCluster * (i / kSubCluster);
}

// level 0: chunk c = sum_{i in chunk} |amp_i|^2 ; one warp per chunk.  Full-size chunks
// stream 128-bit loads, eight in flight per lane; the lane-strided order is fixed.
template <typename R>
__global__ void __launch_bounds__(kThreads) k_chunk_sums(const void *state, int n_active, double *out, uint64_t bstate, uint64_t bout,
                                                         double *sub = nullptr, uint64_t bsub = 0) {
    // sub (optional, full-size chunks only): the 32 lane partials of every chunk -- lane l's partial covers the 16-byte
    // vectors it loaded, sub_vec(l, i): clusters of kSubCluster adjacent vectors (64 bytes), the clusters of a lane
    // 32 * kSubCluster vectors apart, so a warp's loads stay coalesced AND a group is a few whole DRAM atoms.  The
    // sampler picks a group, then one of its 32 amplitudes, instead of scanning all 1024 amplitudes of the chunk
    // (with single-vector strides the leaf reads of 2.5 M shots cost 10 GB of DRAM traffic; clustered: a quarter).
    state = batch_ptr(state, bstate);
    out = batch_ptr(out, bout);
    if (sub) sub = batch_ptr(sub, bsub);
    const int cb = n_active < kChunkBits ? n_active : kChunkBits;
    const uint64_t nchunks = 1ull << (n_active - cb);
    const uint64_t csz = 1ull << cb;
    const int lane = threadIdx.x & 31;
    const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t c = warp0; c < nchunks; c += nwarps) {
        double acc = 0.0;
        if constexpr (sizeof(R) == 4) {
            if (cb == kChunkBits) {
                const float4 *p = reinterpret_cast<const float4 *>(state) + c * (csz / 2);
                constexpr int kIter = (1 << kChunkBits) / 2 / 32;        // 16 vectors per lane
#pragma unroll
                for (int i0 = 0; i0 < kIter; i0 += 8) {
                    float4 t[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) t[k] = __ldcs(p + sub_vec(lane, i0 + k));
#pragma unroll
                    for (int k = 0; k < 8; ++k)
                        acc += ((double)t[k].x * (double)t[k].x + (double)t[k].y * (double)t[k].y) +
                               ((double)t[k].z * (double)t[k].z + (double)t[k].w * (double)t[k].w);
                }
            } else {
                const float2 *p = reinterpret_cast<const float2 *>(state) + c * csz;
                for (uint64_t i = lane; i < csz; i += 32) {
                    const float2 t = p[i];
                    acc += (double)t.x * (double)t.x + (double)t.y * (double)t.y;
                }
            }
        } else {
            const double2 *p = reinterpret_cast<const double2 *>(state) + c * csz;
            if (cb == kChunkBits) {
                constexpr int kIter = (1 << kChunkBits) / 32;            // 32 amplitudes per lane
#pragma unroll
                for (int i0 = 0; i0 < kIter; i0 += 8) {
                    double2 t[8];
#pragma unroll
                    for (int k = 0; k < 8; ++k) t[k] = __ldcs(p + sub_vec(lane, i0 + k));
#pragma unroll
                    for (int k = 0; k < 8; ++k) acc += t[k].x * t[k].x + t[k].y * t[k].y;
                }
            } else {
                for (uint64_t i = lane; i < csz; i += 32) {
                    const double2 t = p[i];
                    acc += t.x * t.x + t.y * t.y;
                }
            }
        }
        if (sub && cb == kChunkBits) sub[c * 32 + lane] = acc;
        acc = warp_sum(acc);
        if (lane == 0) out[c] = acc;
    }
}

// level l+1: node j = sum of up to 1024 children ; one warp per node
static __global__ void __launch_bounds__(kThreads) k_tree_level(const double *in, uint64_t n_in, double *out, uint64_t n_out,
                                                                uint64_t bin = 0, uint64_t bout = 0, int fan_bits = kFanBits) {
    in = batch_ptr(in, bin);
    out = batch_ptr(out, bout);
    const int lane = threadIdx.x & 31;
    const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    for (uint64_t j = warp0; j < n_out; j += nwarps) {
        const uint64_t b = j << fan_bits;
        const uint64_t e = (b + (1ull << fan_bits)) < n_in ? b + (1ull << fan_bits) : n_in;
        double acc = 0.0;
        for (uint64_t i = b + lane; i < e; i += 32) acc += in[i];
        acc = warp_sum(acc);
        if (lane == 0) out[j] = acc;
    }
}

// ----------------------------------------------------------------------------------
// Philox4x32-10 (counter-based RNG; Salmon et al. 2011): key = seed, counter =
// (shot, stream) -> one uniform double in [0,1) per shot, identical on every rank.
// ----------------------------------------------------------------------------------
__host__ __device__ __forceinline__ void philox_round(uint32_t (&c)[4], uint32_t (&k)[2]) {
    const uint64_t p0 = (uint64_t)0xD2511F53u * c[0];
    const uint64_t p1 = (uint64_t)0xCD9E8D57u * c[2];
    const uint32_t n0 = (uint32_t)(p1 >> 32) ^ c[1] ^ k[0];
    const uint32_t n1 = (uint32_t)p1;
    const uint32_t n2 = (uint32_t)(p0 >> 32) ^ c[3] ^ k[1];
    const uint32_t n3 = (uint32_t)p0;
    c[0] = n0; c[1] = n1; c[2] = n2; c[3] = n3;
    k[0] += 0x9E3779B9u; k[1] += 0xBB67AE85u;
}

__host__ __device__ __forceinline__ double philox_uniform(uint64_t seed, uint64_t stream, uint64_t shot) {
    uint32_t c[4] = {(uint32_t)shot, (uint32_t)(shot >> 32), (uint32_t)stream, (uint32_t)(stream >> 32)};
    uint32_t k[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
#pragma unroll
    for (int r = 0; r < 10; ++r) philox_round(c, k);
    const uint64_t bits = ((uint64_t)c[0] << 21) ^ (uint64_t)(c[1] >> 11);   // 53 bits
    return (double)(bits & ((1ull << 53) - 1ull)) * (1.0 / 9007199254740992.0);
}

// Warp-cooperative search inside one node: children [0, cnt) with masses w(i).  Lane l
// owns children l, l+32, l+64, ... (so that a warp's loads are coalesced); the node's
// mass is laid out lane-major: lane 0's children in ascending order, then lane 1's, ...
// Returns the child whose interval contains u (clamped to a child with non-zero mass)
// and subtracts the mass laid out before it from u.  Fixed evaluation order => deterministic.
template <typename F>
__device__ __forceinline__ uint32_t warp_pick(F w, uint32_t cnt, double &u, int lane) {
    double mine = 0.0;
    for (uint32_t i = lane; i < cnt; i += 32u) mine += w(i);
    double incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
        const double t = __shfl_up_sync(0xffffffffu, incl, o);
        if (lane >= o) incl += t;
    }
    const unsigned hit = __ballot_sync(0xffffffffu, incl > u && mine > 0.0);
    const unsigned any = __ballot_sync(0xffffffffu, mine > 0.0);
    int sel;
    if (hit) sel = __ffs(hit) - 1;
    else if (any) sel = 31 - __clz(any);              // rounding pushed u past the total
    else sel = 0;
    const double excl = __shfl_sync(0xffffffffu, incl - mine, sel);
    double rem = u - excl;
    if (cnt <= 32u) {                                 // one child per lane (a 32-ary tree level): the lane IS the child
        u = rem < 0.0 ? 0.0 : rem;
        return (uint32_t)sel < cnt ? (uint32_t)sel : 0u;
    }
    uint32_t child = 0;
    double before = 0.0;
    if (lane == sel) {
        double acc = 0.0;
        uint32_t last_nz = (uint32_t)lane < cnt ? (uint32_t)lane : 0u;
        double last_before = 0.0;
        for (uint32_t i = lane; i < cnt; i += 32u) {
            const double wi = w(i);
            if (wi > 0.0) {
                last_nz = i; last_before = acc;
                if (acc + wi > rem) break;
            }
            acc += wi;
        }
        child = last_nz; before = last_before;
    }
    child = __shfl_sync(0xffffffffu, child, sel);
    before = __shfl_sync(0xffffffffu, before, sel);
    rem -= before;
    u = rem < 0.0 ? 0.0 : rem;
    return child;
}

struct SampleArgs {
    const void *state;
    int32_t n_active;               // qubits the sum tree indexes (its leaves are x < 2^n_active)
    int32_t cond_bits;              // > 0: the state holds 2^cond_bits images of every leaf x, at
                                    // x | a << n_active (an expansion pass ran after the tree was built):
                                    // leaf weight = sum_a |amp|^2, then a is drawn given x
    int32_t cond_low;               // the images are the LOW address bits: (x << cond_bits) | a  (rotated expansion)
    int32_t rot_m, rot_nin;         // rotated storage without a checkpoint tree: the tree indexes physical
                                    // addresses p; logical index = (p >> rot_m) | ((p & (2^rot_m - 1)) << rot_nin)
    int32_t n_levels;               // tree levels above the amplitudes (>= 1)
    const double *sub;              // optional finer level under level[0]: sums over 2^sub_bits amplitudes
    int32_t sub_bits;
    int32_t sub_strided;            // sub holds k_chunk_sums' 32 lane partials per chunk (strided groups, see there)
    uint64_t bsub;                  // batch stride of sub, bytes
    const double *level[8];         // level[0] = chunk sums ... level[n_levels-1] = top
    uint64_t level_n[8];
    uint64_t shots, seed, stream;
    // sharding: rank_lo <= u*total < rank_hi selects this rank (single GPU: [0,total))
    double rank_lo, rank_hi, total;
    uint64_t rank_bits;
    int32_t n_clbits;               // 0 => raw indices
    int8_t clbit_qubit[64];
    uint64_t *keys_out;
    uint8_t *mine_out;              // may be null
    // batch (blockIdx.y = sweep point): strides in bytes of the state, the tree arrays and the keys; per-point
    // Philox streams and total masses (device arrays; null for a plain handle)
    uint64_t bstate, btree, bkeys;
    const uint64_t *streams;
    const double *totals;
    // sharded sampling with the rank masses still on the device (right out of an all-gather): mass of rank r at
    // dev_masses[r * mass_stride]; rank_lo / rank_hi / total are then derived here instead of on the host
    const double *dev_masses;
    int64_t mass_stride;
    int32_t n_ranks, my_rank;
    // cond_low with the rotated pass left unwritten: its input (virt_in, 2^n_active amplitudes) and its arguments;
    // the leaf's images are computed (low_image) instead of loaded
    const void *virt_in;
    ExpandTreeArgs virt;
};

template <typename R>
__global__ void __launch_bounds__(kThreads) k_sample(const __grid_constant__ SampleArgs a) {
    using C2 = typename CplxOf<R>::T;
    // virtual leaf: f_j[bit] of each of the leaf's inputs (at most 2: the finer level sums input pairs) and their
    // diagonal products, worked out once per shot
    __shared__ C2 s_vf[kThreads / 32][2][QCM_MAX_EXPAND][2];
    __shared__ C2 s_vp[kThreads / 32][2];
    const int lane = threadIdx.x & 31;
    const uint64_t warp0 = ((uint64_t)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
    const uint64_t nwarps = ((uint64_t)gridDim.x * blockDim.x) >> 5;
    const int cb = a.n_active < kChunkBits ? a.n_active : kChunkBits;
    const void *const state = batch_ptr(a.state, a.bstate);
    uint64_t *const keys_out = batch_ptr(a.keys_out, a.bkeys);
    const uint64_t stream = a.streams ? a.streams[blockIdx.y] : a.stream;
    double total = a.totals ? a.totals[blockIdx.y] : a.total;
    double rank_lo = a.rank_lo, rank_hi = a.rank_hi;
    if (a.dev_masses) {                              // same left-to-right sums as the host version
        double t = 0.0, lo = 0.0;
        for (int r = 0; r < a.n_ranks; ++r) {
            if (r == a.my_rank) lo = t;
            t += a.dev_masses[(int64_t)r * a.mass_stride];
        }
        total = t;
        rank_lo = lo;
        rank_hi = (a.my_rank == a.n_ranks - 1) ? 1e300 : lo + a.dev_masses[(int64_t)a.my_rank * a.mass_stride];
    }
    for (uint64_t s = warp0; s < a.shots; s += nwarps) {
        double u = philox_uniform(a.seed, stream, s) * total;
        const bool mine = (u >= rank_lo) && (u < rank_hi);
        if (a.mine_out && lane == 0) a.mine_out[s] = mine ? 1 : 0;
        if (!mine) {
            if (lane == 0) keys_out[s] = 0;
            continue;
        }
        u -= rank_lo;
        uint64_t node = 0;
        for (int l = a.n_levels - 1; l >= 0; --l) {
            const double *lv = batch_ptr(a.level[l], a.btree);
            const uint64_t first = node << kFanBits;
            const uint64_t left = a.level_n[l] - first;
            const uint32_t cnt = left < (1ull << kFanBits) ? (uint32_t)left : (1u << kFanBits);
            const uint32_t c = warp_pick([&](uint32_t i) { return lv[first + i]; }, cnt, u, lane);
            node = first + c;
        }
        // node = chunk index; search the amplitudes of the chunk (through the finer level if there is one)
        uint64_t afirst = node << cb;
        uint32_t leaf_cnt = 1u << cb;
        if (a.sub && a.sub_strided) {
            // strided groups (generic tree build): group g = lane partial g of k_chunk_sums, then one of its 32 amplitudes
            const double *sp = batch_ptr(a.sub, a.bsub) + node * 32;
            const uint32_t g = warp_pick([&](uint32_t i) { return sp[i]; }, 32u, u, lane);
            constexpr uint32_t VV = sizeof(R) == 4 ? 2u : 1u;
            auto member = [&](uint32_t i) -> uint64_t { return (uint64_t)VV * sub_vec(g, i / VV) + (i % VV); };
            auto amp_ws = [&](uint32_t i) -> double {
                if constexpr (sizeof(R) == 4) {
                    const float2 t = reinterpret_cast<const float2 *>(state)[afirst + member(i)];
                    return (double)t.x * (double)t.x + (double)t.y * (double)t.y;
                } else {
                    const double2 t = reinterpret_cast<const double2 *>(state)[afirst + member(i)];
                    return t.x * t.x + t.y * t.y;
                }
            };
            const uint32_t c = warp_pick(amp_ws, 32u, u, lane);
            if (lane == 0) {
                uint64_t li = afirst + member(c);
                if (a.rot_m) li = (li >> a.rot_m) | ((li & ((1ull << a.rot_m) - 1ull)) << a.rot_nin);
                const uint64_t gi = li | a.rank_bits;
                uint64_t key = gi;
                if (a.n_clbits > 0) {
                    key = 0;
                    for (int cc = 0; cc < a.n_clbits; ++cc) {
                        const int q = a.clbit_qubit[cc];
                        if (q >= 0) key |= ((gi >> q) & 1ull) << cc;
                    }
                }
                keys_out[s] = key;
            }
            continue;
        }
        if (a.sub) {
            const uint32_t nsub = 1u << (cb - a.sub_bits);
            const double *sp = a.sub + (node << (cb - a.sub_bits));      // (fused checkpoint only: never batched)
            const uint32_t c = warp_pick([&](uint32_t i) { return sp[i]; }, nsub, u, lane);
            afirst += (uint64_t)c << a.sub_bits;
            leaf_cnt = 1u << a.sub_bits;
        }
        const int nb = 1 << a.cond_bits;
        auto amp_w = [&](uint64_t i) -> double {
            if constexpr (sizeof(R) == 4) {
                const float2 t = reinterpret_cast<const float2 *>(state)[i];
                return (double)t.x * (double)t.x + (double)t.y * (double)t.y;
            } else {
                const double2 t = reinterpret_cast<const double2 *>(state)[i];
                return t.x * t.x + t.y * t.y;
            }
        };
        // leaf: the remaining x's, each with its 2^cond_bits images -- one flat, lane-strided search over
        // the (x, image) pairs (image-major, so that consecutive lanes read consecutive amplitudes)
        uint64_t within;
        if (a.cond_low && a.virt_in) {
            // rotated expansion, left unwritten: the same flat search, over computed images
            const int wl = threadIdx.x >> 5;
            const uint32_t k = (uint32_t)lane >> 4, j = ((uint32_t)lane >> 1) & 7u;
            const uint64_t gi = (afirst + k) | a.rank_bits;
            __syncwarp();                                 // the previous shot is done with the factors
            if (k < leaf_cnt && (int)j < a.virt.M) {
                C2 f;
                low_fac_global<R>(a.virt, (int)j, gi, lane & 1, f.x, f.y);
                s_vf[wl][k][j][lane & 1] = f;
            }
            if ((lane & 15) == 0 && k < leaf_cnt) {
                C2 p = reinterpret_cast<const C2 *>(a.virt_in)[afirst + k];
                low_diag(a.virt, gi, [&](int d, uint32_t idx) { return low_diag_global<R>(a.virt, d, idx); }, p.x, p.y);
                s_vp[wl][k] = p;
            }
            __syncwarp();
            auto img_w = [&](uint32_t i) -> double {
                const uint32_t x = i >> a.cond_bits;
                auto fac = [&](int m, int bit, R &fr, R &fi) {
                    const C2 f = s_vf[wl][x][m][bit];
                    fr = f.x; fi = f.y;
                };
                const C2 p = s_vp[wl][x];
                R o_r, o_i;
                low_image<R, sizeof(R) == 4 ? 2 : 1>(fac, a.cond_bits, p.x, p.y, i & (uint32_t)(nb - 1), o_r, o_i);
                return (double)o_r * (double)o_r + (double)o_i * (double)o_i;
            };
            const uint32_t c = warp_pick(img_w, leaf_cnt * (uint32_t)nb, u, lane);
            within = (uint64_t)(c >> a.cond_bits) + ((uint64_t)(c & (uint32_t)(nb - 1)) << a.n_active);
        } else if (a.cond_low) {
            // rotated expansion: the (x, image) pairs of the leaf are one contiguous run, x-major
            const uint32_t c = warp_pick([&](uint32_t i) { return amp_w((afirst << a.cond_bits) + i); },
                                         leaf_cnt * (uint32_t)nb, u, lane);
            within = (uint64_t)(c >> a.cond_bits) + ((uint64_t)(c & (uint32_t)(nb - 1)) << a.n_active);
        } else {
            const uint32_t lbits = 31u - (uint32_t)__clz(leaf_cnt);
            const uint32_t c = warp_pick(
                [&](uint32_t i) { return amp_w(afirst + (i & (leaf_cnt - 1u)) + ((uint64_t)(i >> lbits) << a.n_active)); },
                leaf_cnt * (uint32_t)nb, u, lane);
            within = (uint64_t)(c & (leaf_cnt - 1u)) + ((uint64_t)(c >> lbits) << a.n_active);
        }
        if (lane == 0) {
            uint64_t li = afirst + within;
            if (a.rot_m && !a.cond_bits) li = (li >> a.rot_m) | ((li & ((1ull << a.rot_m) - 1ull)) << a.rot_nin);
            const uint64_t gi = li | a.rank_bits;
            uint64_t key = gi;
            if (a.n_clbits > 0) {
                key = 0;
                for (int c = 0; c < a.n_clbits; ++c) {
                    const int q = a.clbit_qubit[c];
                    if (q >= 0) key |= ((gi >> q) & 1ull) << c;
                }
            }
            keys_out[s] = key;
        }
    }
}

// ----------------------------------------------------------------------------------
// Sampling a PRODUCT state (the program was INIT_PRODUCT and nothing else: e.g. the stored qubits of a QCMRF at
// measure-and-release width, whose clique sweeps are all released -- DESIGN.md 2a): the qubits are independent, so a
// shot is one Bernoulli draw per qubit from its 2-vector -- no sum tree, no pass over the state at all.  One thread per
// shot; Philox4x32-10 keyed (seed ^ kProductKey, stream) at counter (shot, qubit / 4) yields four 32-bit draws per call.
// ----------------------------------------------------------------------------------
constexpr uint64_t kProductKey = 0xC2B2AE3D27D4EB4Full;

__device__ __forceinline__ void philox4(uint64_t seed, uint64_t stream, uint64_t ctr, uint32_t (&out)[4]) {
    uint32_t c[4] = {(uint32_t)ctr, (uint32_t)(ctr >> 32), (uint32_t)stream, (uint32_t)(stream >> 32)};
    uint32_t k[2] = {(uint32_t)seed, (uint32_t)(seed >> 32)};
#pragma unroll
    for (int r = 0; r < 10; ++r) philox_round(c, k);
    out[0] = c[0]; out[1] = c[1]; out[2] = c[2]; out[3] = c[3];
}

struct ProductSampleArgs {
    const double *qv;               // device: n * 4 doubles per point (amp0.re, amp0.im, amp1.re, amp1.im per qubit)
    int32_t n;                      // qubits of the product state (<= 64)
    uint64_t shots, seed, stream;
    const uint64_t *streams;        // batched: per-point streams (or null)
    uint64_t bqv, bkeys;            // batch strides, bytes
    int32_t n_clbits;               // 0 => raw indices
    int8_t clbit_qubit[64];
    uint64_t *keys_out;
};

static __global__ void __launch_bounds__(kThreads) k_sample_product(const __grid_constant__ ProductSampleArgs a) {
    __shared__ double p1[64];
    const double *qv = batch_ptr(a.qv, a.bqv);
    if (threadIdx.x < (unsigned)a.n) {
        const double w0 = qv[4 * threadIdx.x] * qv[4 * threadIdx.x] + qv[4 * threadIdx.x + 1] * qv[4 * threadIdx.x + 1];
        const double w1 = qv[4 * threadIdx.x + 2] * qv[4 * threadIdx.x + 2] + qv[4 * threadIdx.x + 3] * qv[4 * threadIdx.x + 3];
        p1[threadIdx.x] = (w0 + w1) > 0.0 ? w1 / (w0 + w1) : 0.0;
    }
    __syncthreads();
    const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= a.shots) return;
    const uint64_t stream = a.streams ? a.streams[blockIdx.y] : a.stream;
    uint64_t idx = 0;
    for (int q0 = 0; q0 < a.n; q0 += 4) {
        uint32_t r[4];
        philox4(a.seed ^ kProductKey, stream, s * 16ull + (uint64_t)(q0 >> 2), r);
#pragma unroll
        for (int j = 0; j < 4; ++j) {
            const int q = q0 + j;
            if (q < a.n && (double)r[j] * (1.0 / 4294967296.0) < p1[q]) idx |= 1ull << q;
        }
    }
    uint64_t key = idx;
    if (a.n_clbits > 0) {
        key = 0;
        for (int c = 0; c < a.n_clbits; ++c) {
            const int q = a.clbit_qubit[c];
            if (q >= 0) key |= ((idx >> q) & 1ull) << c;
        }
    }
    batch_ptr(a.keys_out, a.bkeys)[s] = key;
}

// total[y] = sum of the top tree level of sweep point y, in index order (one thread per point)
static __global__ void k_batch_totals(const double *top, uint64_t n_top, uint64_t btree, double *totals, int batch) {
    const int y = blockIdx.x * blockDim.x + threadIdx.x;
    if (y >= batch) return;
    const double *p = reinterpret_cast<const double *>(reinterpret_cast<const unsigned char *>(top) + (uint64_t)y * btree);
    double t = 0.0;
    for (uint64_t i = 0; i < n_top; ++i) t += p[i];
    totals[y] = t;
}

// ----------------------------------------------------------------------------------
// Measure-and-release width (DESIGN.md 2a): full-width keys from the sampled basis states of the
// stored qubits.  A released qubit k (never stored: one sweep materialised it from |0> and nothing
// used it again) reads 1 with probability p1_k[index bits of the sampled state at ctrl_k]; its
// uniform is Philox keyed by (seed ^ kReleasedKey, stream) at counter shot * nv + k, independent of
// the sampler's stream.  One thread per shot, in place over the sampler's output.
// ----------------------------------------------------------------------------------
constexpr uint64_t kReleasedKey = 0x9E3779B97F4A7C15ull;
constexpr int kMaxReleased = 64;

struct ReleasedArgs {
    uint64_t *keys;                 // in: raw basis-state indices (k_sample without a clbit map); out: keys
    uint64_t shots, seed, stream;
    const double *p1;               // device: concatenated tables, p1_off[k] their starts
    int32_t nv, n_clbits;
    int32_t p1_off[kMaxReleased];
    int8_t n_ctrl[kMaxReleased];
    int8_t ctrl[kMaxReleased][QCM_MAX_CTRL];
    int8_t vclbit[kMaxReleased];    // clbit of released qubit k, or -1
    int8_t clbit_pos[64];           // physical position feeding clbit c, or -1
    uint64_t bkeys, bp1;            // batch strides in bytes (keys, p1 tables); per-point Philox streams (or null)
    const uint64_t *streams;
};

static __global__ void __launch_bounds__(kThreads) k_released_keys(const __grid_constant__ ReleasedArgs a) {
    const uint64_t s = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x;
    if (s >= a.shots) return;
    uint64_t *const keys = batch_ptr(a.keys, a.bkeys);
    const double *const p1 = batch_ptr(a.p1, a.bp1);
    const uint64_t stream = a.streams ? a.streams[blockIdx.y] : a.stream;
    const uint64_t r = keys[s];
    uint64_t key = 0;
    for (int c = 0; c < a.n_clbits; ++c) {
        const int p = a.clbit_pos[c];
        if (p >= 0) key |= ((r >> p) & 1ull) << c;
    }
    for (int k = 0; k < a.nv; ++k) {
        if (a.vclbit[k] < 0) continue;
        uint32_t idx = 0;
        for (int j = 0; j < a.n_ctrl[k]; ++j) idx |= (uint32_t)((r >> a.ctrl[k][j]) & 1ull) << j;
        const double u = philox_uniform(a.seed ^ kReleasedKey, stream, s * (uint64_t)a.nv + (uint64_t)k);
        if (u < p1[a.p1_off[k] + idx]) key |= 1ull << a.vclbit[k];
    }
    keys[s] = key;
}

// ----------------------------------------------------------------------------------
// Post-selection.
// ----------------------------------------------------------------------------------
// contiguous kept set (QCMRF: the first 2^n amplitudes): probs[i] = |amp_i|^2 and a
// deterministic two-stage sum (per-block partials, then k_tree_level).
// VIRT: the rotated pass that produced the state was left unwritten; `state` is its input and amplitude i is image 0
// of input i, computed with the pass's arguments `va` (same loop, same order of the sums).
template <typename R, bool VIRT>
__global__ void __launch_bounds__(kThreads) k_probs_prefix(const void *state, uint64_t count, int shift, double *probs, double *partial,
                                                           uint64_t bstate, uint64_t bprobs, uint64_t bpartial,
                                                           const __grid_constant__ ExpandTreeArgs va) {
    __shared__ double wsum[kThreads / 32];
    state = batch_ptr(state, bstate);
    if (probs) probs = batch_ptr(probs, bprobs);
    partial = batch_ptr(partial, bpartial);
    double acc = 0.0;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
        double w;
        if constexpr (VIRT) {
            using C2 = typename CplxOf<R>::T;
            C2 p = reinterpret_cast<const C2 *>(state)[i];
            const uint64_t gi = i | va.rank_bits;
            low_diag(va, gi, [&](int d, uint32_t idx) { return low_diag_global<R>(va, d, idx); }, p.x, p.y);
            R o_r, o_i;
            low_image<R, sizeof(R) == 4 ? 2 : 1>([&](int m, int bit, R &fr, R &fi) { low_fac_global<R>(va, m, gi, bit, fr, fi); },
                                                 va.M, p.x, p.y, 0u, o_r, o_i);
            w = (double)o_r * (double)o_r + (double)o_i * (double)o_i;
        } else if constexpr (sizeof(R) == 4) {
            const float2 t = reinterpret_cast<const float2 *>(state)[i << shift];
            w = (double)t.x * (double)t.x + (double)t.y * (double)t.y;
        } else {
            const double2 t = reinterpret_cast<const double2 *>(state)[i << shift];
            w = t.x * t.x + t.y * t.y;
        }
        if (probs) probs[i] = w;
        acc += w;
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < kThreads / 32; ++i) t += wsum[i];
        partial[blockIdx.x] = t;
    }
}

// general mask/value: fp64 atomics into probs, per-block partials for the kept mass
template <typename R>
__global__ void __launch_bounds__(kThreads) k_postselect_general(const void *state, int n_active, uint64_t rank_bits,
                                                                  uint64_t mask, uint64_t value, uint64_t out_mask,
                                                                  int rot_m, int rot_nin, double *probs, double *partial,
                                                                  uint64_t bstate = 0, uint64_t bprobs = 0, uint64_t bpartial = 0) {
    __shared__ double wsum[kThreads / 32];
    state = batch_ptr(state, bstate);
    if (probs) probs = batch_ptr(probs, bprobs);
    partial = batch_ptr(partial, bpartial);
    double acc = 0.0;
    const uint64_t count = 1ull << n_active;
    const uint64_t stride = (uint64_t)gridDim.x * blockDim.x;
    for (uint64_t i = (uint64_t)blockIdx.x * blockDim.x + threadIdx.x; i < count; i += stride) {
        // i walks physical addresses; rotated storage: logical = (i >> rot_m) | ((i & (2^rot_m - 1)) << rot_nin)
        const uint64_t li = rot_m ? ((i >> rot_m) | ((i & ((1ull << rot_m) - 1ull)) << rot_nin)) : i;
        const uint64_t gi = li | rank_bits;
        if ((gi & mask) != value) continue;
        double w;
        if constexpr (sizeof(R) == 4) {
            const float2 t = reinterpret_cast<const float2 *>(state)[i];
            w = (double)t.x * (double)t.x + (double)t.y * (double)t.y;
        } else {
            const double2 t = reinterpret_cast<const double2 *>(state)[i];
            w = t.x * t.x + t.y * t.y;
        }
        if (probs && w != 0.0) atomicAdd(probs + (gi & out_mask), w);
        acc += w;
    }
    acc = warp_sum(acc);
    if ((threadIdx.x & 31) == 0) wsum[threadIdx.x >> 5] = acc;
    __syncthreads();
    if (threadIdx.x == 0) {
        double t = 0.0;
        for (int i = 0; i < kThreads / 32; ++i) t += wsum[i];
        partial[blockIdx.x] = t;
    }
}

}  // namespace qcm
