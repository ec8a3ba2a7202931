// Batched small-circuit path: one thread block per circuit, the whole statevector in
// shared memory, gate program + post-selection + prefix sums + shot sampling in ONE
// launch.  This is how the fixture-sized models of the reference's experiment
// (70 circuits of 3..10 qubits, /root/reference/run_experiment.py:44-57) are served:
// at those sizes a per-gate launch would be pure launch latency.
#include <cuda_runtime.h>

#include <algorithm>
#include <cstdio>
#include <cstring>
#include <mutex>
#include <string>
#include <vector>

#include "qcm_kernels.cuh"
#include "qcm_noise.h"
#include "qcmrf_b200.h"

using namespace qcm;

namespace {

struct SmallArgs {
    int n_circuits;
    const int32_t *n_qubits;
    const int64_t *op_begin;
    const qcm_op *ops;
    const double *tables;
    const int32_t *clbit_qubit;   // [n_circuits][64]
    const int32_t *n_clbits;
    const uint64_t *ps_mask, *ps_value;
    const int32_t *ps_bits;
    const int64_t *probs_begin;   // offsets into probs_out
    const uint64_t *stream_ids;   // may be null
    uint64_t shots, seed;
    uint64_t *keys_out;
    double *probs_out;
    double *kept_out;
    int32_t *status_out;          // per circuit: 0 ok, else offending op index + 1
};

template <typename R> struct Cx { R x, y; };

template <typename R>
__global__ void __launch_bounds__(kThreads) k_small(const SmallArgs a) {
    extern __shared__ __align__(16) unsigned char smem_raw[];
    const int c = blockIdx.x;
    const int N = a.n_qubits[c];
    const uint32_t dim = 1u << N;
    Cx<R> *psi = reinterpret_cast<Cx<R> *>(smem_raw);
    double *pre = reinterpret_cast<double *>(smem_raw + sizeof(Cx<R>) * dim);
    __shared__ double wpart[kThreads];
    __shared__ int bad;
    const int tid = threadIdx.x;
    if (tid == 0) bad = 0;
    // |0...0> unless the program starts with INIT_PRODUCT
    for (uint32_t i = tid; i < dim; i += kThreads) { psi[i].x = (i == 0) ? R(1) : R(0); psi[i].y = R(0); }
    __syncthreads();

    for (int64_t oi = a.op_begin[c]; oi < a.op_begin[c + 1]; ++oi) {
        const qcm_op op = a.ops[oi];
        const double *tab = a.tables + op.table_off;
        if (op.kind == QCM_OP_INIT_PRODUCT) {
            for (uint32_t i = tid; i < dim; i += kThreads) {
                double re = 1.0, im = 0.0;
                for (int q = 0; q < N; ++q) {
                    const int b = (i >> q) & 1;
                    const double fr = tab[4 * q + 2 * b], fi = tab[4 * q + 2 * b + 1];
                    const double nr = re * fr - im * fi;
                    im = re * fi + im * fr;
                    re = nr;
                }
                psi[i].x = (R)re; psi[i].y = (R)im;
            }
        } else if (op.kind == QCM_OP_MUX1Q) {
            const int t = op.target;
            for (uint32_t p = tid; p < (dim >> 1); p += kThreads) {
                const uint32_t i0 = (uint32_t)insert_zero(p, t), i1 = i0 | (1u << t);
                uint32_t idx = 0;
                for (int j = 0; j < op.n_ctrl; ++j) idx |= ((i0 >> op.ctrl[j]) & 1u) << j;
                const double *m = tab + 8 * idx;
                const R x0 = psi[i0].x, y0 = psi[i0].y, x1 = psi[i1].x, y1 = psi[i1].y;
                const R m0 = (R)m[0], m1 = (R)m[1], m2 = (R)m[2], m3 = (R)m[3];
                const R m4 = (R)m[4], m5 = (R)m[5], m6 = (R)m[6], m7 = (R)m[7];
                psi[i0].x = m0 * x0 - m1 * y0 + m2 * x1 - m3 * y1;
                psi[i0].y = m0 * y0 + m1 * x0 + m2 * y1 + m3 * x1;
                psi[i1].x = m4 * x0 - m5 * y0 + m6 * x1 - m7 * y1;
                psi[i1].y = m4 * y0 + m5 * x0 + m6 * y1 + m7 * x1;
            }
        } else if (op.kind == QCM_OP_DIAG) {
            for (uint32_t i = tid; i < dim; i += kThreads) {
                uint32_t idx = 0;
                for (int j = 0; j < op.n_ctrl; ++j) idx |= ((i >> op.ctrl[j]) & 1u) << j;
                const R cr = (R)tab[2 * idx], ci = (R)tab[2 * idx + 1];
                const R x = psi[i].x, y = psi[i].y;
                psi[i].x = cr * x - ci * y;
                psi[i].y = cr * y + ci * x;
            }
        } else if (op.kind == QCM_OP_SWAP) {
            const int qa = min(op.target, op.ctrl[0]), qb = max(op.target, op.ctrl[0]);
            if (qa != qb)
                for (uint32_t p = tid; p < (dim >> 2); p += kThreads) {
                    const uint32_t b = (uint32_t)insert_zero(insert_zero(p, qa), qb);
                    const uint32_t i10 = b | (1u << qa), i01 = b | (1u << qb);
                    const Cx<R> t = psi[i10];
                    psi[i10] = psi[i01];
                    psi[i01] = t;
                }
        } else if (op.kind == QCM_OP_BLOCK || op.kind == QCM_OP_EXTEND) {
            // members follow as plain MUX1Q ops; the state is always fully materialised here
        } else {
            if (tid == 0) bad = (int)(oi - a.op_begin[c]) + 1;
        }
        __syncthreads();
    }
    if (tid == 0) a.status_out[c] = bad;

    // ---- probabilities, inclusive prefix (fixed order) ---------------------------------
    const uint32_t per = (dim + kThreads - 1) / kThreads;          // contiguous segment per thread
    const uint32_t s0 = min(dim, tid * per), s1 = min(dim, s0 + per);
    double acc = 0.0;
    for (uint32_t i = s0; i < s1; ++i) {
        const double w = (double)psi[i].x * (double)psi[i].x + (double)psi[i].y * (double)psi[i].y;
        acc += w;
        pre[i] = acc;
    }
    wpart[tid] = acc;
    __syncthreads();
    if (tid == 0) {
        double run = 0.0;
        for (int i = 0; i < kThreads; ++i) { const double t = wpart[i]; wpart[i] = run; run += t; }
    }
    __syncthreads();
    const double off = wpart[tid];
    for (uint32_t i = s0; i < s1; ++i) pre[i] += off;
    __syncthreads();
    const double total = pre[dim - 1];

    // ---- post-selection ------------------------------------------------------------------
    {
        const uint64_t mask = a.ps_mask[c], value = a.ps_value[c];
        const uint32_t omask = (1u << a.ps_bits[c]) - 1u;
        double *pout = a.probs_out ? a.probs_out + a.probs_begin[c] : nullptr;
        double kept = 0.0;
        for (uint32_t i = tid; i < dim; i += kThreads) {
            if (((uint64_t)i & mask) != value) continue;
            const double w = pre[i] - (i ? pre[i - 1] : 0.0);
            const double wx = (double)psi[i].x * (double)psi[i].x + (double)psi[i].y * (double)psi[i].y;
            (void)w;
            kept += wx;
            if (pout && wx != 0.0) atomicAdd(pout + (i & omask), wx);
        }
        kept = warp_sum(kept);
        __syncthreads();
        if ((tid & 31) == 0) wpart[tid >> 5] = kept;
        __syncthreads();
        if (tid == 0) {
            double t = 0.0;
            for (int i = 0; i < kThreads / 32; ++i) t += wpart[i];
            a.kept_out[c] = t;
        }
    }

    // ---- shots --------------------------------------------------------------------------------
    if (a.keys_out) {
        const int ncl = a.n_clbits[c];
        const int32_t *cq = a.clbit_qubit + 64 * c;
        for (uint64_t s = tid; s < a.shots; s += kThreads) {
            const double u = philox_uniform(a.seed, a.stream_ids ? a.stream_ids[c] : (uint64_t)c, s) * total;
            uint32_t lo = 0, hi = dim - 1;             // first i with pre[i] > u
            while (lo < hi) {
                const uint32_t mid = (lo + hi) >> 1;
                if (pre[mid] > u) hi = mid; else lo = mid + 1;
            }
            // rounding guard: never return a zero-probability state
            while (lo > 0 && pre[lo] == pre[lo - 1]) --lo;
            uint64_t key = lo;
            if (ncl > 0) {
                key = 0;
                for (int b = 0; b < ncl; ++b) {
                    const int q = cq[b];
                    if (q >= 0) key |= (uint64_t)((lo >> q) & 1u) << b;
                }
            }
            a.keys_out[(uint64_t)c * a.shots + s] = key;
        }
    }
}

thread_local std::string g_small_error;

}  // namespace

namespace qcm {

SmallArena g_arena[64];

cudaError_t arena_reserve(SmallArena &A, size_t dev_bytes, size_t pin_bytes) {
    cudaError_t e;
    if (!A.st) {
        if ((e = cudaStreamCreateWithFlags(&A.st, cudaStreamNonBlocking)) != cudaSuccess) return e;
        if ((e = cudaEventCreate(&A.e0)) != cudaSuccess) return e;
        if ((e = cudaEventCreate(&A.e1)) != cudaSuccess) return e;
    }
    if (A.dev_cap < dev_bytes) {
        if (A.dev) cudaFree(A.dev);
        A.dev = nullptr; A.dev_cap = 0;
        if ((e = cudaMalloc(&A.dev, dev_bytes + dev_bytes / 4)) != cudaSuccess) return e;
        A.dev_cap = dev_bytes + dev_bytes / 4;
    }
    if (A.pin_cap < pin_bytes) {
        if (A.pin) cudaFreeHost(A.pin);
        A.pin = nullptr; A.pin_cap = 0;
        if ((e = cudaMallocHost(&A.pin, pin_bytes + pin_bytes / 4)) != cudaSuccess) return e;
        A.pin_cap = pin_bytes + pin_bytes / 4;
    }
    return cudaSuccess;
}

}  // namespace qcm

namespace {

// qcm_run_batch_small; with `readout` (qcm_run_batch_small_readout) the keys are flipped on the device before the copy.
int run_batch_small(int device, int precision, int n_circuits, const int32_t *n_qubits, const int64_t *op_begin,
                    const qcm_op *ops, const double *tables, size_t n_tables, const int32_t *clbit_qubit,
                    const int32_t *n_clbits, const double *readout, const uint64_t *ps_mask, const uint64_t *ps_value,
                    const int32_t *ps_bits, const uint64_t *stream_ids, uint64_t shots, uint64_t seed, uint64_t *keys_out,
                    double *probs_out, double *kept_out, double *device_ms_out) {
    if (n_circuits <= 0 || !n_qubits || !op_begin || !ops || !ps_mask || !ps_value || !ps_bits || !kept_out) return QCM_ERR_INVALID;
    if (precision != QCM_C64 && precision != QCM_C128) return QCM_ERR_INVALID;
    if (shots && (!keys_out || !clbit_qubit || !n_clbits)) return QCM_ERR_INVALID;
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0) return QCM_ERR_NO_DEVICE;
    if (device < 0 || device >= ndev || device >= 64) return QCM_ERR_INVALID;
    int maxq = 0;
    std::vector<int64_t> pbeg(n_circuits + 1, 0);
    for (int c = 0; c < n_circuits; ++c) {
        if (n_qubits[c] < 0 || n_qubits[c] > kSmallMaxQubits) return QCM_ERR_UNSUPPORTED;
        if (ps_bits[c] < 0 || ps_bits[c] > n_qubits[c]) return QCM_ERR_INVALID;
        if (op_begin[c + 1] < op_begin[c]) return QCM_ERR_INVALID;
        maxq = std::max(maxq, n_qubits[c]);
        pbeg[c + 1] = pbeg[c] + (1ll << ps_bits[c]);
    }
    const int64_t n_ops = op_begin[n_circuits];
    for (int64_t i = 0; i < n_ops; ++i) {
        const qcm_op &op = ops[i];
        if (op.n_ctrl < 0 || (op.kind != QCM_OP_BLOCK && op.n_ctrl > QCM_MAX_CTRL)) return QCM_ERR_INVALID;
        size_t need = op.kind == QCM_OP_MUX1Q ? (8ull << op.n_ctrl) : op.kind == QCM_OP_DIAG ? (2ull << op.n_ctrl) : 0;
        if (need && (op.table_off < 0 || (size_t)op.table_off + need > n_tables)) return QCM_ERR_INVALID;
    }
#define SM_CUDA(call)                                                                  \
    do {                                                                                \
        cudaError_t e_ = (call);                                                        \
        if (e_ != cudaSuccess) {                                                        \
            g_small_error = std::string(#call) + ": " + cudaGetErrorString(e_);         \
            rc = (e_ == cudaErrorMemoryAllocation) ? QCM_ERR_NOMEM : QCM_ERR_CUDA;      \
            goto done;                                                                  \
        }                                                                               \
    } while (0)
    int rc = QCM_OK;
    SmallArgs a{};
    SmallArena &A = g_arena[device];
    std::lock_guard<std::mutex> lock(A.mu);
    std::vector<int32_t> status(n_circuits, 0);
    const size_t amp = precision == QCM_C64 ? 8 : 16;
    const size_t smem = ((size_t)amp + 8) << maxq;
    const size_t nc = (size_t)n_circuits;
    // input blob (host pinned, mirrored at the start of the device buffer), then the outputs
    size_t off = 0;
    auto take = [&](size_t bytes) { const size_t o = off; off += up256(std::max<size_t>(bytes, 1)); return o; };
    const size_t o_nq = take(nc * 4), o_ob = take((nc + 1) * 8), o_ops = take((size_t)n_ops * sizeof(qcm_op)),
                 o_tab = take(n_tables * 8), o_pm = take(nc * 8), o_pv = take(nc * 8), o_psb = take(nc * 4),
                 o_pb = take((nc + 1) * 8), o_sid = take(stream_ids ? nc * 8 : 0), o_cq = take(shots ? 64 * nc * 4 : 0),
                 o_ncl = take(shots ? nc * 4 : 0);
    const size_t o_ro = (shots && readout) ? take(nc * 128 * 8) : 0;
    const size_t in_bytes = off;
    const size_t o_keys = take(shots ? shots * nc * 8 : 0), o_kept = take(nc * 8), o_status = take(nc * 4),
                 o_probs = take(probs_out ? (size_t)pbeg[n_circuits] * 8 : 0);
    const size_t dev_bytes = off;
    char *hp, *dp;
    SM_CUDA(cudaSetDevice(device));
    SM_CUDA(arena_reserve(A, dev_bytes, in_bytes));
    hp = (char *)A.pin;
    dp = (char *)A.dev;
    memcpy(hp + o_nq, n_qubits, nc * 4);
    memcpy(hp + o_ob, op_begin, (nc + 1) * 8);
    memcpy(hp + o_ops, ops, (size_t)n_ops * sizeof(qcm_op));
    if (n_tables) memcpy(hp + o_tab, tables, n_tables * 8);
    memcpy(hp + o_pm, ps_mask, nc * 8);
    memcpy(hp + o_pv, ps_value, nc * 8);
    memcpy(hp + o_psb, ps_bits, nc * 4);
    memcpy(hp + o_pb, pbeg.data(), (nc + 1) * 8);
    if (stream_ids) memcpy(hp + o_sid, stream_ids, nc * 8);
    if (shots) {
        memcpy(hp + o_cq, clbit_qubit, 64 * nc * 4);
        memcpy(hp + o_ncl, n_clbits, nc * 4);
        if (readout) memcpy(hp + o_ro, readout, nc * 128 * 8);
    }
    SM_CUDA(cudaMemcpyAsync(dp, hp, in_bytes, cudaMemcpyHostToDevice, A.st));
    if (probs_out) SM_CUDA(cudaMemsetAsync(dp + o_probs, 0, (size_t)pbeg[n_circuits] * 8, A.st));
    a.n_circuits = n_circuits;
    a.n_qubits = (const int32_t *)(dp + o_nq);
    a.op_begin = (const int64_t *)(dp + o_ob);
    a.ops = (const qcm_op *)(dp + o_ops);
    a.tables = (const double *)(dp + o_tab);
    a.clbit_qubit = shots ? (const int32_t *)(dp + o_cq) : nullptr;
    a.n_clbits = shots ? (const int32_t *)(dp + o_ncl) : nullptr;
    a.ps_mask = (const uint64_t *)(dp + o_pm);
    a.ps_value = (const uint64_t *)(dp + o_pv);
    a.ps_bits = (const int32_t *)(dp + o_psb);
    a.probs_begin = (const int64_t *)(dp + o_pb);
    a.shots = shots;
    a.seed = seed;
    a.keys_out = shots ? (uint64_t *)(dp + o_keys) : nullptr;
    a.probs_out = probs_out ? (double *)(dp + o_probs) : nullptr;
    a.kept_out = (double *)(dp + o_kept);
    a.status_out = (int32_t *)(dp + o_status);
    a.stream_ids = stream_ids ? (const uint64_t *)(dp + o_sid) : nullptr;
    if (precision == QCM_C64) {
        SM_CUDA(cudaFuncSetAttribute(k_small<float>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        SM_CUDA(cudaEventRecord(A.e0, A.st));
        k_small<float><<<n_circuits, kThreads, smem, A.st>>>(a);
    } else {
        SM_CUDA(cudaFuncSetAttribute(k_small<double>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        SM_CUDA(cudaEventRecord(A.e0, A.st));
        k_small<double><<<n_circuits, kThreads, smem, A.st>>>(a);
    }
    SM_CUDA(cudaGetLastError());
    if (shots && readout)
        SM_CUDA(launch_readout_keys(A.st, n_circuits, shots, seed, a.stream_ids, a.n_clbits, (const double *)(dp + o_ro),
                                    a.keys_out));
    SM_CUDA(cudaEventRecord(A.e1, A.st));
    SM_CUDA(cudaMemcpyAsync(kept_out, dp + o_kept, nc * sizeof(double), cudaMemcpyDeviceToHost, A.st));
    SM_CUDA(cudaMemcpyAsync(status.data(), dp + o_status, nc * sizeof(int32_t), cudaMemcpyDeviceToHost, A.st));
    if (probs_out) SM_CUDA(cudaMemcpyAsync(probs_out, dp + o_probs, (size_t)pbeg[n_circuits] * sizeof(double), cudaMemcpyDeviceToHost, A.st));
    if (shots) SM_CUDA(cudaMemcpyAsync(keys_out, dp + o_keys, shots * nc * sizeof(uint64_t), cudaMemcpyDeviceToHost, A.st));
    SM_CUDA(cudaStreamSynchronize(A.st));
    if (device_ms_out) {
        float ms = 0.f;
        SM_CUDA(cudaEventElapsedTime(&ms, A.e0, A.e1));
        *device_ms_out = ms;
    }
    for (int c = 0; c < n_circuits; ++c)
        if (status[c]) { g_small_error = "circuit " + std::to_string(c) + ": unsupported op at position " + std::to_string(status[c] - 1); rc = QCM_ERR_INVALID; }
done:
    return rc;
#undef SM_CUDA
}

}  // namespace

extern "C" {

int qcm_small_max_qubits(int precision) {
    return (precision == QCM_C64 || precision == QCM_C128) ? kSmallMaxQubits : 0;
}

int qcm_run_batch_small(int device, int precision, int n_circuits, const int32_t *n_qubits, const int64_t *op_begin,
                        const qcm_op *ops, const double *tables, size_t n_tables, const int32_t *clbit_qubit,
                        const int32_t *n_clbits, const uint64_t *ps_mask, const uint64_t *ps_value, const int32_t *ps_bits,
                        const uint64_t *stream_ids, uint64_t shots, uint64_t seed, uint64_t *keys_out, double *probs_out, double *kept_out,
                        double *device_ms_out) {
    return run_batch_small(device, precision, n_circuits, n_qubits, op_begin, ops, tables, n_tables, clbit_qubit, n_clbits,
                           nullptr, ps_mask, ps_value, ps_bits, stream_ids, shots, seed, keys_out, probs_out, kept_out,
                           device_ms_out);
}

int qcm_run_batch_small_readout(int device, int precision, int n_circuits, const int32_t *n_qubits, const int64_t *op_begin,
                                const qcm_op *ops, const double *tables, size_t n_tables, const int32_t *clbit_qubit,
                                const int32_t *n_clbits, const double *readout, const uint64_t *ps_mask,
                                const uint64_t *ps_value, const int32_t *ps_bits, const uint64_t *stream_ids, uint64_t shots,
                                uint64_t seed, uint64_t *keys_out, double *probs_out, double *kept_out,
                                double *device_ms_out) {
    return run_batch_small(device, precision, n_circuits, n_qubits, op_begin, ops, tables, n_tables, clbit_qubit, n_clbits,
                           readout, ps_mask, ps_value, ps_bits, stream_ids, shots, seed, keys_out, probs_out, kept_out,
                           device_ms_out);
}

}  // extern "C"
