// C ABI of the qcmrf_b200 engine (see include/qcmrf_b200.h for the contract).
// Host-side program validation, kernel selection and launch; no CPU compute path.
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <mutex>
#include <set>
#include <string>
#include <vector>

#include "qcm_kernels.cuh"
#include "qcmrf_b200.h"

using namespace qcm;

namespace {

thread_local std::string g_last_error;

struct DevBuf {
    void *p = nullptr;
    size_t cap = 0;
};

}  // namespace

struct qcm_sim_s {
    int device = 0;
    int n_local = 0;
    int prec = QCM_C64;
    int n_active = 0;
    int n_global = 0;
    uint64_t rank = 0;
    int batch = 1;                  // sweep points held by this handle (qcm_create_batched); kernels run with gridDim.y = batch
    int cur_point = 0;              // point addressed by qcm_get_amplitudes / qcm_set_amplitudes (qcm_batch_select)
    bool deferred = false;          // qcm_set_deferred: calls enqueue their work and return without synchronising
    // the last program was INIT_PRODUCT and nothing else: the state is a product state over product_n qubits whose
    // 2-vectors sit at tab_f64 + product_off (per point); shots are then drawn per qubit (k_sample_product)
    int product_n = -1;
    int64_t product_off = 0;
    double product_mass = 0.0;      // norm^2 of point 0's product state
    size_t tab_stride = 0;          // doubles per point in the uploaded tables
    uint64_t tree_total = 0;        // doubles per point in the sum-tree buffer
    uint64_t probs_n = 0;           // entries per point of the resident post-selected block (qcm_postselect_resident)
    void *state = nullptr;
    bool own_state = false;
    cudaStream_t stream = nullptr;
    int num_sms = 148;
    std::string err;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr;
    qcm_timing timing{};
    DevBuf tab_f64, tab_real, init_lo, init_hi, probs, partial, keys, mine, tree, ctab, tilectr, subtree;
    DevBuf scratch;                 // input copy of a rotated expansion pass
    DevBuf lowpart;                 // its per-CTA partial sums when a CTA covers fewer inputs than a tree chunk
    DevBuf relp1;                   // released-qubit probability tables (qcm_sample_released)
    DevBuf streams, totals;         // batched sampling: per-point Philox streams and total masses
    DevBuf errflag;                 // in-place fused exchange: spin-timeout flag
    // rotated storage (QCM_FLAG_ROTATED_OUTPUT_OK): logical index i of the 2^n_active state lives at
    // physical address ((i & (2^rot_nin - 1)) << rot_m) | (i >> rot_nin); rot_m == 0: identity
    int rot_m = 0, rot_nin = 0;
    bool tree_cond_low = false;     // the checkpoint tree's conditional images are the low address bits
    // virtual last pass (QCM_VIRTUAL_LAST): the rotated result was left unwritten.  Its input stays in `scratch`, and
    // readers compute the images they need from it with these arguments (low_image); materialise_last() writes it
    // out for the readers that need the state itself.
    bool virt = false;
    ExpandTreeArgs virt_args{};
    size_t virt_smem = 0;
    std::vector<double> h_top;
    // sum tree (built by qcm_sample_prepare)
    int tree_levels = 0;
    double *tree_ptr[8] = {nullptr};
    uint64_t tree_n[8] = {0};
    int tree_for_active = -1;       // n_active of the state the tree describes
    int tree_base_bits = 0;         // qubits the tree indexes (tree_for_active - tree_cond_bits)
    int tree_cond_bits = 0;         // expansion qubits materialised after the tree was built
    int tree_sub_bits = 0;          // subtree holds sums over 2^tree_sub_bits amplitudes ...
    bool tree_has_sub = false;      // ... when this is set (fused checkpoint only)
    bool tree_sub_input = false;    // ... not stored: the sampler computes it from the input in `scratch` (virtual pass)
    bool tree_sub_strided = false;  // generic tree build: subtree holds k_chunk_sums' 32 lane partials per chunk
    uint64_t n_expand = 0, n_checkpoint = 0;
    double local_mass = 0.0;
    bool tree_valid = false;
    // per-op profile of the last program
    std::vector<cudaEvent_t> op_ev;
    std::vector<int32_t> op_kind;
    std::vector<uint64_t> op_rd, op_wr;
    std::vector<float> op_ms;
    std::vector<std::string> op_kernel;    // kernel that ran each op of the last program
    std::string cur_kernel;                // set by the launchers, collected per op
    bool op_ms_pending = false;            // the last program ran deferred: its per-op events have not been read yet
    // qcm_mark / qcm_wait: a ring of events; ticket t lives in slot t % kMarks (a later ticket in the same slot
    // implies t has completed: one stream)
    static constexpr int kMarks = 16;
    cudaEvent_t marks[kMarks] = {nullptr};
    uint64_t n_marks = 0;
};

namespace {

int fail(qcm_handle h, int code, const char *fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_last_error = buf;
    if (h) h->err = buf;
    return code;
}

#define QCM_CUDA(h, call)                                                                     \
    do {                                                                                       \
        cudaError_t e_ = (call);                                                               \
        if (e_ != cudaSuccess)                                                                 \
            return fail(h, e_ == cudaErrorMemoryAllocation ? QCM_ERR_NOMEM : QCM_ERR_CUDA,    \
                        "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e_), __FILE__, __LINE__); \
    } while (0)

int ensure(qcm_handle h, DevBuf &b, size_t bytes) {
    if (b.cap >= bytes) return QCM_OK;
    if (b.p) QCM_CUDA(h, cudaFree(b.p));
    b.p = nullptr;
    b.cap = 0;
    QCM_CUDA(h, cudaMalloc(&b.p, bytes));
    b.cap = bytes;
    return QCM_OK;
}

inline size_t amp_bytes(int prec) { return prec == QCM_C64 ? 8 : 16; }
inline size_t real_bytes(const qcm_sim_s *h) { return h->prec == QCM_C64 ? 4 : 8; }
// the program's tables in the state's real type: a float copy for complex64, the fp64 upload itself for complex128
inline const void *tabreal(const qcm_sim_s *h) { return h->prec == QCM_C64 ? h->tab_real.p : h->tab_f64.p; }
// batch strides (bytes) of the state and of the per-point tables in the state's real type / in fp64
inline uint64_t bstate(const qcm_sim_s *h) { return (uint64_t)amp_bytes(h->prec) << h->n_local; }
inline uint64_t btab(const qcm_sim_s *h) { return (uint64_t)h->tab_stride * real_bytes(h); }
inline uint64_t btab64(const qcm_sim_s *h) { return (uint64_t)h->tab_stride * sizeof(double); }
inline dim3 bgrid(const qcm_sim_s *h, uint64_t gx) { return dim3((unsigned)gx, (unsigned)h->batch, 1u); }
inline uint64_t rank_bits(const qcm_sim_s *h) { return h->n_global ? (h->rank << h->n_local) : 0ull; }
template <typename R> constexpr const char *real_name() { return sizeof(R) == 4 ? "float" : "double"; }
// the op's kernel with its template arguments, for qcm_op_kernel_name
inline void name_kernel(qcm_handle h, const char *fmt, ...) {
    char nm[96];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(nm, sizeof nm, fmt, ap);
    va_end(ap);
    h->cur_kernel = nm;
}

int grid_mult() {
    static int v = [] {
        // Streaming kernels run one tile per CTA, in launch (= address) order: resident CTAs then share
        // a compact window of the state, which keeps DRAM pages open.  A persistent grid-stride grid of
        // 148 x occupancy CTAs measured 5.7-5.8 TB/s on the dense in-place pass, this 6.9-7.0 TB/s
        // (profiles/r01_notes.md).  QCM_GRID_MULT=k caps the grid at k waves of resident CTAs (tuning knob).
        const char *e = getenv("QCM_GRID_MULT");
        int t = e ? atoi(e) : 65536;
        return (t < 1 || t > 65536) ? 65536 : t;
    }();
    return v;
}

template <typename K>
int grid_for(qcm_handle h, K kernel, size_t smem, uint64_t work_items_per_block, uint64_t items) {
    int occ = 0;
    cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kernel, kThreads, smem);
    if (occ < 1) occ = 1;
    uint64_t need = (items + work_items_per_block - 1) / work_items_per_block;
    uint64_t cap = (uint64_t)h->num_sms * (uint64_t)occ * (uint64_t)grid_mult();
    if (need < 1) need = 1;
    return (int)std::min<uint64_t>(need, cap);
}

// ---- block / mux launch -----------------------------------------------------------
template <typename R, int V, int M, int U, bool LAZY>
int launch_block_t(qcm_handle h, const BlockArgs &a, size_t smem) {
    auto kern = k_block<R, V, M, U, LAZY>;
    if (smem > 48 * 1024) QCM_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const uint64_t nvec = (1ull << (a.n_out - M)) / V;
    const int grid = grid_for(h, kern, smem, (uint64_t)kThreads * U, nvec);
    kern<<<bgrid(h, grid), kThreads, smem, h->stream>>>(a);
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    name_kernel(h, "k_block<%s,%d,M=%d,U=%d,LAZY=%d>", real_name<R>(), V, M, U, LAZY ? 1 : 0);
    return QCM_OK;
}

template <typename R, int V, bool LAZY>
int launch_block_m(qcm_handle h, int M, const BlockArgs &a, size_t smem) {
    switch (M) {
        case 1: return launch_block_t<R, V, 1, 4, LAZY>(h, a, smem);
        case 2: return launch_block_t<R, V, 2, 2, LAZY>(h, a, smem);
        case 3: return launch_block_t<R, V, 3, 1, LAZY>(h, a, smem);
        case 4: return launch_block_t<R, V, 4, 1, LAZY>(h, a, smem);
        case 5: return launch_block_t<R, V, 5, 1, LAZY>(h, a, smem);
    }
    return fail(h, QCM_ERR_INVALID, "block size %d out of range", M);
}

int expand_threads() {
    static int v = [] {
        const char *e = getenv("QCM_EXPAND_THREADS");          // tuning knob for profiling runs
        int t = e ? atoi(e) : 512;
        if (t < 64 || t > kExpandThreadsMax || (t & (t - 1))) t = 512;
        return t;
    }();
    return v;
}

// How k_expand's tiles are handed out (both in address order, see the kernel): 1 = persistent CTAs
// pulling from a global counter (the coefficient table is staged once per CTA), 0 = one tile per CTA
// in launch order.  QCM_EXPAND_SCHED=launch|counter overrides (tuning knob).
int rotate_enabled() {
    // QCM_ROTATE=0: keep the last expansion pass in logical address order (A/B measurement knob)
    static int v = [] {
        const char *e = getenv("QCM_ROTATE");
        return (e && e[0] == '0') ? 0 : 1;
    }();
    return v;
}

int expand_use_counter() {
    static int v = [] {
        const char *e = getenv("QCM_EXPAND_SCHED");
        if (e && !strcmp(e, "launch")) return 0;
        if (e && !strcmp(e, "counter")) return 1;
        return 0;                    // measured: launch order 11.9 ms vs counter 12.1 ms on the 29->33 qubit pass
    }();
    return v;
}

template <typename R, int V, int M, int U, bool Q0>
int launch_expand_t(qcm_handle h, const ExpandArgs &a, size_t smem) {
    auto kern = k_expand<R, V, M, U, Q0>;
    if (smem > 48 * 1024) QCM_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const int threads = a.tree_out ? (1 << kChunkBits) / V : expand_threads();    // fused tree: sub-tile == chunk
    const uint64_t nvec = (1ull << a.n_in) / V;
    const uint64_t need = std::max<uint64_t>(1, (nvec + (uint64_t)threads * U - 1) / ((uint64_t)threads * U));
    uint64_t grid = need;
    if (a.tile_counter) {
        int occ = 0;
        cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, kern, threads, smem);
        if (occ < 1) occ = 1;
        grid = std::min<uint64_t>(need, (uint64_t)h->num_sms * occ);
    }
    grid = std::min<uint64_t>(grid, 0x7fffffffull);
    kern<<<bgrid(h, grid), threads, smem, h->stream>>>(a);
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    name_kernel(h, "k_expand<%s,%d,M=%d,U=%d,Q0=%d>", real_name<R>(), V, M, U, Q0 ? 1 : 0);
    return QCM_OK;
}

template <typename R, int V, bool Q0>
int launch_expand_m(qcm_handle h, int M, const ExpandArgs &a, size_t smem) {
    switch (M) {
        case 1: return launch_expand_t<R, V, 1, 4, Q0>(h, a, smem);
        case 2: return launch_expand_t<R, V, 2, 4, Q0>(h, a, smem);
        case 3: return launch_expand_t<R, V, 3, 2, Q0>(h, a, smem);
        case 4: return launch_expand_t<R, V, 4, 2, Q0>(h, a, smem);
        case 5: return launch_expand_t<R, V, 5, 2, Q0>(h, a, smem);
    }
    return fail(h, QCM_ERR_INVALID, "expansion of %d qubits out of range", M);
}

struct BlockPlan {
    BlockArgs args{};
    int M = 0;
    size_t smem = 0;
    bool expand = false;            // eligible for the expansion fast path
    ExpandTableArgs targs{};
    ExpandArgs eargs{};
    bool tree = false;              // wide expansion: product-tree kernel
    ExpandTreeArgs trargs{};
    size_t tree_smem = 0;
    bool norm_preserving = false;   // expansion without diagonal members: sum_a |out[x,a]|^2 == |in[x]|^2
    bool rotate = false;            // store the result rotated (k_expand_low); decided by the program loop
    bool input_in_scratch = false;  // ... and its input already lives in h->scratch (the program prefix ran there)
    bool virt = false;              // ... and is left unwritten: only the checkpoint sums run (see qcm_sim_s::virt)
};

// members: ops[0..n_mem) are MUX1Q (or DIAG: a diagonal factor applied in the same sweep);
// tq: block qubits ascending.  Validates and fills `bp`; launches nothing.
int plan_block(qcm_handle h, const int *tq, int M, const qcm_op *members, int n_mem, int n_in, int n_out,
               size_t n_tables, BlockPlan &bp) {
    // a block whose qubits are all new (n_in .. n_in+M-1) may be wider than a general one
    const bool all_new = (n_out - n_in == M) && M >= 1 && tq[0] == n_in;
    const int max_m = all_new ? QCM_MAX_EXPAND : QCM_MAX_BLOCK;
    if (M < 1 || M > max_m) return fail(h, QCM_ERR_INVALID, "block of %d qubits unsupported (max %d)", M, max_m);
    if (n_mem > QCM_MAX_MEMBERS) return fail(h, QCM_ERR_INVALID, "block has %d members (max %d)", n_mem, QCM_MAX_MEMBERS);
    if (n_out > h->n_local || n_in > n_out || n_in < 0) return fail(h, QCM_ERR_INVALID, "bad active range %d -> %d (n_local %d)", n_in, n_out, h->n_local);
    BlockArgs &a = bp.args;
    bp.M = M;
    a.state = h->state;
    a.tables = tabreal(h);
    a.n_in = n_in;
    a.n_out = n_out;
    a.n_members = n_mem;
    a.ctrl_below_32 = 1;
    a.rank_bits = rank_bits(h);
    a.bstate = bstate(h);
    a.btab = btab(h);
    for (int j = 0; j < M; ++j) {
        if (tq[j] < 0 || tq[j] >= n_out) return fail(h, QCM_ERR_INVALID, "block qubit %d outside the active state (%d)", tq[j], n_out);
        if (j && tq[j] <= tq[j - 1]) return fail(h, QCM_ERR_INVALID, "block qubits must be strictly ascending");
        if (j < QCM_MAX_BLOCK) a.tq[j] = tq[j];
    }
    for (int q = n_in; q < n_out; ++q)
        if (!std::binary_search(tq, tq + M, q))
            return fail(h, QCM_ERR_INVALID, "qubit %d is materialised by this op but is not one of its targets", q);
    size_t smem_reals = 0;
    int per_target[QCM_MAX_EXPAND] = {0};
    int n_diag = 0;
    for (int g = 0; g < n_mem; ++g) {
        const qcm_op &op = members[g];
        const bool diag = op.kind == QCM_OP_DIAG;
        if (op.kind != QCM_OP_MUX1Q && !diag) return fail(h, QCM_ERR_INVALID, "block member %d is neither MUX1Q nor DIAG", g);
        if (op.n_ctrl < 0 || op.n_ctrl > QCM_MAX_CTRL) return fail(h, QCM_ERR_INVALID, "member %d: n_ctrl %d out of range", g, op.n_ctrl);
        if (diag) {
            a.mem[g].pos = -1;
            ++n_diag;
        } else {
            const int *pp = std::lower_bound(tq, tq + M, op.target);
            if (pp == tq + M || *pp != op.target) return fail(h, QCM_ERR_INVALID, "member %d targets qubit %d which is not a block qubit", g, op.target);
            a.mem[g].pos = (int8_t)(pp - tq);
            per_target[pp - tq]++;
        }
        a.mem[g].n_ctrl = (int8_t)op.n_ctrl;
        a.mem[g].low_bit = 0;
        for (int j = 0; j < op.n_ctrl; ++j) {
            const int c = op.ctrl[j];
            if (c == 0) a.mem[g].low_bit = (uint16_t)(1u << j);
            if (c >= 32) a.ctrl_below_32 = 0;
            if (c < 0 || c >= h->n_local + h->n_global) return fail(h, QCM_ERR_INVALID, "member %d: index qubit %d out of range", g, c);
            if (std::binary_search(tq, tq + M, c)) return fail(h, QCM_ERR_INVALID, "member %d: index qubit %d is a block target", g, c);
            a.mem[g].ctrl[j] = (int8_t)c;
        }
        const size_t need = (diag ? 2ull : 8ull) << op.n_ctrl;
        if (op.table_off < 0 || (size_t)op.table_off + need > n_tables)
            return fail(h, QCM_ERR_INVALID, "member %d: table [%lld, +%llu) outside tables (%zu)", g, (long long)op.table_off,
                        (unsigned long long)need, n_tables);
        a.mem[g].src_off = (int32_t)op.table_off;
        a.mem[g].tab_off = (int32_t)smem_reals;
        smem_reals += (need + 3) & ~size_t(3);          // keep every table 16-byte aligned
    }
    const size_t real_sz = h->prec == QCM_C64 ? 4 : 8;
    bp.smem = smem_reals * real_sz;
    if (bp.smem > 160 * 1024) return fail(h, QCM_ERR_UNSUPPORTED, "block coefficient tables need %zu B of shared memory", bp.smem);

    // expansion fast path: every block qubit is new (known |0>) and the target of exactly one member
    bool expand = all_new;
    for (int j = 0; j < M && expand; ++j) expand = per_target[j] == 1;
    if (M > QCM_MAX_BLOCK && !expand)
        return fail(h, QCM_ERR_INVALID, "a block of %d qubits must materialise every one of them with exactly one MUX1Q", M);
    // wide expansions (and ones whose index-qubit union overflows the precombined table) use the product tree
    bool tree = expand && M >= kTreeLow && n_diag <= 4;
    if (tree) {
        ExpandTreeArgs &t = bp.trargs;
        t.state = h->state;
        t.tables = tabreal(h);
        t.n_in = n_in;
        t.M = M;
        t.n_diag = 0;
        t.ctrl_below_32 = a.ctrl_below_32;
        t.rank_bits = rank_bits(h);
        t.bstate = bstate(h);
        t.btab = btab(h);
        size_t off = 0;
        for (int g = 0; g < n_mem; ++g) {
            TreeMember &m = a.mem[g].pos < 0 ? t.diag[t.n_diag++] : t.mem[a.mem[g].pos];
            m.n_ctrl = a.mem[g].n_ctrl;
            for (int j = 0; j < m.n_ctrl; ++j) m.ctrl[j] = a.mem[g].ctrl[j];
            m.low_bit = a.mem[g].low_bit;
            m.src_off = a.mem[g].src_off;
            m.tab_off = (int32_t)off;
            off += (a.mem[g].pos < 0 ? 2ull : 4ull) << m.n_ctrl;
            off = (off + 3) & ~size_t(3);
        }
        bp.tree_smem = off * real_sz;
        if (bp.tree_smem > 160 * 1024) tree = false;
    }
    bp.tree = tree;
    if (M > QCM_MAX_BLOCK && !tree)
        return fail(h, QCM_ERR_UNSUPPORTED, "wide expansion of %d qubits cannot be served", M);
    if (expand) {
        // union of the members' index qubits, ascending: the qubits that differ between the lanes
        // of a warp get the low cidx bits (conflict-free shared loads), qubit 0 gets bit 0
        int8_t cu[QCM_MAX_MEMBERS * QCM_MAX_CTRL];
        int nu = 0;
        ExpandTableArgs &t = bp.targs;
        for (int g = 0; g < n_mem; ++g)
            for (int j = 0; j < a.mem[g].n_ctrl; ++j) {
                const int8_t c = a.mem[g].ctrl[j];
                if (std::find(cu, cu + nu, c) == cu + nu) cu[nu++] = c;
            }
        std::sort(cu, cu + nu);
        if (nu + M > kExpandMaxBits || M > QCM_MAX_BLOCK) expand = false;
        for (int g = 0; g < n_mem && expand; ++g) {
            t.mpos[g] = a.mem[g].pos;
            t.mnc[g] = a.mem[g].n_ctrl;
            t.moff[g] = members[g].table_off;
            for (int j = 0; j < a.mem[g].n_ctrl; ++j)
                t.mbit[g][j] = (int8_t)(std::find(cu, cu + nu, a.mem[g].ctrl[j]) - cu);
        }
        if (expand) {
            t.M = M; t.nu = nu; t.n_members = n_mem; t.is_double = h->prec == QCM_C128;
            ExpandArgs &e = bp.eargs;
            e.state = h->state;
            e.n_in = n_in;
            e.nu = nu;
            for (int k = 0; k < nu; ++k) e.cu[k] = cu[k];
            e.cu_below_32 = (nu == 0 || cu[nu - 1] < 32) ? 1 : 0;
            e.rank_bits = rank_bits(h);
            e.bstate = bstate(h);
            e.bctab = (uint64_t)amp_bytes(h->prec) << (M + nu);
            t.btab64 = btab64(h);
            t.bctab = e.bctab;
        }
    }
    if (expand && tree && M >= 5) expand = false;             // M <= 4: the precombined table wins; wider: the tree
    if (expand) bp.tree = false;
    bp.expand = expand;
    bp.norm_preserving = (expand || bp.tree) && n_diag == 0;
    return QCM_OK;
}

int low_shape() {
    // QCM_LOW_SHAPE = <warps per CTA>x<log2 inputs per CTA> of the rotated expansion pass: tuning knob.  Measured on the
    // q34 last pass (profiles/r02_notes.md): 8x8 9.74 ms, 4x7 9.77, 1x5 9.87, 8x10 9.86, 2x6 10.02 -- a bare sequential
    // writer gains 5 % when a CTA's region shrinks from 512 KiB to 32 KiB (tools/membench4.cu), but here the smaller
    // CTAs pay more for their start-up (table staging, first input load) than the compacter write window returns.
    static int v = [] {
        const char *e = getenv("QCM_LOW_SHAPE");
        int w = 8, tb = 8;
        if (e && sscanf(e, "%dx%d", &w, &tb) == 2) {
            const bool ok = (w == 8 && (tb == 8 || tb == 10)) || (w == 4 && tb == 7) || (w == 2 && tb == 6) || (w == 1 && tb == 5);
            if (!ok) { w = 8; tb = 8; }
        }
        return w * 100 + tb;
    }();
    return v;
}

// QCM_LOW_CTAS = resident CTAs per SM of the rotated expansion pass (0 = whatever fits).  A write-only stream is FASTER
// with fewer resident warps (tools/membench5.cu: a bare sequential writer 7.29 TB/s at 64 warps per SM, 7.42 at 32, 7.57
// at 8), the kernel needs enough of them to cover its store-free phase A: the launcher pads the dynamic shared memory
// so that only this many CTAs fit.
int low_ctas() {
    static int v = [] {
        const char *e = getenv("QCM_LOW_CTAS");
        return e ? std::max(0, std::min(32, atoi(e))) : -1;
    }();
    return v;
}

// QCM_VIRTUAL_LAST = 0: always write the rotated last pass; 1: leave it unwritten (virtual) at any size; unset: leave it
// unwritten when its output has more than 2^30 amplitudes -- the rotated states qcm_get_amplitudes never returned.
int virtual_last() {
    static int v = [] {
        const char *e = getenv("QCM_VIRTUAL_LAST");
        return (e && (e[0] == '0' || e[0] == '1')) ? e[0] - '0' : -1;
    }();
    return v;
}

// Raises a kernel's dynamic shared-memory limit to the device's opt-in maximum, once per kernel and device, before its
// first launch there.  Changing a function's attributes while an instance of it runs holds the call back until that
// instance ends (another rank's kernel on this GPU waiting for signals, or this stream's previous pass), and handles
// that share a process get here concurrently, so the check and the set happen under one lock.
int raise_smem_limit(qcm_handle h, const void *kern) {
    static std::mutex mu;
    static std::set<std::pair<int, const void *>> done;
    std::lock_guard<std::mutex> lock(mu);
    if (done.count({h->device, kern})) return QCM_OK;
    int optin = 0;
    QCM_CUDA(h, cudaDeviceGetAttribute(&optin, cudaDevAttrMaxSharedMemoryPerBlockOptin, h->device));
    QCM_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, optin));
    done.insert({h->device, kern});
    return QCM_OK;
}

template <typename R, int V, int MH, int TB, int NW>
static int launch_low_tb(qcm_handle h, int n_in, BlockPlan &bp) {
    auto kern = k_expand_low<R, V, MH, TB, NW>;
    constexpr int warps = NW;
    size_t smem = low_warp_bytes<R, MH>() * warps + bp.tree_smem;
    {
        // default: 24 resident warps per SM for complex64 (q34 last pass, profiles/r02_low_ctas_sweep.txt: 8x8 at 5 / 4 / 3 /
        // 2 CTAs per SM 9.72 / 9.67 / 9.65 / 10.02 ms, 4x7 at 10 / 8 / 6 / 5 / 4: 9.78 / 9.72 / 9.66 / 9.74 / 10.00);
        // complex128 CTAs (4 warps, twice the shared memory) already sit at 6 per SM
        const int want = low_ctas() >= 0 ? low_ctas() : (sizeof(R) == 4 ? std::max(1, 24 / warps) : 0);
        if (want > 0) {
            const size_t per_cta = ((size_t)227 * 1024 / want - 1024) & ~(size_t)127;    // 1 KiB per CTA is the system's
            if (per_cta > smem) smem = per_cta;
        }
    }
    int rc;
    if (smem > 48 * 1024 && (rc = raise_smem_limit(h, (const void *)kern))) return rc;
    ExpandTreeArgs args = bp.trargs;
    double *level0 = args.tree_out;
    if (level0) {                                          // per-warp partial sums, grouped into level 0 below
        rc = ensure(h, h->lowpart, (sizeof(double) * warps) << (n_in - TB));
        if (rc) return rc;
        args.tree_out = (double *)h->lowpart.p;
    }
    kern<<<1u << (n_in - TB), NW * 32, smem, h->stream>>>(args, h->scratch.p);
    name_kernel(h, "k_expand_low<%s,%d,MH=%d,TB=%d,NW=%d>", sizeof(R) == 4 ? "float" : "double", V, MH, TB, NW);
    QCM_CUDA(h, cudaGetLastError());
    if (level0) {
        int wbits = 0;
        while ((1 << wbits) < warps) ++wbits;
        const uint64_t n_out = 1ull << (n_in - kChunkBits);
        k_group_sum<<<(unsigned)((n_out + kThreads - 1) / kThreads), kThreads, 0, h->stream>>>((const double *)h->lowpart.p, kChunkBits - TB + wbits, n_out, level0);
        QCM_CUDA(h, cudaGetLastError());
        h->timing.kernel_launches++;
    }
    return QCM_OK;
}

// the shape of the materialising launch (QCM_LOW_SHAPE), as NW * 100 + TB; complex128 CTAs have always been 4 warps
// (twice the shared memory per warp)
template <typename R>
static int low_shape_for() {
    return (sizeof(R) == 8 && low_shape() == 808) ? 407 : low_shape();
}

template <typename R, int V, int MH>
static int launch_low(qcm_handle h, int n_in, BlockPlan &bp) {
    switch (low_shape_for<R>()) {
        case 810: return launch_low_tb<R, V, MH, 10, 8>(h, n_in, bp);
        case 407: return launch_low_tb<R, V, MH, 7, 4>(h, n_in, bp);
        case 206: return launch_low_tb<R, V, MH, 6, 2>(h, n_in, bp);
        case 105: return launch_low_tb<R, V, MH, 5, 1>(h, n_in, bp);
        default: return launch_low_tb<R, V, MH, 8, 8>(h, n_in, bp);
    }
}

// the sums-only launch of a virtual last pass: level 0, with the association of the materialising launch's shape
// (k_expand_low_sums)
template <typename R, int TB, int NW>
static int launch_low_sums_tb(qcm_handle h, int n_in, const BlockPlan &bp) {
    const uint64_t chunks = 1ull << (n_in - kChunkBits);
    k_expand_low_sums<R, TB, NW><<<(unsigned)chunks, kSumsThreads, 0, h->stream>>>(h->scratch.p, bp.trargs.tree_out);
    name_kernel(h, "k_expand_low_sums<%s,%d,TB=%d,NW=%d>", sizeof(R) == 4 ? "float" : "double", sizeof(R) == 4 ? 2 : 1, TB, NW);
    return QCM_OK;
}

template <typename R>
static int launch_low_sums(qcm_handle h, int n_in, const BlockPlan &bp) {
    switch (low_shape_for<R>()) {
        case 810: return launch_low_sums_tb<R, 10, 8>(h, n_in, bp);
        case 407: return launch_low_sums_tb<R, 7, 4>(h, n_in, bp);
        case 206: return launch_low_sums_tb<R, 6, 2>(h, n_in, bp);
        case 105: return launch_low_sums_tb<R, 5, 1>(h, n_in, bp);
        default: return launch_low_sums_tb<R, 8, 8>(h, n_in, bp);
    }
}

template <typename R, int V>
static int launch_low_mh(qcm_handle h, int MH, int n_in, BlockPlan &bp) {
    switch (MH) {
        case 0: return launch_low<R, V, 0>(h, n_in, bp);
        case 1: return launch_low<R, V, 1>(h, n_in, bp);
        case 2: return launch_low<R, V, 2>(h, n_in, bp);
        case 3:
            if constexpr (V == 1) return launch_low<R, V, 3>(h, n_in, bp);
    }
    return fail(h, QCM_ERR_INVALID, "rotated expansion: %d loop levels out of range", MH);
}

// ---- low-order-target pass ------------------------------------------------------------
int lowq_enabled() {
    // QCM_LOWQ=0: serve low targets with k_block (A/B measurement knob)
    static int v = [] {
        const char *e = getenv("QCM_LOWQ");
        return (e && e[0] == '0') ? 0 : 1;
    }();
    return v;
}

template <typename R, int V, int UB, int MH>
static int launch_lowq_t(qcm_handle h, const LowqArgs &a, size_t smem) {
    auto kern = k_lowq<R, V, UB, MH>;
    if (smem > 48 * 1024) QCM_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    constexpr int LB = (V == 2 ? 1 : 0) + 5 + UB;
    const uint64_t nrows = 1ull << (a.n - LB - MH);
    const uint64_t grid = std::min<uint64_t>(std::max<uint64_t>(1, (nrows + kThreads / 32 - 1) / (kThreads / 32)), 0x7fffffffull);
    kern<<<bgrid(h, grid), kThreads, smem, h->stream>>>(a);
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    char nm[64];
    snprintf(nm, sizeof nm, "k_lowq<%s,%d,UB=%d,MH=%d>", sizeof(R) == 4 ? "float" : "double", V, UB, MH);
    h->cur_kernel = nm;
    return QCM_OK;
}

// Serves an in-place block whose lowest target sits inside a warp's coalesced access.  Returns 1 when the
// pass was launched, 0 when k_block should take it, < 0 on error.
static int try_lowq(qcm_handle h, const BlockPlan &bp) {
    const BlockArgs &b = bp.args;
    const int M = bp.M, n = b.n_out;
    if (!lowq_enabled() || b.n_in != b.n_out || M > QCM_MAX_BLOCK || b.tq[0] >= 6) return 0;
    const int VB = h->prec == QCM_C64 ? 1 : 0;
    int MH = -1;
    for (int mh = 0; mh <= kLowqMaxHigh && MH < 0; ++mh) {
        const int LB = VB + 5 + (3 - mh);
        int high = 0;
        for (int j = 0; j < M; ++j) high += b.tq[j] >= LB;
        if (high == mh && n >= LB + mh) MH = mh;
    }
    if (MH < 0) return 0;
    const int UB = 3 - MH, LB = VB + 5 + UB;
    LowqArgs a{};
    a.state = b.state;
    a.tables = b.tables;
    a.n = n;
    a.n_members = b.n_members;
    a.rank_bits = b.rank_bits;
    a.bstate = b.bstate;
    a.btab = b.btab;
    for (int k = 0; k < MH; ++k) a.th[k] = b.tq[M - MH + k];
    for (int g = 0; g < b.n_members; ++g) {
        const MemberDesc &s = b.mem[g];
        LowqMember &m = a.mem[g];
        if (s.pos < 0) m.pos = -1;
        else {
            const int t = b.tq[s.pos];
            m.pos = (int8_t)(t < LB ? t : LB + (s.pos - (M - MH)));
        }
        m.n_ctrl = s.n_ctrl;
        m.tab_off = s.tab_off;
        m.src_off = s.src_off;
        m.rany = 0;
        for (int j = 0; j < s.n_ctrl; ++j) {
            const int c = s.ctrl[j];
            m.ctrl[j] = (int8_t)c;
            int rb = -1;                                   // register-index bit this qubit is, if any
            if (VB && c == 0) rb = 0;
            else if (c >= VB + 5 && c < LB) rb = c - 5;
            if (rb >= 0) {
                m.rbit[rb] = (uint16_t)(1u << j);
                m.rany |= m.rbit[rb];
            }
        }
    }
    int rc;
    if (h->prec == QCM_C64) {
        rc = MH == 0 ? launch_lowq_t<float, 2, 3, 0>(h, a, bp.smem)
           : MH == 1 ? launch_lowq_t<float, 2, 2, 1>(h, a, bp.smem)
                     : launch_lowq_t<float, 2, 1, 2>(h, a, bp.smem);
    } else {
        rc = MH == 0 ? launch_lowq_t<double, 1, 3, 0>(h, a, bp.smem)
           : MH == 1 ? launch_lowq_t<double, 1, 2, 1>(h, a, bp.smem)
                     : launch_lowq_t<double, 1, 1, 2>(h, a, bp.smem);
    }
    return rc ? rc : 1;
}

int launch_block_plan(qcm_handle h, BlockPlan &bp) {
    const BlockArgs &a = bp.args;
    const int M = bp.M, n_in = a.n_in, n_out = a.n_out;
    int rc;
    if (bp.tree && bp.rotate) {
        // sequential-write variant: input from a scratch copy, output rotated (see k_expand_low)
        const size_t in_bytes = amp_bytes(h->prec) << n_in;
        if (!bp.input_in_scratch) {
            if ((rc = ensure(h, h->scratch, in_bytes))) return rc;
            QCM_CUDA(h, cudaMemcpyAsync(h->scratch.p, h->state, in_bytes, cudaMemcpyDeviceToDevice, h->stream));
            h->timing.bytes_read += in_bytes;      // the scratch copy: one more read and write of the input
            h->timing.bytes_written += in_bytes;
        }
        // a virtual pass runs the checkpoint sums only, with the materialising launch's association (the same tree), and
        // nothing at all without the checkpoint
        const bool launch = !bp.virt || bp.trargs.tree_out;
        if (!launch) rc = QCM_OK;
        else if (bp.virt) rc = h->prec == QCM_C64 ? launch_low_sums<float>(h, n_in, bp) : launch_low_sums<double>(h, n_in, bp);
        else if (h->prec == QCM_C64) rc = launch_low_mh<float, 2>(h, M - 6, n_in, bp);
        else rc = launch_low_mh<double, 1>(h, M - 5, n_in, bp);
        if (rc) return rc;
        QCM_CUDA(h, cudaGetLastError());
        if (launch) h->timing.kernel_launches++;
        h->n_expand++;
        h->rot_m = M;
        h->rot_nin = n_in;
        if (bp.virt) {
            h->virt = true;
            h->virt_args = bp.trargs;
            h->virt_args.tree_out = nullptr;     // materialise_last: the tree exists already
            h->virt_smem = bp.tree_smem;
            if (launch) {                        // algorithmic traffic: the input read, level 0 written
                h->timing.bytes_read += in_bytes;
                h->timing.bytes_written += sizeof(double) << (n_in - kChunkBits);
            }
            return QCM_OK;
        }
    } else if (bp.tree) {
        const int V = (h->prec == QCM_C64 && n_in >= 1) ? 2 : 1;
        name_kernel(h, "k_expand_tree<%s,%d>", h->prec == QCM_C64 ? "float" : "double", V);
        const int threads = bp.trargs.tree_out ? (1 << kChunkBits) / V : 256;     // fused tree: tile == chunk
        const uint64_t nvec = (1ull << n_in) / V;
        const uint64_t grid = std::min<uint64_t>(std::max<uint64_t>(1, (nvec + threads - 1) / threads), 0x7fffffffull);
        const size_t smem = bp.tree_smem;
        if (h->prec == QCM_C64) {
            if (V == 2) {
                if (smem > 48 * 1024) QCM_CUDA(h, cudaFuncSetAttribute(k_expand_tree<float, 2>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                k_expand_tree<float, 2><<<bgrid(h, grid), threads, smem, h->stream>>>(bp.trargs);
            } else {
                if (smem > 48 * 1024) QCM_CUDA(h, cudaFuncSetAttribute(k_expand_tree<float, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
                k_expand_tree<float, 1><<<bgrid(h, grid), threads, smem, h->stream>>>(bp.trargs);
            }
        } else {
            if (smem > 48 * 1024) QCM_CUDA(h, cudaFuncSetAttribute(k_expand_tree<double, 1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
            k_expand_tree<double, 1><<<bgrid(h, grid), threads, smem, h->stream>>>(bp.trargs);
        }
        QCM_CUDA(h, cudaGetLastError());
        h->timing.kernel_launches++;
        h->n_expand++;
    } else if (bp.expand) {
        const size_t centry = h->prec == QCM_C64 ? 8 : 16;
        const size_t nent = 1ull << (M + bp.targs.nu);
        if ((rc = ensure(h, h->ctab, nent * centry * h->batch))) return rc;
        if ((rc = ensure(h, h->tilectr, sizeof(unsigned long long)))) return rc;
        bp.targs.tables = (const double *)h->tab_f64.p;
        bp.targs.ctab = h->ctab.p;
        bp.targs.tile_counter = expand_use_counter() ? (unsigned long long *)h->tilectr.p : nullptr;
        bp.eargs.tile_counter = bp.targs.tile_counter;
        k_expand_table<<<bgrid(h, (nent + 255) / 256), 256, 0, h->stream>>>(bp.targs);
        QCM_CUDA(h, cudaGetLastError());
        h->timing.kernel_launches++;
        bp.eargs.ctab = h->ctab.p;
        const size_t smem = nent * centry;
        const bool q0 = bp.eargs.nu > 0 && bp.eargs.cu[0] == 0;
        if (h->prec == QCM_C64) {
            if (n_in >= 1) rc = q0 ? launch_expand_m<float, 2, true>(h, M, bp.eargs, smem) : launch_expand_m<float, 2, false>(h, M, bp.eargs, smem);
            else rc = launch_expand_m<float, 1, false>(h, M, bp.eargs, smem);
        } else {
            rc = launch_expand_m<double, 1, false>(h, M, bp.eargs, smem);
        }
        if (rc) return rc;
        h->n_expand++;
    } else {
        const bool lazy = n_in != n_out;
        rc = try_lowq(h, bp);
        if (rc < 0) return rc;
        if (rc == 1) {
            rc = QCM_OK;
        } else if (h->prec == QCM_C64) {
            const bool vec2 = a.tq[0] >= 1 && (n_out - M) >= 1;
            if (vec2) rc = lazy ? launch_block_m<float, 2, true>(h, M, a, bp.smem) : launch_block_m<float, 2, false>(h, M, a, bp.smem);
            else rc = lazy ? launch_block_m<float, 1, true>(h, M, a, bp.smem) : launch_block_m<float, 1, false>(h, M, a, bp.smem);
        } else {
            rc = lazy ? launch_block_m<double, 1, true>(h, M, a, bp.smem) : launch_block_m<double, 1, false>(h, M, a, bp.smem);
        }
        if (rc) return rc;
    }
    // algorithmic traffic: read the materialised input, write the whole output
    h->timing.bytes_read += amp_bytes(h->prec) << n_in;
    h->timing.bytes_written += amp_bytes(h->prec) << n_out;
    return QCM_OK;
}

// Writes out the unwritten result of a virtual last pass (qcm_sim_s::virt), from its input, for the readers that need
// the state itself.  Enqueued on the handle's stream; a no-op for any other state.
int materialise_last(qcm_handle h) {
    if (!h->virt) return QCM_OK;
    h->virt = false;
    BlockPlan bp;
    bp.trargs = h->virt_args;
    bp.tree_smem = h->virt_smem;
    const int M = bp.trargs.M, n_in = bp.trargs.n_in;
    const std::string kernel = h->cur_kernel;            // not an op of a program: leave the per-op record alone
    int rc = h->prec == QCM_C64 ? launch_low_mh<float, 2>(h, M - 6, n_in, bp) : launch_low_mh<double, 1>(h, M - 5, n_in, bp);
    h->cur_kernel = kernel;
    if (rc) return rc;
    h->timing.kernel_launches++;
    return QCM_OK;
}

int launch_diag(qcm_handle h, const qcm_op &op, size_t n_tables) {
    if (op.n_ctrl < 0 || op.n_ctrl > QCM_MAX_CTRL) return fail(h, QCM_ERR_INVALID, "DIAG: n_ctrl %d out of range", op.n_ctrl);
    if (op.table_off < 0 || (size_t)op.table_off + (2ull << op.n_ctrl) > n_tables) return fail(h, QCM_ERR_INVALID, "DIAG: table outside tables");
    if (op.n_active_in != op.n_active_out) return fail(h, QCM_ERR_INVALID, "DIAG cannot materialise qubits");
    DiagArgs a{};
    a.state = h->state;
    a.n_ctrl = op.n_ctrl;
    a.n_active = op.n_active_in;
    a.rank_bits = rank_bits(h);
    a.bstate = bstate(h);
    a.btab = btab(h);
    for (int j = 0; j < op.n_ctrl; ++j) {
        if (op.ctrl[j] < 0 || op.ctrl[j] >= h->n_local + h->n_global) return fail(h, QCM_ERR_INVALID, "DIAG: qubit %d out of range", op.ctrl[j]);
        a.ctrl[j] = (int8_t)op.ctrl[j];
    }
    const size_t real_sz = h->prec == QCM_C64 ? 4 : 8;
    a.table = (const char *)tabreal(h) + (size_t)op.table_off * real_sz;
    const size_t smem = (2ull << op.n_ctrl) * real_sz;
    const uint64_t cta_cap = std::max<uint64_t>((uint64_t)(4 * h->num_sms + h->batch - 1) / h->batch,
                                              (amp_bytes(h->prec) << a.n_active) / (16 * std::max<size_t>(smem, 1024)));
    if (h->prec == QCM_C64) {
        if (a.n_active >= 1) {
            auto k = k_diag<float, 2, 4>;
            int grid = (int)std::min<uint64_t>(grid_for(h, k, smem, kThreads * 4, (1ull << a.n_active) / 2), cta_cap);
            k<<<bgrid(h, grid), kThreads, smem, h->stream>>>(a);
            h->cur_kernel = "k_diag<float,2,U=4>";
        } else {
            auto k = k_diag<float, 1, 4>;
            k<<<bgrid(h, 1), kThreads, smem, h->stream>>>(a);
            h->cur_kernel = "k_diag<float,1,U=4>";
        }
    } else {
        auto k = k_diag<double, 1, 4>;
        int grid = (int)std::min<uint64_t>(grid_for(h, k, smem, kThreads * 4, 1ull << a.n_active), cta_cap);
        k<<<bgrid(h, grid), kThreads, smem, h->stream>>>(a);
        h->cur_kernel = "k_diag<double,1,U=4>";
    }
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    h->timing.bytes_read += amp_bytes(h->prec) << a.n_active;
    h->timing.bytes_written += amp_bytes(h->prec) << a.n_active;
    return QCM_OK;
}

// BLOCK header with zero targets: every member is a DIAG, all applied in one sweep
int launch_diag_multi(qcm_handle h, const qcm_op *members, int n_mem, int n_active, size_t n_tables) {
    if (n_mem < 1 || n_mem > QCM_MAX_MEMBERS) return fail(h, QCM_ERR_INVALID, "diagonal block with %d members (max %d)", n_mem, QCM_MAX_MEMBERS);
    BlockArgs a{};
    a.state = h->state;
    a.tables = tabreal(h);
    a.n_in = a.n_out = n_active;
    a.n_members = n_mem;
    a.rank_bits = rank_bits(h);
    a.bstate = bstate(h);
    a.btab = btab(h);
    size_t reals = 0;
    DiagMultiRuns runs{};
    for (int g = 0; g < n_mem; ++g) {
        const qcm_op &op = members[g];
        if (op.kind != QCM_OP_DIAG) return fail(h, QCM_ERR_INVALID, "a BLOCK without targets may only hold DIAG members");
        if (op.n_ctrl < 0 || op.n_ctrl > QCM_MAX_CTRL) return fail(h, QCM_ERR_INVALID, "DIAG: n_ctrl %d out of range", op.n_ctrl);
        if (op.table_off < 0 || (size_t)op.table_off + (2ull << op.n_ctrl) > n_tables) return fail(h, QCM_ERR_INVALID, "DIAG: table outside tables");
        a.mem[g].pos = -1;
        a.mem[g].n_ctrl = (int8_t)op.n_ctrl;
        a.mem[g].low_bit = 0;
        for (int j = 0; j < op.n_ctrl; ++j) {
            if (op.ctrl[j] < 0 || op.ctrl[j] >= h->n_local + h->n_global) return fail(h, QCM_ERR_INVALID, "DIAG: qubit %d out of range", op.ctrl[j]);
            if (op.ctrl[j] == 0) a.mem[g].low_bit = (uint16_t)(1u << j);
            a.mem[g].ctrl[j] = (int8_t)op.ctrl[j];
        }
        a.mem[g].src_off = (int32_t)op.table_off;
        a.mem[g].tab_off = (int32_t)reals;
        reals += ((2ull << op.n_ctrl) + 3) & ~size_t(3);
        // runs of consecutive ascending index qubits (index bit j+1 <-> qubit ctrl[j] + 1); a run that would need a
        // left shift (qubit below its index position: unsorted index qubits) is split into single bits placed by mask
        IndexRuns &rn = runs.m[g];
        rn.below_32 = 1;
        int run_start = 0, run_pos = 0, run_len = 0;
        auto close_run = [&]() {
            if (!run_len) return;
            if (run_start >= run_pos) {
                rn.mask[rn.n_runs] = ((1u << run_len) - 1u) << run_pos;
                rn.shift[rn.n_runs] = run_start - run_pos;
                rn.n_runs++;
            } else {
                return;                              // handled by the caller below (never for ascending qubits)
            }
            run_len = 0;
        };
        bool ok_runs = true;
        for (int j = 0; j < op.n_ctrl; ++j) {
            if (op.ctrl[j] >= 32) rn.below_32 = 0;
            if (run_len && op.ctrl[j] == run_start + run_len) {
                run_len++;
            } else {
                close_run();
                if (run_len) ok_runs = false;
                run_start = op.ctrl[j];
                run_pos = j;
                run_len = 1;
            }
        }
        close_run();
        if (run_len) ok_runs = false;
        if (!ok_runs) {
            // index qubits in an order the run decomposition cannot express with right shifts: one pass per member
            for (int k = 0; k < n_mem; ++k) {
                int rc2 = launch_diag(h, members[k], n_tables);
                if (rc2) return rc2;
            }
            h->cur_kernel += " (diagonal block, one pass per member)";
            return QCM_OK;
        }
    }
    const size_t smem = reals * real_bytes(h);
    if (smem > 200 * 1024) return fail(h, QCM_ERR_UNSUPPORTED, "diagonal block tables need %zu B of shared memory", smem);
    // every CTA stages all tables (up to 16 KiB each): give it at least 16x that much state to sweep, else the
    // staging traffic rivals the state traffic (a 16 MiB sweep point under 32 KiB of tables: 3.3 -> 6+ TB/s)
    const uint64_t cta_cap = std::max<uint64_t>((uint64_t)(4 * h->num_sms + h->batch - 1) / h->batch,
                                              (amp_bytes(h->prec) << n_active) / (16 * std::max<size_t>(smem, 1024)));
    auto capped = [&](int g) { return (int)std::min<uint64_t>((uint64_t)g, cta_cap); };
    if (h->prec == QCM_C64 && n_active >= 1) {
        auto k = k_diag_multi<float, 2, 4>;
        if (smem > 48 * 1024) QCM_CUDA(h, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k<<<bgrid(h, capped(grid_for(h, k, smem, kThreads * 4, (1ull << n_active) / 2))), kThreads, smem, h->stream>>>(a, runs);
        h->cur_kernel = "k_diag_multi<float,2,U=4>";
    } else if (h->prec == QCM_C64) {
        auto k = k_diag_multi<float, 1, 4>;
        if (smem > 48 * 1024) QCM_CUDA(h, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k<<<bgrid(h, 1), kThreads, smem, h->stream>>>(a, runs);
        h->cur_kernel = "k_diag_multi<float,1,U=4>";
    } else {
        auto k = k_diag_multi<double, 1, 4>;
        if (smem > 48 * 1024) QCM_CUDA(h, cudaFuncSetAttribute(k, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        k<<<bgrid(h, capped(grid_for(h, k, smem, kThreads * 4, 1ull << n_active))), kThreads, smem, h->stream>>>(a, runs);
        h->cur_kernel = "k_diag_multi<double,1,U=4>";
    }
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    h->timing.bytes_read += amp_bytes(h->prec) << n_active;
    h->timing.bytes_written += amp_bytes(h->prec) << n_active;
    return QCM_OK;
}

int launch_init(qcm_handle h, const qcm_op &op, size_t n_tables, const double *host_tables) {
    const int n = op.n_active_out;
    if (n < 0 || n > h->n_local) return fail(h, QCM_ERR_INVALID, "INIT_PRODUCT over %d qubits (n_local %d)", n, h->n_local);
    if (op.table_off < 0 || (size_t)op.table_off + 4ull * (size_t)std::max(n, 1) > n_tables)
        return fail(h, QCM_ERR_INVALID, "INIT_PRODUCT: table (max(n,1)*4 doubles) outside tables");
    const int L = n >= 1 ? std::max(1, n / 2) : 0;   // a 2-amplitude vector must share one `hi` factor
    int rc;
    const uint64_t blo = sizeof(double2) << L, bhi = sizeof(double2) << (n - L), bst = bstate(h);
    if ((rc = ensure(h, h->init_lo, blo * h->batch))) return rc;
    if ((rc = ensure(h, h->init_hi, bhi * h->batch))) return rc;
    const double *qv = (const double *)h->tab_f64.p + op.table_off;
    const uint64_t nt = (1ull << L) + (1ull << (n - L));
    k_init_tables<<<bgrid(h, (nt + 255) / 256), 256, 0, h->stream>>>(qv, n, L, h->init_lo.p, (double2 *)h->init_hi.p, h->prec == QCM_C64 ? 1 : 0,
                                                                     btab64(h), blo, bhi);
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    if (h->prec == QCM_C64) {
        if (n >= 1) {
            auto k = k_init<float, 2>;
            int grid = grid_for(h, k, 0, (uint64_t)kThreads * kInitU, (1ull << n) / 2);
            k<<<bgrid(h, grid), kThreads, 0, h->stream>>>(h->state, h->init_lo.p, (const double2 *)h->init_hi.p, n, L, bst, blo, bhi);
            h->cur_kernel = "k_init<float,2>";
        } else {
            k_init<float, 1><<<bgrid(h, 1), kThreads, 0, h->stream>>>(h->state, h->init_lo.p, (const double2 *)h->init_hi.p, n, L, bst, blo, bhi);
            h->cur_kernel = "k_init<float,1>";
        }
    } else {
        auto k = k_init<double, 1>;
        int grid = grid_for(h, k, 0, (uint64_t)kThreads * kInitU, 1ull << n);
        k<<<bgrid(h, grid), kThreads, 0, h->stream>>>(h->state, h->init_lo.p, (const double2 *)h->init_hi.p, n, L, bst, blo, bhi);
        h->cur_kernel = "k_init<double,1>";
    }
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    h->timing.bytes_written += amp_bytes(h->prec) << n;
    h->product_n = n;
    h->product_off = op.table_off;
    h->product_mass = 1.0;
    for (int q = 0; q < n; ++q) {
        const double *v = host_tables + op.table_off + 4 * q;
        h->product_mass *= v[0] * v[0] + v[1] * v[1] + v[2] * v[2] + v[3] * v[3];
    }
    return QCM_OK;
}

int product_sampling_enabled() {
    // QCM_PRODUCT_SAMPLE=0: sample product states through the sum tree like any other state (A/B knob)
    static int v = [] {
        const char *e = getenv("QCM_PRODUCT_SAMPLE");
        return (e && e[0] == '0') ? 0 : 1;
    }();
    return v;
}

// the state is a product state the sampler may draw qubit by qubit (unsharded, at most 64 qubits, not rotated)
bool product_state(const qcm_sim_s *h) {
    return product_sampling_enabled() && h->product_n >= 0 && h->product_n == h->n_active && h->product_n <= 64 &&
           h->n_global == 0 && !h->rot_m;
}

int launch_extend(qcm_handle h, int n_in, int n_out) {
    if (n_in < 0 || n_out > h->n_local || n_in > n_out) return fail(h, QCM_ERR_INVALID, "EXTEND %d -> %d invalid", n_in, n_out);
    if (n_in == n_out) return QCM_OK;
    const uint64_t first = 1ull << n_in, count = (1ull << n_out) - first;
    if (h->prec == QCM_C64) {
        auto k = k_zero<float>;
        k<<<bgrid(h, grid_for(h, k, 0, (uint64_t)kThreads * kInitU, count)), kThreads, 0, h->stream>>>(h->state, first, count, bstate(h));
        h->cur_kernel = "k_zero<float>";
    } else {
        auto k = k_zero<double>;
        k<<<bgrid(h, grid_for(h, k, 0, (uint64_t)kThreads * kInitU, count)), kThreads, 0, h->stream>>>(h->state, first, count, bstate(h));
        h->cur_kernel = "k_zero<double>";
    }
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    h->timing.bytes_written += amp_bytes(h->prec) * count;
    return QCM_OK;
}

int launch_swap(qcm_handle h, const qcm_op &op) {
    int qa = std::min(op.target, op.ctrl[0]), qb = std::max(op.target, op.ctrl[0]);
    const int n = op.n_active_in;
    if (qa == qb) return QCM_OK;
    if (qa < 0 || qb >= n || op.n_active_in != op.n_active_out) return fail(h, QCM_ERR_INVALID, "SWAP(%d,%d) outside the active state (%d)", qa, qb, n);
    const uint64_t quads = 1ull << (n - 2);
    if (h->prec == QCM_C64) {
        if (qa >= 1 && n >= 3) {
            auto k = k_swap<float, 2>;
            k<<<bgrid(h, grid_for(h, k, 0, kThreads, quads / 2)), kThreads, 0, h->stream>>>(h->state, qa, qb, n, bstate(h));
            h->cur_kernel = "k_swap<float,2>";
        } else {
            auto k = k_swap<float, 1>;
            k<<<bgrid(h, grid_for(h, k, 0, kThreads, quads)), kThreads, 0, h->stream>>>(h->state, qa, qb, n, bstate(h));
            h->cur_kernel = "k_swap<float,1>";
        }
    } else {
        auto k = k_swap<double, 1>;
        k<<<bgrid(h, grid_for(h, k, 0, kThreads, quads)), kThreads, 0, h->stream>>>(h->state, qa, qb, n, bstate(h));
        h->cur_kernel = "k_swap<double,1>";
    }
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    h->timing.bytes_read += (amp_bytes(h->prec) << n) / 2;
    h->timing.bytes_written += (amp_bytes(h->prec) << n) / 2;
    return QCM_OK;
}

int upload_tables(qcm_handle h, const double *tables, size_t n_per_point) {
    h->tab_stride = n_per_point;
    const size_t n_tables = n_per_point * (size_t)h->batch;      // batched handle: `batch` consecutive table sets
    if (!n_tables) return QCM_OK;
    int rc;
    if ((rc = ensure(h, h->tab_f64, n_tables * sizeof(double)))) return rc;
    QCM_CUDA(h, cudaMemcpyAsync(h->tab_f64.p, tables, n_tables * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    if (h->prec == QCM_C64) {
        std::vector<float> f(n_tables);
        for (size_t i = 0; i < n_tables; ++i) f[i] = (float)tables[i];
        if ((rc = ensure(h, h->tab_real, n_tables * sizeof(float)))) return rc;
        // pageable source: the runtime stages it before the call returns, so `f` may go out of scope (no synchronisation)
        QCM_CUDA(h, cudaMemcpyAsync(h->tab_real.p, f.data(), n_tables * sizeof(float), cudaMemcpyHostToDevice, h->stream));
    }                                  // complex128: the fp64 upload IS the table in the state's real type (tabreal)
    return QCM_OK;
}

// ---- sum tree -----------------------------------------------------------------------
// level sizes + buffers for a tree over 2^na amplitudes
int tree_layout(qcm_handle h, int na) {
    const int cb = std::min(na, kChunkBits);
    uint64_t sizes[8];
    int levels = 0;
    uint64_t n = 1ull << (na - cb), total = 0;
    while (true) {
        if (levels >= 8) return fail(h, QCM_ERR_UNSUPPORTED, "sum tree too deep");
        sizes[levels++] = n;
        total += n;
        if (n <= (1ull << kFanBits)) break;
        n = (n + (1ull << kFanBits) - 1) >> kFanBits;
    }
    int rc;
    h->tree_total = total;
    if ((rc = ensure(h, h->tree, total * sizeof(double) * h->batch))) return rc;
    double *p = (double *)h->tree.p;
    for (int l = 0; l < levels; ++l) {
        h->tree_ptr[l] = p;
        h->tree_n[l] = sizes[l];
        p += sizes[l];
    }
    h->tree_levels = levels;
    return QCM_OK;
}

// level 0 from the state: one warp per chunk, CTAs in address order (see grid_mult)
int tree_level0(qcm_handle h, int na) {
    const uint64_t warps_per_block = kThreads / 32;
    const uint64_t n0 = h->tree_n[0];
    uint64_t blocks = std::min<uint64_t>((n0 + warps_per_block - 1) / warps_per_block, 0x7fffffffull);
    const uint64_t btree = h->tree_total * sizeof(double);
    // finer level (32 strided groups per chunk) while it stays small: 1/32 .. 1/64 of the state
    double *sub = nullptr;
    const uint64_t bsub = (sizeof(double) * 32) << (na - std::min(na, kChunkBits));
    h->tree_sub_strided = false;
    if (na >= kChunkBits && bsub * h->batch <= (512ull << 20) && ensure(h, h->subtree, bsub * h->batch) == QCM_OK) {
        sub = (double *)h->subtree.p;
        h->tree_sub_strided = true;
    } else {
        cudaGetLastError();
    }
    if (h->prec == QCM_C64) k_chunk_sums<float><<<bgrid(h, blocks), kThreads, 0, h->stream>>>(h->state, na, h->tree_ptr[0], bstate(h), btree, sub, bsub);
    else k_chunk_sums<double><<<bgrid(h, blocks), kThreads, 0, h->stream>>>(h->state, na, h->tree_ptr[0], bstate(h), btree, sub, bsub);
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    return QCM_OK;
}

// upper levels, total mass; the tree then describes a state of `na` base qubits
int tree_finish(qcm_handle h, int na) {
    const uint64_t warps_per_block = kThreads / 32;
    const int levels = h->tree_levels;
    const uint64_t btree = h->tree_total * sizeof(double);
    for (int l = 1; l < levels; ++l) {
        uint64_t blocks = std::min<uint64_t>((h->tree_n[l] + warps_per_block - 1) / warps_per_block, (uint64_t)h->num_sms * 8);
        k_tree_level<<<bgrid(h, blocks), kThreads, 0, h->stream>>>(h->tree_ptr[l - 1], h->tree_n[l - 1], h->tree_ptr[l], h->tree_n[l], btree, btree);
        QCM_CUDA(h, cudaGetLastError());
        h->timing.kernel_launches++;
    }
    const uint64_t ntop = h->tree_n[levels - 1];
    if (h->batch > 1) {
        // per-point totals stay on the device (k_sample reads them): no host round trip in a sweep
        int rc;
        if ((rc = ensure(h, h->totals, sizeof(double) * h->batch))) return rc;
        k_batch_totals<<<(h->batch + 127) / 128, 128, 0, h->stream>>>(h->tree_ptr[levels - 1], ntop, btree, (double *)h->totals.p, h->batch);
        QCM_CUDA(h, cudaGetLastError());
        h->timing.kernel_launches++;
        h->local_mass = 0.0;
        h->tree_valid = true;
        h->tree_for_active = na;
        h->tree_base_bits = na;
        h->tree_cond_bits = 0;
        h->tree_sub_bits = 0;
        h->tree_has_sub = false;
        h->tree_sub_input = false;
        return QCM_OK;
    }
    if (h->deferred) {
        // deferred mode: nothing is read back (qcm_tree_total_device sums the top level on the device for callers that
        // continue there); the local mass is unknown on the host
        h->local_mass = std::nan("");
    } else {
        h->h_top.resize(ntop);
        QCM_CUDA(h, cudaMemcpyAsync(h->h_top.data(), h->tree_ptr[levels - 1], ntop * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        QCM_CUDA(h, cudaStreamSynchronize(h->stream));
        double m = 0.0;
        for (uint64_t i = 0; i < ntop; ++i) m += h->h_top[i];
        h->local_mass = m;
    }
    h->tree_valid = true;
    h->tree_for_active = na;
    h->tree_base_bits = na;
    h->tree_cond_bits = 0;
    h->tree_sub_bits = 0;
    h->tree_has_sub = false;
    h->tree_sub_input = false;
    return QCM_OK;
}

int build_tree(qcm_handle h) {
    const int na = h->n_active;
    int rc;
    if ((rc = materialise_last(h))) return rc;
    if ((rc = tree_layout(h, na))) return rc;
    if ((rc = tree_level0(h, na))) return rc;
    return tree_finish(h, na);
}

static int env_int(const char *name, int dflt) {
    const char *v = getenv(name);
    return (v && *v) ? atoi(v) : dflt;
}

template <typename R, int V, int M, int U>
static int launch_gather_ldg(qcm_handle h, const GatherArgs &a, size_t smem) {
    auto kern = k_block_gather<R, V, M, U>;
    const uint64_t nvec = (1ull << (a.n_local - M)) / V;
    const uint64_t grid = std::min<uint64_t>(std::max<uint64_t>(1, (nvec + (uint64_t)kThreads * U - 1) / ((uint64_t)kThreads * U)), 0x7fffffffull);
    kern<<<(unsigned)grid, kThreads, smem, h->stream>>>(a);
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    return QCM_OK;
}

// stages of the TMA ring: as deep as keeps the ring at 64-96 KB for U = 1 (two CTAs per SM)
template <int M> struct GatherStages { static constexpr int value = M == 1 ? 8 : (M == 2 ? 6 : 3); };

template <typename R, int V, int M, int U>
static int launch_gather_tma(qcm_handle h, const GatherArgs &a, size_t tab_bytes, int tiles_per_cta) {
    constexpr int S = GatherStages<M>::value;
    auto kern = k_block_gather_tma<R, V, M, U, S>;
    const size_t smem = 256 + (size_t)S * (1 << M) * kGatherTileBytes * U + tab_bytes;
    if (smem > 227 * 1024) return fail(h, QCM_ERR_UNSUPPORTED, "gather ring needs %zu B of shared memory", smem);
    QCM_CUDA(h, cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    const uint64_t tiles = ((1ull << (a.n_local - M)) / V) / ((uint64_t)kThreads * U);
    while (tiles_per_cta > 1 && (tiles % tiles_per_cta || tiles / tiles_per_cta < 1)) tiles_per_cta >>= 1;
    const uint64_t grid = tiles / tiles_per_cta;
    if (grid > 0x7fffffffull) return fail(h, QCM_ERR_UNSUPPORTED, "gather grid too large");
    kern<<<(unsigned)grid, kThreads + 32, smem, h->stream>>>(a, tiles_per_cta);
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    return QCM_OK;
}

// QCM_GATHER = tma | ldg, QCM_GATHER_U = vectors per thread per tile, QCM_GATHER_K = tiles per CTA (tma): tuning knobs
template <typename R, int V, int M>
static int launch_gather_t(qcm_handle h, const GatherArgs &a, size_t tab_bytes) {
    const char *mode = getenv("QCM_GATHER");
    const bool want_tma = !(mode && !strcmp(mode, "ldg"));
    const uint64_t nvec = (1ull << (a.n_local - M)) / V;
    int U = env_int("QCM_GATHER_U", want_tma ? 1 : 2);
    if (want_tma && nvec >= (uint64_t)kThreads * 2 && nvec % ((uint64_t)kThreads * 2) == 0) {
        int K = env_int("QCM_GATHER_K", 16);
        if (K < 1) K = 1;
        int p2 = 1;
        while (p2 * 2 <= K) p2 *= 2;                      // power of two, so it divides the tile count
        if (U >= 2) return launch_gather_tma<R, V, M, 2>(h, a, tab_bytes, p2);
        return launch_gather_tma<R, V, M, 1>(h, a, tab_bytes, p2);
    }
    if (U >= 4) return launch_gather_ldg<R, V, M, 4>(h, a, tab_bytes);
    if (U <= 1) return launch_gather_ldg<R, V, M, 1>(h, a, tab_bytes);
    return launch_gather_ldg<R, V, M, 2>(h, a, tab_bytes);
}

template <typename R, int V>
static int launch_gather_m(qcm_handle h, int M, const GatherArgs &a, size_t smem) {
    switch (M) {
        case 1: return launch_gather_t<R, V, 1>(h, a, smem);
        case 2: return launch_gather_t<R, V, 2>(h, a, smem);
        case 3: return launch_gather_t<R, V, 3>(h, a, smem);
    }
    return fail(h, QCM_ERR_INVALID, "gather block of %d qubits out of range", M);
}

// tiles of the in-place fused exchange: one 16-byte vector per consumer thread (U = 1), K consecutive tiles per CTA
static uint64_t gather_inplace_tiles(int n_local, int s, int prec) {
    const uint64_t vec = (1ull << (n_local - s)) / (prec == QCM_C64 ? 2 : 1);
    return vec / kThreads;
}

template <typename R, int V, int M>
static int launch_gather_inplace(qcm_handle h, const GatherArgs &a, const GatherFlags &f, size_t tab_bytes) {
    constexpr int S = GatherStages<M>::value;
    auto kern = k_block_gather_inplace<R, V, M, 1, S>;
    const size_t smem = 256 + (size_t)S * (1 << M) * kGatherTileBytes + tab_bytes;
    if (smem > 227 * 1024) return fail(h, QCM_ERR_UNSUPPORTED, "gather ring needs %zu B of shared memory", smem);
    // set once, before the first launch: another rank's instance may already be waiting for signals (raise_smem_limit)
    int rc;
    if ((rc = raise_smem_limit(h, (const void *)kern))) return rc;
    const uint64_t tiles = ((1ull << (a.n_local - M)) / V) / kThreads;
    int K = env_int("QCM_GATHER_K", 16);
    int p2 = 1;
    while (p2 * 2 <= K) p2 *= 2;
    while (p2 > 1 && (tiles % p2 || tiles / p2 < 1)) p2 >>= 1;
    const uint64_t grid = tiles / p2;
    if (grid > 0x7fffffffull) return fail(h, QCM_ERR_UNSUPPORTED, "gather grid too large");
    kern<<<(unsigned)grid, kThreads + 96, smem, h->stream>>>(a, f, p2);
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    return QCM_OK;
}

int check_device(qcm_handle h) {
    QCM_CUDA(h, cudaSetDevice(h->device));
    return QCM_OK;
}

}  // namespace

// =====================================================================================
extern "C" {

int qcm_abi_version(void) { return QCM_ABI_VERSION; }

int qcm_device_count(int *n_out) {
    if (!n_out) return fail(nullptr, QCM_ERR_INVALID, "n_out is NULL");
    int n = 0;
    cudaError_t e = cudaGetDeviceCount(&n);
    if (e != cudaSuccess) {
        *n_out = 0;
        return fail(nullptr, QCM_ERR_NO_DEVICE, "cudaGetDeviceCount: %s", cudaGetErrorString(e));
    }
    *n_out = n;
    return QCM_OK;
}

int qcm_enable_peer_access(int device, int peer) {
    if (device == peer) return QCM_OK;
    int can = 0;
    cudaError_t e = cudaDeviceCanAccessPeer(&can, device, peer);
    if (e != cudaSuccess || !can) return fail(nullptr, QCM_ERR_UNSUPPORTED, "device %d cannot access device %d directly", device, peer);
    e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaDeviceEnablePeerAccess(peer, 0);
    if (e == cudaErrorPeerAccessAlreadyEnabled) {
        cudaGetLastError();
        e = cudaSuccess;
    }
    if (e != cudaSuccess) return fail(nullptr, QCM_ERR_CUDA, "cudaDeviceEnablePeerAccess(%d -> %d): %s", device, peer, cudaGetErrorString(e));
    return QCM_OK;
}

int qcm_ipc_export(int device, const void *dev_ptr, unsigned char *handle_out, uint64_t *offset_out) {
    if (!dev_ptr || !handle_out || !offset_out) return fail(nullptr, QCM_ERR_INVALID, "NULL argument");
    static_assert(sizeof(cudaIpcMemHandle_t) == QCM_IPC_HANDLE_BYTES, "IPC handle size");
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return fail(nullptr, QCM_ERR_CUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(e));
    // base of the containing allocation: driver entry point through the runtime (no libcuda link dependency)
    typedef int (*range_fn)(unsigned long long *, size_t *, unsigned long long);
    void *fp = nullptr;
    cudaDriverEntryPointQueryResult qr;
    e = cudaGetDriverEntryPoint("cuMemGetAddressRange", &fp, cudaEnableDefault, &qr);
    if (e != cudaSuccess || !fp) return fail(nullptr, QCM_ERR_CUDA, "cuMemGetAddressRange entry point: %s", cudaGetErrorString(e));
    unsigned long long base = 0;
    size_t size = 0;
    const int cr = reinterpret_cast<range_fn>(fp)(&base, &size, (unsigned long long)(uintptr_t)dev_ptr);
    if (cr != 0) return fail(nullptr, QCM_ERR_CUDA, "cuMemGetAddressRange failed (CUresult %d)", cr);
    cudaIpcMemHandle_t hd;
    e = cudaIpcGetMemHandle(&hd, reinterpret_cast<void *>((uintptr_t)base));
    if (e != cudaSuccess) return fail(nullptr, QCM_ERR_CUDA, "cudaIpcGetMemHandle: %s", cudaGetErrorString(e));
    memcpy(handle_out, &hd, sizeof(hd));
    *offset_out = (uint64_t)((uintptr_t)dev_ptr - (uintptr_t)base);
    return QCM_OK;
}

int qcm_ipc_open(int device, const unsigned char *handle, void **base_out) {
    if (!handle || !base_out) return fail(nullptr, QCM_ERR_INVALID, "NULL argument");
    *base_out = nullptr;
    cudaError_t e = cudaSetDevice(device);
    if (e != cudaSuccess) return fail(nullptr, QCM_ERR_CUDA, "cudaSetDevice(%d): %s", device, cudaGetErrorString(e));
    cudaIpcMemHandle_t hd;
    memcpy(&hd, handle, sizeof(hd));
    e = cudaIpcOpenMemHandle(base_out, hd, cudaIpcMemLazyEnablePeerAccess);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, QCM_ERR_CUDA, "cudaIpcOpenMemHandle on device %d: %s", device, cudaGetErrorString(e));
    }
    return QCM_OK;
}

int qcm_ipc_close(int device, void *base) {
    if (!base) return QCM_OK;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaIpcCloseMemHandle(base);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, QCM_ERR_CUDA, "cudaIpcCloseMemHandle: %s", cudaGetErrorString(e));
    }
    return QCM_OK;
}

const char *qcm_last_error(qcm_handle h) { return h ? h->err.c_str() : g_last_error.c_str(); }

int qcm_create(qcm_handle *out, int device, int n_local, int precision, void *ext_state, void *ext_stream) {
    return qcm_create_batched(out, device, n_local, precision, 1, ext_state, ext_stream);
}

int qcm_create_batched(qcm_handle *out, int device, int n_local, int precision, int batch, void *ext_state, void *ext_stream) {
    if (!out) return fail(nullptr, QCM_ERR_INVALID, "out is NULL");
    *out = nullptr;
    if (batch < 1 || batch > 65535) return fail(nullptr, QCM_ERR_INVALID, "batch %d out of range [1, 65535]", batch);
    if (precision != QCM_C64 && precision != QCM_C128) return fail(nullptr, QCM_ERR_INVALID, "precision must be 32 or 64");
    if (n_local < 0 || n_local > 40) return fail(nullptr, QCM_ERR_INVALID, "n_local %d out of range [0, 40]", n_local);
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(nullptr, QCM_ERR_NO_DEVICE, "no CUDA device available: qcmrf_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(nullptr, QCM_ERR_INVALID, "device %d out of range (%d devices)", device, ndev);
    qcm_sim_s *h = new (std::nothrow) qcm_sim_s();
    if (!h) return fail(nullptr, QCM_ERR_NOMEM, "host allocation failed");
    h->device = device;
    h->n_local = n_local;
    h->prec = precision;
    h->batch = batch;
    h->stream = (cudaStream_t)ext_stream;
    cudaError_t e = cudaSetDevice(device);
    if (e == cudaSuccess) e = cudaDeviceGetAttribute(&h->num_sms, cudaDevAttrMultiProcessorCount, device);
    if (e == cudaSuccess) e = cudaEventCreate(&h->ev0);
    if (e == cudaSuccess) e = cudaEventCreate(&h->ev1);
    if (e == cudaSuccess) {
        // allocated up front: a cudaMalloc between the launches of two co-operating kernels would serialise them
        e = cudaMalloc(&h->errflag.p, sizeof(int));
        if (e == cudaSuccess) h->errflag.cap = sizeof(int);
    }
    if (e == cudaSuccess) {
        if (ext_state) {
            h->state = ext_state;
        } else {
            e = cudaMalloc(&h->state, (amp_bytes(precision) << n_local) * (size_t)batch);
            h->own_state = (e == cudaSuccess);
        }
    }
    if (e != cudaSuccess) {
        int code = fail(nullptr, e == cudaErrorMemoryAllocation ? QCM_ERR_NOMEM : QCM_ERR_CUDA, "qcm_create: %s", cudaGetErrorString(e));
        if (h->ev0) cudaEventDestroy(h->ev0);
        if (h->ev1) cudaEventDestroy(h->ev1);
        delete h;
        return code;
    }
    *out = h;
    return QCM_OK;
}

int qcm_destroy(qcm_handle h) {
    if (!h) return QCM_OK;
    cudaSetDevice(h->device);
    cudaStreamSynchronize(h->stream);
    DevBuf *bufs[] = {&h->tab_f64, &h->tab_real, &h->init_lo, &h->init_hi, &h->probs, &h->partial, &h->keys, &h->mine, &h->tree, &h->ctab, &h->tilectr, &h->subtree, &h->scratch, &h->lowpart, &h->relp1, &h->streams, &h->totals, &h->errflag};
    for (DevBuf *b : bufs)
        if (b->p) cudaFree(b->p);
    if (h->own_state && h->state) cudaFree(h->state);
    if (h->ev0) cudaEventDestroy(h->ev0);
    if (h->ev1) cudaEventDestroy(h->ev1);
    for (cudaEvent_t e : h->op_ev) cudaEventDestroy(e);
    for (cudaEvent_t e : h->marks) if (e) cudaEventDestroy(e);
    delete h;
    return QCM_OK;
}

int qcm_set_shard(qcm_handle h, int n_global_qubits, uint64_t rank) {
    if (!h) return fail(nullptr, QCM_ERR_INVALID, "handle is NULL");
    if (n_global_qubits < 0 || h->n_local + n_global_qubits > 62) return fail(h, QCM_ERR_INVALID, "bad n_global_qubits %d", n_global_qubits);
    if (n_global_qubits < 64 && rank >> n_global_qubits) return fail(h, QCM_ERR_INVALID, "rank %llu does not fit %d global qubits", (unsigned long long)rank, n_global_qubits);
    h->n_global = n_global_qubits;
    h->rank = rank;                 // the sum tree holds |amp|^2 of local amplitudes: unaffected
    return QCM_OK;
}

int qcm_synchronize(qcm_handle h) {
    if (!h) return fail(nullptr, QCM_ERR_INVALID, "handle is NULL");
    int rc = check_device(h);
    if (rc) return rc;
    QCM_CUDA(h, cudaStreamSynchronize(h->stream));
    return QCM_OK;
}

int qcm_get_amplitudes(qcm_handle h, uint64_t first, uint64_t count, void *host_out) {
    if (!h || !host_out) return fail(h, QCM_ERR_INVALID, "NULL argument");
    if (first + count > (1ull << h->n_local)) return fail(h, QCM_ERR_INVALID, "amplitude range outside the state");
    int rc = check_device(h);
    if (rc) return rc;
    const size_t ab = amp_bytes(h->prec);
    const uint64_t valid = 1ull << h->n_active;          // beyond: implicit zeros
    const uint64_t vend = std::min(first + count, valid);
    const char *const st = (const char *)h->state + (size_t)h->cur_point * bstate(h);
    if (h->rot_m && first < vend) {
        // rotated storage: fetch the active state and undo the rotation on the host (inspection path)
        if (h->n_active > 30) return fail(h, QCM_ERR_UNSUPPORTED, "qcm_get_amplitudes on a rotated state of %d qubits", h->n_active);
        if ((rc = materialise_last(h))) return rc;
        std::vector<char> tmp((size_t)valid * ab);
        QCM_CUDA(h, cudaMemcpyAsync(tmp.data(), st, (size_t)valid * ab, cudaMemcpyDeviceToHost, h->stream));
        QCM_CUDA(h, cudaStreamSynchronize(h->stream));
        const uint64_t lowm = (1ull << h->rot_nin) - 1ull;
        for (uint64_t i = first; i < vend; ++i) {
            const uint64_t phys = ((i & lowm) << h->rot_m) | (i >> h->rot_nin);
            memcpy((char *)host_out + (i - first) * ab, tmp.data() + phys * ab, ab);
        }
    } else if (first < vend)
        QCM_CUDA(h, cudaMemcpyAsync(host_out, st + first * ab, (vend - first) * ab, cudaMemcpyDeviceToHost, h->stream));
    QCM_CUDA(h, cudaStreamSynchronize(h->stream));
    if (first + count > vend) {
        const uint64_t z0 = std::max(first, vend);
        memset((char *)host_out + (z0 - first) * ab, 0, (first + count - z0) * ab);
    }
    return QCM_OK;
}

int qcm_set_amplitudes(qcm_handle h, uint64_t first, uint64_t count, const void *host_in, int n_active) {
    if (!h || !host_in) return fail(h, QCM_ERR_INVALID, "NULL argument");
    if (first + count > (1ull << h->n_local)) return fail(h, QCM_ERR_INVALID, "amplitude range outside the state");
    if (n_active < 0 || n_active > h->n_local) return fail(h, QCM_ERR_INVALID, "n_active out of range");
    int rc = check_device(h);
    if (rc) return rc;
    const size_t ab = amp_bytes(h->prec);
    QCM_CUDA(h, cudaMemcpyAsync((char *)h->state + (size_t)h->cur_point * bstate(h) + first * ab, host_in, count * ab, cudaMemcpyHostToDevice, h->stream));
    QCM_CUDA(h, cudaStreamSynchronize(h->stream));
    h->n_active = n_active;
    h->tree_valid = false;
    h->product_n = -1;
    h->rot_m = h->rot_nin = 0;
    h->virt = false;
    return QCM_OK;
}

int qcm_state_ptr(qcm_handle h, void **dev_ptr_out, uint64_t *bytes_out) {
    if (!h) return fail(nullptr, QCM_ERR_INVALID, "handle is NULL");
    int rc = check_device(h);
    if (rc) return rc;
    if ((rc = materialise_last(h))) return rc;
    if (dev_ptr_out) *dev_ptr_out = h->state;
    if (bytes_out) *bytes_out = (amp_bytes(h->prec) << h->n_local) * (uint64_t)h->batch;
    return QCM_OK;
}

int qcm_tree_level(qcm_handle h, int level, const double **dev_ptr_out, uint64_t *n_out, int *n_levels_out) {
    if (!h) return fail(nullptr, QCM_ERR_INVALID, "handle is NULL");
    if (!h->tree_valid) return fail(h, QCM_ERR_INVALID, "no sum tree");
    if (level < -1 || level >= h->tree_levels) return fail(h, QCM_ERR_INVALID, "tree level %d of %d", level, h->tree_levels);
    const double *p;
    uint64_t n;
    if (level >= 0) {
        p = h->tree_ptr[level];
        n = h->tree_n[level];
    } else if (h->tree_sub_input) {                // not stored: computed here with the sampler's arithmetic
        n = 1ull << (h->tree_base_bits - h->tree_sub_bits);
        int rc = ensure(h, h->subtree, sizeof(double) * n);
        if (rc) return rc;
        const unsigned blocks = (unsigned)((n + kThreads - 1) / kThreads);
        if (h->prec == QCM_C64) k_low_sub_entries<float><<<blocks, kThreads, 0, h->stream>>>(h->scratch.p, n, (double *)h->subtree.p);
        else k_low_sub_entries<double><<<blocks, kThreads, 0, h->stream>>>(h->scratch.p, n, (double *)h->subtree.p);
        QCM_CUDA(h, cudaGetLastError());
        QCM_CUDA(h, cudaStreamSynchronize(h->stream));
        p = (const double *)h->subtree.p;
    } else if (h->tree_has_sub) {                  // the fused checkpoint's level: sums over 2^tree_sub_bits amplitudes
        p = (const double *)h->subtree.p;
        n = 1ull << (h->tree_base_bits - h->tree_sub_bits);
    } else if (h->tree_sub_strided) {              // k_chunk_sums' 32 lane partials per chunk
        p = (const double *)h->subtree.p;
        n = h->tree_n[0] * 32;
    } else {
        return fail(h, QCM_ERR_INVALID, "the tree has no finer level");
    }
    if (dev_ptr_out) *dev_ptr_out = p;
    if (n_out) *n_out = n;
    if (n_levels_out) *n_levels_out = h->tree_levels;
    return QCM_OK;
}

int qcm_set_deferred(qcm_handle h, int deferred) {
    if (!h) return fail(nullptr, QCM_ERR_INVALID, "handle is NULL");
    h->deferred = deferred != 0;
    return QCM_OK;
}

int qcm_mark(qcm_handle h, uint64_t *ticket_out) {
    if (!h || !ticket_out) return fail(h, QCM_ERR_INVALID, "NULL argument");
    int rc = check_device(h);
    if (rc) return rc;
    const uint64_t t = h->n_marks;
    cudaEvent_t &e = h->marks[t % qcm_sim_s::kMarks];
    if (!e) QCM_CUDA(h, cudaEventCreateWithFlags(&e, cudaEventDisableTiming));
    QCM_CUDA(h, cudaEventRecord(e, h->stream));
    h->n_marks = t + 1;
    *ticket_out = t;
    return QCM_OK;
}

int qcm_wait(qcm_handle h, uint64_t ticket) {
    if (!h) return fail(nullptr, QCM_ERR_INVALID, "handle is NULL");
    if (ticket >= h->n_marks) return fail(h, QCM_ERR_INVALID, "ticket %llu was never issued", (unsigned long long)ticket);
    int rc = check_device(h);
    if (rc) return rc;
    // the slot holds this ticket's event or a later one of the same stream: waiting for it is sufficient either way
    QCM_CUDA(h, cudaEventSynchronize(h->marks[ticket % qcm_sim_s::kMarks]));
    return QCM_OK;
}

int qcm_host_alloc(void **host_out, size_t bytes) {
    if (!host_out) return fail(nullptr, QCM_ERR_INVALID, "NULL argument");
    *host_out = nullptr;
    cudaError_t e = cudaHostAlloc(host_out, bytes ? bytes : 1, cudaHostAllocDefault);
    if (e != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, QCM_ERR_NOMEM, "cudaHostAlloc(%zu): %s", bytes, cudaGetErrorString(e));
    }
    return QCM_OK;
}

int qcm_host_free(void *host_ptr) {
    if (host_ptr && cudaFreeHost(host_ptr) != cudaSuccess) {
        cudaGetLastError();
        return fail(nullptr, QCM_ERR_CUDA, "cudaFreeHost failed");
    }
    return QCM_OK;
}

int qcm_batch_size(qcm_handle h, int *batch_out) {
    if (!h || !batch_out) return fail(h, QCM_ERR_INVALID, "NULL argument");
    *batch_out = h->batch;
    return QCM_OK;
}

int qcm_batch_select(qcm_handle h, int point) {
    if (!h) return fail(nullptr, QCM_ERR_INVALID, "handle is NULL");
    if (point < 0 || point >= h->batch) return fail(h, QCM_ERR_INVALID, "point %d outside the batch of %d", point, h->batch);
    h->cur_point = point;
    return QCM_OK;
}

int qcm_set_active(qcm_handle h, int n_active) {
    if (!h) return fail(nullptr, QCM_ERR_INVALID, "handle is NULL");
    if (n_active < 0 || n_active > h->n_local) return fail(h, QCM_ERR_INVALID, "n_active out of range");
    if (h->rot_m && n_active != h->n_active) return fail(h, QCM_ERR_INVALID, "the state is stored rotated; start a new program first");
    h->n_active = n_active;
    h->tree_valid = false;
    h->product_n = -1;
    return QCM_OK;
}

int qcm_get_active(qcm_handle h, int *n_active_out) {
    if (!h || !n_active_out) return fail(h, QCM_ERR_INVALID, "NULL argument");
    *n_active_out = h->n_active;
    return QCM_OK;
}

int qcm_run_program(qcm_handle h, const qcm_op *ops, int n_ops, const double *tables, size_t n_tables) {
    if (!h) return fail(nullptr, QCM_ERR_INVALID, "handle is NULL");
    if (n_ops < 0 || (n_ops && !ops) || (n_tables && !tables)) return fail(h, QCM_ERR_INVALID, "NULL program");
    int rc = check_device(h);
    if (rc) return rc;
    h->tree_valid = false;
    h->product_n = -1;
    if (h->virt) {
        // the unwritten result depends on this handle's tables and scratch buffer, which this program may reuse: a new
        // state drops it, anything else (which is refused below) writes it out first
        if (n_ops > 0 && ops[0].kind == QCM_OP_INIT_PRODUCT) h->virt = false;
        else if ((rc = materialise_last(h))) return rc;
    }
    bool keep_tree = false;
    h->timing.bytes_read = h->timing.bytes_written = 0;
    QCM_CUDA(h, cudaEventRecord(h->ev0, h->stream));
    if ((rc = upload_tables(h, tables, n_tables))) return rc;
    h->op_kind.clear(); h->op_rd.clear(); h->op_wr.clear(); h->op_ms.clear(); h->op_kernel.clear(); h->cur_kernel.clear();
    size_t n_ev = 0;
    auto mark = [&](void) -> cudaError_t {
        if (n_ev >= h->op_ev.size()) {
            cudaEvent_t e;
            cudaError_t r = cudaEventCreate(&e);
            if (r != cudaSuccess) return r;
            h->op_ev.push_back(e);
        }
        return cudaEventRecord(h->op_ev[n_ev++], h->stream);
    };
    QCM_CUDA(h, mark());
    // Rotated last pass (QCM_FLAG_ROTATED_OUTPUT_OK): its kernel reads the input out of place.  When the
    // program starts from INIT_PRODUCT, everything before the last op fits that input buffer, so the
    // whole prefix runs IN the scratch buffer and no copy is needed; otherwise the input is copied.
    struct StateGuard {
        qcm_handle h; void *real;
        ~StateGuard() { if (real) h->state = real; }
    } guard{h, nullptr};
    int prefix_until = -1;
    bool no_rotate = false;
    {
        int li = -1;
        for (int i = 0; i < n_ops;) {
            li = i;
            i += 1 + (ops[i].kind == QCM_OP_BLOCK ? std::max(0, ops[i].n_ctrl) : 0);
        }
        if (li > 0 && h->batch == 1 && ops[0].kind == QCM_OP_INIT_PRODUCT && ops[li].kind == QCM_OP_BLOCK &&
            (ops[li].flags & QCM_FLAG_ROTATED_OUTPUT_OK) && rotate_enabled() && li + ops[li].n_ctrl == n_ops - 1) {
            const int n_in = ops[li].n_active_in;
            bool fits = n_in >= kChunkBits && n_in <= h->n_local;
            for (int i = 0; i < li && fits; ++i) fits = ops[i].n_active_out <= n_in && ops[i].n_active_in <= n_in;
            if (fits && ensure(h, h->scratch, amp_bytes(h->prec) << n_in) != QCM_OK) {
                cudaGetLastError();                       // no room for the scratch buffer: plain in-place schedule
                fits = false;
                no_rotate = true;
            }
            if (fits) {
                guard.real = h->state;
                h->state = h->scratch.p;
                prefix_until = li;
            }
        }
    }
    for (int i = 0; i < n_ops; ++i) {
        const qcm_op &op = ops[i];
        const uint64_t rd0 = h->timing.bytes_read, wr0 = h->timing.bytes_written;
        bool input_in_scratch = false;
        if (i == prefix_until) {                          // the last op: back to the real state buffer
            h->state = guard.real;
            guard.real = nullptr;
            input_in_scratch = true;
        }
        if (op.kind != QCM_OP_INIT_PRODUCT && op.n_active_in != h->n_active)
            return fail(h, QCM_ERR_INVALID, "op %d expects %d materialised qubits, state has %d", i, op.n_active_in, h->n_active);
        if (op.kind != QCM_OP_INIT_PRODUCT && h->rot_m)
            return fail(h, QCM_ERR_INVALID, "op %d: the state is stored rotated (the previous program ended with "
                        "QCM_FLAG_ROTATED_OUTPUT_OK); start with INIT_PRODUCT", i);
        if (op.kind == QCM_OP_INIT_PRODUCT) h->rot_m = h->rot_nin = 0;
        switch (op.kind) {
            case QCM_OP_INIT_PRODUCT:
                if ((rc = launch_init(h, op, n_tables, tables))) return rc;
                break;
            case QCM_OP_MUX1Q:
            case QCM_OP_BLOCK: {
                BlockPlan bp;
                int n_mem = 1;
                if (op.kind == QCM_OP_MUX1Q) {
                    int tq[1] = {op.target};
                    if ((rc = plan_block(h, tq, 1, &op, 1, op.n_active_in, op.n_active_out, n_tables, bp))) return rc;
                } else if (op.target == 0) {
                    // no targets: a diagonal block (every member DIAG), one sweep for all of them
                    n_mem = op.n_ctrl;
                    if (n_mem < 0 || i + n_mem > n_ops - 1) return fail(h, QCM_ERR_INVALID, "op %d: block members run past the program", i);
                    if (op.n_active_in != op.n_active_out) return fail(h, QCM_ERR_INVALID, "op %d: a diagonal block cannot materialise qubits", i);
                    if ((rc = launch_diag_multi(h, ops + i + 1, n_mem, op.n_active_in, n_tables))) return rc;
                    i += n_mem;
                    break;
                } else {
                    const int M = op.target;
                    n_mem = op.n_ctrl;
                    if (M < 1 || M > QCM_MAX_EXPAND) return fail(h, QCM_ERR_INVALID, "op %d: block of %d qubits (max %d)", i, M, QCM_MAX_EXPAND);
                    if (n_mem < 0 || i + n_mem > n_ops - 1) return fail(h, QCM_ERR_INVALID, "op %d: block members run past the program", i);
                    if ((rc = plan_block(h, op.ctrl, M, ops + i + 1, n_mem, op.n_active_in, op.n_active_out, n_tables, bp))) return rc;
                }
                // Sampling checkpoint: the final pass only multiplies every stored amplitude
                // into 2^M images whose squared moduli add up to the original, so the sum tree
                // can be built on the 2^M-times smaller input instead of re-reading the result.
                const bool last = (i + (op.kind == QCM_OP_BLOCK ? n_mem : 0)) == n_ops - 1;
                bool checkpoint = last && (op.flags & QCM_FLAG_SAMPLE_CHECKPOINT) && bp.norm_preserving &&
                                  op.n_active_in >= kChunkBits && h->batch == 1;
                // rotated output: last op, wide expansion on the product-tree path, enough image bits for a warp store
                bp.rotate = last && !no_rotate && h->batch == 1 && (op.flags & QCM_FLAG_ROTATED_OUTPUT_OK) && bp.tree && rotate_enabled() &&
                            op.n_active_in >= kChunkBits && bp.M >= (h->prec == QCM_C64 ? 6 : 5) &&
                            op.n_active_out - op.n_active_in == bp.M;
                if (bp.rotate) {                          // its product tables + the member tables must fit shared memory
                    const int mh = bp.M - (h->prec == QCM_C64 ? 6 : 5);
                    const size_t per_warp = ((size_t)512 << mh) + 12 * kLowRow * 2 * (h->prec == QCM_C64 ? 4 : 8);
                    if (per_warp * (h->prec == QCM_C64 ? 8 : 4) + bp.tree_smem > 200 * 1024) bp.rotate = false;
                }
                if (bp.rotate && !input_in_scratch && ensure(h, h->scratch, amp_bytes(h->prec) << op.n_active_in) != QCM_OK) {
                    cudaGetLastError();                   // no room for the input copy: keep the in-place kernel
                    bp.rotate = false;
                }
                // virtual: the result is left unwritten, its readers compute the images they use from the input (the
                // sampler on the checkpoint tree: one leaf's images per shot, the prefix post-selection: image 0 of
                // each kept input); without the checkpoint a sampler rebuilds the tree and writes the result out first
                bp.virt = bp.rotate && (virtual_last() == 1 || (virtual_last() < 0 && op.n_active_out > 30));
                bp.input_in_scratch = input_in_scratch;
                if (input_in_scratch && !bp.rotate) {     // the prefix ran in the scratch buffer after all: bring it home
                    QCM_CUDA(h, cudaMemcpyAsync(h->state, h->scratch.p, amp_bytes(h->prec) << op.n_active_in,
                                                cudaMemcpyDeviceToDevice, h->stream));
                }
                int sub_bits = 0;
                if (checkpoint) {
                    // level 0 of the tree: fused into the expansion pass (it reads every input amplitude
                    // anyway); a generic block pass cannot be norm-preserving, so an expansion kernel runs here.
                    // Finer level: per warp (table kernel) or per vector (tree kernel, whose input is small).
                    const int vbits = (h->prec == QCM_C64) ? 1 : 0;
                    sub_bits = bp.tree ? vbits : vbits + 5;
                    if ((rc = tree_layout(h, op.n_active_in))) return rc;
                    // a virtual pass stores no finer level: its input stays in `scratch` as long as the tree is valid
                    // (only a next program writes there), and the sampler computes the entries it reads from it
                    if (!bp.virt && (rc = ensure(h, h->subtree, sizeof(double) << (op.n_active_in - sub_bits)))) return rc;
                    bp.eargs.tree_out = bp.trargs.tree_out = h->tree_ptr[0];
                    bp.eargs.sub_out = bp.trargs.sub_out = bp.virt ? nullptr : (double *)h->subtree.p;
                }
                if ((rc = launch_block_plan(h, bp))) return rc;
                if (checkpoint) {
                    if ((rc = tree_finish(h, op.n_active_in))) return rc;
                    h->tree_sub_strided = false;
                    h->tree_cond_bits = bp.M;
                    h->tree_cond_low = bp.rotate;
                    h->tree_sub_bits = sub_bits;
                    h->tree_has_sub = true;
                    h->tree_sub_input = bp.virt;
                    h->tree_for_active = op.n_active_out;
                    h->n_checkpoint++;
                    keep_tree = true;
                }
                if (op.kind == QCM_OP_BLOCK) i += n_mem;
                break;
            }
            case QCM_OP_DIAG:
                if ((rc = launch_diag(h, op, n_tables))) return rc;
                break;
            case QCM_OP_SWAP:
                if ((rc = launch_swap(h, op))) return rc;
                break;
            case QCM_OP_EXTEND:
                if ((rc = launch_extend(h, op.n_active_in, op.n_active_out))) return rc;
                break;
            default:
                return fail(h, QCM_ERR_INVALID, "op %d: unknown kind %d", i, op.kind);
        }
        h->n_active = op.n_active_out;
        if (op.kind != QCM_OP_INIT_PRODUCT) h->product_n = -1;
        if (!keep_tree) h->tree_valid = false;
        QCM_CUDA(h, mark());
        h->op_kind.push_back(op.kind);
        h->op_kernel.push_back(h->cur_kernel);
        h->cur_kernel.clear();
        h->op_rd.push_back((h->timing.bytes_read - rd0) * (uint64_t)h->batch);
        h->op_wr.push_back((h->timing.bytes_written - wr0) * (uint64_t)h->batch);
    }
    h->timing.bytes_read *= (uint64_t)h->batch;
    h->timing.bytes_written *= (uint64_t)h->batch;
    QCM_CUDA(h, cudaEventRecord(h->ev1, h->stream));
    h->op_ms.assign(h->op_kind.size(), 0.f);
    h->op_ms_pending = h->deferred;
    if (h->deferred) return QCM_OK;          // enqueued; qcm_get_op_profile collects the per-op timings on demand
    QCM_CUDA(h, cudaEventSynchronize(h->ev1));
    float ms = 0.f;
    QCM_CUDA(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->timing.program_ms = ms;
    for (size_t k = 0; k < h->op_kind.size(); ++k) QCM_CUDA(h, cudaEventElapsedTime(&h->op_ms[k], h->op_ev[k], h->op_ev[k + 1]));
    return QCM_OK;
}

static int gather_block_impl(qcm_handle h, const qcm_op *ops, int n_ops, const double *tables, size_t n_tables,
                             const void *const *src_slabs, int s, void *dst_state, void *const *flag_ptrs, uint64_t flag_words,
                             uint32_t epoch);

int qcm_run_gather_block(qcm_handle h, const qcm_op *ops, int n_ops, const double *tables, size_t n_tables,
                         const void *const *src_slabs, int s, void *dst_state) {
    return gather_block_impl(h, ops, n_ops, tables, n_tables, src_slabs, s, dst_state, nullptr, 0, 0);
}

int qcm_gather_flag_words(int n_local, int s, int precision, uint64_t *words_out) {
    if (!words_out || s < 1 || s > QCM_MAX_GATHER || s >= n_local || (precision != QCM_C64 && precision != QCM_C128))
        return fail(nullptr, QCM_ERR_INVALID, "bad argument");
    *words_out = std::max<uint64_t>(1, gather_inplace_tiles(n_local, s, precision)) << s;
    return QCM_OK;
}

int qcm_run_gather_block_inplace(qcm_handle h, const qcm_op *ops, int n_ops, const double *tables, size_t n_tables,
                                 const void *const *src_slabs, int s, void *const *flag_ptrs, uint64_t flag_words, uint32_t epoch) {
    if (!flag_ptrs || !epoch) return fail(h, QCM_ERR_INVALID, "NULL flag array / zero epoch");
    return gather_block_impl(h, ops, n_ops, tables, n_tables, src_slabs, s, h ? h->state : nullptr, flag_ptrs, flag_words, epoch);
}

static int gather_block_impl(qcm_handle h, const qcm_op *ops, int n_ops, const double *tables, size_t n_tables,
                             const void *const *src_slabs, int s, void *dst_state, void *const *flag_ptrs, uint64_t flag_words,
                             uint32_t epoch) {
    if (!h || !ops || n_ops < 1 || !src_slabs || !dst_state) return fail(h, QCM_ERR_INVALID, "NULL argument");
    if (s < 1 || s > QCM_MAX_GATHER || s > h->n_global || s >= h->n_local) return fail(h, QCM_ERR_INVALID, "cannot gather %d qubits", s);
    if (h->n_active != h->n_local) return fail(h, QCM_ERR_INVALID, "gather needs a fully materialised shard");
    if (h->batch != 1) return fail(h, QCM_ERR_UNSUPPORTED, "gather on a batched handle");
    if (h->rot_m) return fail(h, QCM_ERR_INVALID, "gather on a rotated state");
    if (h->own_state) return fail(h, QCM_ERR_INVALID, "gather needs a caller-owned state buffer (ext_state): peers map it");
    int rc = check_device(h);
    if (rc) return rc;
    const qcm_op &hd = ops[0];
    const qcm_op *members = &hd;
    int n_mem = 1;
    int tq[QCM_MAX_GATHER];
    if (hd.kind == QCM_OP_BLOCK) {
        if (hd.target != s || hd.n_ctrl != n_ops - 1) return fail(h, QCM_ERR_INVALID, "gather block header does not match");
        members = ops + 1;
        n_mem = hd.n_ctrl;
        for (int j = 0; j < s; ++j) tq[j] = hd.ctrl[j];
    } else if (hd.kind == QCM_OP_MUX1Q && s == 1 && n_ops == 1) {
        tq[0] = hd.target;
    } else {
        return fail(h, QCM_ERR_INVALID, "gather block must be a MUX1Q (s = 1) or a BLOCK over the s swapped-in qubits");
    }
    for (int j = 0; j < s; ++j)
        if (tq[j] != h->n_local - s + j) return fail(h, QCM_ERR_INVALID, "gather block targets must be the %d highest local qubits", s);
    BlockPlan bp;
    if ((rc = plan_block(h, tq, s, members, n_mem, h->n_local, h->n_local, n_tables, bp))) return rc;
    h->tree_valid = false;
    h->product_n = -1;
    QCM_CUDA(h, cudaEventRecord(h->ev0, h->stream));
    if ((rc = upload_tables(h, tables, n_tables))) return rc;
    GatherArgs a{};
    for (int r = 0; r < (1 << s); ++r) {
        if (!src_slabs[r]) return fail(h, QCM_ERR_INVALID, "src_slabs[%d] is NULL", r);
        a.src[r] = src_slabs[r];
    }
    a.dst = dst_state;
    a.tables = tabreal(h);
    a.n_local = h->n_local;
    a.s = s;
    a.n_members = n_mem;
    a.ctrl_below_32 = bp.args.ctrl_below_32;
    a.rank_bits = rank_bits(h);
    for (int g = 0; g < n_mem; ++g) a.mem[g] = bp.args.mem[g];
    if (flag_ptrs) {
        // in place: the output overwrites this rank's own slabs, ordered against the peers' reads by per-tile flags
        const uint64_t tiles = gather_inplace_tiles(h->n_local, s, h->prec);
        if (tiles < 1 || (tiles << s) > flag_words) return fail(h, QCM_ERR_INVALID, "flag arrays too small: %llu words needed", (unsigned long long)(tiles << s));
        GatherFlags f{};
        int c_me = 0;
        for (int r = 0; r < (1 << s); ++r) {
            if (!flag_ptrs[r]) return fail(h, QCM_ERR_INVALID, "flag_ptrs[%d] is NULL", r);
            f.flags[r] = (uint32_t *)flag_ptrs[r];
            if ((const char *)src_slabs[r] >= (const char *)h->state && (const char *)src_slabs[r] < (const char *)h->state + bstate(h)) c_me = r;
        }
        f.c_me = c_me;                           // the source that lies inside this rank's own state is its own coordinate
        f.epoch = epoch;
        if ((rc = ensure(h, h->errflag, sizeof(int)))) return rc;
        QCM_CUDA(h, cudaMemsetAsync(h->errflag.p, 0, sizeof(int), h->stream));
        f.err = (int32_t *)h->errflag.p;
        int khz = 1900000;
        cudaDeviceGetAttribute(&khz, cudaDevAttrClockRate, h->device);
        f.spin_limit = (long long)khz * 1000ll * (long long)std::max(1, env_int("QCM_GATHER_SPIN_S", 5));
        if (h->prec == QCM_C64) {
            rc = s == 1 ? launch_gather_inplace<float, 2, 1>(h, a, f, bp.smem) : s == 2 ? launch_gather_inplace<float, 2, 2>(h, a, f, bp.smem)
                                                                                        : launch_gather_inplace<float, 2, 3>(h, a, f, bp.smem);
        } else {
            rc = s == 1 ? launch_gather_inplace<double, 1, 1>(h, a, f, bp.smem) : s == 2 ? launch_gather_inplace<double, 1, 2>(h, a, f, bp.smem)
                                                                                         : launch_gather_inplace<double, 1, 3>(h, a, f, bp.smem);
        }
        if (rc) return rc;
        int err = 0;
        QCM_CUDA(h, cudaMemcpyAsync(&err, h->errflag.p, sizeof(int), cudaMemcpyDeviceToHost, h->stream));
        QCM_CUDA(h, cudaStreamSynchronize(h->stream));
        if (err) return fail(h, QCM_ERR_CUDA, "in-place fused exchange: a peer did not signal within the spin limit (ranks out of step?)");
    } else if (h->prec == QCM_C64) rc = launch_gather_m<float, 2>(h, s, a, bp.smem);
    else rc = launch_gather_m<double, 1>(h, s, a, bp.smem);
    if (rc) return rc;
    QCM_CUDA(h, cudaEventRecord(h->ev1, h->stream));
    QCM_CUDA(h, cudaEventSynchronize(h->ev1));
    float ms = 0.f;
    QCM_CUDA(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->timing.program_ms = ms;
    h->timing.bytes_read = amp_bytes(h->prec) << h->n_local;
    h->timing.bytes_written = amp_bytes(h->prec) << h->n_local;
    h->state = dst_state;                   // the handle continues on the gathered buffer (caller-owned, like the old one)
    h->op_kind.assign(1, hd.kind);
    h->op_rd.assign(1, h->timing.bytes_read);
    h->op_wr.assign(1, h->timing.bytes_written);
    h->op_ms.assign(1, ms);
    return QCM_OK;
}

const char *qcm_op_kernel_name(qcm_handle h, int index) {
    if (!h || index < 0 || (size_t)index >= h->op_kernel.size()) return "";
    return h->op_kernel[index].c_str();
}

int qcm_get_op_profile(qcm_handle h, int cap, int32_t *kind_out, float *ms_out, uint64_t *bytes_read_out,
                       uint64_t *bytes_written_out, int *n_out) {
    if (!h || !n_out) return fail(h, QCM_ERR_INVALID, "NULL argument");
    const int n = (int)h->op_ms.size();
    *n_out = n;
    if (h->op_ms_pending && cap > 0 && (size_t)n < h->op_ev.size()) {
        // the last program was only enqueued (deferred mode): wait for its last op and read the events now
        int rc = check_device(h);
        if (rc) return rc;
        QCM_CUDA(h, cudaEventSynchronize(h->op_ev[n]));
        for (int k = 0; k < n; ++k) QCM_CUDA(h, cudaEventElapsedTime(&h->op_ms[k], h->op_ev[k], h->op_ev[k + 1]));
        h->op_ms_pending = false;
    }
    for (int k = 0; k < n && k < cap; ++k) {
        if (kind_out) kind_out[k] = h->op_kind[k];
        if (ms_out) ms_out[k] = h->op_ms[k];
        if (bytes_read_out) bytes_read_out[k] = h->op_rd[k];
        if (bytes_written_out) bytes_written_out[k] = h->op_wr[k];
    }
    return QCM_OK;
}

// mode 0: results to host buffers; 1: to caller-provided DEVICE buffers, no synchronisation (unbatched handles);
// 2: kept to the host, the probability block stays in the handle's device buffer (qcm_fetch_probs).
// Batched handle: kept_out holds `batch` doubles, probs_out `batch` consecutive blocks of 2^n_out_bits.
static int postselect_impl(qcm_handle h, uint64_t mask, uint64_t value, int n_out_bits, double *probs_out, double *kept_out, int mode) {
    const bool dev = mode == 1, resident = mode == 2;
    if (!h || !kept_out) return fail(h, QCM_ERR_INVALID, "NULL argument");
    if (n_out_bits < 0 || n_out_bits > h->n_local || n_out_bits > 30) return fail(h, QCM_ERR_INVALID, "n_out_bits %d out of range", n_out_bits);
    if (value & ~mask) return fail(h, QCM_ERR_INVALID, "value has bits outside mask");
    if (dev && h->batch != 1) return fail(h, QCM_ERR_UNSUPPORTED, "device-resident post-selection on a batched handle: use qcm_postselect_resident");
    int rc = check_device(h);
    if (rc) return rc;
    QCM_CUDA(h, cudaEventRecord(h->ev0, h->stream));
    const uint64_t nprob = 1ull << n_out_bits;
    const uint64_t B = (uint64_t)h->batch;
    const uint64_t local_all = (h->n_local >= 64) ? ~0ull : ((1ull << h->n_local) - 1ull);
    const uint64_t act_all = (1ull << h->n_active) - 1ull;
    const uint64_t rb = rank_bits(h);
    const bool want_probs = probs_out != nullptr || resident;
    if (dev) {
        QCM_CUDA(h, cudaMemsetAsync(kept_out, 0, sizeof(double), h->stream));
    } else {
        for (uint64_t y = 0; y < B; ++y) kept_out[y] = 0.0;
        if (probs_out) memset(probs_out, 0, nprob * B * sizeof(double));
    }
    if (!dev && want_probs) h->probs_n = 0;  // the handle's block buffer is about to be overwritten
    // global (rank) bits and never-materialised bits decide emptiness up front
    bool empty = ((rb & mask & ~local_all) != (value & ~local_all));
    if (value & local_all & ~act_all) empty = true;       // demands a 1 on a qubit known |0>
    if (!dev && want_probs && (rc = ensure(h, h->probs, nprob * B * sizeof(double)))) return rc;
    double *dprobs = want_probs ? (dev ? probs_out : (double *)h->probs.p) : nullptr;
    if (!empty) {
        const uint64_t lmask = mask & act_all, lval = value & act_all;
        const int nb = std::min(n_out_bits, h->n_active);
        const uint64_t out_all = (1ull << nb) - 1ull;
        const bool contiguous = (lval == 0) && (lmask == (act_all & ~out_all));
        // rotated storage: logical i lives at ((i & low) << rot_m) | (i >> rot_nin); the kept prefix
        // (i < 2^nb <= 2^rot_nin) is then the stride-2^rot_m sequence i << rot_m
        const int pshift = (h->rot_m && nb <= h->rot_nin) ? h->rot_m : 0;
        // a batched sweep spreads its points over the grid: fewer blocks per point
        const int blocks = B > 1 ? std::max(8, (int)((uint64_t)h->num_sms * 8 / B)) : h->num_sms * 4;
        const uint64_t bpart = (uint64_t)(blocks + 1) * sizeof(double), bprobs = nprob * sizeof(double);
        if ((rc = ensure(h, h->partial, bpart * B))) return rc;
        if (contiguous && (!h->rot_m || pshift)) {
            const uint64_t count = 1ull << nb;
            if (dprobs && count < nprob) QCM_CUDA(h, cudaMemsetAsync(dprobs, 0, nprob * B * sizeof(double), h->stream));
            double *const part = (double *)h->partial.p;
            if (h->virt) {                        // image 0 of each kept input, from the unwritten pass's input
                if (h->prec == QCM_C64) k_probs_prefix<float, true><<<bgrid(h, blocks), kThreads, 0, h->stream>>>(h->scratch.p, count, 0, dprobs, part, 0, bprobs, bpart, h->virt_args);
                else k_probs_prefix<double, true><<<bgrid(h, blocks), kThreads, 0, h->stream>>>(h->scratch.p, count, 0, dprobs, part, 0, bprobs, bpart, h->virt_args);
            } else if (h->prec == QCM_C64) {
                k_probs_prefix<float, false><<<bgrid(h, blocks), kThreads, 0, h->stream>>>(h->state, count, pshift, dprobs, part, bstate(h), bprobs, bpart, ExpandTreeArgs{});
            } else {
                k_probs_prefix<double, false><<<bgrid(h, blocks), kThreads, 0, h->stream>>>(h->state, count, pshift, dprobs, part, bstate(h), bprobs, bpart, ExpandTreeArgs{});
            }
        } else {
            if ((rc = materialise_last(h))) return rc;
            if (dprobs) QCM_CUDA(h, cudaMemsetAsync(dprobs, 0, nprob * B * sizeof(double), h->stream));
            if (h->prec == QCM_C64)
                k_postselect_general<float><<<bgrid(h, blocks), kThreads, 0, h->stream>>>(h->state, h->n_active, rb, mask, value, nprob - 1, h->rot_m, h->rot_nin, dprobs, (double *)h->partial.p, bstate(h), bprobs, bpart);
            else
                k_postselect_general<double><<<bgrid(h, blocks), kThreads, 0, h->stream>>>(h->state, h->n_active, rb, mask, value, nprob - 1, h->rot_m, h->rot_nin, dprobs, (double *)h->partial.p, bstate(h), bprobs, bpart);
        }
        QCM_CUDA(h, cudaGetLastError());
        h->timing.kernel_launches++;
        // per-point kept mass: the block partials summed in index order, written behind them
        k_tree_level<<<bgrid(h, 1), kThreads, 0, h->stream>>>((const double *)h->partial.p, (uint64_t)blocks,
                                                              dev ? kept_out : (double *)h->partial.p + blocks, 1, bpart, dev ? 0 : bpart, 30);
        QCM_CUDA(h, cudaGetLastError());
        h->timing.kernel_launches++;
        if (!dev) {
            QCM_CUDA(h, cudaMemcpy2DAsync(kept_out, sizeof(double), (double *)h->partial.p + blocks, bpart, sizeof(double), B,
                                          cudaMemcpyDeviceToHost, h->stream));
            if (probs_out) QCM_CUDA(h, cudaMemcpyAsync(probs_out, dprobs, nprob * B * sizeof(double), cudaMemcpyDeviceToHost, h->stream));
        }
    } else if (dprobs) {
        QCM_CUDA(h, cudaMemsetAsync(dprobs, 0, nprob * B * sizeof(double), h->stream));
    }
    if (dev) return QCM_OK;                 // results stay on the device, in stream order: no synchronisation
    if (resident) h->probs_n = nprob;
    QCM_CUDA(h, cudaEventRecord(h->ev1, h->stream));
    if (h->deferred) return QCM_OK;         // kept_out / probs_out (pinned host memory) are valid after qcm_synchronize
    QCM_CUDA(h, cudaEventSynchronize(h->ev1));
    float ms = 0.f;
    QCM_CUDA(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->timing.postselect_ms = ms;
    return QCM_OK;
}

int qcm_postselect(qcm_handle h, uint64_t mask, uint64_t value, int n_out_bits, double *probs_out, double *kept_out) {
    return postselect_impl(h, mask, value, n_out_bits, probs_out, kept_out, 0);
}

int qcm_postselect_device(qcm_handle h, uint64_t mask, uint64_t value, int n_out_bits, void *dev_probs_out, void *dev_kept_out) {
    return postselect_impl(h, mask, value, n_out_bits, (double *)dev_probs_out, (double *)dev_kept_out, 1);
}

int qcm_postselect_resident(qcm_handle h, uint64_t mask, uint64_t value, int n_out_bits, double *kept_out) {
    return postselect_impl(h, mask, value, n_out_bits, nullptr, kept_out, 2);
}

int qcm_fetch_probs(qcm_handle h, int point, uint64_t first, uint64_t count, double *host_out) {
    if (!h || !host_out) return fail(h, QCM_ERR_INVALID, "NULL argument");
    if (!h->probs_n) return fail(h, QCM_ERR_INVALID, "no resident post-selected block (call qcm_postselect_resident first)");
    if (point < 0 || point >= h->batch || first + count > h->probs_n) return fail(h, QCM_ERR_INVALID, "range outside the resident block");
    int rc = check_device(h);
    if (rc) return rc;
    QCM_CUDA(h, cudaMemcpyAsync(host_out, (const double *)h->probs.p + (uint64_t)point * h->probs_n + first, count * sizeof(double),
                                cudaMemcpyDeviceToHost, h->stream));
    QCM_CUDA(h, cudaStreamSynchronize(h->stream));
    return QCM_OK;
}

int qcm_sample_prepare(qcm_handle h, double *local_mass_out) {
    if (!h) return fail(nullptr, QCM_ERR_INVALID, "handle is NULL");
    int rc = check_device(h);
    if (rc) return rc;
    if (product_state(h)) {                  // no tree: the sampler draws a product state qubit by qubit
        if (local_mass_out) *local_mass_out = h->product_mass;
        return QCM_OK;
    }
    if (!h->tree_valid || h->tree_for_active != h->n_active)
        if ((rc = build_tree(h))) return rc;
    if (local_mass_out) *local_mass_out = h->local_mass;
    return QCM_OK;
}

// stream_ids: batched handles only -- one Philox stream per sweep point (host array of `batch` entries); the
// keys of point y land at keys_out + y * shots.  Batched sampling is unsharded (n_ranks == 1).
static int sample_sharded_impl(qcm_handle h, uint64_t shots, uint64_t seed, uint64_t stream_id, const double *rank_masses, int n_ranks,
                               const int32_t *clbit_qubit, int n_clbits, uint64_t *keys_out, uint8_t *mine_out, bool dev,
                               const uint64_t *stream_ids = nullptr, const double *dev_masses = nullptr, int64_t mass_stride = 1) {
    if (!h || !keys_out || (!rank_masses && !stream_ids && !dev_masses)) return fail(h, QCM_ERR_INVALID, "NULL argument");
    if ((h->batch > 1) != (stream_ids != nullptr)) return fail(h, QCM_ERR_INVALID, "batched handles sample with qcm_sample_batched (and only they)");
    if (stream_ids && (h->n_global != 0 || mine_out)) return fail(h, QCM_ERR_UNSUPPORTED, "batched sampling on a sharded state");
    if (n_ranks < 1 || (uint64_t)n_ranks != (1ull << h->n_global)) return fail(h, QCM_ERR_INVALID, "n_ranks %d does not match %d global qubits", n_ranks, h->n_global);
    if (n_clbits < 0 || n_clbits > 64 || (n_clbits && !clbit_qubit)) return fail(h, QCM_ERR_INVALID, "bad clbit map");
    int rc = check_device(h);
    if (rc) return rc;
    if (product_state(h) && n_ranks == 1 && !dev_masses) {
        if (shots == 0) return QCM_OK;
        QCM_CUDA(h, cudaEventRecord(h->ev0, h->stream));
        const uint64_t Bp = (uint64_t)h->batch;
        ProductSampleArgs pa{};
        pa.qv = (const double *)h->tab_f64.p + h->product_off;
        pa.n = h->product_n;
        pa.shots = shots;
        pa.seed = seed;
        pa.stream = stream_id;
        pa.bqv = btab64(h);
        pa.bkeys = shots * sizeof(uint64_t);
        if (stream_ids) {
            if ((rc = ensure(h, h->streams, sizeof(uint64_t) * Bp))) return rc;
            QCM_CUDA(h, cudaMemcpyAsync(h->streams.p, stream_ids, sizeof(uint64_t) * Bp, cudaMemcpyHostToDevice, h->stream));
            pa.streams = (const uint64_t *)h->streams.p;
        }
        pa.n_clbits = n_clbits;
        for (int c = 0; c < n_clbits; ++c) {
            if (clbit_qubit[c] >= h->n_local) return fail(h, QCM_ERR_INVALID, "clbit %d maps to qubit %d out of range", c, clbit_qubit[c]);
            pa.clbit_qubit[c] = (int8_t)(clbit_qubit[c] < 0 ? -1 : clbit_qubit[c]);
        }
        if (dev) {
            pa.keys_out = keys_out;
            if (mine_out) QCM_CUDA(h, cudaMemsetAsync(mine_out, 1, shots, h->stream));
        } else {
            if ((rc = ensure(h, h->keys, shots * Bp * sizeof(uint64_t)))) return rc;
            pa.keys_out = (uint64_t *)h->keys.p;
        }
        k_sample_product<<<bgrid(h, (shots + kThreads - 1) / kThreads), kThreads, 0, h->stream>>>(pa);
        QCM_CUDA(h, cudaGetLastError());
        h->timing.kernel_launches++;
        if (dev) return QCM_OK;
        QCM_CUDA(h, cudaMemcpyAsync(keys_out, h->keys.p, shots * Bp * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->stream));
        if (mine_out) memset(mine_out, 1, shots);
        QCM_CUDA(h, cudaEventRecord(h->ev1, h->stream));
        if (h->deferred) return QCM_OK;
        QCM_CUDA(h, cudaEventSynchronize(h->ev1));
        float pms = 0.f;
        QCM_CUDA(h, cudaEventElapsedTime(&pms, h->ev0, h->ev1));
        h->timing.sample_ms = pms;
        return QCM_OK;
    }
    if (!h->tree_valid || h->tree_for_active != h->n_active)
        if ((rc = build_tree(h))) return rc;
    if (shots == 0) return QCM_OK;
    QCM_CUDA(h, cudaEventRecord(h->ev0, h->stream));
    SampleArgs a{};
    a.state = h->state;
    a.n_active = h->tree_base_bits;
    a.cond_bits = h->tree_cond_bits;
    a.cond_low = (h->tree_cond_bits && h->tree_cond_low) ? 1 : 0;
    a.rot_m = h->rot_m;
    a.rot_nin = h->rot_nin;
    if (h->virt) {                           // the tree is the virtual pass's checkpoint (a rebuilt one materialised it)
        a.virt_in = h->scratch.p;
        a.virt = h->virt_args;
    }
    a.sub = ((h->tree_has_sub && !h->tree_sub_input) || h->tree_sub_strided) ? (const double *)h->subtree.p : nullptr;
    a.sub_in = h->tree_sub_input ? h->scratch.p : nullptr;
    a.sub_bits = h->tree_sub_bits;
    a.sub_strided = (h->tree_sub_strided && !h->tree_has_sub) ? 1 : 0;
    a.bsub = (sizeof(double) * 32) << (h->tree_base_bits - std::min(h->tree_base_bits, kChunkBits));
    a.n_levels = h->tree_levels;
    for (int l = 0; l < h->tree_levels; ++l) {
        a.level[l] = h->tree_ptr[l];
        a.level_n[l] = h->tree_n[l];
    }
    a.shots = shots;
    a.seed = seed;
    a.stream = stream_id;
    double lo = 0.0, total = 0.0;
    const uint64_t B = (uint64_t)h->batch;
    if (stream_ids) {
        // per-point totals were left on the device by the tree build; streams go up here
        if ((rc = ensure(h, h->streams, sizeof(uint64_t) * B))) return rc;
        QCM_CUDA(h, cudaMemcpyAsync(h->streams.p, stream_ids, sizeof(uint64_t) * B, cudaMemcpyHostToDevice, h->stream));
        a.streams = (const uint64_t *)h->streams.p;
        a.totals = (const double *)h->totals.p;
        a.bstate = bstate(h);
        a.btree = h->tree_total * sizeof(double);
        a.bkeys = shots * sizeof(uint64_t);
        a.rank_lo = 0.0;
        a.rank_hi = 1e300;
        a.total = 1.0;
    } else if (dev_masses) {
        a.dev_masses = dev_masses;
        a.mass_stride = mass_stride;
        a.n_ranks = n_ranks;
        a.my_rank = (int)h->rank;
    } else {
        for (int r = 0; r < n_ranks; ++r) {
            if ((uint64_t)r == h->rank) lo = total;
            total += rank_masses[r];
        }
        if (!(total > 0.0)) return fail(h, QCM_ERR_INVALID, "state has zero norm");
        a.rank_lo = lo;
        a.rank_hi = ((int)h->rank == n_ranks - 1) ? 1e300 : lo + rank_masses[h->rank];
        a.total = total;
    }
    a.rank_bits = rank_bits(h);
    a.n_clbits = n_clbits;
    for (int c = 0; c < n_clbits; ++c) {
        if (clbit_qubit[c] >= h->n_local + h->n_global) return fail(h, QCM_ERR_INVALID, "clbit %d maps to qubit %d out of range", c, clbit_qubit[c]);
        a.clbit_qubit[c] = (int8_t)(clbit_qubit[c] < 0 ? -1 : clbit_qubit[c]);
    }
    if (dev) {
        a.keys_out = keys_out;
        a.mine_out = mine_out;
    } else {
        if ((rc = ensure(h, h->keys, shots * B * sizeof(uint64_t)))) return rc;
        if ((rc = ensure(h, h->mine, shots))) return rc;
        a.keys_out = (uint64_t *)h->keys.p;
        a.mine_out = stream_ids ? nullptr : (uint8_t *)h->mine.p;
    }
    const uint64_t wpb = kThreads / 32;
    // a batched sweep spreads its points over the grid: fewer blocks per point
    const uint64_t cap = B > 1 ? std::max<uint64_t>(4, (uint64_t)h->num_sms * 16 / B) : (uint64_t)h->num_sms * 8;
    const unsigned blocks = (unsigned)std::min<uint64_t>((shots + wpb - 1) / wpb, cap);
    if (h->prec == QCM_C64) k_sample<float><<<bgrid(h, blocks), kThreads, 0, h->stream>>>(a);
    else k_sample<double><<<bgrid(h, blocks), kThreads, 0, h->stream>>>(a);
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    if (dev) return QCM_OK;                 // keys / mine stay on the device, in stream order
    QCM_CUDA(h, cudaMemcpyAsync(keys_out, h->keys.p, shots * B * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->stream));
    if (mine_out) QCM_CUDA(h, cudaMemcpyAsync(mine_out, h->mine.p, shots, cudaMemcpyDeviceToHost, h->stream));
    QCM_CUDA(h, cudaEventRecord(h->ev1, h->stream));
    if (h->deferred) return QCM_OK;
    QCM_CUDA(h, cudaEventSynchronize(h->ev1));
    float ms = 0.f;
    QCM_CUDA(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->timing.sample_ms = ms;
    return QCM_OK;
}

int qcm_sample_sharded(qcm_handle h, uint64_t shots, uint64_t seed, uint64_t stream_id, const double *rank_masses, int n_ranks,
                       const int32_t *clbit_qubit, int n_clbits, uint64_t *keys_out, uint8_t *mine_out) {
    return sample_sharded_impl(h, shots, seed, stream_id, rank_masses, n_ranks, clbit_qubit, n_clbits, keys_out, mine_out, false);
}

int qcm_sample_sharded_device(qcm_handle h, uint64_t shots, uint64_t seed, uint64_t stream_id, const double *rank_masses, int n_ranks,
                              const int32_t *clbit_qubit, int n_clbits, void *dev_keys_out, void *dev_mine_out) {
    if (!dev_mine_out) return fail(h, QCM_ERR_INVALID, "NULL argument");
    return sample_sharded_impl(h, shots, seed, stream_id, rank_masses, n_ranks, clbit_qubit, n_clbits, (uint64_t *)dev_keys_out,
                               (uint8_t *)dev_mine_out, true);
}

int qcm_tree_total_device(qcm_handle h, void *dev_total_out) {
    if (!h || !dev_total_out) return fail(h, QCM_ERR_INVALID, "NULL argument");
    int rc = check_device(h);
    if (rc) return rc;
    if (!h->tree_valid || h->tree_for_active != h->n_active)
        if ((rc = build_tree(h))) return rc;
    const int levels = h->tree_levels;
    k_batch_totals<<<(h->batch + 127) / 128, 128, 0, h->stream>>>(h->tree_ptr[levels - 1], h->tree_n[levels - 1],
                                                                  h->tree_total * sizeof(double), (double *)dev_total_out, h->batch);
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    return QCM_OK;
}

int qcm_sample_sharded_devmass(qcm_handle h, uint64_t shots, uint64_t seed, uint64_t stream_id, const void *dev_rank_masses,
                               int64_t mass_stride, int n_ranks, const int32_t *clbit_qubit, int n_clbits, void *dev_keys_out,
                               void *dev_mine_out) {
    if (!dev_mine_out || !dev_rank_masses || mass_stride < 1) return fail(h, QCM_ERR_INVALID, "NULL argument");
    return sample_sharded_impl(h, shots, seed, stream_id, nullptr, n_ranks, clbit_qubit, n_clbits, (uint64_t *)dev_keys_out,
                               (uint8_t *)dev_mine_out, true, nullptr, (const double *)dev_rank_masses, mass_stride);
}

int qcm_sample(qcm_handle h, uint64_t shots, uint64_t seed, uint64_t stream_id, const int32_t *clbit_qubit, int n_clbits,
               uint64_t *keys_out) {
    if (!h) return fail(nullptr, QCM_ERR_INVALID, "handle is NULL");
    if (h->n_global != 0) return fail(h, QCM_ERR_INVALID, "sharded state: use qcm_sample_prepare + qcm_sample_sharded");
    double mass = 0.0;
    int rc = qcm_sample_prepare(h, &mass);
    if (rc) return rc;
    if (h->deferred && h->batch == 1 && !product_state(h)) {
        // deferred mode: the tree's total was not read back; it is summed on the device (same index order as the host
        // sum of the blocking mode, so the shots are identical) and the sampler reads it there
        if ((rc = ensure(h, h->totals, sizeof(double)))) return rc;
        if ((rc = qcm_tree_total_device(h, h->totals.p))) return rc;
        return sample_sharded_impl(h, shots, seed, stream_id, nullptr, 1, clbit_qubit, n_clbits, keys_out, nullptr, false, nullptr,
                                   (const double *)h->totals.p, 1);
    }
    return qcm_sample_sharded(h, shots, seed, stream_id, &mass, 1, clbit_qubit, n_clbits, keys_out, nullptr);
}

int qcm_sample_batched(qcm_handle h, uint64_t shots, uint64_t seed, const uint64_t *stream_ids, const int32_t *clbit_qubit, int n_clbits,
                       uint64_t *keys_out) {
    if (!h || !stream_ids) return fail(h, QCM_ERR_INVALID, "NULL argument");
    double mass = 0.0;
    int rc = qcm_sample_prepare(h, &mass);
    if (rc) return rc;
    return sample_sharded_impl(h, shots, seed, 0, nullptr, 1, clbit_qubit, n_clbits, keys_out, nullptr, false, stream_ids);
}

static int sample_released_impl(qcm_handle h, uint64_t shots, uint64_t seed, uint64_t stream_id, const uint64_t *stream_ids, int nv,
                                const int32_t *n_ctrl, const int32_t *ctrl, int max_ctrl, const double *p1, const int64_t *p1_off,
                                int64_t n_p1, const int32_t *vclbit, const int32_t *clbit_pos, int n_clbits, uint64_t *keys_out);

int qcm_sample_released(qcm_handle h, uint64_t shots, uint64_t seed, uint64_t stream_id, int nv, const int32_t *n_ctrl,
                        const int32_t *ctrl, int max_ctrl, const double *p1, const int64_t *p1_off, int64_t n_p1,
                        const int32_t *vclbit, const int32_t *clbit_pos, int n_clbits, uint64_t *keys_out) {
    if (h && h->batch != 1) return fail(h, QCM_ERR_INVALID, "batched handle: use qcm_sample_released_batched");
    return sample_released_impl(h, shots, seed, stream_id, nullptr, nv, n_ctrl, ctrl, max_ctrl, p1, p1_off, n_p1, vclbit, clbit_pos,
                                n_clbits, keys_out);
}

int qcm_sample_released_batched(qcm_handle h, uint64_t shots, uint64_t seed, const uint64_t *stream_ids, int nv, const int32_t *n_ctrl,
                                const int32_t *ctrl, int max_ctrl, const double *p1, const int64_t *p1_off, int64_t n_p1,
                                const int32_t *vclbit, const int32_t *clbit_pos, int n_clbits, uint64_t *keys_out) {
    if (!stream_ids) return fail(h, QCM_ERR_INVALID, "NULL argument");
    return sample_released_impl(h, shots, seed, 0, stream_ids, nv, n_ctrl, ctrl, max_ctrl, p1, p1_off, n_p1, vclbit, clbit_pos,
                                n_clbits, keys_out);
}

// p1: `batch` consecutive sets of n_p1 probabilities (one set for a plain handle)
static int sample_released_impl(qcm_handle h, uint64_t shots, uint64_t seed, uint64_t stream_id, const uint64_t *stream_ids, int nv,
                                const int32_t *n_ctrl, const int32_t *ctrl, int max_ctrl, const double *p1, const int64_t *p1_off,
                                int64_t n_p1, const int32_t *vclbit, const int32_t *clbit_pos, int n_clbits, uint64_t *keys_out) {
    if (!h || !keys_out || !n_ctrl || !ctrl || !p1 || !p1_off || !vclbit || !clbit_pos) return fail(h, QCM_ERR_INVALID, "NULL argument");
    if (h->n_global != 0) return fail(h, QCM_ERR_UNSUPPORTED, "released-qubit sampling on a sharded state");
    if ((h->batch > 1) != (stream_ids != nullptr)) return fail(h, QCM_ERR_INVALID, "batched handles sample with the _batched entry points (and only they)");
    const uint64_t B = (uint64_t)h->batch;
    if (nv < 0 || nv > kMaxReleased || n_clbits < 0 || n_clbits > 64 || max_ctrl < 1) return fail(h, QCM_ERR_INVALID, "bad released-qubit tables");
    ReleasedArgs a{};
    for (int k = 0; k < nv; ++k) {
        if (n_ctrl[k] < 0 || n_ctrl[k] > QCM_MAX_CTRL || n_ctrl[k] > max_ctrl) return fail(h, QCM_ERR_INVALID, "released qubit %d: n_ctrl out of range", k);
        if (p1_off[k] < 0 || p1_off[k] + (1ll << n_ctrl[k]) > n_p1) return fail(h, QCM_ERR_INVALID, "released qubit %d: table outside p1", k);
        if (vclbit[k] >= 64) return fail(h, QCM_ERR_INVALID, "released qubit %d: clbit out of range", k);
        a.n_ctrl[k] = (int8_t)n_ctrl[k];
        a.p1_off[k] = (int32_t)p1_off[k];
        a.vclbit[k] = (int8_t)(vclbit[k] < 0 ? -1 : vclbit[k]);
        for (int j = 0; j < n_ctrl[k]; ++j) {
            const int c = ctrl[(size_t)k * max_ctrl + j];
            if (c < 0 || c >= h->n_local) return fail(h, QCM_ERR_INVALID, "released qubit %d: index qubit %d out of range", k, c);
            a.ctrl[k][j] = (int8_t)c;
        }
    }
    for (int c = 0; c < 64; ++c) a.clbit_pos[c] = -1;
    for (int c = 0; c < n_clbits; ++c) {
        if (clbit_pos[c] >= h->n_local) return fail(h, QCM_ERR_INVALID, "clbit %d maps to qubit %d out of range", c, clbit_pos[c]);
        a.clbit_pos[c] = (int8_t)(clbit_pos[c] < 0 ? -1 : clbit_pos[c]);
    }
    // raw basis states of the stored qubits, on the device (the sampler's own stream: seed, stream_id)
    double mass = 0.0;
    int rc = qcm_sample_prepare(h, &mass);
    if (rc) return rc;
    if (shots == 0) return QCM_OK;
    if ((rc = ensure(h, h->keys, shots * B * sizeof(uint64_t)))) return rc;
    if ((rc = ensure(h, h->relp1, (size_t)n_p1 * B * sizeof(double)))) return rc;
    if ((rc = sample_sharded_impl(h, shots, seed, stream_id, &mass, 1, nullptr, 0, (uint64_t *)h->keys.p, nullptr, true, stream_ids))) return rc;
    QCM_CUDA(h, cudaMemcpyAsync(h->relp1.p, p1, (size_t)n_p1 * B * sizeof(double), cudaMemcpyHostToDevice, h->stream));
    a.bkeys = shots * sizeof(uint64_t);
    a.bp1 = (uint64_t)n_p1 * sizeof(double);
    a.streams = stream_ids ? (const uint64_t *)h->streams.p : nullptr;
    a.keys = (uint64_t *)h->keys.p;
    a.shots = shots;
    a.seed = seed;
    a.stream = stream_id;
    a.p1 = (const double *)h->relp1.p;
    a.nv = nv;
    a.n_clbits = n_clbits;
    k_released_keys<<<bgrid(h, (shots + kThreads - 1) / kThreads), kThreads, 0, h->stream>>>(a);
    QCM_CUDA(h, cudaGetLastError());
    h->timing.kernel_launches++;
    QCM_CUDA(h, cudaMemcpyAsync(keys_out, h->keys.p, shots * B * sizeof(uint64_t), cudaMemcpyDeviceToHost, h->stream));
    QCM_CUDA(h, cudaEventRecord(h->ev1, h->stream));
    if (h->deferred) return QCM_OK;
    QCM_CUDA(h, cudaEventSynchronize(h->ev1));
    float ms = 0.f;
    QCM_CUDA(h, cudaEventElapsedTime(&ms, h->ev0, h->ev1));
    h->timing.sample_ms = ms;
    return QCM_OK;
}

int qcm_get_timing(qcm_handle h, qcm_timing *out) {
    if (!h || !out) return fail(h, QCM_ERR_INVALID, "NULL argument");
    *out = h->timing;
    return QCM_OK;
}

}  // extern "C"
