/*
 * qcmrf_b200 -- C ABI of the B200-native statevector engine for QCMRF circuits.
 *
 * This is the drop-in boundary: it replaces what the reference reaches through
 *     simulator = Aer.get_backend('qasm_simulator')
 *     result    = simulator.run(T, shots=SHOTS).result()
 *     counts    = result.get_counts()
 * (/root/reference/run_experiment.py:54-57), i.e. qiskit-aer's C++ controller
 * behind the pybind call inside ``.run()``; and the post-selection arithmetic of
 * /root/reference/QCMRF.py:263-284 and /root/reference/eval.py:115-123, which it
 * moves onto the GPU.  The Python side (qcmrf_b200/backend.py) lowers and fuses a
 * circuit into a short list of ``qcm_op`` and calls the functions below through
 * ctypes; INTEGRATION.md shows the binding.
 *
 * Conventions
 *  - every function returns QCM_OK (0) or a negative qcm_status; nothing throws
 *    across the ABI; ``qcm_last_error`` returns a human-readable message.
 *  - all pointers in signatures are HOST pointers owned and sized by the caller,
 *    except ``ext_state`` / ``ext_stream`` of qcm_create (device memory / a
 *    cudaStream_t the caller owns, e.g. a torch tensor and torch's stream).
 *  - a handle is bound to one device and one stream and is not thread-safe.
 *  - basis-state index bit q <-> qubit q (Qiskit little-endian).  For a sharded
 *    state the handle holds the 2^n_local amplitudes whose global index has the
 *    high bits equal to ``rank`` (qcm_set_shard).
 *  - coefficient tables are passed in fp64 and rounded once to the state's
 *    precision, so fp32 kernels get correctly rounded coefficients.
 *  - there is no CPU fallback: without a CUDA device every compute entry point
 *    fails with QCM_ERR_NO_DEVICE.
 */
#ifndef QCMRF_B200_H
#define QCMRF_B200_H

#include <stddef.h>
#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QCM_ABI_VERSION 1
#define QCM_MAX_CTRL 10      /* table-index qubits of one MUX1Q / DIAG op           */
#define QCM_MAX_BLOCK 5      /* target qubits of one BLOCK pass (2^5 vectors/thread) */
#define QCM_MAX_GATHER 3     /* global qubits one fused exchange+gate pass swaps in (8 ranks) */
#define QCM_MAX_EXPAND 8     /* ... of a BLOCK pass whose qubits are all new (one MUX1Q each) */
#define QCM_MAX_MEMBERS 16   /* MUX1Q members of one BLOCK pass                      */

typedef struct qcm_sim_s *qcm_handle;

enum qcm_status {
    QCM_OK = 0,
    QCM_ERR_INVALID = -1,      /* bad argument / malformed program        */
    QCM_ERR_CUDA = -2,         /* a CUDA runtime call failed              */
    QCM_ERR_NOMEM = -3,        /* device or host allocation failed        */
    QCM_ERR_UNSUPPORTED = -4,  /* valid request this build cannot serve   */
    QCM_ERR_NO_DEVICE = -5     /* no usable CUDA device                   */
};

enum qcm_precision { QCM_C64 = 32, QCM_C128 = 64 };   /* bits of the real type */

enum qcm_op_kind {
    /* state <- tensor product of per-qubit 2-vectors over the first n_active_out
     * qubits; table = n_active_out * 4 doubles (amp0.re, amp0.im, amp1.re, amp1.im).
     * The leading H layer of QCMRF._build (QCMRF.py:204-205) folds into this.     */
    QCM_OP_INIT_PRODUCT = 1,
    /* uniformly-controlled single-qubit gate: for every assignment c of the n_ctrl
     * index qubits apply the 2x2 matrix table[c] (8 doubles, row-major re/im) on
     * `target`.  One fused QCMRF clique block (QCMRF.py:216-236) is one of these;
     * so is every h/x/sx/cx/mcx/AND of an unfused program.                        */
    QCM_OP_MUX1Q = 2,
    /* diagonal: amplitude *= table[c] (2 doubles per entry) -- rz, p, cp, cz ...   */
    QCM_OP_DIAG = 3,
    /* header of a blocked pass: the next `n_ctrl` ops (MUX1Q with targets among the
     * block's qubits, pairwise distinct or repeated; or DIAG, a diagonal factor applied
     * in the same sweep; no member's index qubits among the block's targets) are
     * applied in ONE sweep, in order; `ctrl[0..target-1]` lists the block's `target`
     * (= count) distinct target qubits in ascending order.  `target` == 0: a diagonal
     * block -- every member is a DIAG and all of them are applied in one sweep.      */
    QCM_OP_BLOCK = 4,
    /* exchange qubits `target` and `ctrl[0]` (both local)                          */
    QCM_OP_SWAP = 5,
    /* materialise qubits [n_active_in, n_active_out) as |0>: zero-fills the new part  */
    QCM_OP_EXTEND = 6
};

/* Lazy materialisation: before an op the state is valid on the first
 * 2^n_active_in amplitudes (every qubit >= n_active_in is known |0>, its
 * amplitudes are not stored); the op leaves it valid on 2^n_active_out.  Ops
 * never read beyond 2^n_active_in and write all of 2^n_active_out.  Qubits in
 * [n_active_in, n_active_out) must be targets of the op (BLOCK: listed in ctrl[]).
 * A fully materialised program has n_active_in == n_active_out == n_local.       */
/* op.flags, on the LAST op of a program: shots will be drawn from the result.  When that
 * op only materialises new qubits (every block qubit new, one MUX1Q each), the engine
 * builds the sampler's sum tree on its 2^M-times smaller input and samples the new
 * qubits conditionally, instead of re-reading the whole result.                      */
#define QCM_FLAG_SAMPLE_CHECKPOINT 1
/* op.flags, on the LAST op of a program: the engine may store the result of that op in an
 * engine-internal ("rotated") address order -- for a wide expansion pass, with the new qubits as
 * the low address bits, which turns its 2^M write streams into one sequential stream.  Every
 * entry point that reads the state (qcm_postselect*, qcm_sample*, qcm_get_amplitudes) undoes the
 * rotation: callers keep seeing logical indices.  The next program must start with INIT_PRODUCT
 * (or qcm_set_amplitudes); qcm_state_ptr contents are not in logical order until then.
 * The result may also be left UNWRITTEN (by default when it has more than 2^30 amplitudes;
 * QCM_VIRTUAL_LAST in DESIGN.md): the sampler on the QCM_FLAG_SAMPLE_CHECKPOINT tree and the
 * prefix post-selection compute the amplitudes they read from the pass's input, and every other
 * reader (general post-selection, qcm_get_amplitudes, a rebuilt sum tree, qcm_state_ptr) first
 * writes the result out, enqueued on the handle's stream.                                     */
#define QCM_FLAG_ROTATED_OUTPUT_OK 2

typedef struct qcm_op {
    int32_t kind;
    int32_t target;
    int32_t n_ctrl;
    int32_t n_active_in;
    int32_t n_active_out;
    int32_t flags;                 /* QCM_FLAG_* */
    int32_t ctrl[QCM_MAX_CTRL];
    int64_t table_off;             /* offset, in doubles, into `tables` */
} qcm_op;

typedef struct qcm_timing {
    double program_ms;             /* device time of the last qcm_run_program  */
    double sample_ms;              /* device time of the last qcm_sample       */
    double postselect_ms;          /* device time of the last qcm_postselect   */
    uint64_t kernel_launches;      /* kernels launched by this handle so far   */
    uint64_t bytes_read;           /* algorithmic bytes of the last program    */
    uint64_t bytes_written;
} qcm_timing;

#if defined(__GNUC__)
#pragma GCC visibility push(default)
#endif

/* -- library ------------------------------------------------------------------ */
int qcm_abi_version(void);
int qcm_device_count(int *n_out);
const char *qcm_last_error(qcm_handle h);          /* h may be NULL: last global error */

/* -- state -------------------------------------------------------------------- */
/* n_local: qubits stored by this handle.  precision: QCM_C64 | QCM_C128.
 * ext_state: device buffer of 2^n_local complex numbers, or NULL (library allocates).
 * ext_stream: a cudaStream_t, or NULL for the legacy default stream.              */
int qcm_create(qcm_handle *out, int device, int n_local, int precision,
               void *ext_state, void *ext_stream);
int qcm_destroy(qcm_handle h);
/* the global index of local amplitude i is (rank << n_local) | i                  */
int qcm_set_shard(qcm_handle h, int n_global_qubits, uint64_t rank);
int qcm_get_amplitudes(qcm_handle h, uint64_t first, uint64_t count, void *host_out);
int qcm_set_amplitudes(qcm_handle h, uint64_t first, uint64_t count, const void *host_in,
                       int n_active);
int qcm_synchronize(qcm_handle h);

/* -- the hot path ---------------------------------------------------------------- */
/* Executes the fused program (replaces Aer's per-gate statevector sweeps).        */
int qcm_run_program(qcm_handle h, const qcm_op *ops, int n_ops,
                    const double *tables, size_t n_tables);

/* Post-selection (QCMRF.py:263-284 / eval.py:115-123 on exact probabilities):
 * kept = sum |amp_i|^2 over local i with (global(i) & mask) == value;
 * probs_out (optional, 2^n_out_bits doubles) receives, for every kept i, |amp_i|^2
 * accumulated at index (i & (2^n_out_bits - 1)); neither is normalised.
 * For QCMRF: mask = all bits >= n, value = 0, n_out_bits = n  =>  probs/kept is the
 * post-selected pmf with x_0 as MSB and kept is the success probability delta.     */
int qcm_postselect(qcm_handle h, uint64_t mask, uint64_t value, int n_out_bits,
                   double *probs_out, double *kept_out);

/* Shot sampling (replaces Aer's measurement sampling + Result.get_counts keys).
 * Draws `shots` basis states from |amp|^2 with Philox4x32-10 keyed by
 * (seed, stream_id, shot) and returns classical-register integers: bit c of a key is
 * the sampled value of qubit clbit_qubit[c] (negative entry: clbit reads 0, e.g.
 * QCMRF's never-written clbit n).  clbit_qubit == NULL returns raw state indices.  */
int qcm_sample(qcm_handle h, uint64_t shots, uint64_t seed, uint64_t stream_id,
               const int32_t *clbit_qubit, int n_clbits, uint64_t *keys_out);

/* Shot sampling for the measure-and-release width (DESIGN.md 2a): `released` qubits are not
 * stored -- one sweep materialised each from |0> and nothing used it again (a QCMRF clique ancilla,
 * measured right after its block, QCMRF.py:231-239).  The stored qubits' basis state is sampled as
 * in qcm_sample; released qubit k then reads 1 with probability p1[p1_off[k] + idx], idx = the
 * sampled bits at ctrl[k*max_ctrl .. + n_ctrl[k]) (physical positions), drawn on the device from a
 * Philox stream keyed by (seed, stream_id, shot, k).  vclbit[k]: clbit of released qubit k (or -1);
 * clbit_pos[c]: physical position feeding clbit c (or -1).  At most 64 released qubits.        */
int qcm_sample_released(qcm_handle h, uint64_t shots, uint64_t seed, uint64_t stream_id,
                        int n_released, const int32_t *n_ctrl, const int32_t *ctrl, int max_ctrl,
                        const double *p1, const int64_t *p1_off, int64_t n_p1,
                        const int32_t *vclbit, const int32_t *clbit_pos, int n_clbits,
                        uint64_t *keys_out);

/* Sharded sampling, three steps around one all-gather the caller performs:
 *  1. qcm_sample_prepare : builds the local sum tree, returns this rank's mass
 *  2. caller all-gathers the masses of all ranks
 *  3. qcm_sample_sharded : every rank draws the same Philox stream and resolves the
 *     shots that land in its shard; mine_out[s] = 1 where keys_out[s] is valid.    */
int qcm_sample_prepare(qcm_handle h, double *local_mass_out);
int qcm_sample_sharded(qcm_handle h, uint64_t shots, uint64_t seed, uint64_t stream_id,
                       const double *rank_masses, int n_ranks,
                       const int32_t *clbit_qubit, int n_clbits,
                       uint64_t *keys_out, uint8_t *mine_out);

/* Device-resident variants for callers that continue on the GPU (the sharded executor all-gathers
 * pmf blocks and all-reduces keys with NCCL): the outputs are DEVICE pointers, written in stream
 * order on the handle's stream; nothing is copied to the host and nothing synchronises.
 * dev_probs_out: 2^n_out_bits doubles (may be NULL), dev_kept_out: 1 double;
 * dev_keys_out: `shots` uint64, dev_mine_out: `shots` bytes.                                    */
int qcm_postselect_device(qcm_handle h, uint64_t mask, uint64_t value, int n_out_bits,
                          void *dev_probs_out, void *dev_kept_out);
int qcm_sample_sharded_device(qcm_handle h, uint64_t shots, uint64_t seed, uint64_t stream_id,
                              const double *rank_masses, int n_ranks,
                              const int32_t *clbit_qubit, int n_clbits,
                              void *dev_keys_out, void *dev_mine_out);

/* Total |amp|^2 of the local state (per point of a batched handle), summed from the sampler's sum tree on the device
 * into dev_total_out (DEVICE pointer, `batch` doubles), in stream order -- for callers in deferred mode, where
 * qcm_sample_prepare cannot report the mass to the host.                                                   */
int qcm_tree_total_device(qcm_handle h, void *dev_total_out);

/* As qcm_sample_sharded_device, with the rank masses still in DEVICE memory (e.g. straight out of an NCCL
 * all-gather): the mass of rank r is the double at dev_rank_masses[r * mass_stride].  Nothing has to come back
 * to the host between the all-gather and the sampler.                                                       */
int qcm_sample_sharded_devmass(qcm_handle h, uint64_t shots, uint64_t seed, uint64_t stream_id,
                               const void *dev_rank_masses, int64_t mass_stride, int n_ranks,
                               const int32_t *clbit_qubit, int n_clbits,
                               void *dev_keys_out, void *dev_mine_out);

/* Fused qubit-swap + blocked gate pass over NVLink peer memory (sharded states, one box).
 * Replaces "all-to-all that swaps the s global qubits with the s highest local qubits, then the
 * sweeps that target them": ops = a MUX1Q or a BLOCK header + members whose targets are exactly those
 * s highest local qubits (positions n_local-s .. n_local-1 AFTER the swap).  src_slabs[r] (r < 2^s) is a
 * device pointer, valid in this process (CUDA IPC / peer mapped), to the slab with index c_me of the
 * rank with coordinate r, i.e. peer_state + c_me * 2^(n_local-s) amplitudes; dst_state is a local
 * buffer of 2^n_local amplitudes that becomes the handle's state.  The caller must set the shard to the
 * rank bits that hold AFTER the swap (unchanged: the rank keeps its number) and must bracket the
 * call with cross-rank barriers (see qcm_kernels.cuh, k_block_gather).  No CPU fallback.          */
/* cudaDeviceEnablePeerAccess(device -> peer), idempotent; needed before qcm_run_gather_block reads
 * buffers that live on `peer`.                                                                    */
int qcm_enable_peer_access(int device, int peer);

/* CUDA IPC for the peer mappings qcm_run_gather_block reads through (one process per GPU):
 * qcm_ipc_export: handle (64 bytes) of the cudaMalloc allocation that contains dev_ptr + dev_ptr's
 * offset inside it -- works on pointers handed out by a sub-allocator (torch's caching allocator).
 * qcm_ipc_open: maps an exported allocation into THIS process with `device` (the GPU that will read
 * it) current, cudaIpcMemLazyEnablePeerAccess; *base_out is the allocation's base (add the offset).
 * One open per (process, allocation): the caller caches by handle bytes.  qcm_ipc_close unmaps.   */
#define QCM_IPC_HANDLE_BYTES 64
int qcm_ipc_export(int device, const void *dev_ptr, unsigned char *handle_out, uint64_t *offset_out);
int qcm_ipc_open(int device, const unsigned char *handle, void **base_out);
int qcm_ipc_close(int device, void *base);
int qcm_run_gather_block(qcm_handle h, const qcm_op *ops, int n_ops, const double *tables, size_t n_tables,
                         const void *const *src_slabs, int s, void *dst_state);

/* The same fused pass IN PLACE (no second state buffer: serves shards that fill the GPU).  The output overwrites this
 * rank's own slabs; per-(tile, peer) flags in peer-mapped memory order each overwrite behind the peer's read of the
 * same memory (see k_block_gather_inplace).  flag_ptrs[r] (r < 2^s): device pointer, valid in this process, to the flag
 * array (uint32, qcm_gather_flag_words entries, zero-initialised once) of the rank with coordinate r -- the entry of this
 * rank's own coordinate is its local array; epoch: > 0 and larger on every call of the same arrays.  Every rank of the
 * group must make the call (the kernels signal each other); bracket it with cross-rank barriers as for
 * qcm_run_gather_block.  A peer that never signals is reported as QCM_ERR_CUDA after QCM_GATHER_SPIN_S seconds
 * (default 5) instead of hanging the GPU.                                                                  */
int qcm_gather_flag_words(int n_local, int s, int precision, uint64_t *words_out);
int qcm_run_gather_block_inplace(qcm_handle h, const qcm_op *ops, int n_ops, const double *tables, size_t n_tables,
                                 const void *const *src_slabs, int s, void *const *flag_ptrs, uint64_t flag_words,
                                 uint32_t epoch);

/* Batched small circuits (all fixture-sized models in one launch: one thread block
 * per circuit, state resident in shared memory, program + post-selection + sampling
 * fused).  Circuit c has n_qubits[c] <= qcm_small_max_qubits(precision) qubits, ops
 * ops[op_begin[c] .. op_begin[c+1]) (INIT_PRODUCT / MUX1Q / DIAG, fully materialised),
 * clbit map clbit_qubit[64*c ..], post-selection as in qcm_postselect with
 * ps_mask[c], ps_value[c], ps_bits[c]; probs_out is the concatenation of the
 * 2^ps_bits[c] vectors, keys_out is [n_circuits][shots].                           */
int qcm_small_max_qubits(int precision);
int qcm_run_batch_small(int device, int precision, int n_circuits,
                        const int32_t *n_qubits, const int64_t *op_begin,
                        const qcm_op *ops, const double *tables, size_t n_tables,
                        const int32_t *clbit_qubit, const int32_t *n_clbits,
                        const uint64_t *ps_mask, const uint64_t *ps_value,
                        const int32_t *ps_bits,
                        const uint64_t *stream_ids, /* Philox stream per circuit; NULL: index */
                        uint64_t shots, uint64_t seed,
                        uint64_t *keys_out, double *probs_out, double *kept_out,
                        double *device_ms_out);
/* qcm_run_batch_small, then every key's measured clbits flipped by readout errors before the keys are copied out.
 * readout: [n_circuits][64][2] doubles, per clbit P(read 1 | outcome 0), P(read 0 | outcome 1) (zero for an
 * unmeasured clbit); NULL: no flips.  Shot s of circuit c draws clbit b's flip from Philox4x32-10 keyed
 * (seed ^ readout key, stream of c) at counter s * 16 + b / 4 (word b % 4): never a counter of the outcome draw.   */
int qcm_run_batch_small_readout(int device, int precision, int n_circuits,
                                const int32_t *n_qubits, const int64_t *op_begin,
                                const qcm_op *ops, const double *tables, size_t n_tables,
                                const int32_t *clbit_qubit, const int32_t *n_clbits, const double *readout,
                                const uint64_t *ps_mask, const uint64_t *ps_value, const int32_t *ps_bits,
                                const uint64_t *stream_ids, uint64_t shots, uint64_t seed,
                                uint64_t *keys_out, double *probs_out, double *kept_out, double *device_ms_out);

/* -- noisy shots: Pauli-error trajectories of small circuits --------------------------------------------- */
/* One unfused gate: `m` (2x2, row-major re/im, fp64) on `target` wherever (index & ctrl_mask) == ctrl_value; then,
 * when channel >= 0, the Pauli channel channels[channel].                                                        */
typedef struct {
    double m[8];
    int32_t target;
    uint32_t ctrl_mask;
    uint32_t ctrl_value;
    int32_t channel;            /* -1: no error after this gate */
} qcm_gate;

/* A Pauli channel on 1 or 2 qubits: Pauli k (code (k >> 2j) & 3 on qubit[j]: 0 I, 1 X, 2 Y, 3 Z) has probability
 * cum[k] - cum[k-1]; cum[n_paulis - 1] == 1.  qubit[1] == -1 for a 1-qubit channel.                              */
typedef struct {
    double cum[16];
    int32_t n_paulis;           /* 4 or 16 */
    int32_t qubit[2];
    int32_t pad;
} qcm_channel;

/* Noisy shots of many circuits in one call, no fusion: every shot of circuit c (n_qubits[c] <=
 * qcm_small_max_qubits, gates gates[gate_begin[c] .. gate_begin[c+1])) is an independent trajectory from |0..0>:
 * after gate g the channel draws one Pauli from Philox4x32-10 keyed (seed ^ noise key, stream) at counter
 * shot * G_c + g (G_c gates in circuit c); the outcome is drawn from |psi|^2 as qcm_run_batch_small draws it; the
 * key is built from clbit_qubit[64*c ..] and n_clbits[c] as there and flipped by `readout` as in
 * qcm_run_batch_small_readout (NULL: no readout error).  keys_out is [n_circuits][shots].  Channel indices are
 * global (into `channels`).  QCM_ERR_UNSUPPORTED above qcm_small_max_qubits qubits; QCM_ERR_INVALID on a
 * malformed gate, channel or a trajectory whose norm is not finite and positive.  No CPU fallback.              */
int qcm_run_noisy_small(int device, int precision, int n_circuits, const int32_t *n_qubits,
                        const int64_t *gate_begin, const qcm_gate *gates,
                        const qcm_channel *channels, int n_channels,
                        const int32_t *clbit_qubit, const int32_t *n_clbits, const double *readout,
                        const uint64_t *stream_ids, uint64_t shots, uint64_t seed,
                        uint64_t *keys_out, double *device_ms_out);

/* A 1-qubit channel in canonical Kraus form: rho -> sum_i K_i rho K_i^dagger on `qubit`, sum_i K_i^dagger K_i = I
 * within 1e-10.                                                                                                 */
typedef struct {
    double k[4][8];             /* K_i, 2x2 row-major re/im, fp64; entries past n_ops are ignored */
    int32_t n_ops;              /* 1..4 */
    int32_t qubit;
} qcm_kraus;

/* The error after one gate: stages applied in order, each a Pauli channel or a Kraus channel. */
typedef struct {
    int32_t n_stages;           /* 1..4 */
    int32_t kind[4];            /* 0: Pauli channel (index into channels), 1: Kraus (index into krauses) */
    int32_t index[4];
    int32_t pad;
} qcm_gate_error;

/* As qcm_run_noisy_small, but qcm_gate.channel indexes `errors` (-1: no error), and a gate's error applies its
 * stages in order.  Every stage draws one uniform from Philox4x32-10 keyed (seed ^ Kraus key, stream) at counter
 * (shot * G_c + g) * 4 + j for stage j of gate g.  A Pauli stage picks its Pauli from the cumulative table; a
 * Kraus stage picks K_i with probability tr(K_i^dagger K_i rho_q) / sum, rho_q the trajectory's reduced state of
 * the stage's qubit (never an operator of probability 0), and applies K_i / sqrt(p_i).  A Kraus qubit must be one
 * of its gate's qubits (target or control).  QCM_ERR_INVALID on a malformed stage, channel or Kraus record (all
 * checked before any device query) or when a trajectory's norm is not finite and positive.  No CPU fallback. */
int qcm_run_noisy_small_kraus(int device, int precision, int n_circuits, const int32_t *n_qubits,
                              const int64_t *gate_begin, const qcm_gate *gates,
                              const qcm_gate_error *errors, int n_errors,
                              const qcm_channel *channels, int n_channels,
                              const qcm_kraus *krauses, int n_kraus,
                              const int32_t *clbit_qubit, const int32_t *n_clbits, const double *readout,
                              const uint64_t *stream_ids, uint64_t shots, uint64_t seed,
                              uint64_t *keys_out, double *device_ms_out);

/* -- batched sweeps ----------------------------------------------------------------- */
/* A theta / beta sweep over ONE graph (QCMRF's `beta`, /root/reference/QCMRF.py:21,154; BASELINE config 3) is B circuits
 * with the same program structure and different coefficient tables.  A batched handle holds the B states of
 * 2^n_local amplitudes in one allocation and runs every kernel of a program ONCE, with the sweep point as the
 * second grid dimension -- O(10) launches for the whole sweep instead of O(10) per point:
 *   qcm_run_program    : `tables` holds B consecutive table sets of n_tables doubles each (point-major); the ops
 *                        (and every table_off) are shared.  Engine-internal output rotation and the sampling
 *                        checkpoint are not used on batched handles.
 *   qcm_postselect     : kept_out receives B doubles, probs_out (optional) B consecutive blocks of 2^n_out_bits.
 *   qcm_postselect_resident : as qcm_postselect, but the B probability blocks STAY in device memory owned by the
 *                        handle (valid until its next post-selection); qcm_fetch_probs copies (part of) one
 *                        point's block to the host on demand.  Also serves plain handles (B = 1).
 *   qcm_sample_batched / qcm_sample_released_batched : as qcm_sample / qcm_sample_released with one Philox stream
 *                        id per point (stream_ids[B]); keys_out is [B][shots]; released-qubit tables p1 are B
 *                        consecutive sets of n_p1 doubles.
 *   qcm_batch_select   : the point that qcm_get_amplitudes / qcm_set_amplitudes address (default 0).
 * A plain handle is a batched handle with B = 1.                                                       */
int qcm_create_batched(qcm_handle *out, int device, int n_local, int precision, int batch,
                       void *ext_state, void *ext_stream);
/* Deferred mode: qcm_run_program, qcm_postselect*, qcm_sample* enqueue their kernels and copies on the handle's
 * stream and return without synchronising (no timings are collected); host output buffers must then be page-locked
 * (qcm_host_alloc) and are valid after qcm_synchronize.  A sweep becomes ONE synchronisation instead of one per call,
 * and its result copies overlap the kernels that follow.                                                        */
int qcm_set_deferred(qcm_handle h, int deferred);
/* A stream of circuits in deferred mode is a pipeline: qcm_mark records a point in the handle's stream behind
 * everything enqueued so far and returns its ticket; qcm_wait blocks the host until that point has been reached --
 * circuit i's page-locked results are then valid while circuit i+1's program (enqueued after the mark) is still
 * running.  Replaces, for a list of circuits, the blocking result() of the reference's job
 * (run_experiment.py:56: one run() for all circuits).                                                            */
int qcm_mark(qcm_handle h, uint64_t *ticket_out);
int qcm_wait(qcm_handle h, uint64_t ticket);
int qcm_host_alloc(void **host_out, size_t bytes);      /* page-locked host memory (cudaHostAlloc) */
int qcm_host_free(void *host_ptr);
int qcm_batch_size(qcm_handle h, int *batch_out);
int qcm_batch_select(qcm_handle h, int point);
int qcm_postselect_resident(qcm_handle h, uint64_t mask, uint64_t value, int n_out_bits, double *kept_out);
int qcm_fetch_probs(qcm_handle h, int point, uint64_t first, uint64_t count, double *host_out);
int qcm_sample_batched(qcm_handle h, uint64_t shots, uint64_t seed, const uint64_t *stream_ids,
                       const int32_t *clbit_qubit, int n_clbits, uint64_t *keys_out);
int qcm_sample_released_batched(qcm_handle h, uint64_t shots, uint64_t seed, const uint64_t *stream_ids,
                                int n_released, const int32_t *n_ctrl, const int32_t *ctrl, int max_ctrl,
                                const double *p1, const int64_t *p1_off, int64_t n_p1,
                                const int32_t *vclbit, const int32_t *clbit_pos, int n_clbits,
                                uint64_t *keys_out);

/* -- exact MRF inference by enumeration ("px" on the GPU) -------------------------------- */
/* What /root/reference/eval.py:84-93 computes through the proprietary kiopto_native module --
 * lnZ = px.infer(b, task='partition'), p[xid] = exp(px.logpot(b, xid) - lnZ) -- for binary variables:
 * energy(xid) = sum_C weights[off_C + y_C], y_C = sum_j x_{C[j]} 2^(|C|-1-j) (itertools.product order,
 * weights clique-major), x_v = bit n-1-v of xid (x_0 is the most significant bit, eval.py:100-101).
 * clique_size[n_cliques], clique_vars = the cliques' vertices concatenated.  log_z_out: ln Z.
 * pmf_out / energies_out (optional, 2^n doubles each).  Stateless; no CPU fallback.                 */
int qcm_mrf_exact(int device, int n, int n_cliques, const int32_t *clique_size, const int32_t *clique_vars,
                  const double *weights, double *log_z_out, double *pmf_out, double *energies_out,
                  double *device_ms_out);
const char *qcm_mrf_last_error(void);

/* -- multi-GPU plumbing ------------------------------------------------------------ */
/* Packs/unpacks nothing: the qubit-swap all-to-all exchanges contiguous slabs of the
 * top `g` local qubits, which the caller moves with NCCL (torch.distributed).  These
 * two report the device pointer and byte size so the caller can wrap the state.     */
int qcm_state_ptr(qcm_handle h, void **dev_ptr_out, uint64_t *bytes_out);
/* Read-only view of the sampler's sum tree (for tests and diagnostics): the device pointer and
 * entry count (doubles) of level `level`, 0 = the chunk sums over 2^10 amplitudes ... top, and
 * -1 = the finer level under level 0 when the tree has one.  *n_levels_out (optional) receives
 * the number of levels above the amplitudes.  The finer level of an unwritten last pass is not
 * stored (the sampler computes the entries it reads): -1 then writes it, with the sampler's
 * arithmetic, into a handle buffer and synchronises the handle's stream.  Nothing else is built or
 * written: QCM_ERR_INVALID when the handle holds no valid tree or the level does not exist.
 * Batched handles: point 0.                                                                   */
int qcm_tree_level(qcm_handle h, int level, const double **dev_ptr_out, uint64_t *n_out, int *n_levels_out);
int qcm_set_active(qcm_handle h, int n_active);
int qcm_get_active(qcm_handle h, int *n_active_out);

int qcm_get_timing(qcm_handle h, qcm_timing *out);
/* Per-launch record of the last qcm_run_program (one entry per executed op; a BLOCK and
 * its members are one entry): device milliseconds (CUDA events on the handle's stream)
 * and algorithmic bytes read / written.  Up to `cap` entries are copied; *n_out receives
 * the number available.  bench.py derives roofline.achieved from these.                */
int qcm_get_op_profile(qcm_handle h, int cap, int32_t *kind_out, float *ms_out,
                       uint64_t *bytes_read_out, uint64_t *bytes_written_out, int *n_out);
/* Name of the kernel that executed op `index` of the last program (the indices of
 * qcm_get_op_profile), e.g. "k_expand_low<float,2,MH=2,TB=8>"; "" when out of range.  The
 * string lives in the handle until the next program.                                     */
const char *qcm_op_kernel_name(qcm_handle h, int index);

#if defined(__GNUC__)
#pragma GCC visibility pop
#endif

#ifdef __cplusplus
}
#endif
#endif /* QCMRF_B200_H */
