/* qsim_b200 -- C ABI of the B200-native gate-application engine.
 *
 * Drop-in boundary for the gate-application path of the reference's
 * simulators/dv_simulator (abbreviated DV/ below).  The reference is pure
 * Python/NumPy and has no FFI; each entry point replaces the NumPy routine
 * cited beside it, and the Python shim in quantum_computations_b200/ binds the
 * library with ctypes (INTEGRATION.md shows the stub).
 *
 * Conventions
 *  - All functions return 0 on success, a negative QSIM_ERR_* otherwise, never
 *    throw; qsim_last_error() returns a thread-local message.
 *  - State buffers are BORROWED device pointers to interleaved (re, im) double
 *    pairs (numpy/torch complex128), 2^n amplitudes, owned by the caller
 *    (PyTorch).  Work is enqueued on the caller's cudaStream_t (passed as
 *    void*); functions that return a scalar to the host synchronise that stream.
 *  - Qubit numbers are the REFERENCE's: qubit 0 is the most significant bit of
 *    the linear index (DV/numpy_quantum.py:243-247).  For a k-qubit matrix the
 *    first tensor factor acts on targets[0] (DV/gates.py:116-126).
 *  - Matrices are host pointers, row-major, interleaved complex128.
 *  - A density matrix of N qubits is its row-major vec: a 2N-"qubit" buffer in
 *    which row qubit q is qubit q and column qubit q is qubit q+N.
 */
#ifndef QSIM_B200_H
#define QSIM_B200_H

#include <stdint.h>

#ifdef __cplusplus
extern "C" {
#endif

#define QSIM_OK               0
#define QSIM_ERR_ARG         -1   /* invalid argument                        */
#define QSIM_ERR_CUDA        -2   /* a CUDA call failed                      */
#define QSIM_ERR_UNSUPPORTED -3   /* valid request the library cannot serve  */
#define QSIM_ERR_NOMEM       -4

typedef struct qsim_circuit qsim_circuit_t;
typedef struct qsim_plan qsim_plan_t;

typedef struct {
  int32_t tile_bits;        /* T: log2 amplitudes per shared-memory tile (<= 13); 0 = default  */
  int32_t low_bits;         /* L: forced lowest index bits per tile (coalescing);  0 = default  */
  int32_t max_group;        /* 2x2 gates fused per shared-memory round trip (1..4); 0 = default */
  int32_t max_dense_ops;    /* cap on non-diagonal gates per pass;                 0 = default  */
  int32_t lookahead;        /* gates scanned ahead when choosing a tile;           0 = default  */
  int32_t merge_1q;         /* 0 = default (on), 1 = on, 2 = off                                */
  int32_t defer_tail;       /* 1 = do not apply the trailing diagonal / antidiagonal single-qubit
                               products; hand them back through qsim_plan_residual so that the
                               caller can merge them into its next plan (needs merge_1q on)      */
  int32_t max_layers;       /* gate layers per shared-memory round trip (1..8): a qubit whose
                               amplitudes are in registers can take its next gates there;  0 = default */
  int32_t cta_log2;         /* log2 threads per CTA of the tile pass: 7 or 8; 0 = chosen per pass (small CTAs,
                               three to an SM, for passes with many gates; large ones for passes that
                               are bound by HBM)                                                        */
  int32_t reserved0;        /* must be 0 */
  uint64_t apply_tail_mask; /* with defer_tail: qubits (bit q = qubit q) whose trailing products are
                               applied all the same                                              */
} qsim_plan_options_t;

typedef struct {
  int64_t n_input_ops;      /* gates handed to the circuit                                      */
  int64_t n_merged_ops;     /* after single-qubit merging                                       */
  int64_t n_passes;         /* tile passes (one HBM read+write of the state each)               */
  int64_t n_steps;          /* shared-memory round trips over all passes                        */
  int64_t n_dense;          /* matrix applications inside the steps                             */
  int64_t n_sign;           /* CZ/Z sign pairs                                                  */
  int64_t n_generic;        /* gates on 5..10 qubits: one in-place dense-block launch each (DMMA) */
  int64_t n_warp_syncs;     /* steps followed by a warp-level instead of a block-level barrier  */
  int64_t n_layers;         /* gate layers over all steps (n_layers >= n_steps)                 */
} qsim_plan_stats_t;

const char* qsim_last_error(void);
int qsim_version(void);
/* 1 when the library was built with the CUDA kernels, 0 for the host emulator
 * that the CPU tests build from the same planner sources. */
int qsim_has_cuda(void);

/* ---- circuits and fused plans: replace the per-gate loop of
 *      Simulator.run (DV/simulator.py:40-52) -------------------------------- */
int qsim_circuit_create(int n_qubits, qsim_circuit_t** out);
/* Gate.apply ket branch, any k (DV/gates.py:48-50).  Structure (diagonal, CZ,
 * Z) is detected from the matrix values. */
int qsim_circuit_add_matrix(qsim_circuit_t* c, int k, const int* targets, const double* matrix);
/* `count` gates in one call: ks[g] qubits each, targets and row-major complex matrices
 * concatenated in gate order (same checks as qsim_circuit_add_matrix, gate by gate). */
int qsim_circuit_add_many(qsim_circuit_t* c, int64_t count, const int32_t* ks, const int32_t* targets,
                          const double* matrices);
int qsim_circuit_num_ops(const qsim_circuit_t* c);
void qsim_circuit_destroy(qsim_circuit_t* c);

int qsim_plan_compile(const qsim_circuit_t* c, const qsim_plan_options_t* opt, qsim_plan_t** out);
int qsim_plan_stats(const qsim_plan_t* p, qsim_plan_stats_t* out);
/* scratch: unused (kept for ABI stability; every kernel works in place), may be NULL */
int qsim_plan_execute(const qsim_plan_t* p, void* state, int n_qubits, void* scratch, void* stream);
/* With options.defer_tail: the single-qubit gate left over on every qubit, n_qubits x (2x2
 * row-major complex) = 8 doubles per qubit, qubit 0 first; identity where nothing is left.
 * The state after qsim_plan_execute followed by these gates equals the circuit's. */
int qsim_plan_residual(const qsim_plan_t* p, double* out);
void qsim_plan_destroy(qsim_plan_t* p);

/* ---- single operations (each is a one-gate plan) ------------------------------- */
/* expand_gate + `gate @ state` (DV/numpy_quantum.py:243-247, DV/gates.py:50) */
int qsim_apply_matrix(void* state, int n_qubits, const int* targets, int k, const double* matrix,
                      void* scratch, void* stream);
/* same path for diagonal matrices (Z, RZ, P, Pdg, T, Tdg, CZ: DV/gates.py:79-130);
 * diag holds the 2^k diagonal entries */
int qsim_apply_diagonal(void* state, int n_qubits, const int* targets, int k, const double* diag,
                        void* stream);
/* same path for permutation matrices (X, CX, SWAP: DV/gates.py:71-73,116-134);
 * column c of the matrix has its 1 in row perm[c] */
int qsim_apply_permutation(void* state, int n_qubits, const int* targets, int k, const int* perm,
                           void* stream);
/* `gate @ rho @ dagger(gate)` (DV/gates.py:51-52) and Kraus sums
 * (PAPER/tomography.py:21-24) as one 4^k x 4^k matrix on the vec of rho:
 * targets are the k row qubits, the column qubits targets[i]+n are implied. */
int qsim_apply_superop(void* vec_rho, int n_qubits, const int* targets, int k, const double* superop,
                       void* scratch, void* stream);

/* ---- state construction / register resizing -------------------------------------- */
/* tensor(*(s.get() for s in states)) (DV/simulator.py:26); amps = n x 2 complex */
int qsim_init_product(void* state, int n_qubits, const double* amps, void* stream);
/* M.apply (DV/gates.py:165-186): out_norm2[s] = || (I..bra_s..I) psi ||^2 */
int qsim_measure_probs(const void* state, int n_qubits, int qubit, const double* bra0,
                       const double* bra1, double* out_norm2, void* stream);
/* out (2^(n-1) amps) = (I..bra..I) in / norm   (DV/gates.py:185) */
int qsim_collapse(const void* in, void* out, int n_qubits, int qubit, const double* bra, double norm,
                  void* stream);
/* Insert.apply (DV/gates.py:145-153): out has n+1 qubits, the new one at `position` */
int qsim_insert(const void* in, void* out, int n_qubits, int position, const double* amp,
                void* stream);

/* ---- reductions (DV/numpy_quantum.py:131-166); results are host doubles ------------ */
int qsim_reduce_norm2(const void* state, uint64_t n_amps, double* out, void* stream);
int qsim_reduce_inner(const void* a, const void* b, uint64_t n_amps, double* out_re_im, void* stream);
/* <ket| rho |ket> with rho a row-major 2^n x 2^n matrix */
int qsim_reduce_expect(const void* ket, const void* rho, int n_qubits, double* out_re_im, void* stream);
/* tr(rho rho) = sum_ij rho_ij rho_ji  (no Hermiticity assumed) */
int qsim_reduce_purity(const void* rho, int n_qubits, double* out_re_im, void* stream);
int qsim_reduce_trace(const void* rho, int n_qubits, double* out_re_im, void* stream);

/* ---- Pauli-sum expectation values (npq.expect / expecth on Pauli strings) -------------
 * A Pauli string on n qubits is a pair of masks (x, z); bit q of each stands for reference
 * qubit q (as in qsim_plan_options_t::apply_tail_mask).  I = (0,0), X = (1,0), Z = (0,1),
 * Y = (1,1); the operator is P = i^popc(x & z) X^x Z^z (Z applied first), so every string is
 * Hermitian.  Masks with bits at or above n_qubits, and n_qubits outside [1, 63], are
 * QSIM_ERR_ARG; n_terms == 0 does nothing.  Results come back in the caller's term order; a
 * fixed grid and a fixed summation tree make repeated calls bit-identical. */
/* <psi|P_t|psi> for n_terms Pauli strings on a ket (real; P_t Hermitian, see convention above).
 * x_masks/z_masks/out are HOST arrays of n_terms; synchronises the stream.  Terms are grouped
 * by X mask; one read of the state serves up to 32 terms whose X masks span at most 4 dimensions. */
int qsim_expect_pauli(const void* state, int n_qubits, int64_t n_terms, const uint64_t* x_masks,
                      const uint64_t* z_masks, double* out, void* stream);
/* tr(rho P_t) on the row-major vec of an N-qubit density matrix (N <= 31); out = n_terms x (re, im).
 * Reads the 2^N entries rho[c, c^x] per term; no Hermiticity assumed. */
int qsim_expect_pauli_dm(const void* vec_rho, int n_qubits, int64_t n_terms, const uint64_t* x_masks,
                         const uint64_t* z_masks, double* out_re_im, void* stream);

/* ---- Pauli-string rotations (Trotterised evolution under a Pauli sum) ------------------
 * state <- R_{n_rot-1} ... R_1 R_0 state, in place, with R_t = exp(-i angles[t]/2 P_t) and P_t the
 * string (x_masks[t], z_masks[t]) in the convention of qsim_expect_pauli.  Masks and angles are
 * HOST arrays of n_rot.  The rotations are applied in caller order (never reordered); runs of
 * consecutive rotations whose X masks span at most 4 dimensions share one read and one write of
 * the state (up to 32 rotations per pass).  Angle-0 rotations are skipped; x = z = 0 is the global
 * phase exp(-i angle/2).  Null pointers, masks at or above n_qubits, n_qubits outside [1, 63] and a
 * non-finite angle are QSIM_ERR_ARG; n_rot == 0 does nothing.  Allocates nothing and does not
 * synchronise. */
int qsim_apply_pauli_rotations(void* state, int n_qubits, int64_t n_rot, const uint64_t* x_masks,
                               const uint64_t* z_masks, const double* angles, void* stream);
/* rho <- U rho U^dagger, U = R_{n_rot-1} ... R_0, on the row-major vec of an N-qubit density matrix
 * (N <= 31): each rotation acts on the row qubits with its angle and, conjugated, on the column
 * qubits in the same pass. */
int qsim_apply_pauli_rotations_dm(void* vec_rho, int n_qubits, int64_t n_rot, const uint64_t* x_masks,
                                  const uint64_t* z_masks, const double* angles, void* stream);

/* ---- H|psi> for a Pauli sum, and adjoint gradients over Pauli rotations -----------------
 * out <- sum_t c_t P_t in, out of place, with c_t = (coeffs_re_im[2t], coeffs_re_im[2t+1]) and P_t
 * the string (x_masks[t], z_masks[t]) in the convention of qsim_expect_pauli; masks and coefficients
 * are HOST arrays.  Terms are grouped by X mask as for qsim_expect_pauli: one read of `in` and one
 * read-modify-write of `out` per pass of up to 32 terms.  n_terms == 0 writes zeros.  in == out,
 * null pointers, masks at or above n_qubits, n_qubits outside [1, 63] and a non-finite coefficient
 * are QSIM_ERR_ARG.  The vec of an N-qubit density matrix with 2N qubits and masks on qubits
 * 0..N-1 (the row qubits) gives vec(H rho).  Allocates nothing and does not synchronise. */
int qsim_apply_pauli_sum(const void* in, void* out, int n_qubits, int64_t n_terms, const uint64_t* x_masks,
                         const uint64_t* z_masks, const double* coeffs_re_im, void* stream);
/* out <- out + sum_t c_t P_t in: the same passes, every one adding to out (no extra buffer and no
 * extra pass for a sum taken in parts); n_terms == 0 leaves out unchanged.  Same checks. */
int qsim_accumulate_pauli_sum(const void* in, void* out, int n_qubits, int64_t n_terms, const uint64_t* x_masks,
                              const uint64_t* z_masks, const double* coeffs_re_im, void* stream);
/* The backward sweep of the adjoint method over U = R_{n_rot-1} ... R_0, the rotation list of
 * qsim_apply_pauli_rotations.  On entry psi = U psi0 and lam is any state; on return psi holds psi0
 * (within rounding), lam holds U^dagger lam and out[t] = Im<lam_t|P_t|psi_t>, both states taken just
 * after R_t.  With lam = H psi, out[t] = d<H>/d theta_t.  The sweep runs the rotations in reverse
 * order with up to 32 per read and write of both states (X masks spanning at most 3 dimensions);
 * angle-0 rotations are kept.  out: HOST array of n_rot doubles; fixed summation trees, so two calls
 * on the same inputs give bit-identical results.  psi == lam is QSIM_ERR_ARG, the other checks are
 * those of qsim_apply_pauli_rotations; n_rot == 0 does nothing.  Synchronises the stream. */
int qsim_pauli_rotations_adjoint(void* psi, void* lam, int n_qubits, int64_t n_rot, const uint64_t* x_masks,
                                 const uint64_t* z_masks, const double* angles, double* out, void* stream);
/* The same on the row-major vecs of N-qubit density matrices (N <= 31): psi = U rho0 U^dagger,
 * out[t] = d Re<<lam|rho>>/d theta_t with <<A|B>> = tr(A^dagger B). */
int qsim_pauli_rotations_adjoint_dm(void* psi, void* lam, int n_qubits, int64_t n_rot, const uint64_t* x_masks,
                                    const uint64_t* z_masks, const double* angles, double* out, void* stream);

/* ---- Lanczos building blocks: fused H|psi> and dot, and the fused step --------------------
 * out <- prev_scale * prev + sum_t c_t P_t in (strings, coefficients and passes as in
 * qsim_apply_pauli_sum; the first pass reads prev where an accumulating pass reads out).  prev may
 * be out (out <- prev_scale * out + ...) or null (zeros).  The last pass also reduces Re <in|out>
 * with fixed summation trees; *out_dot receives it, so two calls on the same inputs give
 * bit-identical outputs and dots.  n_terms == 0 gives out = prev_scale * prev and its dot.  in ==
 * out, in == prev, a null in, out or out_dot, a non-finite prev_scale and the checks of
 * qsim_apply_pauli_sum are QSIM_ERR_ARG.  Synchronises the stream. */
int qsim_lanczos_apply(const void* in, const void* prev, void* out, int n_qubits, int64_t n_terms,
                       const uint64_t* x_masks, const uint64_t* z_masks, const double* coeffs_re_im, double prev_scale,
                       double* out_dot, void* stream);
/* One streaming pass over n_amps amplitudes: w <- w - a v and, when y is not null, y <- y + b v with
 * b = (b_re_im[0], b_re_im[1]) (a HOST array).  A null w updates y alone.  With out_norm2 (a HOST
 * double) the call reduces |w|^2 after the update (|y|^2 when w is null) with fixed summation trees
 * and synchronises; without it, it does not synchronise.  A null v, w and y both null, a null b_re_im
 * with y, aliased buffers, n_amps == 0 and non-finite a or b are QSIM_ERR_ARG. */
int qsim_lanczos_step(void* w, const void* v, void* y, uint64_t n_amps, double a, const double* b_re_im,
                      double* out_norm2, void* stream);

/* ---- measurement statistics: marginal probabilities and shot sampling -------------------
 * Qubits are the reference's (qubit q is index bit n-1-q).  A marginal over qubits[0..k) has
 * 2^k bins; bit k-1-j of the bin number is the value of qubits[j], so qubits[0] is the most
 * significant bit (the marginal over qubits 0..19 of a 30-qubit ket is bench.py's
 * `state_marginal`).  The probability of basis index i is |psi_i|^2 for a ket and Re rho[i, i]
 * for the vec of an N-qubit density matrix.  The qubits must be distinct, 0 <= k <= n_qubits,
 * 1 <= n_qubits <= 40 (N <= 31 for the _dm variants); anything else is QSIM_ERR_ARG.  Fixed grids
 * and fixed summation / scan trees (no floating-point atomics): repeated calls on the same state
 * give bit-identical marginals and identical outcomes. */
/* out: DEVICE array of 2^k doubles, the raw sums (not normalised).  Does not synchronise. */
int qsim_marginal_probs(const void* state, int n_qubits, int k, const int* qubits, double* out, void* stream);
int qsim_marginal_probs_dm(const void* vec_rho, int n_qubits, int k, const int* qubits, double* out,
                           void* stream);
/* Inverse-CDF sampling of full basis indices.  For the caller's uniform u in [0, 1) (DEVICE array
 * `uniforms`, `shots` doubles) the outcome is the smallest index i with cdf(i) > u * total, where
 * total is the mass the call computed (a ket need not be normalised) and cdf uses the library's
 * fixed summation order; an index with probability 0 is never drawn (a uniform that rounding
 * places past the last nonzero probability takes that index).  For a density matrix a negative
 * diagonal entry counts as 0.  out: DEVICE array of `shots` basis indices.  *total (host) gets the
 * mass sampled from; returning it synchronises the stream.  A total <= 0 (or not finite) is
 * QSIM_ERR_ARG; shots == 0 returns at once; shots must be below 2^31.  workspace: DEVICE buffer of
 * at least qsim_sample_workspace_bytes(n_qubits, shots) bytes (N for the _dm variant), owned by
 * the caller; a shorter one is QSIM_ERR_ARG. */
int qsim_sample_workspace_bytes(int n_qubits, int64_t shots, uint64_t* out_bytes);
int qsim_sample(const void* state, int n_qubits, int64_t shots, const double* uniforms, uint64_t* out,
                double* total, void* workspace, uint64_t workspace_bytes, void* stream);
int qsim_sample_dm(const void* vec_rho, int n_qubits, int64_t shots, const double* uniforms, uint64_t* out,
                   double* total, void* workspace, uint64_t workspace_bytes, void* stream);

/* ---- batched tiny-circuit executor (replaces the sample loop of
 *      PAPER/randomised_benchmarking.py:65-75) --------------------------------------
 * B independent registers of nq <= 2 qubits kept as density matrices (dim = 2^nq).
 * Sequence b applies opcodes[offsets[b] .. offsets[b+1]) (16-bit codes); opcode o multiplies
 * vec(rho) by superops[o] (dim^2 x dim^2) and the ideal ket by unitaries[o]
 * (dim x dim).  Outputs per sequence: fidelity <psi|rho|psi> and purity tr rho^2.
 * All pointers are DEVICE pointers except the scalar arguments. */
int qsim_rb_batch(int nq, int64_t n_seq, const uint16_t* opcodes, const int64_t* offsets,
                  int n_opcodes, const double* superops, const double* unitaries,
                  const double* rho0, const double* psi0, double* out_fidelity, double* out_purity,
                  double* out_rho, void* stream);

/* ---- Pauli-trajectory batch (mechanism of GKP/simulator.py:26-55 at the DV level) ---------
 * `shots` noisy realisations of ONE circuit of 1- and 2-qubit gates on a ket of n_qubits <= 12:
 * after gate g, on each of its qubits, an X and then a Z is applied where the shot's flip bits
 * say so (flips[shot][...], two bytes per gate qubit in gate order: X, Z).  One CTA per shot,
 * state in shared memory; the flips are folded into the gate's rows.  ops = n_ops x {k, bit0,
 * bit1, matrix offset (in complex numbers) into `matrices`} as int32, bits are INDEX bits
 * (reference qubit q is bit n-1-q), bit0 belongs to the first tensor factor.  psi0 /
 * observable: 2^n complex.  out_fidelity[shot] = |<observable|psi>|^2 (optional),
 * out_prob_sum[i] += sum over shots of |psi_i|^2 (optional, caller zeroes it), out_states:
 * shots x 2^n complex (optional, for tests).  All pointers are DEVICE pointers. */
int qsim_traj_batch(int n_qubits, int64_t shots, int n_ops, const int32_t* ops, const double* matrices,
                    const uint8_t* flips, int64_t flips_per_shot, const double* psi0, const double* observable,
                    double* out_fidelity, double* out_prob_sum, double* out_states, void* stream);

/* ---- global<->local qubit exchange helpers for sharded states ----------------------
 * A state of n qubits sharded over 2^g ranks keeps g qubits in the rank number.
 * Exchanging k rank qubits with k local qubits at once is an all-to-all among the 2^k
 * ranks that differ in those rank bits: rank R sends to partner R^d the 2^(n_local-k)
 * amplitudes whose k local bits spell the PARTNER's rank bits, and receives into the
 * same positions (k = 1 is the plain global<->local swap of half a shard).  These two
 * kernels gather such a block into a contiguous send buffer and scatter a received
 * block back; the transfer itself is the caller's (NCCL/gloo send/recv).
 * local_qubits[i] (reference-style numbering inside the shard) is fixed to
 * bit_values[i]; first/count select a chunk of the block; the buffer holds `count`
 * amplitudes.  nbits <= 8. */
int qsim_swap_pack(const void* shard, void* sendbuf, int n_local, int nbits, const int* local_qubits,
                   const int* bit_values, uint64_t first, uint64_t count, void* stream);
int qsim_swap_unpack(void* shard, const void* recvbuf, int n_local, int nbits, const int* local_qubits,
                     const int* bit_values, uint64_t first, uint64_t count, void* stream);

/* ---- exchanges over NVLink peer memory (one process per GPU) -------------------------
 * Every rank exports its shard once through CUDA IPC and maps the other ranks' shards
 * into its own address space; the exchange is then one kernel per rank that reads and
 * writes the partners' shards directly.  Handles are 64-byte cudaIpcMemHandle_t.
 * qsim_ipc_import maps a handle on `device`; qsim_ipc_release unmaps what it returned. */
int qsim_ipc_import(int device, const unsigned char* handle64, void** out_ptr);
int qsim_ipc_release(void* imported_ptr);
/* CUDA-IPC handle of the allocation that holds `ptr` (any cudaMalloc'ed memory, e.g. a
 * PyTorch tensor) and the byte offset of `ptr` inside it: the importer adds the offset to
 * what qsim_ipc_import returns. */
int qsim_ipc_export_ex(void* ptr, unsigned char* handle64, uint64_t* offset);
/* The whole k-qubit exchange as ONE kernel over NVLink peer memory (gather + transfer +
 * scatter fused, in place on both sides, no staging): this rank swaps, with each of the
 * 2^k - 1 partners, the block of `shard` whose k local qubits spell the partner's rank bits
 * against the partner's block whose local qubits spell this rank's.  Pattern d (bit i <->
 * local_qubits[i]) names the partner that differs in those rank bits; peer_shards[d] is
 * that partner's shard mapped into this process (qsim_ipc_import; entry 0 unused),
 * partner_is_lower[d] != 0 if the partner's rank number is below this rank's (the two
 * ranks of a pair split the amplitudes between them by that).  my_bits[i] is this rank's
 * value of the rank bit traded against local_qubits[i].  The caller must make sure, with
 * stream-ordered barriers over the ranks, that every rank's earlier work on its shard is
 * complete before any rank launches, and that every rank's launch is complete before any
 * rank touches its shard again. */
int qsim_exchange_p2p(void* shard, void* const* peer_shards, int n_local, int nbits, const int* local_qubits,
                      const int* my_bits, const int* partner_is_lower, void* stream);

/* Launch statistics since process start (kernels launched by this library). */
int64_t qsim_launch_count(void);

#ifdef __cplusplus
}
#endif
#endif /* QSIM_B200_H */
