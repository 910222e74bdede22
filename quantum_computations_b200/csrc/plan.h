// Pass / step / layer descriptors shared by the host planner, the sm_100a kernels
// and the host emulator used by the CPU tests.
//
// A *pass* streams the whole state through shared memory once (one HBM read +
// one HBM write per amplitude).  The state index is split into T "tile" bits
// and n-T "outer" bits; every CTA owns the 2^T amplitudes of one outer value,
// has them brought into shared memory by TMA (cp.async.bulk.tensor, 128-byte
// swizzle), applies the pass's *steps* there and has TMA write them back in
// place.  Index bits 0..2 are always tile bits, so the unit of every global
// access is one 128-byte row of 8 amplitudes.
//
// A *step* is one shared-memory round trip: every thread pulls 2^r amplitudes
// (spanning r "group" bits of the tile) into registers, runs the step's
// *layers* on them and stores them back.
//
// A *layer* is, in this order: a sign block, a phase table over the 2^r
// amplitudes, and one 2x2 operation per group bit (or one dense 2^r x 2^r
// matrix).  Several layers per step are what lets a qubit receive its next
// non-diagonal gate while its amplitudes are still in registers: the CZ/Z/phase
// gates in between never need other amplitudes.
//
// 2x2 unitaries are applied as  (real rotation) x (phases), the rotation as shears that
// update one amplitude of a pair in place from the other (tile_exec.h):
//   angle <= 45 deg ("TAN"):   c [[1,-t],[t,1]] = [[1,0],[t,1]] [[1,-u],[0,1]] diag(c, c (1 + t^2)),
//                              t = s/c, u = t / (1 + t^2): two FMAs per component pair, the
//                              diagonal is folded into the layer's phase table;
//   up to 90 deg ("SHEAR3"):   [[1,-p],[0,1]] [[1,0],[q,1]] [[1,-p],[0,1]], p = tan(angle/2), q = s:
//                              three FMAs, exact, no scale.
// The merge pass (planner.cpp) splits a quarter turn off every rotation beyond 45 degrees and keeps
// it in its Pauli frame, so SHEAR3 is left for explicit quarter turns (X, Y at the end of a
// circuit); the hot loop runs TAN only, and a layer of sign block + phase table + TAN rotations --
// four out of five layers of a random circuit -- sits behind a single test (tile_exec.h).
//
// Steps are widened to the widest group of their pass with idle group bits (no gate, phase 1):
// ptxas keeps only ONE instantiation of the step body per kernel on the uniform datapath.
//
// Sign blocks.  CZ and Z gates multiply amplitude i by (-1)^q(i), q a quadratic
// form over GF(2) in the index bits -- no memory traffic, any qubits.  They
// commute with every matrix that does not touch their bits, so the planner
// DEFERS each pending pair to the first later layer whose group contains one of
// its bits (or to the pass's final layer).  A layer's sign for amplitude m of
// a work item at local index j0 is
//     parity(m & W(j0)) + qg(m),
//     W_f = z_f + parity(j0 & ng[f])        (f = group factor)
// with ng[f] the in-tile partners of group bit f outside the group, z_f a Z on
// it (a local Z, or a CZ with an outer bit that is 1 for this tile), and qg the
// pairs inside the group (thread independent: the planner folds it into the phase
// table): a few popcounts per work item.  The pass's FINAL layer
// (sign only, last layer of the last step) additionally carries the pairs that
// touch no group bit: a bit common to the work item,
//     g + z.j0 + Q(j0)
// (tile-uniform bit g from pairs of outer bits, linear mask z, quadratic form Q
// with symmetric neighbour masks fin_nsym).
//
// Index-bit convention inside the library: bit b of the linear index.  The
// reference numbers qubits from the most significant end, so reference qubit q
// of an n-qubit register is bit n-1-q (DV/numpy_quantum.py:243-247).
#pragma once
#include <stdint.h>

#define QS_MAX_R        4      // group bits per step (dense 16x16 at most)
#define QS_MAX_STEPS    24     // shared-memory round trips per pass
#define QS_MAX_LAYERS   40     // layers per pass
#define QS_MAX_PAIRS    640    // (outer,outer) and (local,outer) sign pairs per pass
#define QS_MAX_COEF     2560   // doubles of coefficients per pass
// Threads per CTA are chosen per pass (QsPass::cta_log2): 128 or 256.  QS_THREADS_LOG2 is the
// larger of the two (array sizes, default).
#ifndef QS_THREADS_LOG2
#define QS_THREADS_LOG2 8
#endif
#define QS_THREADS_LOG2_MIN 7
// largest tile: 2^13 amplitudes = 128 KiB; a step's per-thread iteration table has 16 entries
#define QS_MAX_T        (QS_THREADS_LOG2 + 5 < 13 ? QS_THREADS_LOG2 + 5 : 13)
#define QS_THREADS      (1 << QS_THREADS_LOG2)
#define QS_MAX_ITER     (1 << (QS_MAX_T - QS_THREADS_LOG2))   // amplitudes per thread in a plain load/store
#define QS_MAX_WORK     16                                    // work items per thread and step (r >= 1)

enum QsLayerKind : uint8_t {
  QS_LAYER_ROT     = 0,   // sign, phase table, per factor none / TAN / SHEAR3
  QS_LAYER_GENERAL = 1,   // sign, phase table, per factor none / any complex 2x2 (8 doubles)
  QS_LAYER_DENSE   = 2    // sign, then one dense 2^r x 2^r complex matrix, or two 4x4 blocks on factors
                          // (0,1) and (2,3) of a 4-bit step (QS_LH_PAIR); only gate layer of its step
};

enum QsFactorForm : uint8_t {
  QS_FORM_NONE = 0,       // nothing on this group bit in this layer
  QS_FORM_TAN    = 1,     // a0 -= u a1 ; a1 += t a0                  (coefficients u, t)
  QS_FORM_SHEAR3 = 2,     // a0 -= p a1 ; a1 += q a0 ; a0 -= p a1     (coefficients p, q)
  QS_FORM_FULL   = 3      // general complex 2x2 (QS_LAYER_GENERAL only)
};

#define QS_LF_SIGN   1u   // the layer has a sign block
#define QS_LF_PHASE  2u   // the layer has a phase table
#define QS_LF_FINAL  4u   // sign block also carries the work-item-common part (final layer)

// head word of a layer (everything the kernel branches on, one uniform load)
#define QS_LH_SIGN     (1u << 0)
#define QS_LH_PHASE    (1u << 1)
#define QS_LH_FINAL    (1u << 2)
#define QS_LH_GENERAL  (1u << 3)
#define QS_LH_DENSE    (1u << 4)
#define QS_LH_SHEAR3ANY (1u << 6)  // some factor of the layer has the three-shear form (rare: quarter turns only)
#define QS_LH_PAIR     (1u << 5)   // dense layer of a 4-bit step holding TWO 4x4 blocks: factors (0,1) and (2,3)
#define QS_LH_TAN(f)    (1u << (8 + (f)))
#define QS_LH_SHEAR3(f) (1u << (12 + (f)))
#define QS_LH_FULL(f)   (1u << (16 + (f)))

struct alignas(16) QsLayer {
  // ---- first 16 bytes: what the kernel reads per layer (one 128-bit uniform load) ----
  uint32_t head;                 // QS_LH_* bits
  uint16_t coef_off;             // ROT: 2 r doubles; GENERAL: 8 r doubles; DENSE: 2 * 4^r doubles (even)
  uint16_t ph_off;               // 2^r complex (amplitude m: matrix factor f is bit r-1-f of m) (even)
  uint32_t ngp[2];               // ng[0] | ng[1] << 16, ng[2] | ng[3] << 16
  // ---- the rest is read by the planner, the emulator and the per-tile sign thread ----
  uint8_t  kind;
  uint8_t  flags;
  uint8_t  form[QS_MAX_R];       // per group factor (QsFactorForm)
  uint8_t  step;                 // the step this layer belongs to
  uint8_t  pad;
  uint16_t pair_off;             // first (local position, outer global bit) pair in QsPass::pairs
  uint16_t n_lo;
  uint16_t zconst;               // local positions carrying a Z
  uint16_t cross;                // paired dense layer (and a final layer behind one): amplitudes m whose sign
                                 // flips because of pairs BETWEEN the two blocks (bit m), which no 4x4 can absorb
  // in-tile partners (local positions outside the group) of group factor f live in ngp; sign
  // pairs inside the group depend on m only and are folded into the phase table (or the
  // dense matrix) by the planner
};
static_assert(sizeof(QsLayer) == 32, "QsLayer layout");

struct QsStep {
  uint8_t  r;                    // number of group bits
  uint8_t  nlayers;
  uint8_t  layer0;               // first layer in QsPass::layers
  uint8_t  block_sync;           // 1: __syncthreads() after this step; 0: the next step only needs data
                                 //    of the same warp (same warp-owned index bits), __syncwarp() is enough
  uint8_t  gpos[QS_MAX_R];       // local position of group factor f (f=0: most significant bit of m)
  uint8_t  fpos[QS_MAX_T];       // the T-r free local positions, in thread-scatter order
  uint8_t  pad[3];
  uint32_t sdepb[1 << QS_MAX_R]; // BYTE offset (swizzled slot * 16) of amplitude m of a work item
  uint32_t hi[QS_MAX_WORK];      // iteration i: jhi | swz(jhi) << 16
};

struct QsPass {
  uint32_t T;                    // tile bits
  uint32_t nsteps;
  uint32_t nlayers;
  uint32_t ncoef;
  uint32_t npairs;
  uint8_t  tile_bits[16];        // ascending global bit numbers of the local positions
  // final layer: the part of its sign that is common to a work item
  uint8_t  has_final;            // the last layer of the last step is a QS_LF_FINAL layer
  uint8_t  cta_log2;             // log2 threads per CTA this pass's thread maps are built for (7 or 8)
  uint16_t fin_pair_off;         // first pair: fin_n_oo (outer, outer), then the layer's own (local, outer)
  uint16_t fin_n_oo;
  uint16_t fin_qhi;              // bit i: Q(jhi_i) for the last step's iteration i
  uint16_t fin_neigh[QS_MAX_WORK];   // XOR of fin_nsym over the bits of jhi_i
  uint16_t fin_nsym[QS_MAX_T];   // fin_nsym[p]: local positions (outside the last group) coupled to p
  QsStep   steps[QS_MAX_STEPS];
  alignas(16) QsLayer layers[QS_MAX_LAYERS];
  uint8_t  pairs[QS_MAX_PAIRS * 2];
  alignas(16) double coef[QS_MAX_COEF];
};

// CUDA kernel parameters are limited to 32764 bytes (CUDA >= 12.1, sm_70+); the pass shares
// them with a 128-byte tensor map and a few scalars.
static_assert(sizeof(QsPass) <= 31000, "QsPass must fit in the kernel parameter space");

// Per-step lookup table built once per kernel launch in shared memory: where the
// thread id lands inside the tile (the only thread-dependent table).
struct QsStepTab {
  uint16_t jA[16];               // local-index bits of thread-id nibble 0
  uint16_t jB[32];               // local-index bits of thread-id bits 4..8
};

// How the TMA boxes of a pass cover a tile (kernel parameter beside the tensor map).
// The state is described to TMA as a 5-dimensional tensor whose dimension i is the
// index-bit range [shift[i], shift[i+1]); a box covers the lowest P tile positions, the
// remaining T-P positions are enumerated by issuing 2^(T-P) boxes per tile.
struct QsTmaGeom {
  int32_t use_tma;               // 0: plain loads / stores (tiny states, unusual tile sets)
  int32_t P;
  int32_t nops;
  int32_t shift[5];
  uint32_t mask[5];
};

// ---- Pauli-sum expectation values on a ket (qsim_expect_pauli) ---------------------------
// A Pauli string is a pair of index-bit masks (x, z): P = i^popc(x & z) X^x Z^z, Z first.
// One *Pauli pass* streams the state once, read only.  Every thread owns the 2^d amplitudes
// base ^ off[m], m < 2^d, where off[m] is the XOR of the pass's generators v_i selected by the
// bits of m; base runs over the indices whose pivot bits (one per generator, chosen so that
// the generators restricted to them are invertible) are zero.  Every term whose x lies in the
// span of the generators -- x = off[xl] -- pairs amplitude m with m ^ xl inside the thread's
// registers.  Terms are grouped by xl; a group forms w[m] = conj(a[m ^ xl]) a[m] once.  A term
// takes the real part of w (even popc(x & z)) or the imaginary part (odd) with the sign
// (-1)^popc((base ^ off[m]) & z) = (outer parity) x (-1)^popc(m & s), where bit i of s is
// parity(generator_i & z): the inner sign is a Walsh function of m.  So a group transforms
// Re w and Im w once (Walsh-Hadamard, D x 2^D additions each) and every term reads ONE entry
// of the spectrum.  The x = 0 group (Z strings) is the case xl = 0: w[m] = |a[m]|^2.
#define QS_PAULI_MAX_D 4
#define QS_PAULI_MAX_TERMS 32          // accumulators per thread, i.e. terms per pass

struct QsPauliGroup {
  uint8_t xl;                    // x of the group in generator coordinates (0: Z strings)
  uint8_t first, count;          // its terms: [first, first + count) of the pass
  uint8_t parts;                 // bit 0: a term takes Re w, bit 1: a term takes Im w
};

struct QsPauliPass {
  uint32_t d;                    // generators = log2 amplitudes per thread
  uint32_t ngroups, nterms;
  uint32_t term0;                // row of the pass's first term in the call's partials
  uint8_t  pivot[QS_PAULI_MAX_D];            // ascending index bits that are zero in every base
  uint64_t off[1 << QS_PAULI_MAX_D];         // XOR of the generators selected by m
  QsPauliGroup groups[1 << QS_PAULI_MAX_D];
  uint64_t z[QS_PAULI_MAX_TERMS];            // index-bit Z mask of each term
  uint8_t  spec[QS_PAULI_MAX_TERMS];         // s: bit i = parity(generator_i & z)
  uint8_t  cls[QS_PAULI_MAX_TERMS];          // bit 0: imaginary part of w; bit 1: negated
};

// ---- Pauli-string rotations (qsim_apply_pauli_rotations / _dm) ------------------------------
// One *rotation pass* applies R_r = exp(-i theta_r / 2 P_r) = c_r - i s_r P_r for a contiguous run
// of rotations, in caller order, with one read and one write of the state.  The thread layout is
// the Pauli pass's (d, pivot, off as in QsPauliPass): every X mask of the run is off[xl] for some
// xl, so P pairs amplitude m with m ^ xl inside the thread's registers, and
//     (P a)[m] = i^popc(x & z) (-1)^(par(base & z) + popc((m ^ xl) & spec)) a[m ^ xl].
// The caller's factor -i i^popc(x & z) is kappa = i^cls.  Rotations of one pass run in a loop, so
// the cap only bounds the descriptor; DESIGN.md section 3.2.3 gives the measurement behind it.
#define QS_PAULI_ROT_MAX 32

struct QsPauliRotPass {
  uint32_t d;                                // generators = log2 amplitudes per thread
  uint32_t nrot;
  uint8_t  pivot[QS_PAULI_MAX_D];            // ascending index bits that are zero in every base
  uint64_t off[1 << QS_PAULI_MAX_D];         // XOR of the generators selected by m
  uint64_t z[QS_PAULI_ROT_MAX];              // index-bit Z mask of each rotation
  double   c[QS_PAULI_ROT_MAX];              // cos(theta / 2)
  double   s[QS_PAULI_ROT_MAX];              // sin(theta / 2)
  uint8_t  xl[QS_PAULI_ROT_MAX];             // X mask in generator coordinates
  uint8_t  spec[QS_PAULI_ROT_MAX];           // bit i = parity(generator_i & z)
  uint8_t  cls[QS_PAULI_ROT_MAX];            // kappa = -i i^popc(x & z) = i^cls
};
static_assert(sizeof(QsPauliRotPass) <= 4096, "QsPauliRotPass is a kernel parameter");

// ---- H|psi> for a Pauli sum (qsim_apply_pauli_sum) -------------------------------------------
// The terms are packed as for the expectation values (QsPauliPass: same grouping, layout and
// spec), and every slot t carries k_t = c_t i^popc(x & z).  With b[m] = in[base ^ off[m ^ xl]]
//     out[m] += sum_t k_t (-1)^(par(base & z_t) + popc((m ^ xl) & spec_t)) b[m] = F[m ^ xl] b[m],
// F the Walsh transform of the spectrum that holds +-k_t at index spec_t: one transform per group,
// whatever the number of its terms.  The first pass of a qsim_apply_pauli_sum call writes out, later
// passes add to it; every pass of a qsim_accumulate_pauli_sum call adds.
//
// A qsim_lanczos_apply call runs the same passes through the kernel's Lanczos instantiation, which
// alone reads the two fields after `accumulate`: its first pass starts from prev_scale x prev
// (QS_APPLY_FROM_PREV) or prev_scale x out when the caller's prev is out (QS_APPLY_FROM_OUT), and
// its last pass (`dot`) also returns the work item's share of Re sum conj(in) out.
#define QS_APPLY_FROM_PREV 2u
#define QS_APPLY_FROM_OUT 3u
struct QsPauliApplyPass {
  QsPauliPass p;
  double   kre[QS_PAULI_MAX_TERMS];          // k_t, slot order of p
  double   kim[QS_PAULI_MAX_TERMS];
  uint32_t accumulate;                       // 0: write out; 1: add to it; QS_APPLY_FROM_PREV / _OUT
  uint32_t dot;                              // Lanczos only: 1 = reduce Re <in|out> after this pass
  double   prev_scale;                       // Lanczos only: p of the first pass
};
static_assert(sizeof(QsPauliApplyPass) <= 4096, "QsPauliApplyPass is a kernel parameter");

// ---- adjoint sweep (qsim_pauli_rotations_adjoint / _dm) ----------------------------------------
// A sweep pass is a QsPauliRotPass whose rotations are in reverse caller order with negated angles,
// applied to two states at once; a work item holds 2^d amplitudes of each, so the kernel keeps four
// times the amplitudes of one state in registers.  Generators per sweep pass (no register spills
// for sm_100a; DESIGN.md section 3.2.4 lists the registers of every d):
#define QS_PAULI_ADJ_MAX_D 3
