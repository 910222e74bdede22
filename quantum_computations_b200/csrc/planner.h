// Host-side circuit container and fusion planner (no CUDA dependency, so the
// same sources also build into the host emulator used by the CPU tests).
#pragma once
#include <complex>
#include <cstdint>
#include <cstdlib>
#include <memory>
#include <string>
#include <vector>

#include "../../include/qsim_b200.h"
#include "plan.h"

namespace qs {

typedef std::complex<double> cplx;

enum OpKind { OP_DENSE = 0, OP_SIGN = 1 };

// One gate in library coordinates: bits[f] is the index bit that matrix factor
// f (f = 0 most significant) acts on.
struct Op {
  int kind = OP_DENSE;
  int k = 0;
  std::vector<int> bits;
  bool diag = false;
  std::vector<cplx> mat;     // 2^k x 2^k row-major (empty for OP_SIGN)
  // k == 1 unitaries emitted by the merge pass as  [[c,-s],[s,c]] . diag(r0, r1)
  bool rot = false;
  double c = 1.0, s = 0.0;
  cplx r0 = cplx(1.0, 0.0), r1 = cplx(1.0, 0.0);
  uint64_t mask() const {
    uint64_t m = 0;
    for (int b : bits) m |= 1ull << b;
    return m;
  }
};

struct PlanItem {
  bool generic = false;      // a dense block on more than QS_MAX_R qubits (own kernel)
  QsPass pass;               // valid when !generic
  Op op;                     // valid when generic
  // device copy of op.mat, made at the first execution and owned by the plan
  // (libqsim_b200.so only; the deleter is cudaFree)
  mutable std::shared_ptr<void> dev_mat;
  mutable int dev_index = -1;
};

}  // namespace qs

struct qsim_circuit {
  int n = 0;
  std::vector<qs::Op> ops;
};

struct qsim_plan {
  int n = 0;
  std::vector<qs::PlanItem> items;
  std::vector<double> residual;          // n x 8 doubles (index bit b first), empty unless defer_tail
  qsim_plan_stats_t stats{};
};

namespace qs {

// Development knobs (A/B switches behind the measurements in DESIGN.md section 5) read the
// environment only in builds with -DQSIM_DEV_KNOBS; the shipped library ignores it.  Every knob
// selects between CORRECT variants; none changes results.
inline int dev_knob(const char* name, int fallback) {
#if defined(QSIM_DEV_KNOBS)
  const char* e = getenv(name);
  return e ? atoi(e) : fallback;
#else
  (void)name;
  return fallback;
#endif
}

void set_error(const std::string& msg);
int fail(int code, const std::string& msg);

// Single-qubit merging pre-pass (returns the reduced op list).
// With `residual` the trailing diagonal / antidiagonal product of every index bit is not
// emitted but written there (8 doubles per bit, identity where nothing is pending).
// Index bits in `apply_mask` are exempt.
std::vector<Op> merge_single_qubit(int n, const std::vector<Op>& in, std::vector<double>* residual = nullptr,
                                   uint64_t apply_mask = 0);

// Greedy tile/pass construction.
int build_plan(int n, const std::vector<Op>& ops, const qsim_plan_options_t& opt, qsim_plan* out);

qsim_plan_options_t resolve_options(const qsim_plan_options_t* opt);

// ---- Pauli-sum expectation values (pauli.cpp; descriptors in plan.h) ----------------------
// Checks of qsim_expect_pauli / _dm: n in [1, 63], masks below 2^n (n_terms == 0 passes).
int check_pauli_args(const char* who, int n, int64_t n_terms, const uint64_t* x_masks, const uint64_t* z_masks,
                     const void* out);
// Reference-qubit masks -> index-bit masks, and popc(x & z) mod 4 of every term.
void pauli_index_masks(int n, int64_t n_terms, const uint64_t* x_masks, const uint64_t* z_masks,
                       std::vector<uint64_t>* xi, std::vector<uint64_t>* zi, std::vector<uint8_t>* phase);

// The passes of one call.  Slot s (pass by pass, term by term) holds caller term order[s].
struct PauliPlan {
  int d = 0;                                 // generators per pass: min(n, QS_PAULI_MAX_D)
  std::vector<QsPauliPass> passes;
  std::vector<int64_t> order;
};
// Greedy grouping by X mask: at most one pass per chunk of <= QS_PAULI_MAX_TERMS terms of one
// non-zero X mask, the Z strings in passes with room (a pass of their own only if none has).
int plan_pauli(int n, int64_t n_terms, const uint64_t* x_masks, const uint64_t* z_masks, PauliPlan* out);
// The passes of one qsim_apply_pauli_sum / qsim_accumulate_pauli_sum call: plan_pauli's, each slot
// with k_t = c_t i^popc(x & z).  The first pass writes out, or adds to it with `accumulate`; with no
// terms one pass that writes zeros (the caller launches nothing when it accumulates).
struct PauliApplyPlan {
  int d = 0;
  std::vector<QsPauliApplyPass> passes;
};
int plan_pauli_apply(int n, int64_t n_terms, const uint64_t* x_masks, const uint64_t* z_masks,
                     const double* coeffs_re_im, bool accumulate, PauliApplyPlan* out);
// The rotation passes of one qsim_apply_pauli_rotations(_dm) call, in caller order, or of one
// adjoint sweep.
struct PauliRotPlan {
  int d = 0;                                 // generators per pass: min(register bits, QS_PAULI_MAX_D
                                             // or, for a sweep, QS_PAULI_ADJ_MAX_D)
  std::vector<QsPauliRotPass> passes;
  // sweeps only: per rotation slot (pass by pass) its caller rotation and the weight of its
  // overlap in that rotation's derivative
  std::vector<int64_t> caller;
  std::vector<double> weight;
};
// Greedy in caller order, never reordered: a rotation joins the open pass while the cap allows and
// its X mask is in the span or the span has room; angle-0 rotations are skipped.  dm: n is N and
// every rotation becomes its row half and its conjugated column half on the 2N-bit vec of rho,
// always in one pass.  adjoint: the sweep of qsim_pauli_rotations_adjoint -- the same packing of
// the rotations in reverse caller order with negated angles, angle-0 rotations kept, at most
// QS_PAULI_ADJ_MAX_D generators per pass.
int plan_pauli_rotations(int n, int64_t n_rot, const uint64_t* x_masks, const uint64_t* z_masks, const double* angles,
                         bool dm, PauliRotPlan* out, bool adjoint = false);
// sums: 2 doubles per slot (re, im) -> out[caller term] (real).
void pauli_finish(const PauliPlan& plan, const double* sums, double* out);
// sums: 2 doubles per sweep slot -> out[caller rotation] = sum of weight x overlap, in slot order.
void pauli_adjoint_finish(const PauliRotPlan& plan, int64_t n_rot, const double* sums, double* out);
// sums: 2 doubles per term, times i^phase -> out_re_im.
void pauli_finish_dm(int64_t n_terms, const std::vector<uint8_t>& phase, const double* sums, double* out_re_im);

}  // namespace qs
