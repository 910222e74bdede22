// The work behind the compute entry points of the C ABI.  capi_host.cpp checks the arguments,
// turns reference qubits into index bits, lowers what it can on the host and then calls one of
// these functions.  libqsim_b200.so links the CUDA implementation (kernels.cu), the host emulator
// of the tests the one that loops over host memory (emu.cpp).  Arguments arrive checked; `stream`
// is the caller's cudaStream_t (the emulator ignores it).
#pragma once
#include "elem_ops.h"
#include "planner.h"

// the 2 x n single-qubit amplitudes travel as a kernel parameter (no allocation, no copy)
struct ProductAmps { double a[4 * 40]; };
struct BraPair { double b[4]; };

namespace qs::dev {

int execute_plan(const qsim_plan& p, qs_c128* state, int n, void* stream);
int init_product(qs_c128* state, int n, const ProductAmps& amps, void* stream);
// pairs = 2^(n-1) amplitude pairs that differ in index bit pos
int measure_probs(const qs_c128* state, int pos, uint64_t pairs, const BraPair& bra0, const BraPair& bra1,
                  double* out_norm2, void* stream);
int collapse(const qs_c128* in, qs_c128* out, int pos, const BraPair& bra, double norm, uint64_t count,
             void* stream);
int insert(const qs_c128* in, qs_c128* out, int pos, const BraPair& amp, uint64_t count, void* stream);
int reduce_norm2(const qs_c128* state, uint64_t n_amps, double* out, void* stream);
int reduce_inner(const qs_c128* a, const qs_c128* b, uint64_t n_amps, double* out_re_im, void* stream);
int reduce_expect(const qs_c128* ket, const qs_c128* rho, int n, double* out_re_im, void* stream);
int reduce_purity(const qs_c128* rho, int n, double* out_re_im, void* stream);
int reduce_trace(const qs_c128* rho, int n, double* out_re_im, void* stream);
// sums: 2 * n_terms doubles (re, im per slot of `plan`), zero on entry
int expect_pauli(const qs_c128* state, int n, const PauliPlan& plan, int64_t n_terms, double* sums, void* stream);
// xi, zi: index-bit masks per term; sums: 2 * n_terms doubles (re, im per term)
int expect_pauli_dm(const qs_c128* rho, int n, int64_t n_terms, const uint64_t* xi, const uint64_t* zi,
                    double* sums, void* stream);
// n index bits (2N for a density matrix); one launch per pass, in place, no allocation, no synchronisation
int apply_pauli_rotations(qs_c128* state, int n, const PauliRotPlan& plan, void* stream);
// out <- sum_t c_t P_t in (or out + ..., as the plan's passes say), n index bits, one launch per pass;
// no allocation, no synchronisation
int apply_pauli_sum(const qs_c128* in, qs_c128* out, int n, const PauliApplyPlan& plan, void* stream);
// the sweep of an adjoint plan on psi and lam (n index bits), one launch per pass plus the final sum;
// sums: 2 doubles per rotation slot of `plan`; synchronises the stream
int pauli_rotations_adjoint(qs_c128* psi, qs_c128* lam, int n, const PauliRotPlan& plan, double* sums, void* stream);
// out: 2^G.k doubles (device memory for the CUDA library)
int marginal_probs(const QsProbSrc& src, const QsMargGeom& G, double* out, void* stream);
// n index bits; ws: the caller's workspace laid out by qs_sample_layout(n, shots); *total gets the
// mass sampled from (the caller refuses a total that is not positive and finite)
int sample(const QsProbSrc& src, int n, int64_t shots, const double* uniforms, uint64_t* out, double* total,
           unsigned char* ws, void* stream);
int rb_batch(int nq, int64_t n_seq, const uint16_t* opcodes, const int64_t* offsets, const double* superops,
             const double* unitaries, const double* rho0, const double* psi0, double* out_fidelity,
             double* out_purity, double* out_rho, void* stream);
int traj_batch(int n, int64_t shots, int n_ops, const QsTrajOp* ops, const double* matrices, const uint8_t* flips,
               int64_t flips_per_shot, const qs_c128* psi0, const qs_c128* observable, double* out_fidelity,
               double* out_prob_sum, qs_c128* out_states, void* stream);
int swap_pack(const qs_c128* shard, qs_c128* buf, const QsBitSel& sel, uint64_t first, uint64_t count, void* stream);
int swap_unpack(qs_c128* shard, const qs_c128* buf, const QsBitSel& sel, uint64_t first, uint64_t count,
                void* stream);

}  // namespace qs::dev
