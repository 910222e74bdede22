// HOST EMULATOR -- TEST INFRASTRUCTURE ONLY.
//
// Builds (g++ only, no CUDA) into tests/_build/libqsim_emu.so and exports the
// same C ABI as libqsim_b200.so, but on HOST pointers.  It runs the very same
// planner (planner.cpp / capi_host.cpp) and the very same per-thread phase
// functions (tile_exec.h, elem_ops.h) as the GPU kernels, looping over thread
// ids where the GPU runs them in parallel.  The CPU test-suite uses it to check
// the plan logic and the index arithmetic without a GPU.  The product package
// never loads it: quantum_computations_b200.engine binds libqsim_b200.so only
// and raises when that library or a CUDA device is missing.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <string>
#include <utility>
#include <vector>

#include "elem_ops.h"
#include "planner.h"

namespace {

int64_t g_launches = 0;

// The emulator runs threads one after the other, so it cannot see a missing
// barrier.  What it can check is the planner's promise behind every
// `block_sync == 0`: in step s and step s+1 each warp touches exactly the same set
// of shared-memory slots.
int g_ownership_violations = 0;

void slots_of_step(const QsPass& P, int s, const QsStepTab& tab, std::vector<int>& owner) {
  const uint32_t nthreads = 1u << P.cta_log2;
  const QsStep& st = P.steps[s];
  const uint32_t nwork = 1u << (P.T - st.r);
  owner.assign((size_t)1 << P.T, -1);
  for (uint32_t tid = 0; tid < nthreads; ++tid) {
    const uint32_t jlo = qs_thread_jlo(tab, tid);
    for (uint32_t i = 0, w = tid; w < nwork; ++i, w += nthreads) {
      const uint32_t j0 = jlo | (st.hi[i] & 0xffffu);
      for (int m = 0; m < (1 << st.r); ++m) {
        uint32_t d = 0;
        for (int f = 0; f < st.r; ++f) d |= (uint32_t)((m >> (st.r - 1 - f)) & 1) << st.gpos[f];
        owner[j0 | d] = (int)(tid >> 5);
      }
    }
  }
}

void check_warp_ownership(const QsPass& P, int s, const QsStepTab& tab_s) {
  static std::vector<int> prev;
  static int prev_step = -2;
  static const QsPass* prev_pass = nullptr;
  std::vector<int> cur;
  slots_of_step(P, s, tab_s, cur);
  // every slot of the tile must be touched exactly by one work item
  for (size_t j = 0; j < cur.size(); ++j)
    if (cur[j] < 0) { ++g_ownership_violations; break; }
  if (prev_pass == &P && prev_step == s - 1 && P.steps[s - 1].block_sync == 0)
    for (size_t j = 0; j < cur.size(); ++j)
      if (cur[j] != prev[j]) { ++g_ownership_violations; break; }
  prev.swap(cur);
  prev_step = s;
  prev_pass = &P;
}

void emu_pass(const QsPass& P, qs_c128* state, int n) {
  const uint32_t nthreads = 1u << P.cta_log2;
  const uint32_t thr_log2 = P.cta_log2;
  const uint64_t ntiles = 1ull << (n - (int)P.T);
  const int nsteps = (int)P.nsteps;
  std::vector<qs_c128> tile((size_t)1 << P.T);
  std::vector<uint32_t> zm(P.nlayers + 1, 0);
  std::vector<QsStepTab> tab(nsteps ? nsteps : 1);
  bool dense = false;
  for (uint32_t l = 0; l < P.nlayers; ++l) dense |= P.layers[l].kind == QS_LAYER_DENSE;
  for (int s = 0; s < nsteps; ++s)
    for (int e = 0; e < QS_TAB_ENTRIES; ++e) qs_build_step_tab(P, s, e, &tab[s], thr_log2);
  std::vector<uint32_t> fin_qlo(nthreads, 0);
  if (P.has_final)
    for (uint32_t tid = 0; tid < nthreads; ++tid)
      fin_qlo[tid] = qs_fin_quad(P, qs_thread_jlo(tab[nsteps - 1], tid));
  for (uint64_t t = 0; t < ntiles; ++t) {
    const uint64_t base = qs_tile_base(P, t);
    for (int l = 0; l < (int)P.nlayers; ++l)
      zm[l] = (P.layers[l].flags & QS_LF_SIGN) ? qs_layer_z(P, l, base) : 0u;
    const uint32_t fin_g = P.has_final ? qs_fin_g(P, base) : 0u;
    for (uint32_t tid = 0; tid < nthreads; ++tid) qs_plain_load(P, state, tile.data(), base, tid, nthreads);
    for (int s = 0; s < nsteps; ++s) {
      for (uint32_t tid = 0; tid < nthreads; ++tid) {
        // same variant selection as launch_pass() in kernels.cu
        // the three dense modes of launch_pass() in kernels.cu run the same step bodies
        if (dense && (t & 1)) qs_phase_step_any<4, 2>(P, s, tile.data(), tid, thr_log2, zm.data(), fin_g, fin_qlo[tid], tab[s]);
        else if (dense) qs_phase_step_any<4, 1>(P, s, tile.data(), tid, thr_log2, zm.data(), fin_g, fin_qlo[tid], tab[s]);
        else qs_phase_step_any<4, 0>(P, s, tile.data(), tid, thr_log2, zm.data(), fin_g, fin_qlo[tid], tab[s]);
      }
      if (t == 0) check_warp_ownership(P, s, tab[s]);
    }
    for (uint32_t tid = 0; tid < nthreads; ++tid) qs_plain_store(P, state, tile.data(), base, tid, nthreads);
  }
  ++g_launches;
}

// dense block on more than QS_MAX_R qubits: the CUDA library runs it in place (k_dense_block);
// here the plain definition with a temporary copy
int emu_generic(const qs::Op& op, qs_c128* state, int n) {
  const int dim = 1 << op.k;
  std::vector<double> flat(2 * (size_t)dim * dim);
  for (int e = 0; e < dim * dim; ++e) { flat[2 * e] = op.mat[e].real(); flat[2 * e + 1] = op.mat[e].imag(); }
  int bits[10];
  for (int f = 0; f < op.k; ++f) bits[f] = op.bits[f];
  const uint64_t count = 1ull << n;
  std::vector<qs_c128> scratch(count);
  for (uint64_t i = 0; i < count; ++i) scratch[i] = qs_generic_amp(state, flat.data(), bits, op.k, i);
  memcpy(state, scratch.data(), sizeof(qs_c128) * count);
  ++g_launches;
  return QSIM_OK;
}

int execute_plan(const qsim_plan* p, void* state, int n, void* scratch) {
  if (!p || !state) return qs::fail(QSIM_ERR_ARG, "qsim_plan_execute: null argument");
  if (g_ownership_violations)
    return qs::fail(QSIM_ERR_UNSUPPORTED, "emulator: a warp-synchronised step reads another warp's amplitudes");
  if (n != p->n) return qs::fail(QSIM_ERR_ARG, "qsim_plan_execute: plan was compiled for a different qubit count");
  for (const qs::PlanItem& it : p->items) {
    if (it.generic) {
      int rc = emu_generic(it.op, (qs_c128*)state, n);
      if (rc != QSIM_OK) return rc;
    } else {
      if ((int)it.pass.T > n) return qs::fail(QSIM_ERR_ARG, "pass tile larger than the state");
      emu_pass(it.pass, (qs_c128*)state, n);
      if (g_ownership_violations)
        return qs::fail(QSIM_ERR_UNSUPPORTED, "emulator: a warp-synchronised step reads another warp's amplitudes");
    }
  }
  return QSIM_OK;
}

int one_gate(void* state, int n, const int* targets, int k, const double* matrix, void* scratch) {
  qsim_circuit_t* c = nullptr;
  int rc = qsim_circuit_create(n, &c);
  if (rc != QSIM_OK) return rc;
  rc = qsim_circuit_add_matrix(c, k, targets, matrix);
  qsim_plan_t* p = nullptr;
  if (rc == QSIM_OK) rc = qsim_plan_compile(c, nullptr, &p);
  if (rc == QSIM_OK) rc = execute_plan(p, state, n, scratch);
  qsim_plan_destroy(p);
  qsim_circuit_destroy(c);
  return rc;
}

}  // namespace

extern "C" {

int qsim_has_cuda(void) { return 0; }
int64_t qsim_launch_count(void) { return g_launches; }

// peer staging: the emulator has one address space; these are plain host operations
int qsim_peer_alloc(int, uint64_t bytes, void** out_ptr) {
  if (!out_ptr || bytes == 0) return qs::fail(QSIM_ERR_ARG, "qsim_peer_alloc: bad argument");
  *out_ptr = malloc(bytes);
  return *out_ptr ? QSIM_OK : qs::fail(QSIM_ERR_NOMEM, "out of host memory");
}
int qsim_peer_free(void* ptr) { free(ptr); return QSIM_OK; }
int qsim_ipc_export(void*, unsigned char*) { return qs::fail(QSIM_ERR_UNSUPPORTED, "no IPC in the host emulator"); }
int qsim_ipc_import(int, const unsigned char*, void**) { return qs::fail(QSIM_ERR_UNSUPPORTED, "no IPC in the host emulator"); }
int qsim_ipc_release(void*) { return QSIM_OK; }
int qsim_ipc_export_ex(void*, unsigned char*, uint64_t*) { return qs::fail(QSIM_ERR_UNSUPPORTED, "no IPC in the host emulator"); }
int qsim_exchange_p2p(void*, void* const*, int, int, const int*, const int*, const int*, void*) {
  return qs::fail(QSIM_ERR_UNSUPPORTED, "no peer memory in the host emulator (the exchange goes through send/recv)");
}
int qsim_peer_copy(void* dst, const void* src, uint64_t bytes, void*) {
  if (!dst || !src) return qs::fail(QSIM_ERR_ARG, "qsim_peer_copy: null argument");
  memcpy(dst, src, bytes);
  return QSIM_OK;
}

int qsim_plan_execute(const qsim_plan_t* p, void* state, int n_qubits, void* scratch, void*) {
  return execute_plan(p, state, n_qubits, scratch);
}

int qsim_apply_matrix(void* state, int n_qubits, const int* targets, int k, const double* matrix,
                      void* scratch, void*) {
  if (!state || !targets || !matrix) return qs::fail(QSIM_ERR_ARG, "qsim_apply_matrix: null argument");
  return one_gate(state, n_qubits, targets, k, matrix, scratch);
}

int qsim_apply_diagonal(void* state, int n_qubits, const int* targets, int k, const double* diag, void*) {
  if (!state || !targets || !diag) return qs::fail(QSIM_ERR_ARG, "qsim_apply_diagonal: null argument");
  if (k < 1 || k > QS_MAX_R) return qs::fail(QSIM_ERR_UNSUPPORTED, "qsim_apply_diagonal: k must be in [1, 4]");
  const int dim = 1 << k;
  std::vector<double> m(2 * (size_t)dim * dim, 0.0);
  for (int d = 0; d < dim; ++d) { m[2 * (d * dim + d)] = diag[2 * d]; m[2 * (d * dim + d) + 1] = diag[2 * d + 1]; }
  return one_gate(state, n_qubits, targets, k, m.data(), nullptr);
}

int qsim_apply_permutation(void* state, int n_qubits, const int* targets, int k, const int* perm, void*) {
  if (!state || !targets || !perm) return qs::fail(QSIM_ERR_ARG, "qsim_apply_permutation: null argument");
  if (k < 1 || k > QS_MAX_R) return qs::fail(QSIM_ERR_UNSUPPORTED, "qsim_apply_permutation: k must be in [1, 4]");
  const int dim = 1 << k;
  std::vector<double> m(2 * (size_t)dim * dim, 0.0);
  std::vector<char> hit(dim, 0);
  for (int c = 0; c < dim; ++c) {
    if (perm[c] < 0 || perm[c] >= dim || hit[perm[c]]) return qs::fail(QSIM_ERR_ARG, "qsim_apply_permutation: not a permutation");
    hit[perm[c]] = 1;
    m[2 * (perm[c] * dim + c)] = 1.0;
  }
  return one_gate(state, n_qubits, targets, k, m.data(), nullptr);
}

int qsim_apply_superop(void* vec_rho, int n_qubits, const int* targets, int k, const double* superop,
                       void* scratch, void*) {
  if (!vec_rho || !targets || !superop) return qs::fail(QSIM_ERR_ARG, "qsim_apply_superop: null argument");
  if (k < 1 || 2 * k > 10) return qs::fail(QSIM_ERR_UNSUPPORTED, "qsim_apply_superop: k must be in [1, 5]");
  std::vector<int> t(2 * k);
  for (int i = 0; i < k; ++i) { t[i] = targets[i]; t[k + i] = targets[i] + n_qubits; }
  return one_gate(vec_rho, 2 * n_qubits, t.data(), 2 * k, superop, scratch);
}

int qsim_init_product(void* state, int n_qubits, const double* amps, void*) {
  if (!state || !amps || n_qubits < 1 || n_qubits > 40) return qs::fail(QSIM_ERR_ARG, "qsim_init_product: bad argument");
  qs_c128* s = (qs_c128*)state;
  for (uint64_t i = 0; i < (1ull << n_qubits); ++i) s[i] = qs_product_amp(amps, n_qubits, i);
  ++g_launches;
  return QSIM_OK;
}

int qsim_measure_probs(const void* state, int n_qubits, int qubit, const double* bra0, const double* bra1,
                       double* out_norm2, void*) {
  if (!state || !bra0 || !bra1 || !out_norm2) return qs::fail(QSIM_ERR_ARG, "qsim_measure_probs: null argument");
  if (n_qubits < 1 || qubit < 0 || qubit >= n_qubits) return qs::fail(QSIM_ERR_ARG, "qsim_measure_probs: qubit out of range");
  const qs_c128* s = (const qs_c128*)state;
  const int pos = n_qubits - 1 - qubit;
  double p0 = 0.0, p1 = 0.0;
  for (uint64_t r = 0; r < (1ull << (n_qubits - 1)); ++r) {
    const qs_c128 u = qs_contract(s, pos, r, bra0), v = qs_contract(s, pos, r, bra1);
    p0 += u.x * u.x + u.y * u.y;
    p1 += v.x * v.x + v.y * v.y;
  }
  out_norm2[0] = p0;
  out_norm2[1] = p1;
  g_launches += 2;
  return QSIM_OK;
}

int qsim_collapse(const void* in, void* out, int n_qubits, int qubit, const double* bra, double norm, void*) {
  if (!in || !out || !bra) return qs::fail(QSIM_ERR_ARG, "qsim_collapse: null argument");
  if (n_qubits < 1 || qubit < 0 || qubit >= n_qubits) return qs::fail(QSIM_ERR_ARG, "qsim_collapse: qubit out of range");
  const int pos = n_qubits - 1 - qubit;
  qs_c128* o = (qs_c128*)out;
  for (uint64_t r = 0; r < (1ull << (n_qubits - 1)); ++r) {
    qs_c128 v = qs_contract((const qs_c128*)in, pos, r, bra);
    v.x /= norm; v.y /= norm;
    o[r] = v;
  }
  ++g_launches;
  return QSIM_OK;
}

int qsim_insert(const void* in, void* out, int n_qubits, int position, const double* amp, void*) {
  if (!in || !out || !amp) return qs::fail(QSIM_ERR_ARG, "qsim_insert: null argument");
  if (n_qubits < 0 || position < 0 || position > n_qubits) return qs::fail(QSIM_ERR_ARG, "qsim_insert: position out of range");
  qs_c128* o = (qs_c128*)out;
  for (uint64_t i = 0; i < (1ull << (n_qubits + 1)); ++i)
    o[i] = qs_insert_amp((const qs_c128*)in, n_qubits - position, i, amp);
  ++g_launches;
  return QSIM_OK;
}

int qsim_reduce_norm2(const void* state, uint64_t n_amps, double* out, void*) {
  if (!state || !out) return qs::fail(QSIM_ERR_ARG, "qsim_reduce_norm2: null argument");
  const qs_c128* s = (const qs_c128*)state;
  double acc = 0.0;
  for (uint64_t i = 0; i < n_amps; ++i) acc += s[i].x * s[i].x + s[i].y * s[i].y;
  *out = acc;
  g_launches += 2;
  return QSIM_OK;
}

int qsim_reduce_inner(const void* a, const void* b, uint64_t n_amps, double* out_re_im, void*) {
  if (!a || !b || !out_re_im) return qs::fail(QSIM_ERR_ARG, "qsim_reduce_inner: null argument");
  const qs_c128 *u = (const qs_c128*)a, *v = (const qs_c128*)b;
  double re = 0.0, im = 0.0;
  for (uint64_t i = 0; i < n_amps; ++i) {
    re += u[i].x * v[i].x + u[i].y * v[i].y;
    im += u[i].x * v[i].y - u[i].y * v[i].x;
  }
  out_re_im[0] = re;
  out_re_im[1] = im;
  g_launches += 2;
  return QSIM_OK;
}

int qsim_reduce_expect(const void* ket, const void* rho, int n_qubits, double* out_re_im, void*) {
  if (!ket || !rho || !out_re_im || n_qubits < 0 || n_qubits > 20) return qs::fail(QSIM_ERR_ARG, "qsim_reduce_expect: bad argument");
  const qs_c128 *k = (const qs_c128*)ket, *r = (const qs_c128*)rho;
  const uint64_t dim = 1ull << n_qubits;
  double re = 0.0, im = 0.0;
  for (uint64_t i = 0; i < dim; ++i)
    for (uint64_t j = 0; j < dim; ++j) {
      const qs_c128 t = qs_cmul(r[i * dim + j], k[j]);
      re += k[i].x * t.x + k[i].y * t.y;
      im += k[i].x * t.y - k[i].y * t.x;
    }
  out_re_im[0] = re;
  out_re_im[1] = im;
  g_launches += 2;
  return QSIM_OK;
}

int qsim_reduce_purity(const void* rho, int n_qubits, double* out_re_im, void*) {
  if (!rho || !out_re_im || n_qubits < 0 || n_qubits > 20) return qs::fail(QSIM_ERR_ARG, "qsim_reduce_purity: bad argument");
  const qs_c128* r = (const qs_c128*)rho;
  const uint64_t dim = 1ull << n_qubits;
  double re = 0.0, im = 0.0;
  for (uint64_t i = 0; i < dim; ++i)
    for (uint64_t j = 0; j < dim; ++j) {
      const qs_c128 t = qs_cmul(r[i * dim + j], r[j * dim + i]);
      re += t.x;
      im += t.y;
    }
  out_re_im[0] = re;
  out_re_im[1] = im;
  g_launches += 2;
  return QSIM_OK;
}

int qsim_reduce_trace(const void* rho, int n_qubits, double* out_re_im, void*) {
  if (!rho || !out_re_im || n_qubits < 0 || n_qubits > 20) return qs::fail(QSIM_ERR_ARG, "qsim_reduce_trace: bad argument");
  const qs_c128* r = (const qs_c128*)rho;
  const uint64_t dim = 1ull << n_qubits;
  double re = 0.0, im = 0.0;
  for (uint64_t i = 0; i < dim; ++i) { re += r[i * dim + i].x; im += r[i * dim + i].y; }
  out_re_im[0] = re;
  out_re_im[1] = im;
  g_launches += 2;
  return QSIM_OK;
}

// Pauli expectation values: the same grouping (pauli.cpp) and the same per-thread bodies
// (elem_ops.h) as the CUDA library; one launch per pass plus the final sum, as there.
int qsim_expect_pauli(const void* state, int n_qubits, int64_t n_terms, const uint64_t* x_masks,
                      const uint64_t* z_masks, double* out, void*) {
  int rc = qs::check_pauli_args("qsim_expect_pauli", n_qubits, n_terms, x_masks, z_masks, out);
  if (rc != QSIM_OK || n_terms == 0) return rc;
  if (!state) return qs::fail(QSIM_ERR_ARG, "qsim_expect_pauli: null state");
  qs::PauliPlan plan;
  rc = qs::plan_pauli(n_qubits, n_terms, x_masks, z_masks, &plan);
  if (rc != QSIM_OK) return rc;
  std::vector<double> sums(2 * (size_t)n_terms, 0.0);
  const uint64_t count = 1ull << (n_qubits - plan.d);
  const qs_c128* s = (const qs_c128*)state;
  for (const QsPauliPass& P : plan.passes) {
    double acc[QS_PAULI_MAX_TERMS] = {0.0}, wal[2 << QS_PAULI_MAX_D];
    for (uint64_t o = 0; o < count; ++o) {
      switch (plan.d) {
        case 1: qs_pauli_item<1>(P, s, o, acc, wal, 1); break;
        case 2: qs_pauli_item<2>(P, s, o, acc, wal, 1); break;
        case 3: qs_pauli_item<3>(P, s, o, acc, wal, 1); break;
        default: qs_pauli_item<4>(P, s, o, acc, wal, 1); break;
      }
    }
    for (uint32_t t = 0; t < P.nterms; ++t) sums[2 * ((size_t)P.term0 + t)] = acc[t];
    ++g_launches;
  }
  ++g_launches;                              // the final sum
  qs::pauli_finish(plan, sums.data(), out);
  return QSIM_OK;
}

int qsim_expect_pauli_dm(const void* vec_rho, int n_qubits, int64_t n_terms, const uint64_t* x_masks,
                         const uint64_t* z_masks, double* out_re_im, void*) {
  int rc = qs::check_pauli_args("qsim_expect_pauli_dm", n_qubits, n_terms, x_masks, z_masks, out_re_im);
  if (rc != QSIM_OK || n_terms == 0) return rc;
  if (!vec_rho) return qs::fail(QSIM_ERR_ARG, "qsim_expect_pauli_dm: null state");
  if (n_qubits > 31) return qs::fail(QSIM_ERR_ARG, "qsim_expect_pauli_dm: n_qubits must be in [1, 31]");
  std::vector<uint64_t> xi, zi;
  std::vector<uint8_t> phase;
  qs::pauli_index_masks(n_qubits, n_terms, x_masks, z_masks, &xi, &zi, &phase);
  std::vector<double> sums(2 * (size_t)n_terms, 0.0);
  const qs_c128* rho = (const qs_c128*)vec_rho;
  for (int64_t t = 0; t < n_terms; ++t)
    for (uint64_t c = 0; c < (1ull << n_qubits); ++c) {
      const qs_c128 v = qs_pauli_dm_elem(rho, n_qubits, xi[t], zi[t], c);
      sums[2 * t] += v.x;
      sums[2 * t + 1] += v.y;
    }
  g_launches += 2;
  qs::pauli_finish_dm(n_terms, phase, sums.data(), out_re_im);
  return QSIM_OK;
}

int qsim_rb_batch(int nq, int64_t n_seq, const uint16_t* opcodes, const int64_t* offsets, int n_opcodes,
                  const double* superops, const double* unitaries, const double* rho0, const double* psi0,
                  double* out_fidelity, double* out_purity, double* out_rho, void*) {
  if (!opcodes || !offsets || !superops || !unitaries || !rho0 || !psi0 || !out_fidelity || !out_purity)
    return qs::fail(QSIM_ERR_ARG, "qsim_rb_batch: null argument");
  if (nq < 1 || nq > 2) return qs::fail(QSIM_ERR_UNSUPPORTED, "qsim_rb_batch: nq must be 1 or 2");
  if (n_seq < 0 || n_opcodes < 1 || n_opcodes > 65536) return qs::fail(QSIM_ERR_ARG, "qsim_rb_batch: bad sizes");
  for (int64_t b = 0; b < n_seq; ++b) {
    const int64_t lo = offsets[b], hi = offsets[b + 1];
    if (nq == 2)
      qs_rb_sequence<4>(opcodes + lo, hi - lo, superops, unitaries, rho0, psi0, out_fidelity + b,
                        out_purity + b, out_rho ? out_rho + (size_t)b * 2 * 16 : nullptr);
    else
      qs_rb_sequence<2>(opcodes + lo, hi - lo, superops, unitaries, rho0, psi0, out_fidelity + b,
                        out_purity + b, out_rho ? out_rho + (size_t)b * 2 * 4 : nullptr);
  }
  ++g_launches;
  return QSIM_OK;
}

int qsim_traj_batch(int n_qubits, int64_t shots, int n_ops, const int32_t* ops, const double* matrices,
                    const uint8_t* flips, int64_t flips_per_shot, const double* psi0, const double* observable,
                    double* out_fidelity, double* out_prob_sum, double* out_states, void*) {
  if (!ops || !matrices || !flips || !psi0) return qs::fail(QSIM_ERR_ARG, "qsim_traj_batch: null argument");
  if (n_qubits < 1 || n_qubits > 12) return qs::fail(QSIM_ERR_UNSUPPORTED, "qsim_traj_batch: 1 <= n_qubits <= 12");
  if (shots < 0 || n_ops < 0 || flips_per_shot < 0) return qs::fail(QSIM_ERR_ARG, "qsim_traj_batch: bad sizes");
  const uint64_t dim = 1ull << n_qubits;
  const QsTrajOp* op = (const QsTrajOp*)ops;
  std::vector<qs_c128> state(dim);
  for (int64_t shot = 0; shot < shots; ++shot) {
    memcpy(state.data(), psi0, sizeof(qs_c128) * dim);
    const uint8_t* fl = flips + shot * flips_per_shot;
    for (int o = 0; o < n_ops; ++o) {
      qs_c128 M[16];
      qs_traj_rows(op[o], matrices, fl, M);
      fl += 2 * op[o].k;
      qs_traj_apply(state.data(), n_qubits, op[o], M, 0, 1);
    }
    if (out_states) memcpy(out_states + 2 * (uint64_t)shot * dim, state.data(), sizeof(qs_c128) * dim);
    double fr = 0.0, fi = 0.0;
    for (uint64_t i = 0; i < dim; ++i) {
      const qs_c128 v = state[i];
      if (out_prob_sum) out_prob_sum[i] += v.x * v.x + v.y * v.y;
      if (observable) {
        const double wx = observable[2 * i], wy = observable[2 * i + 1];
        fr += wx * v.x + wy * v.y;
        fi += wx * v.y - wy * v.x;
      }
    }
    if (observable && out_fidelity) out_fidelity[shot] = fr * fr + fi * fi;
  }
  ++g_launches;
  return QSIM_OK;
}

static int swap_select(const char* who, int n_local, int nbits, const int* local_qubits, const int* bit_values,
                       uint64_t first, uint64_t count, QsBitSel* sel) {
  if (n_local < 1 || nbits < 1 || nbits > 8 || nbits > n_local || !local_qubits || !bit_values)
    return qs::fail(QSIM_ERR_ARG, std::string(who) + ": bad bit list");
  sel->k = nbits;
  for (int i = 0; i < nbits; ++i) {
    if (local_qubits[i] < 0 || local_qubits[i] >= n_local || (bit_values[i] | 1) != 1)
      return qs::fail(QSIM_ERR_ARG, std::string(who) + ": bad qubit or bit");
    sel->pos[i] = n_local - 1 - local_qubits[i];
    sel->val[i] = bit_values[i];
  }
  for (int i = 1; i < nbits; ++i)
    for (int j = i; j > 0 && sel->pos[j] < sel->pos[j - 1]; --j) {
      std::swap(sel->pos[j], sel->pos[j - 1]);
      std::swap(sel->val[j], sel->val[j - 1]);
    }
  for (int i = 1; i < nbits; ++i)
    if (sel->pos[i] == sel->pos[i - 1]) return qs::fail(QSIM_ERR_ARG, std::string(who) + ": repeated qubit");
  if (first + count > (1ull << (n_local - nbits)))
    return qs::fail(QSIM_ERR_ARG, std::string(who) + ": chunk out of range");
  return QSIM_OK;
}

int qsim_swap_pack(const void* shard, void* sendbuf, int n_local, int nbits, const int* local_qubits,
                   const int* bit_values, uint64_t first, uint64_t count, void*) {
  if (!shard || !sendbuf) return qs::fail(QSIM_ERR_ARG, "qsim_swap_pack: null argument");
  QsBitSel sel;
  const int rc = swap_select("qsim_swap_pack", n_local, nbits, local_qubits, bit_values, first, count, &sel);
  if (rc != QSIM_OK) return rc;
  const qs_c128* s = (const qs_c128*)shard;
  qs_c128* b = (qs_c128*)sendbuf;
  for (uint64_t r = 0; r < count; ++r) b[r] = s[qs_deposit(first + r, sel)];
  ++g_launches;
  return QSIM_OK;
}

int qsim_swap_unpack(void* shard, const void* recvbuf, int n_local, int nbits, const int* local_qubits,
                     const int* bit_values, uint64_t first, uint64_t count, void*) {
  if (!shard || !recvbuf) return qs::fail(QSIM_ERR_ARG, "qsim_swap_unpack: null argument");
  QsBitSel sel;
  const int rc = swap_select("qsim_swap_unpack", n_local, nbits, local_qubits, bit_values, first, count, &sel);
  if (rc != QSIM_OK) return rc;
  qs_c128* s = (qs_c128*)shard;
  const qs_c128* b = (const qs_c128*)recvbuf;
  for (uint64_t r = 0; r < count; ++r) s[qs_deposit(first + r, sel)] = b[r];
  ++g_launches;
  return QSIM_OK;
}

// Test-only: shared-memory wavefronts of the 128-bit step accesses of a plan, as the
// hardware serves them (8 lanes per wavefront; lanes conflict when their 16-byte slots
// are equal mod 8).  out[0] = wavefronts, out[1] = the conflict-free minimum.
int qsim_emu_step_wavefronts(const qsim_plan_t* p, double* out) {
  if (!p || !out) return qs::fail(QSIM_ERR_ARG, "qsim_emu_step_wavefronts: null argument");
  double total = 0, ideal = 0;
  int pass_no = 0;
  for (const qs::PlanItem& it : p->items) {
    if (it.generic) continue;
    const QsPass& P = it.pass;
    ++pass_no;
    for (int s = 0; s < (int)P.nsteps; ++s) {
      const double t_before = total, i_before = ideal;
      const QsStep& st = P.steps[s];
      QsStepTab tab;
      const uint32_t nthreads = 1u << P.cta_log2;
      for (int e = 0; e < QS_TAB_ENTRIES; ++e) qs_build_step_tab(P, s, e, &tab, P.cta_log2);
      const uint32_t nwork = 1u << (P.T - st.r);
      for (uint32_t warp = 0; warp < nthreads / 32; ++warp)
        for (uint32_t i = 0, w0 = warp * 32; w0 < nwork; ++i, w0 += nthreads)
          for (int m = 0; m < (1 << st.r); ++m)
            for (int quarter = 0; quarter < 4; ++quarter) {
              int count[8] = {0, 0, 0, 0, 0, 0, 0, 0}, worst = 0;
              for (int l = 0; l < 8; ++l) {
                const uint32_t tid = warp * 32 + quarter * 8 + l;
                if (tid + i * nthreads >= nwork) continue;
                const uint32_t jlo = qs_thread_jlo(tab, tid);
                const uint32_t slo = qs_swz(jlo);
                const uint32_t byte = ((slo ^ (st.hi[i] >> 16)) << 4) ^ st.sdepb[m];
                worst = std::max(worst, ++count[(byte >> 4) & 7u]);
              }
              total += worst;
              ideal += worst ? 1 : 0;
            }
      if (getenv("QSIM_EMU_VERBOSE") && total - t_before > 1.01 * (ideal - i_before)) {
        fprintf(stderr, "pass %d step %d r %d ratio %.2f gpos", pass_no, s, st.r, (total - t_before) / (ideal - i_before));
        for (int f = 0; f < st.r; ++f) fprintf(stderr, " %d", st.gpos[f]);
        fprintf(stderr, " fpos");
        for (int f = 0; f < (int)P.T - st.r; ++f) fprintf(stderr, " %d", st.fpos[f]);
        fprintf(stderr, " sync %d\n", st.block_sync);
      }
    }
  }
  out[0] = total;
  out[1] = ideal;
  return QSIM_OK;
}

// Test-only: per pass (steps, matrices, sign pairs) -> out[3 * pass + {0,1,2}]; returns passes.
int qsim_emu_plan_shape(const qsim_plan_t* p, int* out, int max_passes) {
  if (!p || !out) return -1;
  int k = 0;
  for (const qs::PlanItem& it : p->items) {
    if (it.generic || k >= max_passes) continue;
    int mats = 0;
    for (uint32_t l = 0; l < it.pass.nlayers; ++l) {
      const QsLayer& L = it.pass.layers[l];
      if (L.kind == QS_LAYER_DENSE) { ++mats; continue; }
      for (int f = 0; f < QS_MAX_R; ++f) mats += L.form[f] != QS_FORM_NONE ? 1 : 0;
    }
    out[3 * k] = (int)it.pass.nsteps;
    out[3 * k + 1] = mats;
    out[3 * k + 2] = (int)it.pass.npairs;
    ++k;
  }
  return k;
}

}  // extern "C"

// Test-only: byte offsets (inside the tile) that the 32 lanes of `warp` touch in the
// 128-bit access of amplitude m, iteration i, of step s of pass `pass_no` (0-based).
extern "C" int qsim_emu_step_lane_bytes(const qsim_plan_t* p, int pass_no, int s, int warp, int i, int m, int* out) {
  if (!p || !out) return -1;
  int k = 0;
  for (const qs::PlanItem& it : p->items) {
    if (it.generic) continue;
    if (k++ != pass_no) continue;
    const QsPass& P = it.pass;
    if (s >= (int)P.nsteps) return -2;
    const QsStep& st = P.steps[s];
    QsStepTab tab;
    for (int e = 0; e < QS_TAB_ENTRIES; ++e) qs_build_step_tab(P, s, e, &tab, P.cta_log2);
    for (int l = 0; l < 32; ++l) {
      const uint32_t tid = (uint32_t)warp * 32u + (uint32_t)l;
      const uint32_t slo = qs_swz(qs_thread_jlo(tab, tid));
      out[l] = (int)((((slo ^ (st.hi[i] >> 16)) << 4) ^ st.sdepb[m]));
    }
    return (int)st.r;
  }
  return -3;
}

// Test-only: print the shape of every pass of a plan (tile bits, steps, layers).
extern "C" int qsim_emu_plan_describe(const qsim_plan_t* p) {
  if (!p) return -1;
  int k = 0;
  for (const qs::PlanItem& it : p->items) {
    if (it.generic) { fprintf(stderr, "item %d: generic k=%d\n", k++, it.op.k); continue; }
    const QsPass& P = it.pass;
    fprintf(stderr, "pass %d: T=%u steps=%u layers=%u coef=%u pairs=%u final=%d tile_bits", k++, P.T, P.nsteps, P.nlayers,
            P.ncoef, P.npairs, P.has_final);
    for (uint32_t l = 0; l < P.T; ++l) fprintf(stderr, " %d", P.tile_bits[l]);
    fprintf(stderr, "\n");
    for (uint32_t s = 0; s < P.nsteps; ++s) {
      const QsStep& st = P.steps[s];
      fprintf(stderr, "   step %u: r=%d layers %d..%d sync=%d gpos", s, st.r, st.layer0, st.layer0 + st.nlayers - 1, st.block_sync);
      for (int f = 0; f < st.r; ++f) fprintf(stderr, " %d", st.gpos[f]);
      fprintf(stderr, " fpos");
      for (int f = 0; f < (int)P.T - st.r; ++f) fprintf(stderr, " %d", st.fpos[f]);
      fprintf(stderr, " kinds");
      for (int l = st.layer0; l < st.layer0 + st.nlayers; ++l) fprintf(stderr, " %d/%x", P.layers[l].kind, P.layers[l].flags);
      fprintf(stderr, "\n");
    }
  }
  return k;
}
