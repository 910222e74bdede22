// The C ABI of include/qsim_b200.h apart from the peer, IPC and exchange functions: error
// string, circuit container, plan compile, and every compute entry point.  Shared verbatim by
// libqsim_b200.so (CUDA) and the host emulator of the tests.  Each compute entry point checks
// its arguments, turns reference qubits into index bits (qubit q of n is index bit n-1-q), does
// any lowering on the host and hands the rest to the backend (backend.h).
#include <algorithm>
#include <cmath>
#include <cstring>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "backend.h"

namespace qs {
const char* last_error();
}

namespace {

// One dense gate as a one-gate plan.
int one_gate(void* state, int n, const int* targets, int k, const double* matrix, void* stream) {
  qsim_circuit_t* c = nullptr;
  int rc = qsim_circuit_create(n, &c);
  if (rc != QSIM_OK) return rc;
  rc = qsim_circuit_add_matrix(c, k, targets, matrix);
  qsim_plan_t* p = nullptr;
  if (rc == QSIM_OK) rc = qsim_plan_compile(c, nullptr, &p);
  if (rc == QSIM_OK) rc = qsim_plan_execute(p, state, n, nullptr, stream);
  qsim_plan_destroy(p);
  qsim_circuit_destroy(c);
  return rc;
}

// Fills `sel` (positions ascending) from reference-style local qubit numbers.
int swap_select(const char* who, int n_local, int nbits, const int* local_qubits, const int* bit_values,
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
  for (int i = 1; i < nbits; ++i)                 // insertion sort by position
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

// Checks a marginal's arguments and lays out its pass (elem_ops.h, QsMargGeom): lanes take index
// bits 0..4; of the summed bits above them, the lowest are serial and the highest `gs` number the
// partials, gs chosen so that about 2^15 warp tasks exist and bins x partials stay within
// 2^QS_MARG_PARTIALS_LOG2 (k >= 20: no partials, the pass writes `out`).
int marginal_geom(const char* who, int n, int max_n, int k, const int* qubits, QsMargGeom* G) {
  const std::string w(who);
  if (n < 1 || n > max_n) return qs::fail(QSIM_ERR_ARG, w + ": n_qubits must be in [1, " + std::to_string(max_n) + "]");
  if (k < 0 || k > n) return qs::fail(QSIM_ERR_ARG, w + ": k must be in [0, n_qubits]");
  int binpos[64];
  for (int b = 0; b < 64; ++b) binpos[b] = -1;
  for (int j = 0; j < k; ++j) {
    if (qubits[j] < 0 || qubits[j] >= n) return qs::fail(QSIM_ERR_ARG, w + ": qubit out of range");
    const int bit = n - 1 - qubits[j];
    if (binpos[bit] >= 0) return qs::fail(QSIM_ERR_ARG, w + ": qubits must be distinct");
    binpos[bit] = k - 1 - j;                   // qubits[0] is the most significant bin bit
  }
  memset(G, 0, sizeof(*G));
  const int lane_log2 = n < 5 ? n : 5;
  G->n = n;
  G->k = k;
  G->lanes = 1 << lane_log2;
  int k_hi = 0, hs = 0, high_summed[64];
  for (int b = lane_log2; b < n; ++b) {
    if (binpos[b] >= 0) ++k_hi;
    else high_summed[hs++] = b;
  }
  int gs = std::min(hs, std::min(std::max(0, 15 - k_hi), 14));
  if (k + gs > QS_MARG_PARTIALS_LOG2) gs = std::max(0, QS_MARG_PARTIALS_LOG2 - k);
  G->gs_bits = gs;
  for (int i = 0; i < hs - gs; ++i) G->rmask |= 1ull << high_summed[i];
  for (int b = lane_log2; b < n; ++b)
    if (!(G->rmask >> b & 1)) G->gmask |= 1ull << b;
  G->nserial = 1ull << (hs - gs);
  G->ntasks = 1ull << (n - lane_log2 - (hs - gs));
  for (int b = 0; b < lane_log2; ++b)
    if (binpos[b] < 0) G->lane_sum |= 1u << b;
  for (int l = 0; l < G->lanes; ++l)
    for (int b = 0; b < lane_log2; ++b)
      if (binpos[b] >= 0 && (l >> b & 1)) G->lane_slot[l] += 1ull << (binpos[b] + gs);
  uint64_t contrib[64] = {0};                  // slot contribution of task bit b
  for (int b = lane_log2, g = 0; b < n; ++b) {
    if (binpos[b] >= 0) contrib[b] = 1ull << (binpos[b] + gs);
    else if (!(G->rmask >> b & 1)) contrib[b] = 1ull << g++;
  }
  for (int t = 0; t < QS_MARG_TAB_BYTES; ++t)
    for (int v = 0; v < 256; ++v)
      for (int i = 0; i < 8; ++i)
        if (v >> i & 1 && 5 + 8 * t + i < 64) G->tab[t][v] += contrib[5 + 8 * t + i];
  return QSIM_OK;
}

int marginal(const char* who, const void* state, int n, int max_n, int k, const int* qubits, double* out, bool dm,
             void* stream) {
  if (!state || !out || (k > 0 && !qubits)) return qs::fail(QSIM_ERR_ARG, std::string(who) + ": null argument");
  QsMargGeom G;
  const int rc = marginal_geom(who, n, max_n, k, qubits, &G);
  if (rc != QSIM_OK) return rc;
  const QsProbSrc src{(const qs_c128*)state, dm ? (1ull << n) + 1ull : 1ull, dm ? 1 : 0};
  return qs::dev::marginal_probs(src, G, out, stream);
}

int sample_bytes(const char* who, int n, int max_n, int64_t shots, uint64_t* bytes) {
  const std::string w(who);
  if (n < 1 || n > max_n) return qs::fail(QSIM_ERR_ARG, w + ": n_qubits must be in [1, " + std::to_string(max_n) + "]");
  if (shots < 0 || shots >= (1ll << 31)) return qs::fail(QSIM_ERR_ARG, w + ": shots must be in [0, 2^31)");
  *bytes = qs_sample_layout(n, (uint64_t)shots).bytes;
  return QSIM_OK;
}

int sample(const char* who, const void* state, int n, int max_n, int64_t shots, const double* uniforms, uint64_t* out,
           double* total, void* workspace, uint64_t workspace_bytes, bool dm, void* stream) {
  uint64_t need = 0;
  int rc = sample_bytes(who, n, max_n, shots, &need);
  if (rc != QSIM_OK || shots == 0) return rc;
  const std::string w(who);
  if (!state || !uniforms || !out || !total || !workspace) return qs::fail(QSIM_ERR_ARG, w + ": null argument");
  if (workspace_bytes < need)
    return qs::fail(QSIM_ERR_ARG, w + ": workspace too small (" + std::to_string(need) + " bytes needed)");
  const QsProbSrc src{(const qs_c128*)state, dm ? (1ull << n) + 1ull : 1ull, dm ? 1 : 0};
  double t = 0.0;
  rc = qs::dev::sample(src, n, shots, uniforms, out, &t, (unsigned char*)workspace, stream);
  if (rc != QSIM_OK) return rc;
  if (!(t > 0.0) || !std::isfinite(t)) return qs::fail(QSIM_ERR_ARG, w + ": the state has no probability mass");
  *total = t;
  return QSIM_OK;
}

}  // namespace

extern "C" {

const char* qsim_last_error(void) { return qs::last_error(); }

int qsim_version(void) { return 102; }

int qsim_circuit_create(int n_qubits, qsim_circuit_t** out) {
  if (!out) return qs::fail(QSIM_ERR_ARG, "qsim_circuit_create: out is null");
  if (n_qubits < 1 || n_qubits > 40)
    return qs::fail(QSIM_ERR_ARG, "qsim_circuit_create: n_qubits must be in [1, 40]");
  qsim_circuit* c = new (std::nothrow) qsim_circuit();
  if (!c) return qs::fail(QSIM_ERR_NOMEM, "out of host memory");
  c->n = n_qubits;
  *out = c;
  return QSIM_OK;
}

int qsim_circuit_add_matrix(qsim_circuit_t* c, int k, const int* targets, const double* matrix) {
  if (!c || !targets || !matrix) return qs::fail(QSIM_ERR_ARG, "qsim_circuit_add_matrix: null argument");
  if (k < 1 || k > 10 || k > c->n)
    return qs::fail(QSIM_ERR_ARG, "qsim_circuit_add_matrix: k must be in [1, min(10, n)]");
  qs::Op op;
  op.kind = qs::OP_DENSE;
  op.k = k;
  uint64_t seen = 0;
  for (int f = 0; f < k; ++f) {
    const int q = targets[f];
    if (q < 0 || q >= c->n) return qs::fail(QSIM_ERR_ARG, "qsim_circuit_add_matrix: target out of range");
    if (seen >> q & 1) return qs::fail(QSIM_ERR_ARG, "qsim_circuit_add_matrix: targets must be distinct");
    seen |= 1ull << q;
    op.bits.push_back(c->n - 1 - q);      // reference qubit q is index bit n-1-q
  }
  const int dim = 1 << k;
  op.mat.resize((size_t)dim * dim);
  bool diag = true;
  for (int e = 0; e < dim * dim; ++e) {
    const double re = matrix[2 * e], im = matrix[2 * e + 1];
    if (!std::isfinite(re) || !std::isfinite(im))
      return qs::fail(QSIM_ERR_ARG, "qsim_circuit_add_matrix: non-finite matrix entry");
    op.mat[e] = qs::cplx(re, im);
    if ((e / dim) != (e % dim) && (re != 0.0 || im != 0.0)) diag = false;
  }
  op.diag = diag;
  // CZ is recognised by value: it becomes a sign pair that costs no traffic.
  if (k == 2 && diag && op.mat[0] == qs::cplx(1, 0) && op.mat[5] == qs::cplx(1, 0) &&
      op.mat[10] == qs::cplx(1, 0) && op.mat[15] == qs::cplx(-1, 0)) {
    op.kind = qs::OP_SIGN;
    op.mat.clear();
  }
  c->ops.push_back(std::move(op));
  return QSIM_OK;
}

int qsim_circuit_add_many(qsim_circuit_t* c, int64_t count, const int32_t* ks, const int32_t* targets,
                          const double* matrices) {
  if (!c || count < 0 || (count > 0 && (!ks || !targets || !matrices)))
    return qs::fail(QSIM_ERR_ARG, "qsim_circuit_add_many: null argument");
  for (int64_t g = 0; g < count; ++g) {
    const int k = ks[g];
    const int rc = qsim_circuit_add_matrix(c, k, targets, matrices);
    if (rc != QSIM_OK) return rc;
    targets += k;
    matrices += (size_t)2 << (2 * k);
  }
  return QSIM_OK;
}

int qsim_circuit_num_ops(const qsim_circuit_t* c) { return c ? (int)c->ops.size() : 0; }

void qsim_circuit_destroy(qsim_circuit_t* c) { delete c; }

int qsim_plan_compile(const qsim_circuit_t* c, const qsim_plan_options_t* opt, qsim_plan_t** out) {
  if (!c || !out) return qs::fail(QSIM_ERR_ARG, "qsim_plan_compile: null argument");
  const qsim_plan_options_t o = qs::resolve_options(opt);
  qsim_plan* p = new (std::nothrow) qsim_plan();
  if (!p) return qs::fail(QSIM_ERR_NOMEM, "out of host memory");
  int rc;
  try {
    if (o.merge_1q == 1) {
      uint64_t apply_bits = 0;                       // option mask is by qubit; qubit q is index bit n-1-q
      for (int q = 0; q < c->n; ++q)
        if (o.apply_tail_mask >> q & 1) apply_bits |= 1ull << (c->n - 1 - q);
      std::vector<qs::Op> merged =
          qs::merge_single_qubit(c->n, c->ops, o.defer_tail == 1 ? &p->residual : nullptr, apply_bits);
      rc = qs::build_plan(c->n, merged, o, p);
    } else {
      rc = qs::build_plan(c->n, c->ops, o, p);
    }
  } catch (const std::bad_alloc&) {
    rc = qs::fail(QSIM_ERR_NOMEM, "out of host memory while planning");
  }
  if (rc != QSIM_OK) {
    delete p;
    return rc;
  }
  p->stats.n_input_ops = (int64_t)c->ops.size();
  *out = p;
  return QSIM_OK;
}

int qsim_plan_stats(const qsim_plan_t* p, qsim_plan_stats_t* out) {
  if (!p || !out) return qs::fail(QSIM_ERR_ARG, "qsim_plan_stats: null argument");
  *out = p->stats;
  return QSIM_OK;
}

int qsim_plan_residual(const qsim_plan_t* p, double* out) {
  if (!p || !out) return qs::fail(QSIM_ERR_ARG, "qsim_plan_residual: null argument");
  for (int q = 0; q < p->n; ++q) {
    double* dst = out + (size_t)8 * q;
    if (p->residual.empty()) {
      for (int e = 0; e < 8; ++e) dst[e] = 0.0;
      dst[0] = 1.0; dst[6] = 1.0;
    } else {
      const double* src = p->residual.data() + (size_t)8 * (p->n - 1 - q);   // qubit q is index bit n-1-q
      for (int e = 0; e < 8; ++e) dst[e] = src[e];
    }
  }
  return QSIM_OK;
}

void qsim_plan_destroy(qsim_plan_t* p) { delete p; }

int qsim_plan_execute(const qsim_plan_t* p, void* state, int n_qubits, void* /*scratch*/, void* stream) {
  if (!p || !state) return qs::fail(QSIM_ERR_ARG, "qsim_plan_execute: null argument");
  if (n_qubits != p->n) return qs::fail(QSIM_ERR_ARG, "qsim_plan_execute: plan was compiled for a different qubit count");
  return qs::dev::execute_plan(*p, (qs_c128*)state, n_qubits, stream);
}

int qsim_apply_matrix(void* state, int n_qubits, const int* targets, int k, const double* matrix,
                      void* /*scratch*/, void* stream) {
  if (!state || !targets || !matrix) return qs::fail(QSIM_ERR_ARG, "qsim_apply_matrix: null argument");
  return one_gate(state, n_qubits, targets, k, matrix, stream);
}

int qsim_apply_diagonal(void* state, int n_qubits, const int* targets, int k, const double* diag, void* stream) {
  if (!state || !targets || !diag) return qs::fail(QSIM_ERR_ARG, "qsim_apply_diagonal: null argument");
  if (k < 1 || k > QS_MAX_R) return qs::fail(QSIM_ERR_UNSUPPORTED, "qsim_apply_diagonal: k must be in [1, 4]");
  const int dim = 1 << k;
  std::vector<double> m(2 * (size_t)dim * dim, 0.0);
  for (int d = 0; d < dim; ++d) { m[2 * (d * dim + d)] = diag[2 * d]; m[2 * (d * dim + d) + 1] = diag[2 * d + 1]; }
  return one_gate(state, n_qubits, targets, k, m.data(), stream);
}

int qsim_apply_permutation(void* state, int n_qubits, const int* targets, int k, const int* perm, void* stream) {
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
  return one_gate(state, n_qubits, targets, k, m.data(), stream);
}

// vec(rho) is a 2n-qubit ket: row qubit q is qubit q, column qubit q is qubit q + n
int qsim_apply_superop(void* vec_rho, int n_qubits, const int* targets, int k, const double* superop,
                       void* /*scratch*/, void* stream) {
  if (!vec_rho || !targets || !superop) return qs::fail(QSIM_ERR_ARG, "qsim_apply_superop: null argument");
  if (k < 1 || 2 * k > 10) return qs::fail(QSIM_ERR_UNSUPPORTED, "qsim_apply_superop: k must be in [1, 5]");
  std::vector<int> t(2 * k);
  for (int i = 0; i < k; ++i) { t[i] = targets[i]; t[k + i] = targets[i] + n_qubits; }
  return one_gate(vec_rho, 2 * n_qubits, t.data(), 2 * k, superop, stream);
}

int qsim_init_product(void* state, int n_qubits, const double* amps, void* stream) {
  if (!state || !amps || n_qubits < 1 || n_qubits > 40) return qs::fail(QSIM_ERR_ARG, "qsim_init_product: bad argument");
  ProductAmps pa;
  memset(&pa, 0, sizeof(pa));
  memcpy(pa.a, amps, sizeof(double) * 4 * n_qubits);
  return qs::dev::init_product((qs_c128*)state, n_qubits, pa, stream);
}

int qsim_measure_probs(const void* state, int n_qubits, int qubit, const double* bra0, const double* bra1,
                       double* out_norm2, void* stream) {
  if (!state || !bra0 || !bra1 || !out_norm2) return qs::fail(QSIM_ERR_ARG, "qsim_measure_probs: null argument");
  if (n_qubits < 1 || qubit < 0 || qubit >= n_qubits) return qs::fail(QSIM_ERR_ARG, "qsim_measure_probs: qubit out of range");
  BraPair b0, b1;
  memcpy(b0.b, bra0, sizeof(b0.b));
  memcpy(b1.b, bra1, sizeof(b1.b));
  return qs::dev::measure_probs((const qs_c128*)state, n_qubits - 1 - qubit, 1ull << (n_qubits - 1), b0, b1,
                                out_norm2, stream);
}

int qsim_collapse(const void* in, void* out, int n_qubits, int qubit, const double* bra, double norm, void* stream) {
  if (!in || !out || !bra) return qs::fail(QSIM_ERR_ARG, "qsim_collapse: null argument");
  if (n_qubits < 1 || qubit < 0 || qubit >= n_qubits) return qs::fail(QSIM_ERR_ARG, "qsim_collapse: qubit out of range");
  BraPair b;
  memcpy(b.b, bra, sizeof(b.b));
  return qs::dev::collapse((const qs_c128*)in, (qs_c128*)out, n_qubits - 1 - qubit, b, norm, 1ull << (n_qubits - 1),
                           stream);
}

int qsim_insert(const void* in, void* out, int n_qubits, int position, const double* amp, void* stream) {
  if (!in || !out || !amp) return qs::fail(QSIM_ERR_ARG, "qsim_insert: null argument");
  if (n_qubits < 0 || position < 0 || position > n_qubits) return qs::fail(QSIM_ERR_ARG, "qsim_insert: position out of range");
  BraPair a;
  memcpy(a.b, amp, sizeof(a.b));
  // the new register has n+1 qubits; reference position p is index bit (n+1)-1-p
  return qs::dev::insert((const qs_c128*)in, (qs_c128*)out, n_qubits - position, a, 1ull << (n_qubits + 1), stream);
}

int qsim_reduce_norm2(const void* state, uint64_t n_amps, double* out, void* stream) {
  if (!state || !out) return qs::fail(QSIM_ERR_ARG, "qsim_reduce_norm2: null argument");
  return qs::dev::reduce_norm2((const qs_c128*)state, n_amps, out, stream);
}

int qsim_reduce_inner(const void* a, const void* b, uint64_t n_amps, double* out_re_im, void* stream) {
  if (!a || !b || !out_re_im) return qs::fail(QSIM_ERR_ARG, "qsim_reduce_inner: null argument");
  return qs::dev::reduce_inner((const qs_c128*)a, (const qs_c128*)b, n_amps, out_re_im, stream);
}

int qsim_reduce_expect(const void* ket, const void* rho, int n_qubits, double* out_re_im, void* stream) {
  if (!ket || !rho || !out_re_im || n_qubits < 0 || n_qubits > 20) return qs::fail(QSIM_ERR_ARG, "qsim_reduce_expect: bad argument");
  return qs::dev::reduce_expect((const qs_c128*)ket, (const qs_c128*)rho, n_qubits, out_re_im, stream);
}

int qsim_reduce_purity(const void* rho, int n_qubits, double* out_re_im, void* stream) {
  if (!rho || !out_re_im || n_qubits < 0 || n_qubits > 20) return qs::fail(QSIM_ERR_ARG, "qsim_reduce_purity: bad argument");
  return qs::dev::reduce_purity((const qs_c128*)rho, n_qubits, out_re_im, stream);
}

int qsim_reduce_trace(const void* rho, int n_qubits, double* out_re_im, void* stream) {
  if (!rho || !out_re_im || n_qubits < 0 || n_qubits > 20) return qs::fail(QSIM_ERR_ARG, "qsim_reduce_trace: bad argument");
  return qs::dev::reduce_trace((const qs_c128*)rho, n_qubits, out_re_im, stream);
}

int qsim_expect_pauli(const void* state, int n_qubits, int64_t n_terms, const uint64_t* x_masks,
                      const uint64_t* z_masks, double* out, void* stream) {
  int rc = qs::check_pauli_args("qsim_expect_pauli", n_qubits, n_terms, x_masks, z_masks, out);
  if (rc != QSIM_OK || n_terms == 0) return rc;
  if (!state) return qs::fail(QSIM_ERR_ARG, "qsim_expect_pauli: null state");
  qs::PauliPlan plan;
  std::vector<double> sums;
  try {
    rc = qs::plan_pauli(n_qubits, n_terms, x_masks, z_masks, &plan);
    sums.assign(2 * (size_t)n_terms, 0.0);
  } catch (const std::bad_alloc&) {
    rc = qs::fail(QSIM_ERR_NOMEM, "out of host memory while grouping the Pauli terms");
  }
  if (rc != QSIM_OK) return rc;
  rc = qs::dev::expect_pauli((const qs_c128*)state, n_qubits, plan, n_terms, sums.data(), stream);
  if (rc != QSIM_OK) return rc;
  qs::pauli_finish(plan, sums.data(), out);
  return QSIM_OK;
}

int qsim_expect_pauli_dm(const void* vec_rho, int n_qubits, int64_t n_terms, const uint64_t* x_masks,
                         const uint64_t* z_masks, double* out_re_im, void* stream) {
  int rc = qs::check_pauli_args("qsim_expect_pauli_dm", n_qubits, n_terms, x_masks, z_masks, out_re_im);
  if (rc != QSIM_OK || n_terms == 0) return rc;
  if (!vec_rho) return qs::fail(QSIM_ERR_ARG, "qsim_expect_pauli_dm: null state");
  if (n_qubits > 31) return qs::fail(QSIM_ERR_ARG, "qsim_expect_pauli_dm: n_qubits must be in [1, 31]");
  std::vector<uint64_t> xi, zi;
  std::vector<uint8_t> phase;
  qs::pauli_index_masks(n_qubits, n_terms, x_masks, z_masks, &xi, &zi, &phase);
  std::vector<double> sums(2 * (size_t)n_terms, 0.0);
  rc = qs::dev::expect_pauli_dm((const qs_c128*)vec_rho, n_qubits, n_terms, xi.data(), zi.data(), sums.data(), stream);
  if (rc != QSIM_OK) return rc;
  qs::pauli_finish_dm(n_terms, phase, sums.data(), out_re_im);
  return QSIM_OK;
}

int qsim_marginal_probs(const void* state, int n_qubits, int k, const int* qubits, double* out, void* stream) {
  return marginal("qsim_marginal_probs", state, n_qubits, 40, k, qubits, out, false, stream);
}

int qsim_marginal_probs_dm(const void* vec_rho, int n_qubits, int k, const int* qubits, double* out, void* stream) {
  return marginal("qsim_marginal_probs_dm", vec_rho, n_qubits, 31, k, qubits, out, true, stream);
}

int qsim_sample_workspace_bytes(int n_qubits, int64_t shots, uint64_t* out_bytes) {
  if (!out_bytes) return qs::fail(QSIM_ERR_ARG, "qsim_sample_workspace_bytes: null argument");
  return sample_bytes("qsim_sample_workspace_bytes", n_qubits, 40, shots, out_bytes);
}

int qsim_sample(const void* state, int n_qubits, int64_t shots, const double* uniforms, uint64_t* out, double* total,
                void* workspace, uint64_t workspace_bytes, void* stream) {
  return sample("qsim_sample", state, n_qubits, 40, shots, uniforms, out, total, workspace, workspace_bytes, false,
                stream);
}

int qsim_sample_dm(const void* vec_rho, int n_qubits, int64_t shots, const double* uniforms, uint64_t* out,
                   double* total, void* workspace, uint64_t workspace_bytes, void* stream) {
  return sample("qsim_sample_dm", vec_rho, n_qubits, 31, shots, uniforms, out, total, workspace, workspace_bytes, true,
                stream);
}

int qsim_rb_batch(int nq, int64_t n_seq, const uint16_t* opcodes, const int64_t* offsets, int n_opcodes,
                  const double* superops, const double* unitaries, const double* rho0, const double* psi0,
                  double* out_fidelity, double* out_purity, double* out_rho, void* stream) {
  if (!opcodes || !offsets || !superops || !unitaries || !rho0 || !psi0 || !out_fidelity || !out_purity)
    return qs::fail(QSIM_ERR_ARG, "qsim_rb_batch: null argument");
  if (nq < 1 || nq > 2) return qs::fail(QSIM_ERR_UNSUPPORTED, "qsim_rb_batch: nq must be 1 or 2");
  if (n_seq < 0 || n_opcodes < 1 || n_opcodes > 65536) return qs::fail(QSIM_ERR_ARG, "qsim_rb_batch: bad sizes");
  if (n_seq == 0) return QSIM_OK;
  return qs::dev::rb_batch(nq, n_seq, opcodes, offsets, superops, unitaries, rho0, psi0, out_fidelity, out_purity,
                           out_rho, stream);
}

int qsim_traj_batch(int n_qubits, int64_t shots, int n_ops, const int32_t* ops, const double* matrices,
                    const uint8_t* flips, int64_t flips_per_shot, const double* psi0, const double* observable,
                    double* out_fidelity, double* out_prob_sum, double* out_states, void* stream) {
  if (!ops || !matrices || !flips || !psi0) return qs::fail(QSIM_ERR_ARG, "qsim_traj_batch: null argument");
  if (n_qubits < 1 || n_qubits > 12) return qs::fail(QSIM_ERR_UNSUPPORTED, "qsim_traj_batch: 1 <= n_qubits <= 12");
  if (shots < 0 || n_ops < 0 || flips_per_shot < 0) return qs::fail(QSIM_ERR_ARG, "qsim_traj_batch: bad sizes");
  if (shots == 0) return QSIM_OK;
  return qs::dev::traj_batch(n_qubits, shots, n_ops, (const QsTrajOp*)ops, matrices, flips, flips_per_shot,
                             (const qs_c128*)psi0, (const qs_c128*)observable, out_fidelity, out_prob_sum,
                             (qs_c128*)out_states, stream);
}

int qsim_swap_pack(const void* shard, void* sendbuf, int n_local, int nbits, const int* local_qubits,
                   const int* bit_values, uint64_t first, uint64_t count, void* stream) {
  if (!shard || !sendbuf) return qs::fail(QSIM_ERR_ARG, "qsim_swap_pack: null argument");
  QsBitSel sel;
  const int rc = swap_select("qsim_swap_pack", n_local, nbits, local_qubits, bit_values, first, count, &sel);
  if (rc != QSIM_OK) return rc;
  return qs::dev::swap_pack((const qs_c128*)shard, (qs_c128*)sendbuf, sel, first, count, stream);
}

int qsim_swap_unpack(void* shard, const void* recvbuf, int n_local, int nbits, const int* local_qubits,
                     const int* bit_values, uint64_t first, uint64_t count, void* stream) {
  if (!shard || !recvbuf) return qs::fail(QSIM_ERR_ARG, "qsim_swap_unpack: null argument");
  QsBitSel sel;
  const int rc = swap_select("qsim_swap_unpack", n_local, nbits, local_qubits, bit_values, first, count, &sel);
  if (rc != QSIM_OK) return rc;
  return qs::dev::swap_unpack((qs_c128*)shard, (const qs_c128*)recvbuf, sel, first, count, stream);
}

}  // extern "C"
