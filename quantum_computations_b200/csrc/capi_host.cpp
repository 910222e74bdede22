// Host-only part of the C ABI: error string, circuit container, plan compile.
// Shared verbatim by libqsim_b200.so (CUDA) and the host emulator of the tests.
#include <cmath>
#include <new>

#include "planner.h"

namespace qs {
const char* last_error();
}

extern "C" {

const char* qsim_last_error(void) { return qs::last_error(); }

int qsim_version(void) { return 101; }

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

}  // extern "C"
