// Host half of the Pauli-sum expectation values (qsim_expect_pauli / _dm), of H|psi>
// (qsim_apply_pauli_sum / qsim_accumulate_pauli_sum), of the Pauli-string rotations (qsim_apply_pauli_rotations / _dm) and of
// their adjoint sweep (qsim_pauli_rotations_adjoint / _dm): argument checks, the reference-qubit ->
// index-bit conversion and the packing of the terms into Pauli passes.  Shared verbatim by libqsim_b200.so
// and the host emulator, so the CPU tests check the very grouping the GPU runs.
#include <algorithm>
#include <cmath>
#include <cstring>
#include <map>

#include "planner.h"

namespace qs {

namespace {

// reference qubit q of an n-qubit register is index bit n-1-q
uint64_t to_index_bits(uint64_t m, int n) {
  uint64_t r = 0;
  for (int q = 0; q < n; ++q)
    if (m >> q & 1) r |= 1ull << (n - 1 - q);
  return r;
}

int popc64(uint64_t v) { return __builtin_popcountll(v); }

// Subspace spanned by a pass's generators, with the reduced basis that finds the pivots.
struct Span {
  int d = 0;
  uint64_t gen[QS_PAULI_MAX_D] = {0, 0, 0, 0};
  uint64_t red[QS_PAULI_MAX_D] = {0, 0, 0, 0};     // red[i] has pivot bit piv[i], no other pivot
  int piv[QS_PAULI_MAX_D] = {0, 0, 0, 0};

  uint64_t reduce(uint64_t v) const {
    for (int i = 0; i < d; ++i)
      if (v >> piv[i] & 1) v ^= red[i];
    return v;
  }
  bool contains(uint64_t v) const { return reduce(v) == 0; }
  void add(uint64_t v) {
    const uint64_t r = reduce(v);
    int p = 63;
    while (!(r >> p & 1)) --p;
    for (int i = 0; i < d; ++i)
      if (red[i] >> p & 1) red[i] ^= r;
    gen[d] = v;
    red[d] = r;
    piv[d] = p;
    ++d;
  }
  uint64_t off(int m) const {
    uint64_t o = 0;
    for (int i = 0; i < d; ++i)
      if (m >> i & 1) o ^= gen[i];
    return o;
  }
  int coords(uint64_t v) const {          // m with off(m) == v (v in the span)
    for (int m = 0; m < (1 << d); ++m)
      if (off(m) == v) return m;
    return -1;
  }
};

struct Chunk {                              // up to QS_PAULI_MAX_TERMS terms of one X mask
  uint64_t x;
  std::vector<int64_t> terms;
};

struct PassDraft {
  Span span;
  std::vector<const Chunk*> chunks;
  int nterms = 0;
};

}  // namespace

int check_pauli_args(const char* who, int n, int64_t n_terms, const uint64_t* x_masks, const uint64_t* z_masks,
                     const void* out) {
  if (n_terms < 0) return fail(QSIM_ERR_ARG, std::string(who) + ": n_terms < 0");
  if (n_terms == 0) return QSIM_OK;
  if (!x_masks || !z_masks || !out) return fail(QSIM_ERR_ARG, std::string(who) + ": null argument");
  if (n < 1 || n > 63) return fail(QSIM_ERR_ARG, std::string(who) + ": n_qubits must be in [1, 63]");
  const uint64_t limit = 1ull << n;
  for (int64_t t = 0; t < n_terms; ++t)
    if (x_masks[t] >= limit || z_masks[t] >= limit)
      return fail(QSIM_ERR_ARG, std::string(who) + ": a Pauli mask has a bit at or above n_qubits");
  return QSIM_OK;
}

void pauli_index_masks(int n, int64_t n_terms, const uint64_t* x_masks, const uint64_t* z_masks,
                       std::vector<uint64_t>* xi, std::vector<uint64_t>* zi, std::vector<uint8_t>* phase) {
  xi->resize((size_t)n_terms);
  zi->resize((size_t)n_terms);
  phase->resize((size_t)n_terms);
  for (int64_t t = 0; t < n_terms; ++t) {
    (*xi)[t] = to_index_bits(x_masks[t], n);
    (*zi)[t] = to_index_bits(z_masks[t], n);
    (*phase)[t] = (uint8_t)(popc64(x_masks[t] & z_masks[t]) & 3);
  }
}

int plan_pauli(int n, int64_t n_terms, const uint64_t* x_masks, const uint64_t* z_masks, PauliPlan* out) {
  std::vector<uint64_t> xi, zi;
  std::vector<uint8_t> phase;
  pauli_index_masks(n, n_terms, x_masks, z_masks, &xi, &zi, &phase);
  const int d = std::min(n, QS_PAULI_MAX_D);
  out->d = d;
  out->passes.clear();
  out->order.clear();

  // groups by X mask (ascending mask, terms in caller order), cut into chunks that fit a pass
  std::map<uint64_t, std::vector<int64_t>> groups;
  for (int64_t t = 0; t < n_terms; ++t) groups[xi[t]].push_back(t);
  std::vector<Chunk> chunks;
  for (const auto& kv : groups)
    for (size_t i = 0; i < kv.second.size(); i += QS_PAULI_MAX_TERMS) {
      Chunk c;
      c.x = kv.first;
      c.terms.assign(kv.second.begin() + i, kv.second.begin() + std::min(kv.second.size(), i + QS_PAULI_MAX_TERMS));
      chunks.push_back(std::move(c));
    }

  // Greedy packing.  Chunks with x != 0, widest X mask first: into the first pass whose span
  // holds x already, else into the first pass that can take x as another generator, else a new
  // pass.  Every pass thus opens for one chunk and there are at most as many passes as chunks
  // with x != 0.  The Z strings go where there is room, into a pass of their own only if none
  // has (or there is no other pass).
  std::vector<const Chunk*> order;
  for (const Chunk& c : chunks)
    if (c.x) order.push_back(&c);
  std::stable_sort(order.begin(), order.end(),
                   [](const Chunk* a, const Chunk* b) { return popc64(a->x) > popc64(b->x); });
  std::vector<PassDraft> drafts;
  for (const Chunk* c : order) {
    const int size = (int)c->terms.size();
    PassDraft* home = nullptr;
    for (PassDraft& p : drafts)
      if (p.nterms + size <= QS_PAULI_MAX_TERMS && p.span.contains(c->x)) { home = &p; break; }
    if (!home)
      for (PassDraft& p : drafts)
        if (p.nterms + size <= QS_PAULI_MAX_TERMS && p.span.d < d) { home = &p; break; }
    if (!home) {
      drafts.emplace_back();
      home = &drafts.back();
    }
    if (!home->span.contains(c->x)) home->span.add(c->x);
    home->chunks.push_back(c);
    home->nterms += size;
  }
  for (const Chunk& c : chunks) {
    if (c.x) continue;
    const int size = (int)c.terms.size();
    PassDraft* home = nullptr;
    for (PassDraft& p : drafts)
      if (p.nterms + size <= QS_PAULI_MAX_TERMS) { home = &p; break; }
    if (!home) {
      drafts.emplace_back();
      home = &drafts.back();
    }
    home->chunks.push_back(&c);
    home->nterms += size;
  }

  // descriptors: pad every span to d generators with single bits (more amplitudes per thread),
  // the highest index bits first so that the pivots stay high and neighbouring threads read
  // neighbouring amplitudes (coalesced); groups of a pass in ascending xl, terms of a group in
  // caller order
  uint32_t term0 = 0;
  for (PassDraft& p : drafts) {
    for (int b = n - 1; p.span.d < d && b >= 0; --b)
      if (!p.span.contains(1ull << b)) p.span.add(1ull << b);
    QsPauliPass P;
    memset(&P, 0, sizeof(P));
    P.d = (uint32_t)d;
    P.term0 = term0;
    int piv[QS_PAULI_MAX_D];
    for (int i = 0; i < d; ++i) piv[i] = p.span.piv[i];
    std::sort(piv, piv + d);
    for (int i = 0; i < d; ++i) P.pivot[i] = (uint8_t)piv[i];
    for (int m = 0; m < (1 << d); ++m) P.off[m] = p.span.off(m);
    std::vector<std::pair<int, const Chunk*>> by_xl;
    for (const Chunk* c : p.chunks) by_xl.emplace_back(p.span.coords(c->x), c);
    std::stable_sort(by_xl.begin(), by_xl.end(),
                     [](const std::pair<int, const Chunk*>& a, const std::pair<int, const Chunk*>& b) {
                       return a.first < b.first;
                     });
    uint32_t t = 0;
    for (size_t k = 0; k < by_xl.size(); ++k) {
      const int xl = by_xl[k].first;
      if (P.ngroups == 0 || P.groups[P.ngroups - 1].xl != xl) {
        P.groups[P.ngroups].xl = (uint8_t)xl;
        P.groups[P.ngroups].first = (uint8_t)t;
        ++P.ngroups;
      }
      for (int64_t term : by_xl[k].second->terms) {
        P.z[t] = zi[term];
        uint32_t spec = 0;
        for (int i = 0; i < d; ++i) spec |= (uint32_t)(popc64(P.off[1 << i] & zi[term]) & 1) << i;
        P.spec[t] = (uint8_t)spec;
        const int c = phase[term];
        P.cls[t] = (uint8_t)((c & 1) | ((c == 1 || c == 2) ? 2 : 0));
        P.groups[P.ngroups - 1].parts |= (uint8_t)((c & 1) ? 2 : 1);
        out->order.push_back(term);
        ++P.groups[P.ngroups - 1].count;
        ++t;
      }
    }
    P.nterms = t;
    term0 += t;
    out->passes.push_back(P);
  }
  return QSIM_OK;
}

int plan_pauli_apply(int n, int64_t n_terms, const uint64_t* x_masks, const uint64_t* z_masks,
                     const double* coeffs_re_im, bool accumulate, PauliApplyPlan* out) {
  // no terms: the layout of one identity term, and a pass without groups that writes the zeros
  const uint64_t none = 0;
  PauliPlan plan;
  const int rc = n_terms ? plan_pauli(n, n_terms, x_masks, z_masks, &plan) : plan_pauli(n, 1, &none, &none, &plan);
  if (rc != QSIM_OK) return rc;
  out->d = plan.d;
  out->passes.clear();
  for (const QsPauliPass& P : plan.passes) {
    QsPauliApplyPass A;
    memset(&A, 0, sizeof(A));
    A.p = P;
    A.accumulate = (accumulate || !out->passes.empty()) ? 1u : 0u;
    if (n_terms == 0) A.p.ngroups = A.p.nterms = 0;
    for (uint32_t t = 0; t < A.p.nterms; ++t) {
      const int64_t term = plan.order[P.term0 + t];
      const double re = coeffs_re_im[2 * term], im = coeffs_re_im[2 * term + 1];
      switch (popc64(x_masks[term] & z_masks[term]) & 3) {     // times i^popc(x & z)
        case 0: A.kre[t] = re; A.kim[t] = im; break;
        case 1: A.kre[t] = -im; A.kim[t] = re; break;
        case 2: A.kre[t] = -re; A.kim[t] = -im; break;
        default: A.kre[t] = im; A.kim[t] = -re; break;
      }
    }
    out->passes.push_back(A);
  }
  return QSIM_OK;
}

int plan_pauli_rotations(int n, int64_t n_rot, const uint64_t* x_masks, const uint64_t* z_masks, const double* angles,
                         bool dm, PauliRotPlan* out, bool adjoint) {
  // the rotations on the register, in caller order (an adjoint sweep: reverse caller order, negated
  // angles); a unit is what must share a pass (for a density matrix the row and the column half of
  // one caller rotation: they commute, and one pass holds both)
  struct Rot { uint64_t x, z; double theta; int cls; };
  const int nreg = dm ? 2 * n : n;
  std::vector<Rot> rots;
  std::vector<size_t> unit_end;
  out->caller.clear();
  out->weight.clear();
  for (int64_t i = 0; i < n_rot; ++i) {
    const int64_t t = adjoint ? n_rot - 1 - i : i;
    // the identity; a sweep keeps it, for its derivative
    if (angles[t] == 0.0 && !adjoint) continue;
    const double theta = adjoint ? -angles[t] : angles[t];
    const int c = popc64(x_masks[t] & z_masks[t]) & 3;
    const int cls = (c + 3) & 3;                       // -i i^c
    rots.push_back({to_index_bits(x_masks[t], nreg), to_index_bits(z_masks[t], nreg), theta, cls});
    // column half: conj(exp(-i theta/2 P)) = exp(+i theta/2 conj(P)) and conj(P) = (-1)^c P
    if (dm)
      rots.push_back({to_index_bits(x_masks[t] << n, nreg), to_index_bits(z_masks[t] << n, nreg),
                      (c & 1) ? theta : -theta, cls});
    unit_end.push_back(rots.size());
    if (adjoint) {
      // d/dtheta = d/dtheta_row + (+-1) d/dtheta_col, each half's overlap twice its derivative of
      // the linear Re<<lam|rho>>
      out->caller.push_back(t);
      out->weight.push_back(dm ? 0.5 : 1.0);
      if (dm) {
        out->caller.push_back(t);
        out->weight.push_back((c & 1) ? 0.5 : -0.5);
      }
    }
  }
  const int d = std::min(nreg, adjoint ? QS_PAULI_ADJ_MAX_D : QS_PAULI_MAX_D);
  out->d = d;
  out->passes.clear();

  // Greedy in caller order: a unit joins the open pass if the cap allows and its X masks lie in the
  // span or fit as further generators; otherwise it opens the next pass.
  struct Draft { Span span; size_t first, last; };
  std::vector<Draft> drafts;
  size_t begin = 0;
  for (size_t end : unit_end) {
    bool fits = !drafts.empty() && end - drafts.back().first <= QS_PAULI_ROT_MAX;
    Span grown;
    if (fits) {
      grown = drafts.back().span;
      for (size_t r = begin; r < end && fits; ++r)
        if (!grown.contains(rots[r].x)) {
          if (grown.d < d) grown.add(rots[r].x);
          else fits = false;
        }
    }
    if (fits) {
      drafts.back().span = grown;
      drafts.back().last = end;
    } else {
      Draft dr;
      for (size_t r = begin; r < end; ++r)
        if (!dr.span.contains(rots[r].x)) dr.span.add(rots[r].x);
      dr.first = begin;
      dr.last = end;
      drafts.push_back(dr);
    }
    begin = end;
  }

  // descriptors: spans padded and pivots chosen as in plan_pauli
  for (Draft& p : drafts) {
    for (int b = nreg - 1; p.span.d < d && b >= 0; --b)
      if (!p.span.contains(1ull << b)) p.span.add(1ull << b);
    QsPauliRotPass P;
    memset(&P, 0, sizeof(P));
    P.d = (uint32_t)d;
    int piv[QS_PAULI_MAX_D];
    for (int i = 0; i < d; ++i) piv[i] = p.span.piv[i];
    std::sort(piv, piv + d);
    for (int i = 0; i < d; ++i) P.pivot[i] = (uint8_t)piv[i];
    for (int m = 0; m < (1 << d); ++m) P.off[m] = p.span.off(m);
    for (size_t r = p.first; r < p.last; ++r) {
      const Rot& R = rots[r];
      const uint32_t k = P.nrot++;
      P.xl[k] = (uint8_t)p.span.coords(R.x);
      P.z[k] = R.z;
      uint32_t spec = 0;
      for (int i = 0; i < d; ++i) spec |= (uint32_t)(popc64(P.off[1 << i] & R.z) & 1) << i;
      P.spec[k] = (uint8_t)spec;
      P.cls[k] = (uint8_t)R.cls;
      P.c[k] = std::cos(0.5 * R.theta);
      P.s[k] = std::sin(0.5 * R.theta);
    }
    out->passes.push_back(P);
  }
  return QSIM_OK;
}

void pauli_finish(const PauliPlan& plan, const double* sums, double* out) {
  for (size_t s = 0; s < plan.order.size(); ++s) out[plan.order[s]] = sums[2 * s];
}

void pauli_adjoint_finish(const PauliRotPlan& plan, int64_t n_rot, const double* sums, double* out) {
  for (int64_t t = 0; t < n_rot; ++t) out[t] = 0.0;
  for (size_t s = 0; s < plan.caller.size(); ++s) out[plan.caller[s]] += plan.weight[s] * sums[2 * s];
}

void pauli_finish_dm(int64_t n_terms, const std::vector<uint8_t>& phase, const double* sums, double* out_re_im) {
  for (int64_t t = 0; t < n_terms; ++t) {
    const double re = sums[2 * t], im = sums[2 * t + 1];
    double* o = out_re_im + 2 * t;
    switch (phase[t]) {                      // times i^phase
      case 0: o[0] = re; o[1] = im; break;
      case 1: o[0] = -im; o[1] = re; break;
      case 2: o[0] = -re; o[1] = -im; break;
      default: o[0] = im; o[1] = -re; break;
    }
  }
}

}  // namespace qs
