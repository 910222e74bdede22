// Element-wise bodies of the non-tiled kernels, shared by the device kernels
// (grid-stride loops in kernels.cu) and the host emulator of the CPU tests.
// Bit convention: reference qubit q of an n-qubit register is index bit n-1-q.
#pragma once
#include <cmath>

#include "tile_exec.h"

QS_HD qs_c128 qs_cmul(qs_c128 a, qs_c128 b) {
  qs_c128 o;
  o.x = a.x * b.x - a.y * b.y;
  o.y = a.x * b.y + a.y * b.x;
  return o;
}

QS_HD uint64_t qs_insert_bit(uint64_t r, int pos, uint64_t bit) {
  const uint64_t low = r & ((1ull << pos) - 1ull);
  return ((r >> pos) << (pos + 1)) | (bit << pos) | low;
}

// Index of travelling amplitude r of a k-bit exchange: the k bits at positions pos[]
// (ascending) are fixed to val[], the other bits are r's, in order.
struct QsBitSel { int k; int pos[8]; int val[8]; };
QS_HD uint64_t qs_deposit(uint64_t r, const QsBitSel& sel) {
  for (int i = 0; i < sel.k; ++i) r = qs_insert_bit(r, sel.pos[i], (uint64_t)sel.val[i]);
  return r;
}

// parse_state for list[State] (DV/simulator.py:26): amplitude i of the product
// of n single-qubit kets; amps = n x 2 complex, qubit q first.
QS_HD qs_c128 qs_product_amp(const double* amps, int n, uint64_t i) {
  qs_c128 v; v.x = 1.0; v.y = 0.0;
  for (int q = 0; q < n; ++q) {
    const int bit = (int)((i >> (n - 1 - q)) & 1ull);
    qs_c128 a; a.x = amps[4 * q + 2 * bit]; a.y = amps[4 * q + 2 * bit + 1];
    v = qs_cmul(v, a);
  }
  return v;
}

// (I .. bra .. I) psi at reduced index r (DV/gates.py:173-181): bra is NOT conjugated.
QS_HD qs_c128 qs_contract(const qs_c128* in, int pos, uint64_t r, const double* bra) {
  const qs_c128 a0 = in[qs_insert_bit(r, pos, 0)];
  const qs_c128 a1 = in[qs_insert_bit(r, pos, 1)];
  qs_c128 o;
  o.x = bra[0] * a0.x - bra[1] * a0.y + bra[2] * a1.x - bra[3] * a1.y;
  o.y = bra[0] * a0.y + bra[1] * a0.x + bra[2] * a1.y + bra[3] * a1.x;
  return o;
}

// Insert.apply (DV/gates.py:145-153): out index i has the new qubit at bit `pos`.
QS_HD qs_c128 qs_insert_amp(const qs_c128* in, int pos, uint64_t i, const double* amp) {
  const uint64_t bit = (i >> pos) & 1ull;
  const uint64_t low = i & ((1ull << pos) - 1ull);
  const uint64_t r = ((i >> (pos + 1)) << pos) | low;
  qs_c128 a; a.x = amp[2 * bit]; a.y = amp[2 * bit + 1];
  return qs_cmul(in[r], a);
}

// Generic k-qubit matrix, out of place: out[i] = sum_c M[row(i), c] in[i with targets <- c].
// bits[f] = index bit of matrix factor f (f = 0 most significant).
QS_HD qs_c128 qs_generic_amp(const qs_c128* in, const double* mat, const int* bits, int k, uint64_t i) {
  const int dim = 1 << k;
  int row = 0;
  uint64_t cleared = i;
  for (int f = 0; f < k; ++f) {
    row |= (int)((i >> bits[f]) & 1ull) << (k - 1 - f);
    cleared &= ~(1ull << bits[f]);
  }
  double re = 0.0, im = 0.0;
  for (int c = 0; c < dim; ++c) {
    uint64_t src = cleared;
    for (int f = 0; f < k; ++f) src |= (uint64_t)((c >> (k - 1 - f)) & 1) << bits[f];
    const qs_c128 a = in[src];
    const double mr = mat[2 * (row * dim + c)], mi = mat[2 * (row * dim + c) + 1];
    re += mr * a.x - mi * a.y;
    im += mr * a.y + mi * a.x;
  }
  qs_c128 o; o.x = re; o.y = im;
  return o;
}

// One RB sequence (PAPER/randomised_benchmarking.py:65-75, DV part): vec(rho)
// times a dim^2 x dim^2 superoperator per opcode, ideal ket times a dim x dim
// unitary per opcode; then fidelity <psi|rho|psi> and purity tr(rho rho).
template <int DIM>
QS_HD void qs_rb_sequence(const uint16_t* codes, int64_t len, const double* superops,
                          const double* unitaries, const double* rho0, const double* psi0,
                          double* out_fid, double* out_pur, double* out_rho) {
  constexpr int D2 = DIM * DIM;
  qs_c128 rho[D2], psi[DIM];
  for (int e = 0; e < D2; ++e) { rho[e].x = rho0[2 * e]; rho[e].y = rho0[2 * e + 1]; }
  for (int e = 0; e < DIM; ++e) { psi[e].x = psi0[2 * e]; psi[e].y = psi0[2 * e + 1]; }
  for (int64_t t = 0; t < len; ++t) {
    const double* S = superops + (size_t)codes[t] * 2 * D2 * D2;
    const double* U = unitaries + (size_t)codes[t] * 2 * DIM * DIM;
    qs_c128 nr[D2];
    for (int r = 0; r < D2; ++r) {
      double re = 0.0, im = 0.0;
      for (int c = 0; c < D2; ++c) {
        const double mr = S[2 * (r * D2 + c)], mi = S[2 * (r * D2 + c) + 1];
        re += mr * rho[c].x - mi * rho[c].y;
        im += mr * rho[c].y + mi * rho[c].x;
      }
      nr[r].x = re; nr[r].y = im;
    }
    for (int e = 0; e < D2; ++e) rho[e] = nr[e];
    qs_c128 np_[DIM];
    for (int r = 0; r < DIM; ++r) {
      double re = 0.0, im = 0.0;
      for (int c = 0; c < DIM; ++c) {
        const double mr = U[2 * (r * DIM + c)], mi = U[2 * (r * DIM + c) + 1];
        re += mr * psi[c].x - mi * psi[c].y;
        im += mr * psi[c].y + mi * psi[c].x;
      }
      np_[r].x = re; np_[r].y = im;
    }
    for (int e = 0; e < DIM; ++e) psi[e] = np_[e];
  }
  // fidelity = Re sum_ij conj(psi_i) rho_ij psi_j  (npq.fidelity ket/matrix branch)
  double fid = 0.0;
  for (int i = 0; i < DIM; ++i)
    for (int j = 0; j < DIM; ++j) {
      const qs_c128 rp = qs_cmul(rho[i * DIM + j], psi[j]);
      fid += psi[i].x * rp.x + psi[i].y * rp.y;
    }
  // purity = Re tr(rho rho) = Re sum_ij rho_ij rho_ji
  double pur = 0.0;
  for (int i = 0; i < DIM; ++i)
    for (int j = 0; j < DIM; ++j) {
      const qs_c128 a = rho[i * DIM + j], b = rho[j * DIM + i];
      pur += a.x * b.x - a.y * b.y;
    }
  *out_fid = fid;
  *out_pur = pur;
  if (out_rho)
    for (int e = 0; e < D2; ++e) { out_rho[2 * e] = rho[e].x; out_rho[2 * e + 1] = rho[e].y; }
}


// ---- Pauli-trajectory batch (trajectories.py; mechanism of GKP/simulator.py:26-55 at the DV
//      level): one shot = the circuit on a small ket with, after every gate and on each of its
//      qubits, an X flip and then a Z flip where the shot's flip bits say so -------------------
// A gate of the shared circuit: k = 1 or 2 qubits on index bits b0 (matrix factor 0, the
// most significant bit of the row index) and b1; `mat` = offset of its row-major complex
// matrix in the matrix table (in complex numbers).
struct QsTrajOp { int32_t k, b0, b1, mat; };

// Row r of (Z^z X^x M): X on a qubit swaps the rows that differ in its bit, Z negates the
// rows where its bit is 1.  flips = {x0, z0[, x1, z1]} for the gate's qubits in order.
QS_HD void qs_traj_rows(const QsTrajOp& op, const double* mats, const uint8_t* flips, qs_c128* M) {
  const int dim = 1 << op.k;
  int xmask = 0, zmask = 0;
  for (int f = 0; f < op.k; ++f) {
    xmask |= (flips[2 * f] ? 1 : 0) << (op.k - 1 - f);
    zmask |= (flips[2 * f + 1] ? 1 : 0) << (op.k - 1 - f);
  }
  const double* src = mats + 2 * (size_t)op.mat;
  for (int r = 0; r < dim; ++r) {
    const double sgn = (qs_par((uint32_t)(r & zmask)) ? -1.0 : 1.0);
    for (int c = 0; c < dim; ++c) {
      M[r * dim + c].x = sgn * src[2 * ((r ^ xmask) * dim + c)];
      M[r * dim + c].y = sgn * src[2 * ((r ^ xmask) * dim + c) + 1];
    }
  }
}

// Work items tid, tid + nthreads, ... of one gate on the 2^n amplitudes in `state`.
QS_HD void qs_traj_apply(qs_c128* state, int n, const QsTrajOp& op, const qs_c128* M, uint32_t tid, uint32_t nthreads) {
  if (op.k == 1) {
    const uint64_t bit = 1ull << op.b0;
    for (uint64_t w = tid; w < (1ull << (n - 1)); w += nthreads) {
      const uint64_t i0 = qs_insert_bit(w, op.b0, 0);
      const qs_c128 a0 = state[i0], a1 = state[i0 | bit];
      qs_c128 o0, o1;
      o0.x = M[0].x * a0.x - M[0].y * a0.y + M[1].x * a1.x - M[1].y * a1.y;
      o0.y = M[0].x * a0.y + M[0].y * a0.x + M[1].x * a1.y + M[1].y * a1.x;
      o1.x = M[2].x * a0.x - M[2].y * a0.y + M[3].x * a1.x - M[3].y * a1.y;
      o1.y = M[2].x * a0.y + M[2].y * a0.x + M[3].x * a1.y + M[3].y * a1.x;
      state[i0] = o0;
      state[i0 | bit] = o1;
    }
  } else {
    const int lo = op.b0 < op.b1 ? op.b0 : op.b1, hi = op.b0 < op.b1 ? op.b1 : op.b0;
    for (uint64_t w = tid; w < (1ull << (n - 2)); w += nthreads) {
      const uint64_t base = qs_insert_bit(qs_insert_bit(w, lo, 0), hi, 0);
      uint64_t idx[4];
      qs_c128 a[4];
      for (int r = 0; r < 4; ++r) {
        idx[r] = base | ((uint64_t)((r >> 1) & 1) << op.b0) | ((uint64_t)(r & 1) << op.b1);
        a[r] = state[idx[r]];
      }
      for (int r = 0; r < 4; ++r) {
        double re = 0.0, im = 0.0;
        for (int c = 0; c < 4; ++c) {
          re += M[4 * r + c].x * a[c].x - M[4 * r + c].y * a[c].y;
          im += M[4 * r + c].x * a[c].y + M[4 * r + c].y * a[c].x;
        }
        state[idx[r]].x = re;
        state[idx[r]].y = im;
      }
    }
  }
}

// ---- Pauli-sum expectation values (qsim_expect_pauli, qsim_expect_pauli_dm; plan.h) --------
QS_HD uint32_t qs_par64(uint64_t v) {
#if defined(__CUDA_ARCH__)
  return (uint32_t)__popcll(v) & 1u;
#else
  return (uint32_t)__builtin_popcountll(v) & 1u;
#endif
}

// In-place Walsh-Hadamard transform: v[s] <- sum_m (-1)^popc(m & s) v[m].
template <int D>
QS_HD void qs_walsh(double* v) {
#pragma unroll
  for (int h = 0; h < D; ++h)
#pragma unroll
    for (int m = 0; m < (1 << D); ++m)
      if (!((m >> h) & 1)) {
        const double x = v[m], y = v[m | (1 << h)];
        v[m] = x + y;
        v[m | (1 << h)] = x - y;
      }
}

// One work item (outer index o) of a Pauli pass: acc[t * stride] += this item's share of term t;
// wal[k * stride], k < 2^(D+1), is the thread's spectrum scratch (Re, then Im).
// For a group, b[m] = a[m ^ xl] comes from a conditional swap per generator bit (uniform
// branches, so a[] and b[] stay in registers for any xl), and w[m] = conj(b[m]) a[m].  Summing
// over all m visits each pair (u, u ^ xl) from both ends: w[u ^ xl] = conj(w[u]) and the signs
// differ by (-1)^popc(x & z), so the real parts add up for an even popc(x & z) and the
// imaginary parts for an odd one -- the part the term takes -- while the other part cancels
// exactly by never being accumulated.
template <int D>
QS_HD void qs_pauli_item(const QsPauliPass& P, const qs_c128* __restrict__ state, uint64_t o, double* acc,
                         double* wal, uint32_t stride) {
  uint64_t base = o;
#pragma unroll
  for (int i = 0; i < D; ++i) base = qs_insert_bit(base, P.pivot[i], 0);
  qs_c128 a[1 << D];
#pragma unroll
  for (int m = 0; m < (1 << D); ++m) a[m] = state[base ^ P.off[m]];
  for (uint32_t g = 0; g < P.ngroups; ++g) {
    const QsPauliGroup G = P.groups[g];
    const uint32_t t1 = (uint32_t)G.first + G.count;
    qs_c128 b[1 << D];
#pragma unroll
    for (int m = 0; m < (1 << D); ++m) b[m] = a[m];
#pragma unroll
    for (int k = 0; k < D; ++k) {
      if ((G.xl >> k) & 1) {
#pragma unroll
        for (int m = 0; m < (1 << D); ++m)
          if (!((m >> k) & 1)) {
            const qs_c128 tmp = b[m];
            b[m] = b[m | (1 << k)];
            b[m | (1 << k)] = tmp;
          }
      }
    }
    if (G.parts & 1u) {
      double w[1 << D];
#pragma unroll
      for (int m = 0; m < (1 << D); ++m) w[m] = b[m].x * a[m].x + b[m].y * a[m].y;
      qs_walsh<D>(w);
#pragma unroll
      for (int m = 0; m < (1 << D); ++m) wal[m * stride] = w[m];
    }
    if (G.parts & 2u) {
      double w[1 << D];
#pragma unroll
      for (int m = 0; m < (1 << D); ++m) w[m] = b[m].x * a[m].y - b[m].y * a[m].x;
      qs_walsh<D>(w);
#pragma unroll
      for (int m = 0; m < (1 << D); ++m) wal[((1 << D) + m) * stride] = w[m];
    }
    for (uint32_t t = G.first; t < t1; ++t) {
      const uint32_t cls = P.cls[t];
      const double v = wal[((cls & 1u) << D | P.spec[t]) * stride];
      const uint32_t neg = qs_par64(base & P.z[t]) ^ (cls >> 1);
      acc[t * stride] += neg ? -v : v;
    }
  }
}

// Density matrix: entry c of tr(rho X^x Z^z) = sum_c (-1)^popc(c & z) rho[c, c ^ x] (the phase
// i^popc(x & z) is applied by the host).  rho is the row-major vec of an N-qubit matrix.
QS_HD qs_c128 qs_pauli_dm_elem(const qs_c128* __restrict__ rho, int N, uint64_t x, uint64_t z, uint64_t c) {
  qs_c128 v = rho[(c << N) | (c ^ x)];
  if (qs_par64(c & z)) { v.x = -v.x; v.y = -v.y; }
  return v;
}

// ---- measurement statistics (qsim_marginal_probs / qsim_sample and their _dm variants) ---------
// The probability of basis index i: |a[i]|^2 for a ket (stride 1), Re a[i * stride] for the vec of
// a density matrix (stride 2^N + 1 walks the diagonal).
struct QsProbSrc { const qs_c128* a; uint64_t stride; int dm; };
QS_HD double qs_prob(const QsProbSrc& s, uint64_t i) {
  const qs_c128 v = s.a[i * s.stride];
  return s.dm ? v.x : v.x * v.x + v.y * v.y;
}
// what sampling draws from: a negative diagonal entry (rounding) counts as 0
QS_HD double qs_prob_clamped(const QsProbSrc& s, uint64_t i) {
  const double p = qs_prob(s, i);
  return p > 0.0 ? p : 0.0;
}
struct QsProbFn {
  QsProbSrc s;
  QS_HD double operator()(uint64_t i) const { return qs_prob(s, i); }
};

// Bits of v deposited, lowest first, into the set bits of mask.
QS_HD uint64_t qs_deposit_mask(uint64_t v, uint64_t mask) {
  uint64_t out = 0;
  for (int b = 0; b < 64 && v; ++b)
    if (mask >> b & 1ull) { out |= (v & 1ull) << b; v >>= 1; }
  return out;
}

// Geometry of the marginal pass (built on the host, capi_host.cpp).  A warp task reads 32 lanes x
// nserial probabilities: index bits 0..4 are the lane number whatever they are (every warp load
// covers 512 contiguous bytes of a ket), the serial bits (rmask) are summed in registers and the
// task bits (gmask) number the tasks.  Lane bits that are summed bits reduce by a shuffle-xor tree
// (lane_sum); lane bits that are bin bits stay in separate lanes.  A task writes one value per bin
// of its lanes, into slot lane_slot[lane] + slot(task), slot(task) being the task bits looked up
// byte by byte in tab.  gs_bits == 0: the slot is the bin and the pass writes `out` itself.
// Otherwise a slot is (bin << gs_bits | g), g = the task's summed task bits, and a final kernel
// sums the 2^gs_bits partials of every bin in a fixed tree (qs_marg_final_ref).
constexpr int QS_MARG_TAB_BYTES = 5;         // task bits 5 .. 44
constexpr int QS_MARG_PARTIALS_LOG2 = 20;    // bins x partials per bin when gs_bits > 0
struct QsMargGeom {
  int32_t n, k, gs_bits, lanes;              // lanes = 2^min(n, 5)
  uint32_t lane_sum, pad;
  uint64_t rmask, gmask, nserial, ntasks;
  uint64_t lane_slot[32];
  uint64_t tab[QS_MARG_TAB_BYTES][256];
};

// Lane `lane`'s sum over the serial bits of the task at `base` (its task bits deposited): serial
// element e (ascending index) goes to accumulator e & 7, eight loads in flight, and the eight
// accumulators are added in a fixed tree.
template <class P>
QS_HD double qs_marg_lane(const QsMargGeom& G, const P& prob, uint64_t base, uint32_t lane) {
  double acc[8] = {0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0, 0.0};
  const uint64_t rm = G.rmask;
  uint64_t s = 0;                             // next serial bits: submasks of rm in ascending order
  if (G.nserial >= 8) {
    for (uint64_t e = 0; e < G.nserial; e += 8) {
      uint64_t idx[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) { idx[u] = base | s | lane; s = (s - rm) & rm; }
      double p[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) p[u] = prob(idx[u]);
#pragma unroll
      for (int u = 0; u < 8; ++u) acc[u] += p[u];
    }
  } else {
#pragma unroll
    for (int u = 0; u < 8; ++u)
      if ((uint64_t)u < G.nserial) { acc[u] += prob(base | s | lane); s = (s - rm) & rm; }
  }
  return ((acc[0] + acc[1]) + (acc[2] + acc[3])) + ((acc[4] + acc[5]) + (acc[6] + acc[7]));
}

QS_HD uint64_t qs_marg_task_slot(const QsMargGeom& G, uint64_t base) {
  const uint64_t t = base >> 5;
  uint64_t slot = 0;
  for (int b = 0; b < QS_MARG_TAB_BYTES; ++b) slot += G.tab[b][(t >> (8 * b)) & 255u];
  return slot;
}

// Inverse-CDF step of one level: the smallest s in [0, K) with X(s) > *t (binary search over the
// level's inclusive scan X), and *t becomes the target inside s.  An s with mass(s) == 0 can only
// come from rounding between differently ordered sums: then the next s with nonzero mass is taken
// and the target becomes 0 (its first nonzero entry).  With no such s (the target at or past the
// end of the scan, by rounding) the last s with nonzero mass is taken and the target becomes +inf
// (its last nonzero entry).  The parent has nonzero mass, so one of its parts has.
template <class FX, class FM>
QS_HD int qs_cdf_pick(const FX& X, const FM& mass, int K, double* t) {
  int lo = 0, hi = K;
  while (lo < hi) {
    const int mid = (lo + hi) >> 1;
    if (X(mid) > *t) hi = mid;
    else lo = mid + 1;
  }
  if (lo < K && mass(lo) > 0.0) {
    if (lo > 0) *t = *t - X(lo - 1);           // >= 0: X(lo - 1) <= *t
    return lo;
  }
  if (lo < K)
    for (int r = lo + 1; r < K; ++r)
      if (mass(r) > 0.0) { *t = 0.0; return r; }
  for (int r = K - 1; r >= 0; --r)
    if (mass(r) > 0.0) { *t = HUGE_VAL; return r; }
  *t = HUGE_VAL;
  return K - 1;
}

// Sampling: 256 amplitudes per sub-tile, 256 sub-tiles per chunk, up to 1024 shots per work item
// of the resolving kernel.  The caller's workspace (byte offsets, 256-aligned) holds per sub-tile
// and per chunk the masses, the chunk scan and the total, per chunk the shot counts, bucket ends and
// work-item offsets, and per shot its chunk, its target inside the chunk and its bucketed order.
constexpr int QS_SUB_LOG2 = 8, QS_CHUNK_LOG2 = 16, QS_SAMPLE_ITEM = 1024;
struct QsSampleLayout {
  uint64_t nchunks, sub_mass, chunk_mass, chunk_incl, total, counts, ends, items, shot_chunk, shot_t, order,
      bytes;
};
inline QsSampleLayout qs_sample_layout(int n, uint64_t shots) {
  QsSampleLayout L;
  L.nchunks = n > QS_CHUNK_LOG2 ? 1ull << (n - QS_CHUNK_LOG2) : 1ull;
  uint64_t off = 0;
  auto take = [&off](uint64_t bytes) { const uint64_t at = off; off += (bytes + 255ull) & ~255ull; return at; };
  L.sub_mass = take(8 * (L.nchunks << (QS_CHUNK_LOG2 - QS_SUB_LOG2)));
  L.chunk_mass = take(8 * L.nchunks);
  L.chunk_incl = take(8 * L.nchunks);
  L.total = take(8);
  L.counts = take(4 * L.nchunks);
  L.ends = take(4 * L.nchunks);
  L.items = take(4 * (L.nchunks + 1));
  L.shot_chunk = take(4 * shots);
  L.shot_t = take(8 * shots);
  L.order = take(4 * shots);
  L.bytes = off;
  return L;
}

// ---- host reference of the kernels' summation orders (the emulator runs these) ------------------
// Kogge-Stone inclusive scan of 32 values: what __shfl_up_sync gives lane by lane.
inline void qs_ks32(double* x) {
  for (int d = 1; d < 32; d <<= 1) {
    double o[32];
    for (int l = 0; l < 32; ++l) o[l] = x[l];
    for (int l = d; l < 32; ++l) x[l] = o[l] + o[l - d];
  }
}

// The library's inclusive scan of v[0 .. count) by `threads` threads (a multiple of 32, <= 1024):
// thread r sums its segment [r * seg, (r + 1) * seg) serially (seg = ceil(count / threads)), the
// thread totals are scanned by a Kogge-Stone tree inside each warp and the warp totals by the same
// tree, and element i of segment r is excl(r) + its serial prefix, with
// excl(r) = (warp's exclusive part) + (lane's exclusive part).
inline void qs_scan_ref(const double* v, uint64_t count, int threads, double* incl) {
  const uint64_t seg = (count + threads - 1) / threads;
  double li[1024], wt[32];
  for (int r = 0; r < threads; ++r) {
    double s = 0.0;
    for (uint64_t e = 0; e < seg; ++e)
      if (r * seg + e < count) s += v[r * seg + e];
    li[r] = s;
  }
  for (int w = 0; w < threads / 32; ++w) qs_ks32(li + 32 * w);
  for (int w = 0; w < 32; ++w) wt[w] = w < threads / 32 ? li[32 * w + 31] : 0.0;
  qs_ks32(wt);
  for (int r = 0; r < threads; ++r) {
    const int w = r >> 5, l = r & 31;
    const double ex = (w ? wt[w - 1] : 0.0) + (l ? li[r - 1] : 0.0);
    double s = 0.0;
    for (uint64_t e = 0; e < seg; ++e)
      if (r * seg + e < count) { s += v[r * seg + e]; incl[r * seg + e] = ex + s; }
  }
}

// out[bin] of the final marginal kernel: thread r of 256 sums the partials r, r + 256, ... serially,
// a shuffle-xor tree (16, 8, 4, 2, 1) combines each warp, and the 8 warp sums go in a fixed tree.
inline double qs_marg_final_ref(const double* row, uint64_t count) {
  double v[256], w[8];
  for (int r = 0; r < 256; ++r) {
    double s = 0.0;
    for (uint64_t i = r; i < count; i += 256) s += row[i];
    v[r] = s;
  }
  for (int off = 16; off > 0; off >>= 1) {
    double o[256];
    for (int r = 0; r < 256; ++r) o[r] = v[r];
    for (int r = 0; r < 256; ++r) v[r] = o[r] + o[r ^ off];
  }
  for (int i = 0; i < 8; ++i) w[i] = v[32 * i];
  return ((w[0] + w[1]) + (w[2] + w[3])) + ((w[4] + w[5]) + (w[6] + w[7]));
}
