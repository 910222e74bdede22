// HOST EMULATOR -- TEST INFRASTRUCTURE ONLY.
//
// Builds (g++ only, no CUDA) into tests/_build/libqsim_emu.so and exports the
// same C ABI as libqsim_b200.so, but on HOST pointers.  It links the very same
// C ABI layer (capi_host.cpp: argument checks, qubit conversion, host lowering),
// planner (planner.cpp, pauli.cpp) and per-thread phase functions (tile_exec.h,
// elem_ops.h) as the CUDA library; this file holds only the backend (backend.h),
// which loops over thread ids where the GPU runs them in parallel, and the
// functions that have no host equivalent.  The CPU test-suite uses it to check
// the plan logic and the index arithmetic without a GPU.  The product package
// never loads it: quantum_computations_b200.engine binds libqsim_b200.so only
// and raises when that library or a CUDA device is missing.
#include <algorithm>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <vector>

#include "backend.h"

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

}  // namespace

// =====================================================================================
// Backend of the compute entry points (backend.h; checks and lowering in capi_host.cpp):
// the per-thread bodies of the CUDA kernels, looped over the work items
// =====================================================================================
namespace qs::dev {

int execute_plan(const qsim_plan& p, qs_c128* state, int n, void*) {
  if (g_ownership_violations)
    return qs::fail(QSIM_ERR_UNSUPPORTED, "emulator: a warp-synchronised step reads another warp's amplitudes");
  for (const qs::PlanItem& it : p.items) {
    if (it.generic) {
      int rc = emu_generic(it.op, state, n);
      if (rc != QSIM_OK) return rc;
    } else {
      if ((int)it.pass.T > n) return qs::fail(QSIM_ERR_ARG, "pass tile larger than the state");
      emu_pass(it.pass, state, n);
      if (g_ownership_violations)
        return qs::fail(QSIM_ERR_UNSUPPORTED, "emulator: a warp-synchronised step reads another warp's amplitudes");
    }
  }
  return QSIM_OK;
}

int init_product(qs_c128* state, int n, const ProductAmps& amps, void*) {
  for (uint64_t i = 0; i < (1ull << n); ++i) state[i] = qs_product_amp(amps.a, n, i);
  ++g_launches;
  return QSIM_OK;
}

int measure_probs(const qs_c128* state, int pos, uint64_t pairs, const BraPair& bra0, const BraPair& bra1,
                  double* out_norm2, void*) {
  double p0 = 0.0, p1 = 0.0;
  for (uint64_t r = 0; r < pairs; ++r) {
    const qs_c128 u = qs_contract(state, pos, r, bra0.b), v = qs_contract(state, pos, r, bra1.b);
    p0 += u.x * u.x + u.y * u.y;
    p1 += v.x * v.x + v.y * v.y;
  }
  out_norm2[0] = p0;
  out_norm2[1] = p1;
  g_launches += 2;
  return QSIM_OK;
}

int collapse(const qs_c128* in, qs_c128* out, int pos, const BraPair& bra, double norm, uint64_t count, void*) {
  for (uint64_t r = 0; r < count; ++r) {
    qs_c128 v = qs_contract(in, pos, r, bra.b);
    v.x /= norm; v.y /= norm;
    out[r] = v;
  }
  ++g_launches;
  return QSIM_OK;
}

int insert(const qs_c128* in, qs_c128* out, int pos, const BraPair& amp, uint64_t count, void*) {
  for (uint64_t i = 0; i < count; ++i) out[i] = qs_insert_amp(in, pos, i, amp.b);
  ++g_launches;
  return QSIM_OK;
}

int reduce_norm2(const qs_c128* s, uint64_t n_amps, double* out, void*) {
  double acc = 0.0;
  for (uint64_t i = 0; i < n_amps; ++i) acc += s[i].x * s[i].x + s[i].y * s[i].y;
  *out = acc;
  g_launches += 2;
  return QSIM_OK;
}

int reduce_inner(const qs_c128* u, const qs_c128* v, uint64_t n_amps, double* out_re_im, void*) {
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

int reduce_expect(const qs_c128* k, const qs_c128* r, int n, double* out_re_im, void*) {
  const uint64_t dim = 1ull << n;
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

int reduce_purity(const qs_c128* r, int n, double* out_re_im, void*) {
  const uint64_t dim = 1ull << n;
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

int reduce_trace(const qs_c128* r, int n, double* out_re_im, void*) {
  const uint64_t dim = 1ull << n;
  double re = 0.0, im = 0.0;
  for (uint64_t i = 0; i < dim; ++i) { re += r[i * dim + i].x; im += r[i * dim + i].y; }
  out_re_im[0] = re;
  out_re_im[1] = im;
  g_launches += 2;
  return QSIM_OK;
}

// one launch per pass plus the final sum, as in the CUDA library
int expect_pauli(const qs_c128* s, int n, const PauliPlan& plan, int64_t, double* sums, void*) {
  const uint64_t count = 1ull << (n - plan.d);
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
  return QSIM_OK;
}

// one launch per pass, as in the CUDA library
int apply_pauli_rotations(qs_c128* s, int n, const PauliRotPlan& plan, void*) {
  const uint64_t count = 1ull << (n - plan.d);
  for (const QsPauliRotPass& P : plan.passes) {
    for (uint64_t o = 0; o < count; ++o) {
      switch (plan.d) {
        case 1: qs_pauli_rot_item<1>(P, s, o); break;
        case 2: qs_pauli_rot_item<2>(P, s, o); break;
        case 3: qs_pauli_rot_item<3>(P, s, o); break;
        default: qs_pauli_rot_item<4>(P, s, o); break;
      }
    }
    ++g_launches;
  }
  return QSIM_OK;
}

// one launch per pass, as in the CUDA library
int apply_pauli_sum(const qs_c128* in, qs_c128* out, int n, const PauliApplyPlan& plan, void*) {
  const uint64_t count = 1ull << (n - plan.d);
  double spec[2 << QS_PAULI_MAX_D];
  for (const QsPauliApplyPass& A : plan.passes) {
    for (uint64_t o = 0; o < count; ++o) {
      switch (plan.d) {
        case 1: qs_pauli_apply_item<1>(A, in, nullptr, out, o, spec, 1); break;
        case 2: qs_pauli_apply_item<2>(A, in, nullptr, out, o, spec, 1); break;
        case 3: qs_pauli_apply_item<3>(A, in, nullptr, out, o, spec, 1); break;
        default: qs_pauli_apply_item<4>(A, in, nullptr, out, o, spec, 1); break;
      }
    }
    ++g_launches;
  }
  return QSIM_OK;
}

// one launch per pass plus the final sum, as in the CUDA library
int lanczos_apply(const qs_c128* in, const qs_c128* prev, qs_c128* out, int n, const PauliApplyPlan& plan,
                  double* out_dot, void*) {
  const uint64_t count = 1ull << (n - plan.d);
  double spec[2 << QS_PAULI_MAX_D], dot = 0.0;
  for (const QsPauliApplyPass& A : plan.passes) {
    for (uint64_t o = 0; o < count; ++o) {
      switch (plan.d) {
        case 1: dot += qs_pauli_apply_item<1, true>(A, in, prev, out, o, spec, 1); break;
        case 2: dot += qs_pauli_apply_item<2, true>(A, in, prev, out, o, spec, 1); break;
        case 3: dot += qs_pauli_apply_item<3, true>(A, in, prev, out, o, spec, 1); break;
        default: dot += qs_pauli_apply_item<4, true>(A, in, prev, out, o, spec, 1); break;
      }
    }
    ++g_launches;
  }
  ++g_launches;                              // the final sum
  *out_dot = dot;
  return QSIM_OK;
}

// the step pass, and the final sum when the caller wants the norm, as in the CUDA library
int lanczos_step(qs_c128* w, const qs_c128* v, qs_c128* y, uint64_t n_amps, double a, double bre, double bim,
                 double* out_norm2, void*) {
  double acc = 0.0;
  for (uint64_t i = 0; i < n_amps; ++i) acc += qs_lanczos_step_elem(w, v, y, i, a, bre, bim);
  ++g_launches;
  if (out_norm2) {
    *out_norm2 = acc;
    ++g_launches;
  }
  return QSIM_OK;
}

// one launch per pass plus the final sum, as in the CUDA library
int pauli_rotations_adjoint(qs_c128* psi, qs_c128* lam, int n, const PauliRotPlan& plan, double* sums, void*) {
  const uint64_t count = 1ull << (n - plan.d);
  size_t row0 = 0;
  for (const QsPauliRotPass& P : plan.passes) {
    double acc[QS_PAULI_ROT_MAX] = {0.0};
    for (uint64_t o = 0; o < count; ++o) {
      switch (plan.d) {
        case 1: qs_pauli_adjoint_item<1>(P, psi, lam, o, acc, 1); break;
        case 2: qs_pauli_adjoint_item<2>(P, psi, lam, o, acc, 1); break;
        default: qs_pauli_adjoint_item<QS_PAULI_ADJ_MAX_D>(P, psi, lam, o, acc, 1); break;
      }
    }
    for (uint32_t r = 0; r < P.nrot; ++r) sums[2 * (row0 + r)] = acc[r];
    row0 += P.nrot;
    ++g_launches;
  }
  ++g_launches;                              // the final sum
  return QSIM_OK;
}

int expect_pauli_dm(const qs_c128* rho, int n, int64_t n_terms, const uint64_t* xi, const uint64_t* zi,
                    double* sums, void*) {
  for (int64_t t = 0; t < n_terms; ++t)
    for (uint64_t c = 0; c < (1ull << n); ++c) {
      const qs_c128 v = qs_pauli_dm_elem(rho, n, xi[t], zi[t], c);
      sums[2 * t] += v.x;
      sums[2 * t + 1] += v.y;
    }
  g_launches += 2;
  return QSIM_OK;
}

// The warp tasks of k_marginal one after the other, lane by lane, in the kernel's summation order
// (the lane shuffle tree and the final sum as qs_marg_final_ref): bit-identical to the GPU.
int marginal_probs(const QsProbSrc& src, const QsMargGeom& G, double* out, void*) {
  const QsProbFn prob{src};
  std::vector<double> partials;
  if (G.gs_bits) partials.assign((size_t)1 << (G.k + G.gs_bits), 0.0);
  double* dst = G.gs_bits ? partials.data() : out;
  uint64_t base = 0;
  for (uint64_t t = 0; t < G.ntasks; ++t) {
    double v[32];
    for (uint32_t l = 0; l < 32; ++l) v[l] = l < (uint32_t)G.lanes ? qs_marg_lane(G, prob, base, l) : 0.0;
    for (int b = 0; b < 5; ++b)
      if (G.lane_sum >> b & 1) {
        double o[32];
        for (int l = 0; l < 32; ++l) o[l] = v[l];
        for (int l = 0; l < 32; ++l) v[l] = o[l] + o[l ^ (1 << b)];
      }
    const uint64_t slot = qs_marg_task_slot(G, base);
    for (uint32_t l = 0; l < (uint32_t)G.lanes; ++l)
      if ((l & G.lane_sum) == 0) dst[G.lane_slot[l] + slot] = v[l];
    base = ((base | ~G.gmask) + 1) & G.gmask;
  }
  ++g_launches;
  if (G.gs_bits) {
    for (uint64_t b = 0; b < (1ull << G.k); ++b)
      out[b] = qs_marg_final_ref(partials.data() + (b << G.gs_bits), 1ull << G.gs_bits);
    ++g_launches;
  }
  return QSIM_OK;
}

// The six kernels of the CUDA sampler as host loops, with the same scans (qs_scan_ref) and the
// same inverse-CDF steps (qs_cdf_pick): the same uniforms give the same outcomes.  The bucketing of
// the shots by chunk and sub-tile only orders the work, so the loops here go shot by shot.
int sample(const QsProbSrc& src, int n, int64_t shots, const double* uniforms, uint64_t* out, double* total,
           unsigned char* ws, void*) {
  const QsSampleLayout L = qs_sample_layout(n, (uint64_t)shots);
  const uint64_t n_amps = 1ull << n, subs = 1ull << (QS_CHUNK_LOG2 - QS_SUB_LOG2);
  double* sub_mass = (double*)(ws + L.sub_mass);
  double* chunk_mass = (double*)(ws + L.chunk_mass);
  double* chunk_incl = (double*)(ws + L.chunk_incl);
  double* shot_t = (double*)(ws + L.shot_t);
  uint32_t* shot_chunk = (uint32_t*)(ws + L.shot_chunk);
  auto sub_probs = [&](uint64_t c, uint64_t s, double* p) {
    for (int e = 0; e < 256; ++e) {
      const uint64_t i = (c << QS_CHUNK_LOG2) | (s << QS_SUB_LOG2) | (uint64_t)e;
      p[e] = i < n_amps ? qs_prob_clamped(src, i) : 0.0;
    }
  };
  double p[256], incl[256];
  for (uint64_t c = 0; c < L.nchunks; ++c) {             // k_sample_masses
    for (uint64_t s = 0; s < subs; ++s) {
      sub_probs(c, s, p);
      qs_scan_ref(p, 256, 32, incl);
      sub_mass[c * subs + s] = incl[255];
    }
    qs_scan_ref(sub_mass + c * subs, subs, 32, incl);
    chunk_mass[c] = incl[255];
  }
  qs_scan_ref(chunk_mass, L.nchunks, 1024, chunk_incl);   // k_sample_scan
  const double tot = chunk_incl[L.nchunks - 1];
  *total = tot;
  g_launches += 6;
  if (!(tot > 0.0) || !std::isfinite(tot)) return QSIM_OK;
  const int K = (int)L.nchunks;
  for (int64_t i = 0; i < shots; ++i) {                    // k_sample_locate
    double t = uniforms[i] * tot;
    shot_chunk[i] = (uint32_t)qs_cdf_pick([&](int c) { return chunk_incl[c]; }, [&](int c) { return chunk_mass[c]; },
                                          K, &t);
    shot_t[i] = t;
  }
  uint64_t cached = ~0ull;
  double sub_incl[256];
  for (int64_t i = 0; i < shots; ++i) {                    // k_sample_resolve
    const uint64_t c = shot_chunk[i];
    const double* sm = sub_mass + c * subs;
    if (c != cached) { qs_scan_ref(sm, subs, 32, sub_incl); cached = c; }
    double t = shot_t[i];
    const int s = qs_cdf_pick([&](int j) { return sub_incl[j]; }, [&](int j) { return sm[j]; }, 256, &t);
    sub_probs(c, (uint64_t)s, p);
    qs_scan_ref(p, 256, 32, incl);
    const int j = qs_cdf_pick([&](int e) { return incl[e]; }, [&](int e) { return p[e]; }, 256, &t);
    out[i] = (c << QS_CHUNK_LOG2) | ((uint64_t)s << QS_SUB_LOG2) | (uint64_t)j;
  }
  return QSIM_OK;
}

int rb_batch(int nq, int64_t n_seq, const uint16_t* opcodes, const int64_t* offsets, const double* superops,
             const double* unitaries, const double* rho0, const double* psi0, double* out_fidelity,
             double* out_purity, double* out_rho, void*) {
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

int traj_batch(int n, int64_t shots, int n_ops, const QsTrajOp* op, const double* matrices, const uint8_t* flips,
               int64_t flips_per_shot, const qs_c128* psi0, const qs_c128* observable, double* out_fidelity,
               double* out_prob_sum, qs_c128* out_states, void*) {
  const uint64_t dim = 1ull << n;
  std::vector<qs_c128> state(dim);
  for (int64_t shot = 0; shot < shots; ++shot) {
    memcpy(state.data(), psi0, sizeof(qs_c128) * dim);
    const uint8_t* fl = flips + shot * flips_per_shot;
    for (int o = 0; o < n_ops; ++o) {
      qs_c128 M[16];
      qs_traj_rows(op[o], matrices, fl, M);
      fl += 2 * op[o].k;
      qs_traj_apply(state.data(), n, op[o], M, 0, 1);
    }
    if (out_states) memcpy(out_states + (uint64_t)shot * dim, state.data(), sizeof(qs_c128) * dim);
    double fr = 0.0, fi = 0.0;
    for (uint64_t i = 0; i < dim; ++i) {
      const qs_c128 v = state[i];
      if (out_prob_sum) out_prob_sum[i] += v.x * v.x + v.y * v.y;
      if (observable) {
        const qs_c128 w = observable[i];
        fr += w.x * v.x + w.y * v.y;
        fi += w.x * v.y - w.y * v.x;
      }
    }
    if (observable && out_fidelity) out_fidelity[shot] = fr * fr + fi * fi;
  }
  ++g_launches;
  return QSIM_OK;
}

int swap_pack(const qs_c128* shard, qs_c128* buf, const QsBitSel& sel, uint64_t first, uint64_t count, void*) {
  for (uint64_t r = 0; r < count; ++r) buf[r] = shard[qs_deposit(first + r, sel)];
  ++g_launches;
  return QSIM_OK;
}

int swap_unpack(qs_c128* shard, const qs_c128* buf, const QsBitSel& sel, uint64_t first, uint64_t count, void*) {
  for (uint64_t r = 0; r < count; ++r) shard[qs_deposit(first + r, sel)] = buf[r];
  ++g_launches;
  return QSIM_OK;
}

}  // namespace qs::dev

extern "C" {

int qsim_has_cuda(void) { return 0; }
int64_t qsim_launch_count(void) { return g_launches; }

// peer memory: the emulator has no IPC; its exchanges go through qsim_swap_pack / _unpack
int qsim_ipc_import(int, const unsigned char*, void**) { return qs::fail(QSIM_ERR_UNSUPPORTED, "no IPC in the host emulator"); }
int qsim_ipc_release(void*) { return QSIM_OK; }
int qsim_ipc_export_ex(void*, unsigned char*, uint64_t*) { return qs::fail(QSIM_ERR_UNSUPPORTED, "no IPC in the host emulator"); }
int qsim_exchange_p2p(void*, void* const*, int, int, const int*, const int*, const int*, void*) {
  return qs::fail(QSIM_ERR_UNSUPPORTED, "no peer memory in the host emulator (the exchange goes through send/recv)");
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
