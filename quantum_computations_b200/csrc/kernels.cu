// sm_100a kernels, the CUDA backend of the compute entry points (backend.h) and the peer, IPC and
// exchange functions of the C ABI (include/qsim_b200.h).
//
// Almost everything here is memory-bound complex128 work: TMA-staged 2^T-amplitude
// tiles in shared memory so that many gates apply per HBM pass, 16-byte (128-bit)
// accesses per amplitude, persistent grids sized to the SM count.  Tensor cores
// appear once: dense blocks on 5..10 qubits are FP64 MMAs (k_dense_block); tcgen05
// has no f64 kind and the 2x2 / 4x4 updates of the tile pass have no GEMM shape.
#include <cuda.h>
#include <cuda_runtime.h>
#include <cudaTypedefs.h>

#include <algorithm>

#include <atomic>
#include <cstdio>
#include <cstdlib>
#include <cstring>
#include <memory>
#include <mutex>
#include <new>
#include <string>
#include <utility>
#include <vector>

#include "backend.h"

namespace {

std::atomic<int64_t> g_launches{0};

struct DevCtx {
  std::once_flag once;
  int init_rc = 0;                // cudaError_t of the one-time initialisation
  int sms = 0;
  // scratch of the reductions: one set per device, serialised by reduce_lock (a reduction
  // synchronises its stream anyway, so concurrent callers lose nothing)
  std::mutex reduce_lock;
  double* d_partials = nullptr;   // [kReduceBlocks][2]
  double* d_out = nullptr;        // [2]
  double* h_out = nullptr;        // pinned [2]
  // scratch of the Pauli expectation values (qsim_expect_pauli / _dm), also under reduce_lock;
  // allocated at the first such call and grown when a call has more terms than any before
  double* d_pauli_partials = nullptr;   // [terms][blocks][2]
  double* d_pauli_sums = nullptr;       // [terms][2]
  double* h_pauli_sums = nullptr;       // pinned [terms][2]
  uint64_t* d_pauli_masks = nullptr;    // [terms][2] (density matrices: x, z)
  size_t pauli_partials_cap = 0, pauli_terms_cap = 0;
  // partials of the marginals with few bins (2^QS_MARG_PARTIALS_LOG2 doubles, allocated at the first
  // such call).  A marginal does not synchronise: the next one waits on the device for marg_done.
  std::mutex marg_lock;
  double* d_marg_partials = nullptr;
  cudaEvent_t marg_done = nullptr;
  std::mutex occ_lock;
  int occ[12] = {0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0, 0};   // resident CTAs/SM of the k_tile_pass variants at the last smem size
  int occ_smem = -1;
};

constexpr int kMaxDevices = 16;
constexpr int kReduceThreads = 256;
constexpr int kReduceBlocks = 148 * 8;
DevCtx g_ctx[kMaxDevices];

#define QS_CUDA(call)                                                                  \
  do {                                                                                 \
    cudaError_t e_ = (call);                                                           \
    if (e_ != cudaSuccess)                                                             \
      return qs::fail(QSIM_ERR_CUDA, std::string(#call) + ": " + cudaGetErrorString(e_)); \
  } while (0)

// Counts `n` kernel launches and reports a launch that failed.
int launched(int n = 1) {
  g_launches.fetch_add(n, std::memory_order_relaxed);
  QS_CUDA(cudaGetLastError());
  return QSIM_OK;
}

// The device a buffer lives on, made current for the lifetime of this object (the caller's
// current device is restored afterwards: torch keeps its own idea of it).
struct Bound {
  DevCtx* ctx = nullptr;
  int device = -1;
  int prev = -1;
  ~Bound() {
    if (prev >= 0 && prev != device) cudaSetDevice(prev);
  }
};

int bind_device(const void* ptr, Bound* b) {
  cudaPointerAttributes at;
  cudaError_t e = cudaPointerGetAttributes(&at, ptr);
  if (e != cudaSuccess) {
    cudaGetLastError();
    return qs::fail(QSIM_ERR_CUDA, std::string("cudaPointerGetAttributes: ") + cudaGetErrorString(e));
  }
  if (at.type != cudaMemoryTypeDevice && at.type != cudaMemoryTypeManaged)
    return qs::fail(QSIM_ERR_ARG, "buffer is not device memory (no CPU path exists in this library)");
  if (at.device < 0 || at.device >= kMaxDevices) return qs::fail(QSIM_ERR_ARG, "device index out of range");
  if (cudaGetDevice(&b->prev) != cudaSuccess) b->prev = -1;
  b->device = at.device;
  if (b->prev != at.device) QS_CUDA(cudaSetDevice(at.device));
  DevCtx& c = g_ctx[at.device];
  std::call_once(c.once, [&c, &at] {
    cudaDeviceProp prop;
    cudaError_t rc = cudaGetDeviceProperties(&prop, at.device);
    if (rc == cudaSuccess) c.sms = prop.multiProcessorCount;
    if (rc == cudaSuccess) rc = cudaMalloc(&c.d_partials, sizeof(double) * 2 * kReduceBlocks);
    if (rc == cudaSuccess) rc = cudaMalloc(&c.d_out, sizeof(double) * 2);
    if (rc == cudaSuccess) rc = cudaMallocHost(&c.h_out, sizeof(double) * 2);
    c.init_rc = (int)rc;
  });
  if (c.init_rc != 0)
    return qs::fail(QSIM_ERR_CUDA, std::string("device initialisation: ") + cudaGetErrorString((cudaError_t)c.init_rc));
  b->ctx = &c;
  return QSIM_OK;
}

// =====================================================================================
// Tile pass: the fused multi-gate kernel (plan.h / tile_exec.h)
// =====================================================================================
// TMA + mbarrier primitives (sm_90+ PTX; SASS: UTMALDG / UTMASTG / SYNCS).
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }
__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n"
      ".reg .pred p;\n"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
      "selp.u32 %0, 1, 0, p;\n"
      "}\n"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* map, const void* src, int c0, int c1, int c2, int c3,
                                             int c4) {
  asm volatile("cp.async.bulk.tensor.5d.global.shared::cta.tile.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];" ::"l"(map),
               "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
               : "memory");
}
__device__ __forceinline__ void tma_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_wait_read0() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }

// Box `o` of the tile at `base`: its tile positions P.. are the bits of o.
__device__ __forceinline__ void tma_box_coords(const QsPass& P, const QsTmaGeom& G, uint64_t base, int o, int* c) {
  uint64_t b = base;
  for (int q = 0; q < (int)P.T - G.P; ++q) b |= (uint64_t)((o >> q) & 1) << P.tile_bits[G.P + q];
  c[0] = (int)(((b >> G.shift[0]) & G.mask[0]) * 2);       // dimension 0 counts doubles
#pragma unroll
  for (int i = 1; i < 5; ++i) c[i] = (int)((b >> G.shift[i]) & G.mask[i]);
}

// One pass of the fused plan.  Persistent grid: every CTA loops over tiles; TMA brings a
// tile into shared memory (one mbarrier per CTA), the steps run on it, TMA writes it back.
// The three CTAs of an SM are in different phases, so one CTA's fill and drain overlap
// the steps of the other two.
// TL2 = log2 threads per CTA (QsPass::cta_log2): 128-thread CTAs run three (smem-limited) or four
// to an SM, 256-thread CTAs two (16 amplitudes per thread) or three (8 per thread).
template <int MAXR, int DENSE, int TL2>
__global__ void __launch_bounds__(1 << TL2, (TL2 == 7 ? (MAXR <= 3 ? 6 : 4) : (MAXR <= 3 ? 3 : 2)))
k_tile_pass(qs_c128* state, const __grid_constant__ QsPass P, const __grid_constant__ CUtensorMap tmap,
            const __grid_constant__ QsTmaGeom G, uint64_t ntiles) {
  extern __shared__ __align__(1024) unsigned char qs_smem[];
  qs_c128* tile = reinterpret_cast<qs_c128*>(qs_smem);
  __shared__ QsStepTab s_tab[QS_MAX_STEPS];
  __shared__ uint32_t s_zm[QS_MAX_LAYERS + 1];     // per layer qs_layer_z; [QS_MAX_LAYERS] = final g
  __shared__ __align__(8) uint64_t s_bar;
  const uint32_t tid = threadIdx.x;
  const int nsteps = (int)P.nsteps;
  const int nlayers = (int)P.nlayers;
  const bool use_tma = G.use_tma != 0;

  // tile-independent thread tables, once per launch (the grid is persistent)
  for (int e = (int)tid; e < nsteps * QS_TAB_ENTRIES; e += (1 << TL2))
    qs_build_step_tab(P, e / QS_TAB_ENTRIES, e % QS_TAB_ENTRIES, &s_tab[e / QS_TAB_ENTRIES], TL2);
  if (tid == 0) {
    mbar_init(&s_bar, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  __syncthreads();
  const uint32_t fin_qlo = P.has_final ? qs_fin_quad(P, qs_thread_jlo(s_tab[nsteps - 1], tid)) : 0u;
  uint32_t phase = 0;
  const uint32_t box_bytes = 16u << G.P;

  for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    uint64_t base = 0;
    if (!use_tma || tid < 96) base = qs_tile_base(P, t);
    if (use_tma) {
      if (tid < 32) {
        tma_wait_read0();                        // my stores of the previous tile have left the buffer
        __syncwarp();
        if (tid == 0) mbar_expect_tx(&s_bar, 16u << P.T);
        __syncwarp();
        for (int o = (int)tid; o < G.nops; o += 32) {
          int c[5];
          tma_box_coords(P, G, base, o, c);
          tma_load_5d(qs_smem + (size_t)o * box_bytes, &tmap, &s_bar, c[0], c[1], c[2], c[3], c[4]);
        }
      }
    } else {
      qs_plain_load(P, state, tile, base, tid, (1u << TL2));
    }
    // per-tile sign data, one thread per layer (warps 1 and 2)
    if (tid >= 32 && (int)tid < 32 + nlayers) {
      const int l = (int)tid - 32;
      if (P.layers[l].flags & QS_LF_SIGN) s_zm[l] = qs_layer_z(P, l, base);
    } else if (tid == 95 && P.has_final) {
      s_zm[QS_MAX_LAYERS] = qs_fin_g(P, base);
    }
    __syncthreads();
    if (use_tma) {
      while (!mbar_try_wait(&s_bar, phase)) {}
      phase ^= 1u;
    }
    const uint32_t fin_g = s_zm[QS_MAX_LAYERS];
    for (int s = 0; s < nsteps; ++s) {
      qs_phase_step_any<MAXR, DENSE>(P, s, tile, tid, TL2, s_zm, fin_g, fin_qlo, s_tab[s]);
      // the tile goes back through the async proxy: order this thread's writes before it
      if (s == nsteps - 1 && use_tma) fence_async_smem();
      // inside a run the next step touches only amplitudes of the same warp (plan.h)
      if (P.steps[s].block_sync) __syncthreads();
      else __syncwarp();
    }
    if (use_tma) {
      if (tid < 32) {
        for (int o = (int)tid; o < G.nops; o += 32) {
          int c[5];
          tma_box_coords(P, G, base, o, c);
          tma_store_5d(&tmap, qs_smem + (size_t)o * box_bytes, c[0], c[1], c[2], c[3], c[4]);
        }
        tma_commit();
      }
    } else {
      qs_plain_store(P, state, tile, base, tid, (1u << TL2));
      __syncthreads();
    }
  }
  if (use_tma && tid < 32) tma_wait_read0();
}

typedef void (*TileKernel)(qs_c128*, const QsPass, const CUtensorMap, const QsTmaGeom, uint64_t);

PFN_cuTensorMapEncodeTiled tensor_map_encoder() {
  static PFN_cuTensorMapEncodeTiled fn = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    cudaGetLastError();
    return (PFN_cuTensorMapEncodeTiled)p;
  }();
  return fn;
}

// Describe the state to TMA so that one box covers the lowest tile positions of the pass
// (plan.h, QsTmaGeom).  Dimension 0 is the index-bit range [0, cut1) with a box of bits
// 0..2 (one 128-byte row, the swizzle span); dimensions 1..4 start at the four lowest runs
// of tile bits above bit 2 (a run longer than 8 bits is cut: boxes are at most 256 wide).
// Returns use_tma = 0 when the pass has to use plain loads.
void make_tma_geom(const QsPass& P, qs_c128* state, int n, QsTmaGeom* G, CUtensorMap* map) {
  memset(G, 0, sizeof(*G));
  memset(map, 0, sizeof(*map));
  static const bool off = qs::dev_knob("QSIM_NO_TMA", 0) != 0;
  PFN_cuTensorMapEncodeTiled enc = tensor_map_encoder();
  const int T = (int)P.T;
  if (off || !enc || n < 12 || n > 40 || T < 6) return;
  if (P.tile_bits[0] != 0 || P.tile_bits[1] != 1 || P.tile_bits[2] != 2) return;
  bool is_tile[64] = {false};
  for (int l = 0; l < T; ++l) is_tile[P.tile_bits[l]] = true;
  int cuts[4], ncuts = 0;
  {
    int run = 0;
    for (int b = 3; b < n && ncuts < 4; ++b) {
      if (is_tile[b] && (run == 0 || run == 8)) { cuts[ncuts++] = b; run = 1; }
      else if (is_tile[b]) ++run;
      else run = 0;
    }
    for (int b = n - 1; b > 3 && ncuts < 4; --b) {     // fillers: any other positions
      bool used = false;
      for (int i = 0; i < ncuts; ++i) used |= cuts[i] == b;
      if (!used) cuts[ncuts++] = b;
    }
    if (ncuts != 4) return;
    std::sort(cuts, cuts + 4);
  }
  const int start[6] = {0, cuts[0], cuts[1], cuts[2], cuts[3], n};
  cuuint64_t gdim[5], gstride[4];
  cuuint32_t box[5], estr[5] = {1, 1, 1, 1, 1};
  int covered = 3;
  bool prefix = true;         // the box must cover the LOWEST tile positions, in order
  for (int i = 0; i < 5; ++i) {
    const int lo = start[i], hi = start[i + 1];
    if (hi - lo > 31) return;
    int nb = 0;
    if (i == 0) {
      nb = 3;
      for (int b = 3; b < hi; ++b)
        if (is_tile[b]) return;                        // cannot happen: cut 1 is the first tile bit above 2
    } else {
      if (prefix)
        while (lo + nb < hi && is_tile[lo + nb] && nb < 8) ++nb;
      for (int b = lo + nb; b < hi; ++b)
        if (is_tile[b]) prefix = false;
      covered += nb;
    }
    G->shift[i] = lo;
    G->mask[i] = (uint32_t)((1ull << (hi - lo)) - 1ull);
    gdim[i] = (1ull << (hi - lo)) * (i == 0 ? 2 : 1);
    box[i] = (1u << nb) * (i == 0 ? 2 : 1);
    if (i > 0) gstride[i - 1] = 16ull << lo;
  }
  if (covered < 6 || T - covered > 6) return;
  if (enc(map, CU_TENSOR_MAP_DATA_TYPE_FLOAT64, 5, state, gdim, gstride, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
          CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
          CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) != CUDA_SUCCESS)
    return;
  G->P = covered;
  G->nops = 1 << (T - covered);
  G->use_tma = 1;
}

int launch_pass(DevCtx* ctx, const QsPass& P, qs_c128* state, int n, cudaStream_t stream) {
  if ((int)P.T > n) return qs::fail(QSIM_ERR_ARG, "pass tile larger than the state");
  const uint64_t ntiles = 1ull << (n - (int)P.T);
  const int smem = (int)(sizeof(qs_c128) << P.T);
  int maxr = 1;
  bool dense = false;
  for (uint32_t s = 0; s < P.nsteps; ++s) maxr = P.steps[s].r > maxr ? P.steps[s].r : maxr;
  int dense_steps = 0;
  for (uint32_t s = 0; s < P.nsteps; ++s) dense_steps += P.layers[P.steps[s].layer0].kind == QS_LAYER_DENSE ? 1 : 0;
  dense = dense_steps > 0;
  // dense mode of the kernel (tile_exec.h, qs_phase_step_any): mostly dense steps -> all inline
  int dense_mode = dense_steps == 0 ? 0 : (2 * dense_steps > (int)P.nsteps ? 2 : 1);
  static const int force_dense = qs::dev_knob("QSIM_FORCE_DENSE_VARIANT", 0);
  if (force_dense == 1 || force_dense == 2) dense_mode = std::max(dense_mode, force_dense);   // development knob
  // [cta size][MAXR 3 / 4][dense mode 0 / 1 / 2]
  static const TileKernel variants[12] = {
      k_tile_pass<3, 0, 8>, k_tile_pass<3, 1, 8>, k_tile_pass<3, 2, 8>,
      k_tile_pass<4, 0, 8>, k_tile_pass<4, 1, 8>, k_tile_pass<4, 2, 8>,
      k_tile_pass<3, 0, 7>, k_tile_pass<3, 1, 7>, k_tile_pass<3, 2, 7>,
      k_tile_pass<4, 0, 7>, k_tile_pass<4, 1, 7>, k_tile_pass<4, 2, 7>};
  if (P.cta_log2 != QS_THREADS_LOG2_MIN && P.cta_log2 != QS_THREADS_LOG2)
    return qs::fail(QSIM_ERR_ARG, "pass built for an unsupported CTA size");
  const int threads = 1 << P.cta_log2;
  const int vi = (P.cta_log2 == QS_THREADS_LOG2 ? 0 : 6) + (maxr <= 3 ? 0 : 3) + dense_mode;
  int occ;
  {
    std::lock_guard<std::mutex> guard(ctx->occ_lock);
    if (ctx->occ_smem != smem) {
      for (int v = 0; v < 12; ++v) {
        QS_CUDA(cudaFuncSetAttribute(variants[v], cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
        QS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&ctx->occ[v], variants[v], v < 6 ? 256 : 128, smem));
      }
      ctx->occ_smem = smem;
    }
    occ = ctx->occ[vi];
  }
  if (occ < 1) return qs::fail(QSIM_ERR_CUDA, "tile pass does not fit on an SM");
  uint64_t grid = (uint64_t)ctx->sms * (uint64_t)occ;
  if (grid > ntiles) grid = ntiles;
  QsTmaGeom geom;
  CUtensorMap map;
  make_tma_geom(P, state, n, &geom, &map);
  variants[vi]<<<(unsigned)grid, threads, smem, stream>>>(state, P, map, geom, ntiles);
  return launched();
}

// =====================================================================================
// Simple streaming kernels
// =====================================================================================
__global__ void k_init_product(qs_c128* state, int n, const __grid_constant__ ProductAmps amps, uint64_t count) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < count;
       i += (uint64_t)gridDim.x * blockDim.x)
    state[i] = qs_product_amp(amps.a, n, i);
}

// n >= 16: the index splits into (o2 | o1 | tid) = (bits 16.., bits 8..15, bits 0..7) and the
// amplitude into three factors: one per thread (registers), a 256-entry table per block
// (shared memory) and one per o2 (uniform) -- two complex multiplications per amplitude
// instead of n, so the kernel runs at the HBM write rate.
__device__ __forceinline__ qs_c128 product_bits(const ProductAmps& amps, int n, uint32_t v, int first_bit, int nbits) {
  qs_c128 p; p.x = 1.0; p.y = 0.0;
  for (int b = 0; b < nbits; ++b) {
    const int q = n - 1 - (first_bit + b);
    const int bit = (int)((v >> b) & 1u);
    qs_c128 a; a.x = amps.a[4 * q + 2 * bit]; a.y = amps.a[4 * q + 2 * bit + 1];
    p = qs_cmul(p, a);
  }
  return p;
}

__global__ void __launch_bounds__(256) k_init_product_big(qs_c128* state, int n, const __grid_constant__ ProductAmps amps) {
  __shared__ qs_c128 t1[256];
  const uint32_t tid = threadIdx.x;
  const qs_c128 lo = product_bits(amps, n, tid, 0, 8);
  t1[tid] = product_bits(amps, n, tid, 8, 8);
  __syncthreads();
  const uint64_t n2 = 1ull << (n - 16);
  for (uint64_t o2 = blockIdx.x; o2 < n2; o2 += gridDim.x) {
    const qs_c128 pl = qs_cmul(product_bits(amps, n, (uint32_t)o2, 16, n - 16), lo);
    qs_c128* dst = state + (o2 << 16) + tid;
#pragma unroll 4
    for (uint32_t o1 = 0; o1 < 256; ++o1) dst[(uint64_t)o1 << 8] = qs_cmul(pl, t1[o1]);
  }
}

__global__ void k_collapse(const qs_c128* __restrict__ in, qs_c128* __restrict__ out, int pos,
                           BraPair bra, double norm, uint64_t count) {
  for (uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; r < count;
       r += (uint64_t)gridDim.x * blockDim.x) {
    qs_c128 v = qs_contract(in, pos, r, bra.b);
    v.x /= norm; v.y /= norm;
    out[r] = v;
  }
}

__global__ void k_insert(const qs_c128* __restrict__ in, qs_c128* __restrict__ out, int pos,
                         BraPair amp, uint64_t count) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < count;
       i += (uint64_t)gridDim.x * blockDim.x)
    out[i] = qs_insert_amp(in, pos, i, amp.b);
}

__global__ void k_swap_pack(const qs_c128* __restrict__ shard, qs_c128* __restrict__ buf, QsBitSel sel,
                            uint64_t first, uint64_t count) {
  for (uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; r < count;
       r += (uint64_t)gridDim.x * blockDim.x)
    buf[r] = shard[qs_deposit(first + r, sel)];
}

__global__ void k_swap_unpack(qs_c128* __restrict__ shard, const qs_c128* __restrict__ buf, QsBitSel sel,
                              uint64_t first, uint64_t count) {
  for (uint64_t r = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; r < count;
       r += (uint64_t)gridDim.x * blockDim.x)
    shard[qs_deposit(first + r, sel)] = buf[r];
}

// One k-qubit exchange as ONE kernel over NVLink peer memory: gather, transfer and scatter
// fused.  With k rank qubits trading places with k local qubits, rank R swaps, with each of the
// 2^k - 1 partners R ^ d, the block of its shard whose k local bits spell the PARTNER's rank
// bits against the partner's block whose local bits spell R's -- in place on both sides.
// Every pair of amplitudes is handled by exactly one of the two ranks (alternating 512-byte
// runs: the lower rank takes the even ones), which loads its own element and the partner's
// (P2P load), and stores them crosswise (P2P store): each element crosses NVLink once, is
// read from HBM once and written once, and no staging buffer exists.  The caller brackets the
// launch with two stream-ordered barriers over the ranks (sharded.py).
struct ExchGeom {
  int k, n_local;
  int pos[8];                 // local bit positions, ascending
  int mine[8];                // this rank's value of the rank bit traded against pos[i]
  qs_c128* peer[256];         // peer[d]: partner shard for the bit pattern d (over pos[] order); [0] unused
  unsigned char higher[256];  // higher[d] = 1 if this rank's number is above the partner's
  int chunk_log2;             // > 0: work is dealt to the partners in chunks of 2^chunk_log2 pairs (round robin),
                              // so that all 2^k - 1 partners are being talked to at any time; 0: partner after partner
};
constexpr int kExchSplitBit = 5;

// U pairs per thread and trip: all 2 U loads (U of them over NVLink) are issued before the
// first store, which is what keeps enough bytes in flight to cover the NVLink round trip.
template <int U>
__global__ void __launch_bounds__(256)
k_exchange_p2p(qs_c128* __restrict__ shard, const __grid_constant__ ExchGeom G) {
  const int k = G.k;
  const uint64_t half = 1ull << (G.n_local - k - 1);          // amplitudes per partner that THIS rank moves
  const uint64_t total = half * ((1ull << k) - 1ull);
  const uint64_t stride = (uint64_t)gridDim.x * blockDim.x * U;
  for (uint64_t w0 = (uint64_t)blockIdx.x * blockDim.x * U + threadIdx.x; w0 < total; w0 += stride) {
    qs_c128* mine[U];
    qs_c128* remote[U];
    qs_c128 x[U], y[U];
#pragma unroll
    for (int u = 0; u < U; ++u) {
      const uint64_t w = w0 + (uint64_t)u * blockDim.x;
      mine[u] = nullptr;
      if (w >= total) continue;
      int d;
      uint64_t q;
      if (G.chunk_log2 > 0) {
        const uint64_t chunk = w >> G.chunk_log2, nd = (1ull << k) - 1ull;
        d = 1 + (int)(chunk % nd);
        q = ((chunk / nd) << G.chunk_log2) | (w & ((1ull << G.chunk_log2) - 1ull));
      } else {
        d = 1 + (int)(w / half);
        q = w % half;
      }
      // r: index inside the block; bit kExchSplitBit says which of the two ranks moves it
      const uint64_t low = q & ((1ull << kExchSplitBit) - 1ull);
      const uint64_t r = ((q >> kExchSplitBit) << (kExchSplitBit + 1)) | ((uint64_t)G.higher[d] << kExchSplitBit) | low;
      uint64_t mine_idx = r, theirs_idx = r;
#pragma unroll 1
      for (int i = 0; i < k; ++i) {
        const uint64_t lo_m = mine_idx & ((1ull << G.pos[i]) - 1ull);
        const uint64_t lo_t = theirs_idx & ((1ull << G.pos[i]) - 1ull);
        const uint64_t vd = (uint64_t)(G.mine[i] ^ ((d >> i) & 1));    // partner's rank bit
        mine_idx = ((mine_idx >> G.pos[i]) << (G.pos[i] + 1)) | (vd << G.pos[i]) | lo_m;
        theirs_idx = ((theirs_idx >> G.pos[i]) << (G.pos[i] + 1)) | ((uint64_t)G.mine[i] << G.pos[i]) | lo_t;
      }
      mine[u] = shard + mine_idx;
      remote[u] = G.peer[d] + theirs_idx;
    }
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (mine[u]) { y[u] = *remote[u]; x[u] = *mine[u]; }
#pragma unroll
    for (int u = 0; u < U; ++u)
      if (mine[u]) { *remote[u] = x[u]; *mine[u] = y[u]; }
  }
}

unsigned stream_grid(const DevCtx* ctx, uint64_t count, int threads) {
  uint64_t blocks = (count + threads - 1) / threads;
  const uint64_t cap = (uint64_t)ctx->sms * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return (unsigned)blocks;
}

// =====================================================================================
// Reductions: fixed grid, fixed tree -> bit-reproducible results run to run
// =====================================================================================
struct FnNorm2 {
  const qs_c128* a;
  __device__ void operator()(uint64_t i, double& s0, double& s1) const {
    const qs_c128 v = a[i];
    s0 += v.x * v.x + v.y * v.y;
  }
};
struct FnInner {   // sum conj(a_i) b_i
  const qs_c128 *a, *b;
  __device__ void operator()(uint64_t i, double& s0, double& s1) const {
    const qs_c128 u = a[i], v = b[i];
    s0 += u.x * v.x + u.y * v.y;
    s1 += u.x * v.y - u.y * v.x;
  }
};
struct FnMeasure {  // s0 += |bra0 . pair|^2, s1 += |bra1 . pair|^2
  const qs_c128* a;
  int pos;
  BraPair b0, b1;
  __device__ void operator()(uint64_t r, double& s0, double& s1) const {
    const qs_c128 u = qs_contract(a, pos, r, b0.b);
    const qs_c128 v = qs_contract(a, pos, r, b1.b);
    s0 += u.x * u.x + u.y * u.y;
    s1 += v.x * v.x + v.y * v.y;
  }
};
struct FnExpect {   // sum_ij conj(k_i) rho_ij k_j ; element e = i * dim + j
  const qs_c128 *ket, *rho;
  int n;
  __device__ void operator()(uint64_t e, double& s0, double& s1) const {
    const uint64_t i = e >> n, j = e & ((1ull << n) - 1ull);
    const qs_c128 t = qs_cmul(rho[e], ket[j]);
    const qs_c128 k = ket[i];
    s0 += k.x * t.x + k.y * t.y;
    s1 += k.x * t.y - k.y * t.x;
  }
};
struct FnPurity {   // sum_ij rho_ij rho_ji
  const qs_c128* rho;
  int n;
  __device__ void operator()(uint64_t e, double& s0, double& s1) const {
    const uint64_t i = e >> n, j = e & ((1ull << n) - 1ull);
    const qs_c128 t = qs_cmul(rho[e], rho[(j << n) | i]);
    s0 += t.x;
    s1 += t.y;
  }
};
struct FnTrace {
  const qs_c128* rho;
  int n;
  __device__ void operator()(uint64_t i, double& s0, double& s1) const {
    const qs_c128 v = rho[(i << n) | i];
    s0 += v.x;
    s1 += v.y;
  }
};

__device__ __forceinline__ void block_reduce2(double& s0, double& s1) {
  __shared__ double w0[kReduceThreads / 32], w1[kReduceThreads / 32];
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) {
    s0 += __shfl_down_sync(0xffffffffu, s0, off);
    s1 += __shfl_down_sync(0xffffffffu, s1, off);
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  if (lane == 0) { w0[warp] = s0; w1[warp] = s1; }
  __syncthreads();
  if (warp == 0) {
    s0 = lane < kReduceThreads / 32 ? w0[lane] : 0.0;
    s1 = lane < kReduceThreads / 32 ? w1[lane] : 0.0;
#pragma unroll
    for (int off = 4; off > 0; off >>= 1) {
      s0 += __shfl_down_sync(0xffffffffu, s0, off);
      s1 += __shfl_down_sync(0xffffffffu, s1, off);
    }
  }
}

template <class F>
__global__ void __launch_bounds__(kReduceThreads) k_reduce(F f, uint64_t count, double* partials) {
  double s0 = 0.0, s1 = 0.0;
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < count;
       i += (uint64_t)gridDim.x * blockDim.x)
    f(i, s0, s1);
  block_reduce2(s0, s1);
  if (threadIdx.x == 0) { partials[2 * blockIdx.x] = s0; partials[2 * blockIdx.x + 1] = s1; }
}

__global__ void __launch_bounds__(kReduceThreads) k_reduce_final(const double* partials, int nblocks, double* out) {
  double s0 = 0.0, s1 = 0.0;
  for (int i = threadIdx.x; i < nblocks; i += blockDim.x) { s0 += partials[2 * i]; s1 += partials[2 * i + 1]; }
  block_reduce2(s0, s1);
  if (threadIdx.x == 0) { out[0] = s0; out[1] = s1; }
}

template <class F>
int reduce_to_host(DevCtx* ctx, F f, uint64_t count, double* out2, cudaStream_t stream) {
  uint64_t blocks = (count + kReduceThreads - 1) / kReduceThreads;
  if (blocks > (uint64_t)kReduceBlocks) blocks = kReduceBlocks;
  if (blocks < 1) blocks = 1;
  std::lock_guard<std::mutex> guard(ctx->reduce_lock);
  k_reduce<F><<<(unsigned)blocks, kReduceThreads, 0, stream>>>(f, count, ctx->d_partials);
  k_reduce_final<<<1, kReduceThreads, 0, stream>>>(ctx->d_partials, (int)blocks, ctx->d_out);
  int rc = launched(2);
  if (rc != QSIM_OK) return rc;
  QS_CUDA(cudaMemcpyAsync(ctx->h_out, ctx->d_out, 2 * sizeof(double), cudaMemcpyDeviceToHost, stream));
  QS_CUDA(cudaStreamSynchronize(stream));
  out2[0] = ctx->h_out[0];
  out2[1] = ctx->h_out[1];
  return QSIM_OK;
}

// =====================================================================================
// Pauli-sum expectation values (plan.h, elem_ops.h, pauli.cpp)
// =====================================================================================
constexpr int kPauliThreads = 64;         // 32 KiB of accumulators and spectra per CTA (static shared memory)
constexpr int kPauliBlocksPerSM = 5;       // 195 registers: 5 x 64 threads x 16 loads of 16 B in flight per SM
constexpr int kPauliDmBlocks = 64;         // per term

// Sum of col[0 .. kPauliThreads-1] in a fixed order (lane 0 of the calling warp holds it).
__device__ __forceinline__ double pauli_warp_sum(const double* col) {
  const int lane = threadIdx.x & 31;
  double s = col[lane];
#pragma unroll
  for (int k = 1; k < kPauliThreads / 32; ++k) s += col[lane + 32 * k];
#pragma unroll
  for (int off = 16; off > 0; off >>= 1) s += __shfl_down_sync(0xffffffffu, s, off);
  return s;
}

// One Pauli pass over a ket: every thread keeps one accumulator per term and its group spectra in
// shared memory ([entry][thread]: conflict-free), the block writes one partial per term.
template <int D>
__global__ void __launch_bounds__(kPauliThreads)
k_pauli_expect(const qs_c128* __restrict__ state, const __grid_constant__ QsPauliPass P, uint64_t count,
               double* __restrict__ partials) {
  __shared__ double acc[QS_PAULI_MAX_TERMS * kPauliThreads];
  __shared__ double wal[(2 << D) * kPauliThreads];
  for (uint32_t t = 0; t < P.nterms; ++t) acc[t * kPauliThreads + threadIdx.x] = 0.0;
  for (uint64_t o = blockIdx.x * (uint64_t)kPauliThreads + threadIdx.x; o < count;
       o += (uint64_t)gridDim.x * kPauliThreads)
    qs_pauli_item<D>(P, state, o, acc + threadIdx.x, wal + threadIdx.x, kPauliThreads);
  __syncthreads();
  const int warp = threadIdx.x >> 5;
  for (uint32_t t = warp; t < P.nterms; t += kPauliThreads / 32) {
    const double s = pauli_warp_sum(acc + t * kPauliThreads);
    if ((threadIdx.x & 31) == 0) {
      double* dst = partials + 2 * ((uint64_t)(P.term0 + t) * gridDim.x + blockIdx.x);
      dst[0] = s;
      dst[1] = 0.0;
    }
  }
}

// Density matrix: all terms in one launch, blockIdx.y strides over the terms, one thread per
// (term, c); masks = [term][x, z] in index bits.
__global__ void __launch_bounds__(kReduceThreads)
k_pauli_expect_dm(const qs_c128* __restrict__ rho, int N, const uint64_t* __restrict__ masks, int64_t n_terms,
                  double* __restrict__ partials) {
  const uint64_t dim = 1ull << N;
  for (int64_t t = blockIdx.y; t < n_terms; t += gridDim.y) {
    const uint64_t x = masks[2 * t], z = masks[2 * t + 1];
    double s0 = 0.0, s1 = 0.0;
    for (uint64_t c = blockIdx.x * (uint64_t)kReduceThreads + threadIdx.x; c < dim;
         c += (uint64_t)gridDim.x * kReduceThreads) {
      const qs_c128 v = qs_pauli_dm_elem(rho, N, x, z, c);
      s0 += v.x;
      s1 += v.y;
    }
    block_reduce2(s0, s1);
    if (threadIdx.x == 0) {
      double* dst = partials + 2 * ((uint64_t)t * gridDim.x + blockIdx.x);
      dst[0] = s0;
      dst[1] = s1;
    }
    __syncthreads();                       // block_reduce2's shared words are reused next term
  }
}

// sums[t] = partials[t][0] + ... + partials[t][nblocks - 1], fixed tree: bit-reproducible.
__global__ void __launch_bounds__(kReduceThreads)
k_pauli_final(const double* __restrict__ partials, int nblocks, int64_t n_terms, double* __restrict__ sums) {
  for (int64_t t = blockIdx.x; t < n_terms; t += gridDim.x) {
    const double* row = partials + 2 * (uint64_t)t * nblocks;
    double s0 = 0.0, s1 = 0.0;
    for (int i = threadIdx.x; i < nblocks; i += blockDim.x) { s0 += row[2 * i]; s1 += row[2 * i + 1]; }
    block_reduce2(s0, s1);
    if (threadIdx.x == 0) { sums[2 * t] = s0; sums[2 * t + 1] = s1; }
    __syncthreads();
  }
}

// Grows the per-device Pauli scratch (caller holds reduce_lock).  Growing frees the old
// buffers, which waits for the device: it happens only when a call has more terms than any before.
int pauli_scratch(DevCtx* ctx, size_t terms, size_t blocks) {
  const size_t partials = terms * blocks * 2;
  if (partials > ctx->pauli_partials_cap) {
    if (ctx->d_pauli_partials) QS_CUDA(cudaFree(ctx->d_pauli_partials));
    ctx->d_pauli_partials = nullptr;
    ctx->pauli_partials_cap = 0;
    QS_CUDA(cudaMalloc(&ctx->d_pauli_partials, sizeof(double) * partials));
    ctx->pauli_partials_cap = partials;
  }
  if (terms > ctx->pauli_terms_cap) {
    if (ctx->d_pauli_sums) QS_CUDA(cudaFree(ctx->d_pauli_sums));
    if (ctx->h_pauli_sums) QS_CUDA(cudaFreeHost(ctx->h_pauli_sums));
    if (ctx->d_pauli_masks) QS_CUDA(cudaFree(ctx->d_pauli_masks));
    ctx->d_pauli_sums = ctx->h_pauli_sums = nullptr;
    ctx->d_pauli_masks = nullptr;
    ctx->pauli_terms_cap = 0;
    QS_CUDA(cudaMalloc(&ctx->d_pauli_sums, sizeof(double) * 2 * terms));
    QS_CUDA(cudaMallocHost(&ctx->h_pauli_sums, sizeof(double) * 2 * terms));
    QS_CUDA(cudaMalloc(&ctx->d_pauli_masks, sizeof(uint64_t) * 2 * terms));
    ctx->pauli_terms_cap = terms;
  }
  return QSIM_OK;
}

// Final sum of a call's partials and the one download into `sums` (2 * n_terms doubles; the
// caller holds reduce_lock, which guards the pinned buffer too); synchronises the stream.
int pauli_sums_to_host(DevCtx* ctx, int64_t n_terms, int nblocks, double* sums, cudaStream_t stream) {
  const unsigned grid = (unsigned)std::min<int64_t>(n_terms, 65535);
  k_pauli_final<<<grid, kReduceThreads, 0, stream>>>(ctx->d_pauli_partials, nblocks, n_terms, ctx->d_pauli_sums);
  const int rc = launched();
  if (rc != QSIM_OK) return rc;
  QS_CUDA(cudaMemcpyAsync(ctx->h_pauli_sums, ctx->d_pauli_sums, sizeof(double) * 2 * n_terms, cudaMemcpyDeviceToHost,
                          stream));
  QS_CUDA(cudaStreamSynchronize(stream));
  memcpy(sums, ctx->h_pauli_sums, sizeof(double) * 2 * n_terms);
  return QSIM_OK;
}

template <int D>
void launch_pauli_pass(const QsPauliPass& P, const qs_c128* state, uint64_t count, unsigned blocks, double* partials,
                       cudaStream_t stream) {
  k_pauli_expect<D><<<blocks, kPauliThreads, 0, stream>>>(state, P, count, partials);
}

// =====================================================================================
// Pauli-string rotations (plan.h, elem_ops.h, pauli.cpp): one in-place pass per run of rotations
// =====================================================================================
// D = 4 takes 222 registers, so two 128-thread CTAs are resident per SM; measured (DESIGN.md section 5),
// one CTA per SM is 1.3x slower and 2, 4 or 8 are equal
constexpr int kRotThreads = 128;
constexpr int kRotBlocksPerSM = 4;

template <int D>
__global__ void __launch_bounds__(kRotThreads)
k_pauli_rotate(qs_c128* __restrict__ state, const __grid_constant__ QsPauliRotPass P, uint64_t count) {
  for (uint64_t o = blockIdx.x * (uint64_t)kRotThreads + threadIdx.x; o < count; o += (uint64_t)gridDim.x * kRotThreads)
    qs_pauli_rot_item<D>(P, state, o);
}

// =====================================================================================
// H|psi> for a Pauli sum and the adjoint sweep (plan.h, elem_ops.h, pauli.cpp)
// =====================================================================================
// The apply pass has the rotation pass's grid; every thread keeps its group spectrum in shared
// memory ([entry][thread]: conflict-free), where the terms scatter by a runtime index.
template <int D>
__global__ void __launch_bounds__(kRotThreads)
k_pauli_apply(const qs_c128* __restrict__ in, qs_c128* __restrict__ out, const __grid_constant__ QsPauliApplyPass A,
              uint64_t count) {
  __shared__ double spec[(2 << D) * kRotThreads];
  for (uint64_t o = blockIdx.x * (uint64_t)kRotThreads + threadIdx.x; o < count; o += (uint64_t)gridDim.x * kRotThreads)
    qs_pauli_apply_item<D>(A, in, out, o, spec + threadIdx.x, kRotThreads);
}

// One sweep pass: psi and lam together, one accumulator per rotation and thread in shared memory;
// the block writes one partial per rotation, to row row0 + r of the call's partials (k_pauli_final
// sums them as it sums the expectation values' terms).
constexpr int kAdjBlocksPerSM = 4;

template <int D>
__global__ void __launch_bounds__(kPauliThreads)
k_pauli_adjoint(qs_c128* __restrict__ psi, qs_c128* __restrict__ lam, const __grid_constant__ QsPauliRotPass P,
                uint64_t count, uint32_t row0, double* __restrict__ partials) {
  __shared__ double acc[QS_PAULI_ROT_MAX * kPauliThreads];
  for (uint32_t r = 0; r < P.nrot; ++r) acc[r * kPauliThreads + threadIdx.x] = 0.0;
  for (uint64_t o = blockIdx.x * (uint64_t)kPauliThreads + threadIdx.x; o < count;
       o += (uint64_t)gridDim.x * kPauliThreads)
    qs_pauli_adjoint_item<D>(P, psi, lam, o, acc + threadIdx.x, kPauliThreads);
  __syncthreads();
  const int warp = threadIdx.x >> 5;
  for (uint32_t r = warp; r < P.nrot; r += kPauliThreads / 32) {
    const double s = pauli_warp_sum(acc + r * kPauliThreads);
    if ((threadIdx.x & 31) == 0) {
      double* dst = partials + 2 * ((uint64_t)(row0 + r) * gridDim.x + blockIdx.x);
      dst[0] = s;
      dst[1] = 0.0;
    }
  }
}

// =====================================================================================
// Marginal probabilities (elem_ops.h, QsMargGeom): one read-only pass, then a fixed-tree final sum
// =====================================================================================
constexpr int kMargThreads = 256;
constexpr int kMargWarpsPerSM = 64;

// Warp w takes the tasks [w * per_warp, (w + 1) * per_warp): each lane sums its serial elements
// (qs_marg_lane), the summed lane bits reduce by shuffles, and the lanes that stand for a bin
// write it to dst (out, or the partials).
__global__ void __launch_bounds__(kMargThreads)
k_marginal(const __grid_constant__ QsMargGeom G, QsProbSrc src, double* __restrict__ dst, uint64_t per_warp) {
  const uint32_t lane = threadIdx.x & 31u;
  const uint64_t warp = (blockIdx.x * (uint64_t)kMargThreads + threadIdx.x) >> 5;
  const uint64_t t0 = warp * per_warp;
  if (t0 >= G.ntasks) return;
  const uint64_t t1 = t0 + per_warp < G.ntasks ? t0 + per_warp : G.ntasks;
  const bool active = lane < (uint32_t)G.lanes;
  const bool writer = active && (lane & G.lane_sum) == 0u;
  const uint64_t lslot = G.lane_slot[lane];
  const QsProbFn prob{src};
  uint64_t base = qs_deposit_mask(t0, G.gmask);
#pragma unroll 2
  for (uint64_t t = t0; t < t1; ++t) {
    double v = active ? qs_marg_lane(G, prob, base, lane) : 0.0;
#pragma unroll
    for (int b = 0; b < 5; ++b)
      if (G.lane_sum >> b & 1u) v += __shfl_xor_sync(0xffffffffu, v, 1 << b);
    if (writer) dst[lslot + qs_marg_task_slot(G, base)] = v;
    base = ((base | ~G.gmask) + 1ull) & G.gmask;
  }
}

// out[b] = the 2^gs_bits partials of bin b in the tree of qs_marg_final_ref.
__global__ void __launch_bounds__(256)
k_marg_final(const double* __restrict__ partials, int gs_bits, uint64_t bins, double* __restrict__ out) {
  __shared__ double w[8];
  const uint64_t per = 1ull << gs_bits;
  for (uint64_t b = blockIdx.x; b < bins; b += gridDim.x) {
    const double* row = partials + (b << gs_bits);
    double s = 0.0;
    for (uint64_t i = threadIdx.x; i < per; i += 256) s += row[i];
#pragma unroll
    for (int off = 16; off > 0; off >>= 1) s += __shfl_xor_sync(0xffffffffu, s, off);
    if ((threadIdx.x & 31u) == 0) w[threadIdx.x >> 5] = s;
    __syncthreads();
    if (threadIdx.x == 0) out[b] = ((w[0] + w[1]) + (w[2] + w[3])) + ((w[4] + w[5]) + (w[6] + w[7]));
    __syncthreads();
  }
}

// =====================================================================================
// Shot sampling: two-level inverse CDF (elem_ops.h: layout, qs_scan_ref orders, qs_cdf_pick)
// =====================================================================================
// Kogge-Stone inclusive scan over the lanes (qs_ks32).
__device__ __forceinline__ double warp_ks32(double x) {
  const int lane = threadIdx.x & 31;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const double y = __shfl_up_sync(0xffffffffu, x, d);
    if (lane >= d) x = x + y;
  }
  return x;
}

// qs_scan_ref(v, 256, 32): v[e] is at v[e + (e >> 3)] (padded: lane l reads its eight values
// without bank conflicts); incl[m] = inclusive value of element 8 * lane + m.
__device__ __forceinline__ void warp_scan256(const double* v, double incl[8]) {
  const int lane = threadIdx.x & 31;
  double s = 0.0;
#pragma unroll
  for (int m = 0; m < 8; ++m) { s += v[9 * lane + m]; incl[m] = s; }
  const double li = warp_ks32(s);
  double ex = __shfl_up_sync(0xffffffffu, li, 1);
  ex = 0.0 + (lane ? ex : 0.0);
#pragma unroll
  for (int m = 0; m < 8; ++m) incl[m] = ex + incl[m];
}

// The 256 probabilities of sub-tile (c, s) into the warp's padded buffer (coalesced loads).
__device__ __forceinline__ void load_sub(const QsProbSrc& src, uint64_t n_amps, uint64_t c, uint64_t s, double* pb) {
  const int lane = threadIdx.x & 31;
  const uint64_t base = (c << QS_CHUNK_LOG2) | (s << QS_SUB_LOG2);
  double p[8];
#pragma unroll
  for (int m = 0; m < 8; ++m) {
    const uint64_t i = base + (uint64_t)(32 * m + lane);
    p[m] = i < n_amps ? qs_prob_clamped(src, i) : 0.0;
  }
#pragma unroll
  for (int m = 0; m < 8; ++m) {
    const int e = 32 * m + lane;
    pb[e + (e >> 3)] = p[m];
  }
  __syncwarp();
}

// Pass 1: every sub-tile's mass and every chunk's mass (the totals of their qs_scan_ref scans).
__global__ void __launch_bounds__(256)
k_sample_masses(QsProbSrc src, uint64_t n_amps, uint64_t nchunks, double* __restrict__ sub_mass,
                double* __restrict__ chunk_mass) {
  __shared__ double pb[8][288];
  __shared__ double sm[288];
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5;
  double incl[8];
  for (uint64_t c = blockIdx.x; c < nchunks; c += gridDim.x) {
    for (int s = w; s < 256; s += 8) {
      load_sub(src, n_amps, c, (uint64_t)s, pb[w]);
      warp_scan256(pb[w], incl);
      if (lane == 31) { sub_mass[(c << 8) + s] = incl[7]; sm[s + (s >> 3)] = incl[7]; }
      __syncwarp();
    }
    __syncthreads();
    if (w == 0) {
      warp_scan256(sm, incl);
      if (lane == 31) chunk_mass[c] = incl[7];
    }
    __syncthreads();
  }
}

// Pass 2 (one CTA of 1024): the chunk scan qs_scan_ref(chunk_mass, nchunks, 1024) and the total.
__global__ void __launch_bounds__(1024)
k_sample_scan(const double* __restrict__ cm, uint64_t count, double* __restrict__ incl, double* __restrict__ total) {
  __shared__ double wt[32];
  const int r = threadIdx.x, lane = r & 31, w = r >> 5;
  const uint64_t seg = (count + 1023) / 1024;
  double s = 0.0;
  for (uint64_t e = 0; e < seg; ++e)
    if (r * seg + e < count) s += cm[r * seg + e];
  const double li = warp_ks32(s);
  if (lane == 31) wt[w] = li;
  __syncthreads();
  if (w == 0) {
    const double x = warp_ks32(wt[lane]);
    wt[lane] = x;
  }
  __syncthreads();
  double lex = __shfl_up_sync(0xffffffffu, li, 1);
  const double ex = (w ? wt[w - 1] : 0.0) + (lane ? lex : 0.0);
  s = 0.0;
  for (uint64_t e = 0; e < seg; ++e) {
    const uint64_t i = r * seg + e;
    if (i < count) {
      s += cm[i];
      incl[i] = ex + s;
      if (i == count - 1) *total = ex + s;
    }
  }
}

__device__ __forceinline__ bool sample_total_ok(double t) { return t > 0.0 && t < HUGE_VAL; }

// atomicAdd(counter, 1) for every calling lane, one atomic per distinct counter in the warp: a
// concentrated distribution sends all shots to one counter, and same-address atomics serialise.
// Returns the lane's old value (its slot).
__device__ __forceinline__ uint32_t warp_claim(uint32_t* counter) {
  const unsigned peers = __match_any_sync(__activemask(), (unsigned long long)counter);
  const int lane = threadIdx.x & 31, leader = __ffs(peers) - 1;
  uint32_t base = 0;
  if (lane == leader) base = atomicAdd(counter, (uint32_t)__popc(peers));
  base = __shfl_sync(peers, base, leader);
  return base + (uint32_t)__popc(peers & ((1u << lane) - 1u));
}

// Pass 3: every shot's chunk (first inverse-CDF level) and its target inside it; shot counts per chunk.
__global__ void __launch_bounds__(256)
k_sample_locate(const double* __restrict__ u, uint64_t shots, const double* __restrict__ chunk_incl,
                const double* __restrict__ chunk_mass, int nchunks, const double* __restrict__ total,
                uint32_t* __restrict__ shot_chunk, double* __restrict__ shot_t, uint32_t* __restrict__ counts) {
  const double tot = *total;
  if (!sample_total_ok(tot)) return;         // refused on the host
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < shots; i += (uint64_t)gridDim.x * blockDim.x) {
    double t = u[i] * tot;
    const int c = qs_cdf_pick([&](int j) { return chunk_incl[j]; }, [&](int j) { return chunk_mass[j]; }, nchunks, &t);
    shot_chunk[i] = (uint32_t)c;
    shot_t[i] = t;
    warp_claim(counts + c);                   // integer counts: exact in any order
  }
}

// Exclusive block scan of one unsigned value per thread (blockDim.x a multiple of 32); *sum = the total.
__device__ __forceinline__ uint32_t block_exscan_u32(uint32_t v, uint32_t* wt, uint32_t* sum) {
  const int lane = threadIdx.x & 31, w = threadIdx.x >> 5, nw = blockDim.x >> 5;
  uint32_t x = v;
#pragma unroll
  for (int d = 1; d < 32; d <<= 1) {
    const uint32_t y = __shfl_up_sync(0xffffffffu, x, d);
    if (lane >= d) x += y;
  }
  if (lane == 31) wt[w] = x;
  __syncthreads();
  if (w == 0) {
    uint32_t z = lane < nw ? wt[lane] : 0u;
#pragma unroll
    for (int d = 1; d < 32; d <<= 1) {
      const uint32_t y = __shfl_up_sync(0xffffffffu, z, d);
      if (lane >= d) z += y;
    }
    if (lane < nw) wt[lane] = z;
  }
  __syncthreads();
  const uint32_t ex = (w ? wt[w - 1] : 0u) + x - v;
  *sum = wt[nw - 1];
  __syncthreads();
  return ex;
}

// Pass 4 (one CTA of 1024): bucket starts per chunk (written to `ends`, which the scatter advances
// to the bucket ends) and work-item offsets (ceil(count / QS_SAMPLE_ITEM) items per chunk).
__global__ void __launch_bounds__(1024)
k_sample_offsets(const uint32_t* __restrict__ counts, uint64_t nchunks, uint32_t* __restrict__ ends,
                 uint32_t* __restrict__ items) {
  __shared__ uint32_t wt[32];
  const int r = threadIdx.x;
  const uint64_t seg = (nchunks + 1023) / 1024;
  uint32_t a = 0, b = 0;
  for (uint64_t e = 0; e < seg; ++e)
    if (r * seg + e < nchunks) {
      const uint32_t c = counts[r * seg + e];
      a += c;
      b += (c + QS_SAMPLE_ITEM - 1) / QS_SAMPLE_ITEM;
    }
  uint32_t tot_a, tot_b;
  uint32_t xa = block_exscan_u32(a, wt, &tot_a);
  uint32_t xb = block_exscan_u32(b, wt, &tot_b);
  for (uint64_t e = 0; e < seg; ++e) {
    const uint64_t i = r * seg + e;
    if (i < nchunks) {
      const uint32_t c = counts[i];
      ends[i] = xa;
      items[i] = xb;
      xa += c;
      xb += (c + QS_SAMPLE_ITEM - 1) / QS_SAMPLE_ITEM;
    }
  }
  if (r == 0) items[nchunks] = tot_b;
}

// Pass 5: the shots bucketed by chunk (the order inside a bucket does not matter: every outcome is a
// function of its own uniform).
__global__ void __launch_bounds__(256)
k_sample_scatter(uint64_t shots, const uint32_t* __restrict__ shot_chunk, uint32_t* __restrict__ ends,
                 uint32_t* __restrict__ order) {
  for (uint64_t i = blockIdx.x * (uint64_t)blockDim.x + threadIdx.x; i < shots; i += (uint64_t)gridDim.x * blockDim.x)
    order[warp_claim(ends + shot_chunk[i])] = (uint32_t)i;
}

struct ResolveSmem {
  double sm[288];                       // the chunk's sub-tile masses (padded)
  double sincl[256];                    // their scan
  double pb[8][288];                    // per warp: a sub-tile's probabilities (padded)
  double ib[8][256];                    // per warp: their scan
  double tl[QS_SAMPLE_ITEM];            // per shot slot: target inside its sub-tile
  uint32_t shot[QS_SAMPLE_ITEM];
  uint16_t bucket[QS_SAMPLE_ITEM];      // shot slots bucketed by sub-tile
  uint8_t sub[QS_SAMPLE_ITEM];
  uint32_t cnt[256], start[257], wt[32];
};

// Pass 6: work item = up to QS_SAMPLE_ITEM shots of one chunk.  The shots find their sub-tile
// (second level, from the stored sub-tile masses), are bucketed by it in shared memory, and only the
// sub-tiles that hold shots are read again: each is scanned by one warp, which then resolves its
// shots by binary search.  Heavy chunks (a basis state, GHZ) simply have many work items.
__global__ void __launch_bounds__(256)
k_sample_resolve(QsProbSrc src, uint64_t n_amps, uint64_t nchunks, const double* __restrict__ sub_mass,
                 const uint32_t* __restrict__ counts, const uint32_t* __restrict__ ends,
                 const uint32_t* __restrict__ items, const uint32_t* __restrict__ order,
                 const double* __restrict__ shot_t, uint64_t* __restrict__ out) {
  extern __shared__ __align__(16) unsigned char qs_resolve_smem[];
  ResolveSmem& S = *reinterpret_cast<ResolveSmem*>(qs_resolve_smem);
  const int tid = threadIdx.x, lane = tid & 31, w = tid >> 5;
  const uint32_t n_items = items[nchunks];
  double incl[8];
  for (uint32_t item = blockIdx.x; item < n_items; item += gridDim.x) {
    uint64_t lo = 0, hi = nchunks;          // the chunk: the last c with items[c] <= item
    while (hi - lo > 1) {
      const uint64_t mid = (lo + hi) >> 1;
      if (items[mid] <= item) lo = mid;
      else hi = mid;
    }
    const uint64_t c = lo;
    const uint32_t j0 = (item - items[c]) * QS_SAMPLE_ITEM;
    const uint32_t first = ends[c] - counts[c] + j0;
    const uint32_t len = min((uint32_t)QS_SAMPLE_ITEM, counts[c] - j0);
    S.sm[tid + (tid >> 3)] = sub_mass[(c << 8) + tid];
    S.cnt[tid] = 0;
    __syncthreads();
    if (w == 0) {
      warp_scan256(S.sm, incl);
#pragma unroll
      for (int m = 0; m < 8; ++m) S.sincl[8 * lane + m] = incl[m];
    }
    __syncthreads();
    for (uint32_t q = tid; q < len; q += 256) {
      const uint32_t i = order[first + q];
      double t = shot_t[i];
      const int s = qs_cdf_pick([&](int j) { return S.sincl[j]; }, [&](int j) { return S.sm[j + (j >> 3)]; }, 256, &t);
      S.shot[q] = i;
      S.tl[q] = t;
      S.sub[q] = (uint8_t)s;
      warp_claim(&S.cnt[s]);
    }
    __syncthreads();
    {
      uint32_t total;
      const uint32_t ex = block_exscan_u32(S.cnt[tid], S.wt, &total);
      S.start[tid] = ex;
      if (tid == 0) S.start[256] = total;
      S.cnt[tid] = ex;                       // from here on: bucket cursors
    }
    __syncthreads();
    for (uint32_t q = tid; q < len; q += 256) S.bucket[warp_claim(&S.cnt[S.sub[q]])] = (uint16_t)q;
    __syncthreads();
    for (int s = w; s < 256; s += 8) {
      const uint32_t b0 = S.start[s], b1 = S.start[s + 1];
      if (b0 == b1) continue;
      load_sub(src, n_amps, c, (uint64_t)s, S.pb[w]);
      warp_scan256(S.pb[w], incl);
#pragma unroll
      for (int m = 0; m < 8; ++m) S.ib[w][8 * lane + m] = incl[m];
      __syncwarp();
      const double* ib = S.ib[w];
      const double* pb = S.pb[w];
      for (uint32_t q = b0 + lane; q < b1; q += 32) {
        const uint32_t slot = S.bucket[q];
        double t = S.tl[slot];
        const int j = qs_cdf_pick([&](int e) { return ib[e]; }, [&](int e) { return pb[e + (e >> 3)]; }, 256, &t);
        out[S.shot[slot]] = (c << QS_CHUNK_LOG2) | ((uint64_t)s << QS_SUB_LOG2) | (uint64_t)j;
      }
      __syncwarp();
    }
    __syncthreads();
  }
}

// =====================================================================================
// Batched tiny-circuit executor
// =====================================================================================
template <int DIM>
__global__ void __launch_bounds__(128) k_rb_batch(int64_t n_seq, const uint16_t* __restrict__ codes,
                                                  const int64_t* __restrict__ offsets,
                                                  const double* __restrict__ superops,
                                                  const double* __restrict__ unitaries,
                                                  const double* __restrict__ rho0,
                                                  const double* __restrict__ psi0, double* out_fid,
                                                  double* out_pur, double* out_rho) {
  const int64_t b = blockIdx.x * (int64_t)blockDim.x + threadIdx.x;
  if (b >= n_seq) return;
  const int64_t lo = offsets[b], hi = offsets[b + 1];
  qs_rb_sequence<DIM>(codes + lo, hi - lo, superops, unitaries, rho0, psi0, out_fid + b, out_pur + b,
                      out_rho ? out_rho + (size_t)b * 2 * DIM * DIM : nullptr);
}

// =====================================================================================
// Pauli-trajectory batch: one CTA per shot, the ket (n <= 12 qubits) lives in shared memory
// =====================================================================================
// Every shot runs the same gate list; its random X / Z flips (bits prepared by the host from
// the caller's generator) are folded into the rows of each gate's matrix, so a noisy shot
// costs exactly what the noiseless circuit costs.  Outputs: |<obs|psi>|^2 per shot and the
// sum over shots of |amplitude|^2 (each CTA accumulates its shots in registers and adds once).
__global__ void __launch_bounds__(256)
k_traj_batch(int n, int64_t shots, int nops, const QsTrajOp* __restrict__ ops, const double* __restrict__ mats,
             const uint8_t* __restrict__ flips, int64_t flips_per_shot, const qs_c128* __restrict__ psi0,
             const qs_c128* __restrict__ obs, double* out_fid, double* out_prob, qs_c128* out_states) {
  extern __shared__ __align__(16) unsigned char qs_traj_smem[];
  qs_c128* state = reinterpret_cast<qs_c128*>(qs_traj_smem);
  __shared__ qs_c128 M[16];
  __shared__ double red[2 * 8];
  const uint32_t tid = threadIdx.x;
  const uint64_t dim = 1ull << n;
  double acc[16];                                   // n <= 12: at most 16 amplitudes per thread
#pragma unroll
  for (int e = 0; e < 16; ++e) acc[e] = 0.0;
  for (int64_t shot = blockIdx.x; shot < shots; shot += gridDim.x) {
    for (uint64_t i = tid; i < dim; i += 256) state[i] = psi0[i];
    const uint8_t* fl = flips + shot * flips_per_shot;
    __syncthreads();
    for (int o = 0; o < nops; ++o) {
      const QsTrajOp op = ops[o];
      if (tid == 0) qs_traj_rows(op, mats, fl, M);
      fl += 2 * op.k;
      __syncthreads();
      qs_traj_apply(state, n, op, M, tid, 256);
      __syncthreads();
    }
    if (out_states)
      for (uint64_t i = tid; i < dim; i += 256) out_states[(uint64_t)shot * dim + i] = state[i];
    double fr = 0.0, fi = 0.0;
    int e = 0;
    for (uint64_t i = tid; i < dim; i += 256, ++e) {
      const qs_c128 v = state[i];
      acc[e] += v.x * v.x + v.y * v.y;
      if (obs) { const qs_c128 w = obs[i]; fr += w.x * v.x + w.y * v.y; fi += w.x * v.y - w.y * v.x; }
    }
    if (obs && out_fid) {
#pragma unroll
      for (int off = 16; off > 0; off >>= 1) {
        fr += __shfl_down_sync(0xffffffffu, fr, off);
        fi += __shfl_down_sync(0xffffffffu, fi, off);
      }
      if ((tid & 31u) == 0) { red[2 * (tid >> 5)] = fr; red[2 * (tid >> 5) + 1] = fi; }
      __syncthreads();
      if (tid == 0) {
        double sr = 0.0, si = 0.0;
        for (int w = 0; w < 8; ++w) { sr += red[2 * w]; si += red[2 * w + 1]; }
        out_fid[shot] = sr * sr + si * si;
      }
    }
    __syncthreads();
  }
  if (out_prob) {
    int e = 0;
    for (uint64_t i = tid; i < dim; i += 256, ++e) atomicAdd(out_prob + i, acc[e]);
  }
}

// =====================================================================================
// Dense k-qubit block, 5 <= k <= 10 (Gate.apply with any k, DV/gates.py:44-54): in place,
// one pass over the state, FP64 tensor-core MMA (DMMA.8x8x4)
// =====================================================================================
// A tile is the 2^k amplitudes of the gate's qubits times 8 "columns" (the three lowest
// index bits the gate does not touch, so rows of 8 amplitudes are 128 contiguous bytes
// whenever the gate leaves bits 0..2 alone).  With the complex matrix split into real and
// imaginary parts the update is the real GEMM
//     out_re = Mr in_re - Mi in_im,   out_im = Mr in_im + Mi in_re        (2^k x 2^k) x (2^k x 8)
// i.e. four m8n8k4 MMAs per 8-row block and 4-column chunk of M.  The whole tile is staged in
// shared memory first, every warp keeps its 8x8 output block in registers and writes it
// straight back to the addresses it came from: no scratch buffer, no second pass.
struct DenseGeom {
  int k, ncol, T;
  uint8_t gate_bits[10];     // index bit of matrix factor f (f = 0: most significant bit of the row index)
  uint8_t col_bits[3];       // ascending
  uint8_t tile_bits[16];     // ascending union of the two
};

__device__ __forceinline__ void dmma_8x8x4(double& d0, double& d1, double a, double b) {
  asm volatile("mma.sync.aligned.m8n8k4.row.col.f64.f64.f64.f64 {%0,%1}, {%2}, {%3}, {%0,%1};"
               : "+d"(d0), "+d"(d1)
               : "d"(a), "d"(b));
}

__device__ __forceinline__ uint64_t dense_index(const DenseGeom& G, uint64_t base, int row, int col) {
  uint64_t idx = base;
  for (int f = 0; f < G.k; ++f) idx |= (uint64_t)((row >> (G.k - 1 - f)) & 1) << G.gate_bits[f];
  for (int b = 0; b < G.ncol; ++b) idx |= (uint64_t)((col >> b) & 1) << G.col_bits[b];
  return idx;
}

__global__ void __launch_bounds__(256)
k_dense_block(qs_c128* state, const double* __restrict__ mat, const __grid_constant__ DenseGeom G, uint64_t ntiles) {
  extern __shared__ __align__(16) unsigned char qs_dense_smem[];
  qs_c128* tile = reinterpret_cast<qs_c128*>(qs_dense_smem);   // slot of (c, col): c * 8 + (col ^ ((c & 3) << 1))
  const int k = G.k, dim = 1 << k, ncols = 1 << G.ncol;
  const int tid = (int)threadIdx.x, lane = tid & 31, warp = tid >> 5, nwarps = (int)blockDim.x >> 5;
  for (uint64_t t = blockIdx.x; t < ntiles; t += gridDim.x) {
    uint64_t base = t;
    for (int l = 0; l < G.T; ++l) {
      const uint32_t pos = G.tile_bits[l];
      const uint64_t low = base & ((1ull << pos) - 1ull);
      base = ((base >> pos) << (pos + 1)) | low;
    }
    for (int e = tid; e < dim * 8; e += (int)blockDim.x) {
      const int c = e >> 3, col = e & 7;
      qs_c128 v; v.x = 0.0; v.y = 0.0;
      if (col < ncols) v = state[dense_index(G, base, c, col)];
      tile[c * 8 + (col ^ ((c & 3) << 1))] = v;
    }
    __syncthreads();
    for (int rb = warp; rb < dim / 8; rb += nwarps) {
      double re0 = 0.0, re1 = 0.0, im0 = 0.0, im1 = 0.0;
      const int row = rb * 8 + (lane >> 2);
      const double2* mrow = reinterpret_cast<const double2*>(mat) + ((size_t)row << k);
      const int colb = lane >> 2;
#pragma unroll 4
      for (int chunk = 0; chunk < dim / 4; ++chunk) {
        const int c = chunk * 4 + (lane & 3);
        const double2 mv = __ldg(mrow + c);                              // M[row][c]
        const qs_c128 b = tile[c * 8 + (colb ^ ((c & 3) << 1))];        // in[c][colb]
        dmma_8x8x4(re0, re1, mv.x, b.x);
        dmma_8x8x4(re0, re1, -mv.y, b.y);
        dmma_8x8x4(im0, im1, mv.x, b.y);
        dmma_8x8x4(im0, im1, mv.y, b.x);
      }
      const int col0 = 2 * (lane & 3);
      if (col0 < ncols) {
        qs_c128 o; o.x = re0; o.y = im0;
        state[dense_index(G, base, row, col0)] = o;
      }
      if (col0 + 1 < ncols) {
        qs_c128 o; o.x = re1; o.y = im1;
        state[dense_index(G, base, row, col0 + 1)] = o;
      }
    }
    __syncthreads();
  }
}

std::mutex g_dense_upload_lock;

int run_dense_block(DevCtx* ctx, const qs::PlanItem& it, qs_c128* state, int n, int device, cudaStream_t stream) {
  const qs::Op& op = it.op;
  const int k = op.k, dim = 1 << k;
  if (k < 5 || k > 10 || k > n) return qs::fail(QSIM_ERR_UNSUPPORTED, "dense block: k must be in [5, min(10, n)]");
  {
    // the matrix goes to the device once per plan (synchronously, like compiling the plan);
    // executions after the first launch without any host synchronisation
    std::lock_guard<std::mutex> guard(g_dense_upload_lock);
    if (!it.dev_mat || it.dev_index != device) {
      std::vector<double> flat(2 * (size_t)dim * dim);
      for (int e = 0; e < dim * dim; ++e) { flat[2 * e] = op.mat[e].real(); flat[2 * e + 1] = op.mat[e].imag(); }
      void* d = nullptr;
      QS_CUDA(cudaMalloc(&d, sizeof(double) * flat.size()));
      it.dev_mat = std::shared_ptr<void>(d, [](void* p) { cudaFree(p); });
      it.dev_index = device;
      QS_CUDA(cudaMemcpy(d, flat.data(), sizeof(double) * flat.size(), cudaMemcpyHostToDevice));
    }
  }
  DenseGeom G;
  memset(&G, 0, sizeof(G));
  G.k = k;
  uint64_t gmask = 0;
  for (int f = 0; f < k; ++f) { G.gate_bits[f] = (uint8_t)op.bits[f]; gmask |= 1ull << op.bits[f]; }
  for (int b = 0; b < n && G.ncol < 3; ++b)
    if (!(gmask >> b & 1)) G.col_bits[G.ncol++] = (uint8_t)b;
  uint64_t tmask = gmask;
  for (int i = 0; i < G.ncol; ++i) tmask |= 1ull << G.col_bits[i];
  for (int b = 0; b < n; ++b)
    if (tmask >> b & 1) G.tile_bits[G.T++] = (uint8_t)b;
  const uint64_t ntiles = 1ull << (n - G.T);
  const int smem = (int)sizeof(qs_c128) * dim * 8;
  const int threads = dim / 8 >= 8 ? 256 : 32 * (dim / 8);
  if (smem > 48 * 1024) QS_CUDA(cudaFuncSetAttribute(k_dense_block, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  int occ = 0;
  QS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_dense_block, threads, smem));
  if (occ < 1) return qs::fail(QSIM_ERR_CUDA, "dense block does not fit on an SM");
  uint64_t grid = (uint64_t)ctx->sms * (uint64_t)occ;
  if (grid > ntiles) grid = ntiles;
  k_dense_block<<<(unsigned)grid, threads, smem, stream>>>(state, (const double*)it.dev_mat.get(), G, ntiles);
  return launched();
}

}  // namespace

// =====================================================================================
// C ABI
// =====================================================================================
extern "C" {

int qsim_has_cuda(void) { return 1; }

int64_t qsim_launch_count(void) { return g_launches.load(std::memory_order_relaxed); }

int qsim_peer_alloc(int device, uint64_t bytes, void** out_ptr) {
  if (!out_ptr || bytes == 0) return qs::fail(QSIM_ERR_ARG, "qsim_peer_alloc: bad argument");
  QS_CUDA(cudaSetDevice(device));
  QS_CUDA(cudaMalloc(out_ptr, bytes));
  return QSIM_OK;
}

int qsim_peer_free(void* ptr) {
  if (ptr) QS_CUDA(cudaFree(ptr));
  return QSIM_OK;
}

int qsim_ipc_export(void* ptr, unsigned char* handle64) {
  static_assert(sizeof(cudaIpcMemHandle_t) == 64, "IPC handle size");
  if (!ptr || !handle64) return qs::fail(QSIM_ERR_ARG, "qsim_ipc_export: null argument");
  cudaIpcMemHandle_t h;
  QS_CUDA(cudaIpcGetMemHandle(&h, ptr));
  memcpy(handle64, &h, 64);
  return QSIM_OK;
}

int qsim_ipc_import(int device, const unsigned char* handle64, void** out_ptr) {
  if (!handle64 || !out_ptr) return qs::fail(QSIM_ERR_ARG, "qsim_ipc_import: null argument");
  cudaIpcMemHandle_t h;
  memcpy(&h, handle64, 64);
  QS_CUDA(cudaSetDevice(device));
  QS_CUDA(cudaIpcOpenMemHandle(out_ptr, h, cudaIpcMemLazyEnablePeerAccess));
  return QSIM_OK;
}

int qsim_ipc_release(void* imported_ptr) {
  if (imported_ptr) QS_CUDA(cudaIpcCloseMemHandle(imported_ptr));
  return QSIM_OK;
}

int qsim_ipc_export_ex(void* ptr, unsigned char* handle64, uint64_t* offset) {
  if (!ptr || !handle64 || !offset) return qs::fail(QSIM_ERR_ARG, "qsim_ipc_export_ex: null argument");
  cudaIpcMemHandle_t h;
  QS_CUDA(cudaIpcGetMemHandle(&h, ptr));
  memcpy(handle64, &h, 64);
  // the handle names the whole allocation: find its base through the driver
  typedef CUresult (*RangeFn)(CUdeviceptr*, size_t*, CUdeviceptr);
  static RangeFn range = [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuMemGetAddressRange", &p, cudaEnableDefault, &q) != cudaSuccess ||
        q != cudaDriverEntryPointSuccess)
      p = nullptr;
    cudaGetLastError();
    return (RangeFn)p;
  }();
  if (!range) return qs::fail(QSIM_ERR_CUDA, "cuMemGetAddressRange is not available");
  CUdeviceptr base = 0;
  size_t size = 0;
  if (range(&base, &size, (CUdeviceptr)ptr) != CUDA_SUCCESS)
    return qs::fail(QSIM_ERR_CUDA, "cuMemGetAddressRange failed");
  *offset = (uint64_t)((CUdeviceptr)ptr - base);
  return QSIM_OK;
}

int qsim_exchange_p2p(void* shard, void* const* peer_shards, int n_local, int nbits, const int* local_qubits,
                      const int* my_bits, const int* partner_is_lower, void* stream) {
  if (!shard || !peer_shards || !local_qubits || !my_bits || !partner_is_lower)
    return qs::fail(QSIM_ERR_ARG, "qsim_exchange_p2p: null argument");
  if (nbits < 1 || nbits > 8 || n_local - nbits - 1 < kExchSplitBit)
    return qs::fail(QSIM_ERR_ARG, "qsim_exchange_p2p: bad sizes (blocks must hold at least 64 amplitudes)");
  ExchGeom G;
  memset(&G, 0, sizeof(G));
  G.k = nbits;
  G.n_local = n_local;
  // order the bits by local position (ascending); pattern bit i of d stays with the caller's bit i
  int order[8];
  for (int i = 0; i < nbits; ++i) order[i] = i;
  for (int i = 1; i < nbits; ++i)
    for (int j = i; j > 0 && local_qubits[order[j]] > local_qubits[order[j - 1]]; --j) std::swap(order[j], order[j - 1]);
  for (int i = 0; i < nbits; ++i) {
    const int q = local_qubits[order[i]];
    if (q < 0 || q >= n_local || (my_bits[order[i]] | 1) != 1) return qs::fail(QSIM_ERR_ARG, "qsim_exchange_p2p: bad qubit or bit");
    G.pos[i] = n_local - 1 - q;                    // reference-style local qubit -> index bit
    G.mine[i] = my_bits[order[i]];
    if (i > 0 && G.pos[i] <= G.pos[i - 1]) return qs::fail(QSIM_ERR_ARG, "qsim_exchange_p2p: repeated qubit");
  }
  for (int d = 1; d < (1 << nbits); ++d) {
    // the caller's pattern d (bit i <-> its bit i) in sorted order
    int ds = 0;
    for (int i = 0; i < nbits; ++i) ds |= ((d >> order[i]) & 1) << i;
    if (!peer_shards[d]) return qs::fail(QSIM_ERR_ARG, "qsim_exchange_p2p: missing peer pointer");
    G.peer[ds] = (qs_c128*)peer_shards[d];
    G.higher[ds] = partner_is_lower[d] ? 1 : 0;
  }
  Bound bound;
  int rc = bind_device(shard, &bound);
  if (rc != QSIM_OK) return rc;
  const uint64_t total = (1ull << (n_local - nbits - 1)) * ((1ull << nbits) - 1ull);
  // development knobs (defaults measured on 2 and 8 B200s): pairs per thread and trip, CTAs per SM
  static const int batch = qs::dev_knob("QSIM_EXCH_BATCH", 4);
  static const int per_sm = qs::dev_knob("QSIM_EXCH_CTAS", 8);
  static const int chunk_log2 = qs::dev_knob("QSIM_EXCH_CHUNK_LOG2", 0);
  G.chunk_log2 = (chunk_log2 > 0 && chunk_log2 <= n_local - nbits - 1 && nbits > 1) ? chunk_log2 : 0;
  const int U = batch >= 8 ? 8 : batch >= 4 ? 4 : batch >= 2 ? 2 : 1;
  uint64_t blocks = (total + 256ull * U - 1) / (256ull * U);
  const uint64_t cap = (uint64_t)bound.ctx->sms * (uint64_t)(per_sm > 0 ? per_sm : 8);
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  cudaStream_t st = (cudaStream_t)stream;
  if (U == 8) k_exchange_p2p<8><<<(unsigned)blocks, 256, 0, st>>>((qs_c128*)shard, G);
  else if (U == 4) k_exchange_p2p<4><<<(unsigned)blocks, 256, 0, st>>>((qs_c128*)shard, G);
  else if (U == 2) k_exchange_p2p<2><<<(unsigned)blocks, 256, 0, st>>>((qs_c128*)shard, G);
  else k_exchange_p2p<1><<<(unsigned)blocks, 256, 0, st>>>((qs_c128*)shard, G);
  return launched();
}

int qsim_peer_copy(void* dst, const void* src, uint64_t bytes, void* stream) {
  if (!dst || !src) return qs::fail(QSIM_ERR_ARG, "qsim_peer_copy: null argument");
  QS_CUDA(cudaMemcpyAsync(dst, src, bytes, cudaMemcpyDefault, (cudaStream_t)stream));
  return QSIM_OK;
}

}  // extern "C"

// =====================================================================================
// Backend of the compute entry points (backend.h; checks and lowering in capi_host.cpp)
// =====================================================================================
namespace qs::dev {

int execute_plan(const qsim_plan& p, qs_c128* state, int n, void* stream) {
  Bound bound;
  int rc = bind_device(state, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  for (const qs::PlanItem& it : p.items) {
    rc = it.generic ? run_dense_block(ctx, it, state, n, bound.device, st) : launch_pass(ctx, it.pass, state, n, st);
    if (rc != QSIM_OK) return rc;
  }
  return QSIM_OK;
}

int init_product(qs_c128* state, int n, const ProductAmps& amps, void* stream) {
  Bound bound;
  int rc = bind_device(state, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  cudaStream_t st = (cudaStream_t)stream;
  const uint64_t count = 1ull << n;
  if (n >= 16) {
    uint64_t blocks = count >> 16;
    if (blocks > (uint64_t)ctx->sms * 8) blocks = (uint64_t)ctx->sms * 8;
    k_init_product_big<<<(unsigned)blocks, 256, 0, st>>>(state, n, amps);
  } else {
    k_init_product<<<stream_grid(ctx, count, 256), 256, 0, st>>>(state, n, amps, count);
  }
  return launched();
}

int measure_probs(const qs_c128* state, int pos, uint64_t pairs, const BraPair& bra0, const BraPair& bra1,
                  double* out_norm2, void* stream) {
  Bound bound;
  int rc = bind_device(state, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  FnMeasure f{state, pos, bra0, bra1};
  return reduce_to_host(ctx, f, pairs, out_norm2, (cudaStream_t)stream);
}

int collapse(const qs_c128* in, qs_c128* out, int pos, const BraPair& bra, double norm, uint64_t count,
             void* stream) {
  Bound bound;
  int rc = bind_device(in, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  k_collapse<<<stream_grid(ctx, count, 256), 256, 0, (cudaStream_t)stream>>>(in, out, pos, bra, norm, count);
  return launched();
}

int insert(const qs_c128* in, qs_c128* out, int pos, const BraPair& amp, uint64_t count, void* stream) {
  Bound bound;
  int rc = bind_device(in, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  k_insert<<<stream_grid(ctx, count, 256), 256, 0, (cudaStream_t)stream>>>(in, out, pos, amp, count);
  return launched();
}

int reduce_norm2(const qs_c128* state, uint64_t n_amps, double* out, void* stream) {
  Bound bound;
  int rc = bind_device(state, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  FnNorm2 f{state};
  double r[2];
  rc = reduce_to_host(ctx, f, n_amps, r, (cudaStream_t)stream);
  if (rc == QSIM_OK) *out = r[0];
  return rc;
}

int reduce_inner(const qs_c128* a, const qs_c128* b, uint64_t n_amps, double* out_re_im, void* stream) {
  Bound bound;
  int rc = bind_device(a, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  FnInner f{a, b};
  return reduce_to_host(ctx, f, n_amps, out_re_im, (cudaStream_t)stream);
}

int reduce_expect(const qs_c128* ket, const qs_c128* rho, int n, double* out_re_im, void* stream) {
  Bound bound;
  int rc = bind_device(rho, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  FnExpect f{ket, rho, n};
  return reduce_to_host(ctx, f, 1ull << (2 * n), out_re_im, (cudaStream_t)stream);
}

int reduce_purity(const qs_c128* rho, int n, double* out_re_im, void* stream) {
  Bound bound;
  int rc = bind_device(rho, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  FnPurity f{rho, n};
  return reduce_to_host(ctx, f, 1ull << (2 * n), out_re_im, (cudaStream_t)stream);
}

int reduce_trace(const qs_c128* rho, int n, double* out_re_im, void* stream) {
  Bound bound;
  int rc = bind_device(rho, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  FnTrace f{rho, n};
  return reduce_to_host(ctx, f, 1ull << n, out_re_im, (cudaStream_t)stream);
}

int expect_pauli(const qs_c128* state, int n, const PauliPlan& plan, int64_t n_terms, double* sums, void* stream) {
  Bound bound;
  int rc = bind_device(state, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  const uint64_t count = 1ull << (n - plan.d);
  uint64_t blocks = (count + kPauliThreads - 1) / kPauliThreads;
  blocks = std::min<uint64_t>(blocks, (uint64_t)ctx->sms * kPauliBlocksPerSM);
  const cudaStream_t st = (cudaStream_t)stream;
  std::lock_guard<std::mutex> guard(ctx->reduce_lock);
  rc = pauli_scratch(ctx, (size_t)n_terms, (size_t)blocks);
  if (rc != QSIM_OK) return rc;
  for (const QsPauliPass& P : plan.passes) {
    switch (plan.d) {
      case 1: launch_pauli_pass<1>(P, state, count, (unsigned)blocks, ctx->d_pauli_partials, st); break;
      case 2: launch_pauli_pass<2>(P, state, count, (unsigned)blocks, ctx->d_pauli_partials, st); break;
      case 3: launch_pauli_pass<3>(P, state, count, (unsigned)blocks, ctx->d_pauli_partials, st); break;
      default: launch_pauli_pass<4>(P, state, count, (unsigned)blocks, ctx->d_pauli_partials, st); break;
    }
    rc = launched();
    if (rc != QSIM_OK) return rc;
  }
  return pauli_sums_to_host(ctx, n_terms, (int)blocks, sums, st);
}

int expect_pauli_dm(const qs_c128* rho, int n, int64_t n_terms, const uint64_t* xi, const uint64_t* zi,
                    double* sums, void* stream) {
  std::vector<uint64_t> masks(2 * (size_t)n_terms);     // upload format of k_pauli_expect_dm: [x, z] per term
  for (int64_t t = 0; t < n_terms; ++t) { masks[2 * t] = xi[t]; masks[2 * t + 1] = zi[t]; }
  Bound bound;
  int rc = bind_device(rho, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  const uint64_t dim = 1ull << n;
  const unsigned bx = (unsigned)std::min<uint64_t>((dim + kReduceThreads - 1) / kReduceThreads, kPauliDmBlocks);
  const unsigned by = (unsigned)std::min<int64_t>(n_terms, 65535);
  const cudaStream_t st = (cudaStream_t)stream;
  std::lock_guard<std::mutex> guard(ctx->reduce_lock);
  rc = pauli_scratch(ctx, (size_t)n_terms, (size_t)bx);
  if (rc != QSIM_OK) return rc;
  QS_CUDA(cudaMemcpyAsync(ctx->d_pauli_masks, masks.data(), sizeof(uint64_t) * masks.size(), cudaMemcpyHostToDevice, st));
  k_pauli_expect_dm<<<dim3(bx, by), kReduceThreads, 0, st>>>(rho, n, ctx->d_pauli_masks, n_terms,
                                                             ctx->d_pauli_partials);
  rc = launched();
  if (rc != QSIM_OK) return rc;
  return pauli_sums_to_host(ctx, n_terms, (int)bx, sums, st);
}

int apply_pauli_rotations(qs_c128* state, int n, const PauliRotPlan& plan, void* stream) {
  Bound bound;
  int rc = bind_device(state, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  const uint64_t count = 1ull << (n - plan.d);
  const int per_sm = qs::dev_knob("QSIM_ROT_BLOCKS_PER_SM", kRotBlocksPerSM);
  const unsigned blocks = (unsigned)std::min<uint64_t>((count + kRotThreads - 1) / kRotThreads,
                                                       (uint64_t)ctx->sms * per_sm);
  const cudaStream_t st = (cudaStream_t)stream;
  for (const QsPauliRotPass& P : plan.passes) {
    switch (plan.d) {
      case 1: k_pauli_rotate<1><<<blocks, kRotThreads, 0, st>>>(state, P, count); break;
      case 2: k_pauli_rotate<2><<<blocks, kRotThreads, 0, st>>>(state, P, count); break;
      case 3: k_pauli_rotate<3><<<blocks, kRotThreads, 0, st>>>(state, P, count); break;
      default: k_pauli_rotate<4><<<blocks, kRotThreads, 0, st>>>(state, P, count); break;
    }
    rc = launched();
    if (rc != QSIM_OK) return rc;
  }
  return QSIM_OK;
}

int apply_pauli_sum(const qs_c128* in, qs_c128* out, int n, const PauliApplyPlan& plan, void* stream) {
  Bound bound;
  int rc = bind_device(out, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  const uint64_t count = 1ull << (n - plan.d);
  const unsigned blocks = (unsigned)std::min<uint64_t>((count + kRotThreads - 1) / kRotThreads,
                                                       (uint64_t)ctx->sms * kRotBlocksPerSM);
  const cudaStream_t st = (cudaStream_t)stream;
  for (const QsPauliApplyPass& A : plan.passes) {
    switch (plan.d) {
      case 1: k_pauli_apply<1><<<blocks, kRotThreads, 0, st>>>(in, out, A, count); break;
      case 2: k_pauli_apply<2><<<blocks, kRotThreads, 0, st>>>(in, out, A, count); break;
      case 3: k_pauli_apply<3><<<blocks, kRotThreads, 0, st>>>(in, out, A, count); break;
      default: k_pauli_apply<4><<<blocks, kRotThreads, 0, st>>>(in, out, A, count); break;
    }
    rc = launched();
    if (rc != QSIM_OK) return rc;
  }
  return QSIM_OK;
}

int pauli_rotations_adjoint(qs_c128* psi, qs_c128* lam, int n, const PauliRotPlan& plan, double* sums, void* stream) {
  Bound bound;
  int rc = bind_device(psi, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  const uint64_t count = 1ull << (n - plan.d);
  const unsigned blocks = (unsigned)std::min<uint64_t>((count + kPauliThreads - 1) / kPauliThreads,
                                                       (uint64_t)ctx->sms * kAdjBlocksPerSM);
  const int64_t rows = (int64_t)plan.caller.size();
  const cudaStream_t st = (cudaStream_t)stream;
  std::lock_guard<std::mutex> guard(ctx->reduce_lock);
  rc = pauli_scratch(ctx, (size_t)rows, blocks);
  if (rc != QSIM_OK) return rc;
  uint32_t row0 = 0;
  for (const QsPauliRotPass& P : plan.passes) {
    double* partials = ctx->d_pauli_partials;
    switch (plan.d) {
      case 1: k_pauli_adjoint<1><<<blocks, kPauliThreads, 0, st>>>(psi, lam, P, count, row0, partials); break;
      case 2: k_pauli_adjoint<2><<<blocks, kPauliThreads, 0, st>>>(psi, lam, P, count, row0, partials); break;
      default:
        k_pauli_adjoint<QS_PAULI_ADJ_MAX_D><<<blocks, kPauliThreads, 0, st>>>(psi, lam, P, count, row0, partials);
        break;
    }
    rc = launched();
    if (rc != QSIM_OK) return rc;
    row0 += P.nrot;
  }
  return pauli_sums_to_host(ctx, rows, (int)blocks, sums, st);
}

int marginal_probs(const QsProbSrc& src, const QsMargGeom& G, double* out, void* stream) {
  Bound bound;
  int rc = bind_device(src.a, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  const cudaStream_t st = (cudaStream_t)stream;
  const uint64_t warps = std::min<uint64_t>(G.ntasks, (uint64_t)ctx->sms * kMargWarpsPerSM);
  const uint64_t blocks = (warps + kMargThreads / 32 - 1) / (kMargThreads / 32);
  const uint64_t slots = blocks * (kMargThreads / 32);
  const uint64_t per_warp = (G.ntasks + slots - 1) / slots;
  if (G.gs_bits == 0) {
    k_marginal<<<(unsigned)blocks, kMargThreads, 0, st>>>(G, src, out, per_warp);
    return launched();
  }
  std::lock_guard<std::mutex> guard(ctx->marg_lock);
  if (!ctx->marg_done) QS_CUDA(cudaEventCreateWithFlags(&ctx->marg_done, cudaEventDisableTiming));
  if (!ctx->d_marg_partials) QS_CUDA(cudaMalloc(&ctx->d_marg_partials, sizeof(double) << QS_MARG_PARTIALS_LOG2));
  QS_CUDA(cudaStreamWaitEvent(st, ctx->marg_done, 0));     // the previous marginal's final sum has read them
  k_marginal<<<(unsigned)blocks, kMargThreads, 0, st>>>(G, src, ctx->d_marg_partials, per_warp);
  const uint64_t bins = 1ull << G.k;
  const unsigned grid = (unsigned)std::min<uint64_t>(bins, (uint64_t)ctx->sms * 8);
  k_marg_final<<<grid, 256, 0, st>>>(ctx->d_marg_partials, G.gs_bits, bins, out);
  rc = launched(2);
  if (rc != QSIM_OK) return rc;
  QS_CUDA(cudaEventRecord(ctx->marg_done, st));
  return QSIM_OK;
}

int sample(const QsProbSrc& src, int n, int64_t shots, const double* uniforms, uint64_t* out, double* total,
           unsigned char* ws, void* stream) {
  Bound bound;
  int rc = bind_device(src.a, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  const cudaStream_t st = (cudaStream_t)stream;
  const QsSampleLayout L = qs_sample_layout(n, (uint64_t)shots);
  double* sub_mass = (double*)(ws + L.sub_mass);
  double* chunk_mass = (double*)(ws + L.chunk_mass);
  double* chunk_incl = (double*)(ws + L.chunk_incl);
  double* d_total = (double*)(ws + L.total);
  uint32_t* counts = (uint32_t*)(ws + L.counts);
  uint32_t* ends = (uint32_t*)(ws + L.ends);
  uint32_t* items = (uint32_t*)(ws + L.items);
  uint32_t* shot_chunk = (uint32_t*)(ws + L.shot_chunk);
  double* shot_t = (double*)(ws + L.shot_t);
  uint32_t* order = (uint32_t*)(ws + L.order);
  const uint64_t n_amps = 1ull << n, nchunks = L.nchunks;
  const int smem = (int)sizeof(ResolveSmem);
  QS_CUDA(cudaFuncSetAttribute(k_sample_resolve, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  int occ = 0;
  QS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_sample_resolve, 256, smem));
  if (occ < 1) return qs::fail(QSIM_ERR_CUDA, "sample resolve kernel does not fit on an SM");
  QS_CUDA(cudaMemsetAsync(counts, 0, sizeof(uint32_t) * nchunks, st));
  const unsigned shot_grid = stream_grid(ctx, (uint64_t)shots, 256);
  k_sample_masses<<<(unsigned)std::min<uint64_t>(nchunks, (uint64_t)ctx->sms * 8), 256, 0, st>>>(
      src, n_amps, nchunks, sub_mass, chunk_mass);
  k_sample_scan<<<1, 1024, 0, st>>>(chunk_mass, nchunks, chunk_incl, d_total);
  k_sample_locate<<<shot_grid, 256, 0, st>>>(uniforms, (uint64_t)shots, chunk_incl, chunk_mass, (int)nchunks, d_total,
                                             shot_chunk, shot_t, counts);
  k_sample_offsets<<<1, 1024, 0, st>>>(counts, nchunks, ends, items);
  k_sample_scatter<<<shot_grid, 256, 0, st>>>((uint64_t)shots, shot_chunk, ends, order);
  k_sample_resolve<<<(unsigned)(ctx->sms * occ), 256, smem, st>>>(src, n_amps, nchunks, sub_mass, counts, ends, items,
                                                                  order, shot_t, out);
  rc = launched(6);
  if (rc != QSIM_OK) return rc;
  std::lock_guard<std::mutex> guard(ctx->reduce_lock);      // guards the pinned word
  QS_CUDA(cudaMemcpyAsync(ctx->h_out, d_total, sizeof(double), cudaMemcpyDeviceToHost, st));
  QS_CUDA(cudaStreamSynchronize(st));
  *total = ctx->h_out[0];
  return QSIM_OK;
}

int rb_batch(int nq, int64_t n_seq, const uint16_t* opcodes, const int64_t* offsets, const double* superops,
             const double* unitaries, const double* rho0, const double* psi0, double* out_fidelity,
             double* out_purity, double* out_rho, void* stream) {
  Bound bound;
  int rc = bind_device(out_fidelity, &bound);
  if (rc != QSIM_OK) return rc;
  const unsigned blocks = (unsigned)((n_seq + 127) / 128);
  cudaStream_t st = (cudaStream_t)stream;
  if (nq == 2)
    k_rb_batch<4><<<blocks, 128, 0, st>>>(n_seq, opcodes, offsets, superops, unitaries, rho0, psi0,
                                         out_fidelity, out_purity, out_rho);
  else
    k_rb_batch<2><<<blocks, 128, 0, st>>>(n_seq, opcodes, offsets, superops, unitaries, rho0, psi0,
                                         out_fidelity, out_purity, out_rho);
  return launched();
}

int traj_batch(int n, int64_t shots, int n_ops, const QsTrajOp* ops, const double* matrices, const uint8_t* flips,
               int64_t flips_per_shot, const qs_c128* psi0, const qs_c128* observable, double* out_fidelity,
               double* out_prob_sum, qs_c128* out_states, void* stream) {
  Bound bound;
  int rc = bind_device(psi0, &bound);
  if (rc != QSIM_OK) return rc;
  const int smem = (int)(sizeof(qs_c128) << n);
  if (smem > 48 * 1024) QS_CUDA(cudaFuncSetAttribute(k_traj_batch, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
  int occ = 0;
  QS_CUDA(cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, k_traj_batch, 256, smem));
  if (occ < 1) return qs::fail(QSIM_ERR_CUDA, "trajectory batch does not fit on an SM");
  int64_t grid = (int64_t)bound.ctx->sms * occ;
  if (grid > shots) grid = shots;
  k_traj_batch<<<(unsigned)grid, 256, smem, (cudaStream_t)stream>>>(n, shots, n_ops, ops, matrices, flips,
                                                                    flips_per_shot, psi0, observable, out_fidelity,
                                                                    out_prob_sum, out_states);
  return launched();
}

int swap_pack(const qs_c128* shard, qs_c128* buf, const QsBitSel& sel, uint64_t first, uint64_t count, void* stream) {
  Bound bound;
  int rc = bind_device(shard, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  if (count == 0) return QSIM_OK;
  k_swap_pack<<<stream_grid(ctx, count, 256), 256, 0, (cudaStream_t)stream>>>(shard, buf, sel, first, count);
  return launched();
}

int swap_unpack(qs_c128* shard, const qs_c128* buf, const QsBitSel& sel, uint64_t first, uint64_t count,
                void* stream) {
  Bound bound;
  int rc = bind_device(shard, &bound);
  DevCtx* ctx = bound.ctx;
  if (rc != QSIM_OK) return rc;
  if (count == 0) return QSIM_OK;
  k_swap_unpack<<<stream_grid(ctx, count, 256), 256, 0, (cudaStream_t)stream>>>(shard, buf, sel, first, count);
  return launched();
}

}  // namespace qs::dev
