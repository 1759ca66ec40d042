// Tensor-core (tcgen05 / TMEM) kernels of the denoiser: 3-product split contractions (3xFP16 or 3xTF32 operands) with
// fp32 accumulation in TMEM.
//
//   tc_edge_kernel<0,..>   — GCL.edge_model + receiver sums                 (egnn_new.py:31-52)
//   tc_edge_kernel<1,..>   — EquivariantUpdate.coord_model                  (egnn_new.py:96-116)
//                            PAIR = true (3xFP16 default): CTA pairs, tcgen05 cta_group::2, second-layer weights resident
//   tc_node_block_kernel   — GCL.node_model + the merged first-layer GEMM that consumes the new h, CTA pairs (egnn_new.py:48-58)
//   tc_node_gemm_kernel    — C = A @ W + bias                               (first block's first layer; single-CTA merged GEMM)
//   tc_node_mlp_kernel     — node_model alone, single CTA                   (3xTF32 / dsb_set_kernel_variants(0))
//
// One persistent CTA per SM, warp-specialised (see dsb_tc.cuh); the roles of the edge kernels:
//   warps 0-3   epilogue: tcgen05.ld accumulator rows (thread = one tile row), bias/SiLU/gate, chunk sums, RED
//   warps 4-11  producers: build the A operand chunk (gather Pa[row]+Pb[col]+radial terms, SiLU, hi/lo split) straight
//               into 128B-swizzled shared memory; fence.proxy.async; arrive on full_x (of the pair's leader CTA)
//   warp 12     MMA issuer: one thread (of the leader CTA) issues 12 tcgen05.mma (4 k-steps x 3 split terms) per K-chunk
//   warp 13     bulk-copy issuer: cp.async.bulk of the pre-split, pre-swizzled weight images (once per launch when resident)
//   warps 14-15 scalar warps: per-edge indices, distances and directions one tile ahead
// Two operand stages and two 256-column TMEM accumulators: the epilogue of tile t overlaps the main loop of tile t+1.
#include <cstdlib>

#include "dsb_tc.cuh"

namespace dsb {
using namespace tc;


// =====================================================================================================
// weight images: B[n][k] (= the reference's own [out][in] Linear layout) split into hi/lo and laid out as
// [n_tile][k_chunk][H rows x 128 B, SWIZZLE_128B] (n-tiles are H = hidden_nf wide) so that one k-chunk is a single bulk copy.
// =====================================================================================================
__global__ void pack_b_image_kernel(float* __restrict__ hi, float* __restrict__ lo, const float* __restrict__ src, int lds,
                                    int scol, int n_rows, int n_dst_off, int K, int chunks, int TN) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)n_rows * K) return;
  const int n = (int)(idx / K), k = (int)(idx - (int64_t)n * K);
  const int nd = n_dst_off + n, nt = nd / TN, nl = nd % TN;
  const int kc = k / TKC, c = (k % TKC) >> 2, j = k & 3;
  const size_t off = ((size_t)nt * chunks + kc) * (size_t)(TN * TKC) + sw128_offset(nl, c) / 4 + j;
  const float w = src[(size_t)n * lds + scol + k];
  const float h = tf32_hi(w);
  hi[off] = h;
  lo[off] = w - h;
}

void launch_pack_b_image(float* hi, float* lo, const float* src, int lds, int scol, int n_rows, int n_dst_off, int K, int tn) {
  const int64_t tot = (int64_t)n_rows * K;
  pack_b_image_kernel<<<(unsigned)((tot + 255) / 256), 256>>>(hi, lo, src, lds, scol, n_rows, n_dst_off, K, K / TKC, tn);
}

// 3xFP16 images: w*scale = w_h + w_l in fp16, [n_tile][K/64][256 rows x 128 B (64 halfs), SWIZZLE_128B]
__global__ void pack_b_image_f16_kernel(__half* __restrict__ hi, __half* __restrict__ lo, const float* __restrict__ src, int lds,
                                        int scol, int n_rows, int n_dst_off, int K, int chunks, float scale, int TN) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)n_rows * K) return;
  const int n = (int)(idx / K), k = (int)(idx - (int64_t)n * K);
  const int nd = n_dst_off + n, nt = nd / TN, nl = nd % TN;
  const int kc = k / TKC16, c16 = (k % TKC16) >> 3, j = k & 7;
  const size_t off = ((size_t)nt * chunks + kc) * (size_t)(TN * 64) + sw128_offset(nl, c16) / 2 + j;
  const float w = src[(size_t)n * lds + scol + k] * scale;
  const __half h = __float2half_rn(w);
  hi[off] = h;
  lo[off] = __float2half_rn(w - __half2float(h));
}

void launch_pack_b_image_f16(float* hi, float* lo, const float* src, int lds, int scol, int n_rows, int n_dst_off, int K, float scale, int tn) {
  const int64_t tot = (int64_t)n_rows * K;
  pack_b_image_f16_kernel<<<(unsigned)((tot + 255) / 256), 256>>>(reinterpret_cast<__half*>(hi), reinterpret_cast<__half*>(lo), src,
                                                                  lds, scol, n_rows, n_dst_off, K, K / TKC16, scale, tn);
}

// max |src[n][scol + k]| over an [n_rows][K] block -> *out (device uint holding the float bits; non-negative floats order as uints)
__global__ void absmax_kernel(const float* __restrict__ src, int lds, int scol, int n_rows, int K, unsigned* __restrict__ out) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  float v = 0.f;
  if (idx < (int64_t)n_rows * K) { const int n = (int)(idx / K), k = (int)(idx - (int64_t)n * K); v = fabsf(src[(size_t)n * lds + scol + k]); }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v = fmaxf(v, __shfl_xor_sync(0xffffffffu, v, o));
  if ((threadIdx.x & 31) == 0) atomicMax(out, __float_as_uint(v));
}
void launch_absmax(const float* src, int lds, int scol, int n_rows, int K, unsigned* out) {
  const int64_t tot = (int64_t)n_rows * K;
  absmax_kernel<<<(unsigned)((tot + 255) / 256), 256>>>(src, lds, scol, n_rows, K, out);
}

// bring-up / diagnosis only (profiles/tc_ablate.py): 1 skip weight copies, 2 skip producer work, 4 skip epilogue work,
// 8 skip MMAs.  Results are garbage when non-zero; never set by the product path.
extern "C" int dsb_debug_set_tc_flags(int flags) {
#if !DSB_TC_INSTRUMENT
  if (flags != 0) return -4;      // product build: no instrumentation compiled in
#endif
  return cudaMemcpyToSymbol(tc::g_tc_debug, &flags, sizeof(int)) == cudaSuccess ? 0 : -3;
}
// reads (and clears) the 64 cycle counters accumulated by kernels run with flag 512
extern "C" int dsb_debug_read_tc_prof(unsigned long long* out32) {
  if (cudaMemcpyFromSymbol(out32, tc::g_tc_prof, 64 * sizeof(unsigned long long)) != cudaSuccess) return -3;
  unsigned long long z[64] = {0};
  return cudaMemcpyToSymbol(tc::g_tc_prof, z, sizeof(z)) == cudaSuccess ? 0 : -3;
}

// ---- common prologue / epilogue of every TC kernel -----------------------------------------------------------------
constexpr size_t kControlBytes = 256;      // keeps the per-kernel extras 16-byte aligned for float4 access
static_assert(sizeof(Control) <= kControlBytes, "Control block grew");
struct Carve {
  char* stages;
  Control* ctl;
  char* extra;
};
template <int H>
__device__ __forceinline__ Carve carve_smem(uint8_t* raw) {
  const uint32_t base = smem_u32(raw);
  const uint32_t pad = (1024u - (base & 1023u)) & 1023u;
  Carve c;
  c.stages = reinterpret_cast<char*>(raw) + pad;
  c.ctl = reinterpret_cast<Control*>(c.stages + NSTAGE * Geo<H>::STAGE_BYTES);
  c.extra = reinterpret_cast<char*>(c.ctl) + kControlBytes;
  return c;
}
template <int H> constexpr size_t tc_smem_base() { return 1024 + (size_t)NSTAGE * Geo<H>::STAGE_BYTES + kControlBytes; }
constexpr int GEMM_T_STRIDE = 36;          // floats; 16-byte aligned rows, conflict-free for row-wise STS.128 and LDS.128

__device__ __forceinline__ void tc_begin(Control* ctl, int warp, int scal_full_count = 1) {
  if (threadIdx.x == 0) control_init(ctl, scal_full_count);
  __syncthreads();
  if (warp == MMA_WARP) tmem_alloc(&ctl->tmem_base, 512);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
}
__device__ __forceinline__ void tc_end(Control* ctl, int warp) {
  tc_fence_before();
  __syncthreads();
  if (warp == MMA_WARP) tmem_dealloc(ctl->tmem_base, 512);
}

template <int H>
__device__ __forceinline__ void tma_role(Control* ctl, char* stages, const float* bhi, const float* blo, uint32_t& g, int chunks) {
  using G = Geo<H>;
  for (int kc = 0; kc < chunks; ++kc, ++g) {
    const int s = g & 1;
    mbar_wait(&ctl->empty[s], ((g >> 1) & 1) ^ 1);
    char* st = stages + (size_t)s * G::STAGE_BYTES + 2 * A_CHUNK_BYTES;
    if (tc_debug() & 1) { mbar_arrive(&ctl->full_w[s]); continue; }
    mbar_arrive_expect_tx(&ctl->full_w[s], 2 * G::B_CHUNK_BYTES);
    bulk_g2s(st, bhi + (size_t)kc * G::B_CHUNK_FLOATS, G::B_CHUNK_BYTES, &ctl->full_w[s]);
    bulk_g2s(st + G::B_CHUNK_BYTES, blo + (size_t)kc * G::B_CHUNK_FLOATS, G::B_CHUNK_BYTES, &ctl->full_w[s]);
  }
}

// =====================================================================================================
// node GEMM
// =====================================================================================================
struct TcGemmArgs {
  const float* A; int lda; int K;
  const float* Bhi; const float* Blo;        // [Nn/256][K/32][8192]
  const float* bias;
  float* C; int ldc; int M; int Nn;
  int dead_mt; int dead_nt;                    // tiles with m-tile >= dead_mt and n-tile < dead_nt are skipped (dead_nt == 0: none)
  float inv_scale;                             // 3xFP16: 1 / (X_SCALE * weight scale); 1 for 3xTF32
  int32_t* status;
};

// live-tile enumeration: region A = m-tiles [0, dead_mt) x all n-tiles, region B = m-tiles [dead_mt, ntm) x n-tiles [dead_nt, ntn)
struct TileMap {
  int ntn, ntm, dead_mt, dead_nt, nA, n_live;
  __device__ TileMap(int M, int Nn, int dmt, int dnt, int TN) {
    ntn = Nn / TN; ntm = (M + TM - 1) / TM;
    dead_nt = dnt; dead_mt = dnt > 0 ? (dmt < ntm ? dmt : ntm) : ntm;
    nA = dead_mt * ntn;
    n_live = nA + (ntm - dead_mt) * (ntn - dead_nt);
  }
  __device__ void get(int t, int& mt, int& nt) const {
    if (t < nA) { mt = t / ntn; nt = t - mt * ntn; }
    else { const int u = t - nA, w = ntn - dead_nt; mt = dead_mt + u / w; nt = dead_nt + (u - (u / w) * w); }
  }
};

template <bool F16, int H>
__global__ void __launch_bounds__(TC_THREADS, 1) tc_node_gemm_kernel(TcGemmArgs g) {
  using G = Geo<H>;
  constexpr int TN = H;
  extern __shared__ uint8_t smem_raw[];
  const Carve cv = carve_smem<H>(smem_raw);
  Control* ctl = cv.ctl;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const TileMap tm(g.M, g.Nn, g.dead_mt, g.dead_nt, TN);
  const int n_tiles = tm.n_live;
  const int n_my = ((int)blockIdx.x < n_tiles) ? (n_tiles - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  if (n_my == 0) return;
  const int halves = g.K / TKC, chunks = F16 ? halves / 2 : halves;
  const bool gprof = (tc_debug() & 512) && blockIdx.x == 0;
  const long long k0 = gprof ? tc_clock() : 0;
  pdl_trigger();
  tc_begin(ctl, warp);
  pdl_wait();
  const long long k1 = gprof ? tc_clock() : 0;
  if (gprof && threadIdx.x == 0) { atomicAdd(&g_tc_prof[16], (unsigned long long)(k1 - k0)); atomicAdd(&g_tc_prof[23], 1ull); }

  if (warp < EPI_WARPS) {
    // Epilogue.  tcgen05.ld gives each thread one accumulator ROW; storing rows directly would make every
    // STG.128 touch 32 different rows (32 L1 wavefronts per 512 bytes).  Each 32x32 block is
    // therefore transposed through a per-warp shared buffer so that 8 lanes cover 128 contiguous bytes of one row
    // (4 rows = 4 wavefronts per instruction).
    float* T = reinterpret_cast<float*>(cv.extra) + warp * (32 * GEMM_T_STRIDE);
    const int tr = lane >> 3, tc4 = (lane & 7) * 4;
    for (int it = 0; it < n_my; ++it) {
      int mt_, nt_;
      tm.get(blockIdx.x + it * gridDim.x, mt_, nt_);
      const int m0 = mt_ * TM, n0 = nt_ * TN;
      const int a = it & 1;
      const long long e0 = gprof ? tc_clock() : 0;
      mbar_wait(&ctl->acc_full[a], (it >> 1) & 1);
      tc_fence_after();
      const long long e1 = gprof ? tc_clock() : 0;
      if (gprof && threadIdx.x == 0) atomicAdd(&g_tc_prof[17], (unsigned long long)(e1 - (it == 0 ? k1 : e0)));   // epilogue waits for the accumulator
      const uint32_t taddr = ctl->tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(a * ACC_STRIDE);
#pragma unroll 1
      for (int cb = 0; cb < ((tc_debug() & 4) ? 0 : TN / 32); ++cb) {
        const int n = n0 + cb * 32 + tc4;
        const float4 bias = __ldg(reinterpret_cast<const float4*>(g.bias + n));
        float v[32];
        tmem_ld32(taddr + cb * 32, v);
#pragma unroll
        for (int q = 0; q < 8; ++q)
          *reinterpret_cast<float4*>(T + lane * GEMM_T_STRIDE + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        __syncwarp();
        const f32x2 ip = pk2(g.inv_scale, g.inv_scale), b01 = pk2(bias.x, bias.y), b23 = pk2(bias.z, bias.w);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int rl = 4 * i + tr;
          const int row = m0 + warp * 32 + rl;
          const float4 x = *reinterpret_cast<const float4*>(T + rl * GEMM_T_STRIDE + tc4);
          if (row < g.M) {
            f32x2 x01 = pk2(x.x, x.y), x23 = pk2(x.z, x.w);
            if (F16) { x01 = fma2(x01, ip, b01); x23 = fma2(x23, ip, b23); }
            else { x01 = add2(x01, b01); x23 = add2(x23, b23); }
            float4 o;
            upk2(x01, o.x, o.y); upk2(x23, o.z, o.w);
            if (!(tc_debug() & 32)) *reinterpret_cast<float4*>(g.C + (size_t)row * g.ldc + n) = o;
          }
        }
        __syncwarp();
      }
      if (gprof && threadIdx.x == 0) atomicAdd(&g_tc_prof[18], (unsigned long long)(tc_clock() - e1));             // epilogue work of one tile
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&ctl->epi_done[a]);
    }
  } else if (warp < MMA_WARP) {
    // same coalesced mapping as the edge kernels: warp pw owns rows [16 pw, 16 pw + 16), lane = (sub-row, 16-byte piece)
    const int ptid = threadIdx.x - EPI_WARPS * 32;
    const int pw = ptid >> 5, sr = lane >> 3, pc = lane & 7;
    uint32_t gc = 0;
    auto load_half = [&](int m0, int hf, float4 (&v)[4]) {
      const int k = hf * TKC + 4 * pc;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int m = m0 + 16 * pw + 4 * sr + i;
        float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
        if (m < g.M && !(tc_debug() & 2)) x = *reinterpret_cast<const float4*>(g.A + (size_t)m * g.lda + k);
        v[i] = x;
      }
    };
    const long long p0 = gprof ? tc_clock() : 0;
    // Two register sets, each holding one K-chunk (a full pipeline stage) of this thread's rows: the loads of chunk q+2 are
    // issued right after chunk q has been converted and stored, i.e. they have a whole chunk period more than the L2
    // latency before they are needed (one-ahead prefetch left the loop bound by that latency: 1.8 k cycles of the MMA
    // thread's 3.5 k per chunk were spent waiting for the operand).
    constexpr int HPC = F16 ? 2 : 1;
    auto tile_m0 = [&](int it) { int mt_, nt_; tm.get(blockIdx.x + it * gridDim.x, mt_, nt_); return mt_ * TM; };
    const int total = n_my * chunks;
    auto load_chunk = [&](int q, float4 (&buf)[HPC][4]) {
      const int it = q / chunks, kc = q - it * chunks;
      const int m0 = tile_m0(it);
#pragma unroll
      for (int h = 0; h < HPC; ++h) load_half(m0, kc * HPC + h, buf[h]);
    };
    auto stage_chunk = [&](int q, float4 (&buf)[HPC][4]) {
      const int s = gc & 1;
      mbar_wait(&ctl->empty[s], ((gc >> 1) & 1) ^ 1);
      char* st = cv.stages + (size_t)s * G::STAGE_BYTES;
#pragma unroll
      for (int h = 0; h < HPC; ++h)
#pragma unroll
        for (int i = 0; i < 4; ++i) store_piece<F16>(st, 16 * pw + 4 * sr + i, h, pc, buf[h][i]);
      // fence.proxy.async waits for every outstanding load of the thread (FENCE.VIEW.ASYNC stalls on the long scoreboard,
      // profiles/r1 source view): loads issued BEFORE it put a full L2 round trip between the stores and the arrive, on the
      // MMA thread's critical path (wait-X 1.8 k cycles/chunk).  Issue the next loads after the hand-off instead.
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&ctl->full_x[s]);
      if (q + 2 < total) load_chunk(q + 2, buf);
      ++gc;
    };
    float4 bufA[HPC][4], bufB[HPC][4];
    load_chunk(0, bufA);
    if (total > 1) load_chunk(1, bufB);
    for (int q = 0; q < total; q += 2) {
      stage_chunk(q, bufA);
      if (q + 1 < total) stage_chunk(q + 1, bufB);
    }
    if (gprof && ptid == 0) atomicAdd(&g_tc_prof[19], (unsigned long long)(tc_clock() - p0));    // producers: all tiles of this CTA
  } else if (warp == MMA_WARP) {
    if (lane == 0) mma_role<F16, H>(ctl, cv.stages, n_my, chunks, 0);
    __syncwarp();
  } else {
    if (lane == 0) {
      uint32_t gc = 0;
      for (int it = 0; it < n_my; ++it) {
        int mt_, nt;
        tm.get(blockIdx.x + it * gridDim.x, mt_, nt);
        tma_role<H>(ctl, cv.stages, g.Bhi + (size_t)nt * chunks * G::B_CHUNK_FLOATS, g.Blo + (size_t)nt * chunks * G::B_CHUNK_FLOATS, gc, chunks);
      }
    }
    __syncwarp();
  }
  const long long k2 = gprof ? tc_clock() : 0;
  tc_end(ctl, warp);
  if (gprof && threadIdx.x == 0) {
    atomicAdd(&g_tc_prof[20], (unsigned long long)(k2 - k1));            // thread 0 (epilogue warp 0): begin -> before teardown
    atomicAdd(&g_tc_prof[21], (unsigned long long)(tc_clock() - k2));    // teardown (syncthreads + TMEM dealloc)
    atomicAdd(&g_tc_prof[22], (unsigned long long)n_my);
  }
}

// =====================================================================================================
// fused node MLP (egnn_new.py:48-58): h <- h + W4 SiLU(W3 [h | agg/norm] + b3) + b4 for one 128-row tile per CTA.
// Phase 1 is a node GEMM as above, its producers build the A operand from h and agg/norm (K = 2H, accumulator 0).  Its
// epilogue does not go to global memory: the four epilogue warps apply bias + SiLU to the accumulator and write the result,
// already split and swizzled, into the A slots of the stage ring, i.e. they ARE the producers of phase 2 (K = H,
// accumulator 1), whose weight chunks the bulk-copy thread streams right behind those of phase 1.  The phase-2 epilogue adds
// bias and residual, stores the new h in place (rows are private to the CTA) and re-arms the aggregate.  One launch and one
// [N,H] round trip through global memory less than two node GEMMs.
// =====================================================================================================
struct TcMlpArgs {
  const float* h; int ldh;                      // A1 of phase 1, residual of phase 2, output (in place)
  const float* agg; int ldagg; float div;       // A2 of phase 1 (exact division), zeroed at the end
  const int32_t* deg;                           // != nullptr ('mean' aggregation): row m is divided by max(deg[m], 1) instead
  const float* W3hi; const float* W3lo;         // [1][2H/kc][8192] images
  const float* W4hi; const float* W4lo;         // [1][H/kc][8192]
  const float* b3; const float* b4;
  float inv3, inv4;                             // 3xFP16: 1 / weight scale; 1 for 3xTF32
  float* hout; float* zero; int M;
  int32_t* status;
};

template <bool F16, int H>
__global__ void __launch_bounds__(TC_THREADS, 1) tc_node_mlp_kernel(TcMlpArgs g) {
  using G = Geo<H>;
  constexpr int TN = H;
  extern __shared__ uint8_t smem_raw[];
  const Carve cv = carve_smem<H>(smem_raw);
  Control* ctl = cv.ctl;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ntm = (g.M + TM - 1) / TM;
  const int n_my = ((int)blockIdx.x < ntm) ? (ntm - (int)blockIdx.x + (int)gridDim.x - 1) / (int)gridDim.x : 0;
  if (n_my == 0) return;
  constexpr int KPC = F16 ? TKC16 : TKC;        // k-values per pipeline chunk
  constexpr int CB_PER_CHUNK = KPC / 32;        // 32-column accumulator blocks per phase-2 chunk
  constexpr int C1 = 2 * H / KPC, C2 = H / KPC, CT = C1 + C2;
  constexpr int HPC = F16 ? 2 : 1;
  pdl_trigger();
  tc_begin(ctl, warp);
  pdl_wait();

  if (warp < EPI_WARPS) {
    float* T = reinterpret_cast<float*>(cv.extra) + warp * (32 * GEMM_T_STRIDE);
    const int tr = lane >> 3, tc4 = (lane & 7) * 4;
    for (int it = 0; it < n_my; ++it) {
      const int m0 = (blockIdx.x + it * gridDim.x) * TM;
      const uint32_t tbase = ctl->tmem_base + ((uint32_t)(warp * 32) << 16);
      // ---- phase-1 epilogue = phase-2 producer
      mbar_wait(&ctl->acc_full[0], it & 1);
      tc_fence_after();
      const uint32_t q0 = (uint32_t)it * CT + C1;             // global index of the first phase-2 chunk
      const int myrow = warp * 32 + lane;
#pragma unroll 1
      for (int cb = 0; cb < TN / 32; ++cb) {
        const uint32_t q = q0 + cb / CB_PER_CHUNK;
        const int s = q & 1;
        if (cb % CB_PER_CHUNK == 0) mbar_wait(&ctl->empty[s], ((q >> 1) & 1) ^ 1);
        char* st = cv.stages + (size_t)s * G::STAGE_BYTES;
        float v[32];
        tmem_ld32(tbase + cb * 32, v);
        const f32x2 ip = pk2(g.inv3, g.inv3);
#pragma unroll
        for (int p8 = 0; p8 < 8; ++p8) {
          const float4 bb = __ldg(reinterpret_cast<const float4*>(g.b3 + cb * 32 + 4 * p8));
          f32x2 x01 = pk2(v[4 * p8], v[4 * p8 + 1]), x23 = pk2(v[4 * p8 + 2], v[4 * p8 + 3]);
          if (F16) { x01 = fma2(x01, ip, pk2(bb.x, bb.y)); x23 = fma2(x23, ip, pk2(bb.z, bb.w)); }
          else { x01 = add2(x01, pk2(bb.x, bb.y)); x23 = add2(x23, pk2(bb.z, bb.w)); }
          x01 = silu2(x01); x23 = silu2(x23);
          float4 x;
          upk2(x01, x.x, x.y); upk2(x23, x.z, x.w);
          store_piece<F16>(st, myrow, cb % CB_PER_CHUNK, p8, x);
        }
        if (cb % CB_PER_CHUNK == CB_PER_CHUNK - 1) {
          fence_proxy_async();
          __syncwarp();
          if (lane == 0) mbar_arrive_n(&ctl->full_x[s], PROD_WARPS / EPI_WARPS);
        }
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&ctl->epi_done[0]);
      // ---- phase-2 epilogue: h <- h + acc * inv4 + b4, aggregate re-armed
      mbar_wait(&ctl->acc_full[1], it & 1);
      tc_fence_after();
      const uint32_t taddr = tbase + (uint32_t)ACC_STRIDE;
      auto load_res = [&](int cb, float4 (&rr)[8]) {
        const int n = cb * 32 + tc4;
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int row = m0 + warp * 32 + 4 * i + tr;
          rr[i] = row < g.M ? *reinterpret_cast<const float4*>(g.h + (size_t)row * g.ldh + n) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
      };
      auto do_block = [&](int cb, const float4 (&rr)[8]) {
        const int n = cb * 32 + tc4;
        const float4 bias = __ldg(reinterpret_cast<const float4*>(g.b4 + n));
        float v[32];
        tmem_ld32(taddr + cb * 32, v);
#pragma unroll
        for (int q = 0; q < 8; ++q)
          *reinterpret_cast<float4*>(T + lane * GEMM_T_STRIDE + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
        __syncwarp();
        const f32x2 ip = pk2(g.inv4, g.inv4), b01 = pk2(bias.x, bias.y), b23 = pk2(bias.z, bias.w);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const int rl = 4 * i + tr;
          const int row = m0 + warp * 32 + rl;
          const float4 x = *reinterpret_cast<const float4*>(T + rl * GEMM_T_STRIDE + tc4);
          if (row < g.M) {
            f32x2 x01 = pk2(x.x, x.y), x23 = pk2(x.z, x.w);
            if (F16) { x01 = fma2(x01, ip, b01); x23 = fma2(x23, ip, b23); }
            else { x01 = add2(x01, b01); x23 = add2(x23, b23); }
            x01 = add2(pk2(rr[i].x, rr[i].y), x01); x23 = add2(pk2(rr[i].z, rr[i].w), x23);
            float4 o;
            upk2(x01, o.x, o.y); upk2(x23, o.z, o.w);
            *reinterpret_cast<float4*>(g.hout + (size_t)row * g.ldh + n) = o;
            *reinterpret_cast<float4*>(g.zero + (size_t)row * g.ldagg + n) = make_float4(0.f, 0.f, 0.f, 0.f);
          }
        }
        __syncwarp();
      };
      float4 ra[8], rb[8];
      load_res(0, ra);
#pragma unroll 1
      for (int cb = 0; cb < TN / 32; cb += 2) {
        load_res(cb + 1, rb);
        do_block(cb, ra);
        if (cb + 2 < TN / 32) load_res(cb + 2, ra);
        do_block(cb + 1, rb);
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(&ctl->epi_done[1]);
    }
  } else if (warp < MMA_WARP) {
    // producers: phase-1 chunks only (global chunk indices it*CT + kc, kc < C1); two register sets, loads two chunks ahead
    const int ptid = threadIdx.x - EPI_WARPS * 32;
    const int pw = ptid >> 5, sr = lane >> 3, pc = lane & 7;
    const int total = n_my * C1;
    auto load_chunk = [&](int j, float4 (&buf)[HPC][4]) {
      const int it = j / C1, kc = j - it * C1;
      const int m0 = (blockIdx.x + it * gridDim.x) * TM;
#pragma unroll
      for (int h = 0; h < HPC; ++h) {
        const int k = (kc * HPC + h) * TKC + 4 * pc;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int m = m0 + 16 * pw + 4 * sr + i;
          float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
          if (m < g.M) x = k < H ? *reinterpret_cast<const float4*>(g.h + (size_t)m * g.ldh + k)
                                    : *reinterpret_cast<const float4*>(g.agg + (size_t)m * g.ldagg + (k - H));
          buf[h][i] = x;
        }
      }
    };
    auto stage_chunk = [&](int j, float4 (&buf)[HPC][4]) {
      const int it = j / C1, kc = j - it * C1;
      const uint32_t q = (uint32_t)it * CT + kc;
      const int s = q & 1;
      mbar_wait(&ctl->empty[s], ((q >> 1) & 1) ^ 1);
      char* st = cv.stages + (size_t)s * G::STAGE_BYTES;
#pragma unroll
      for (int h = 0; h < HPC; ++h) {
        const bool second = (kc * HPC + h) * TKC + 4 * pc >= H;       // aggregate columns: exact division by the normalisation
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float4 x = buf[h][i];
          if (second) {
            const int m = (blockIdx.x + it * gridDim.x) * TM + 16 * pw + 4 * sr + i;
            const float dv = g.deg ? (float)max(m < g.M ? g.deg[m] : 1, 1) : g.div;
            x.x = __fdiv_rn(x.x, dv); x.y = __fdiv_rn(x.y, dv); x.z = __fdiv_rn(x.z, dv); x.w = __fdiv_rn(x.w, dv);
          }
          store_piece<F16>(st, 16 * pw + 4 * sr + i, h, pc, x);
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive(&ctl->full_x[s]);
      if (j + 2 < total) load_chunk(j + 2, buf);      // after the fence: see tc_node_gemm_kernel
    };
    float4 bufA[HPC][4], bufB[HPC][4];
    load_chunk(0, bufA);
    if (total > 1) load_chunk(1, bufB);
    for (int j = 0; j < total; j += 2) {
      stage_chunk(j, bufA);
      if (j + 1 < total) stage_chunk(j + 1, bufB);
    }
  } else if (warp == MMA_WARP) {
    if (lane == 0) {
      uint32_t q = 0;
      for (int it = 0; it < n_my; ++it) {
#pragma unroll 1
        for (int ph = 0; ph < 2; ++ph) {
          mbar_wait(&ctl->epi_done[ph], (it & 1) ^ 1);        // accumulator ph drained by the epilogue of the previous tile
          tc_fence_after();
          const uint32_t d = ctl->tmem_base + (uint32_t)(ph * ACC_STRIDE);
          const int nchunks = ph == 0 ? C1 : C2;
          for (int kc = 0; kc < nchunks; ++kc, ++q) {
            const int s = q & 1;
            const uint32_t par = (q >> 1) & 1;
            mbar_wait(&ctl->full_w[s], par);
            mbar_wait(&ctl->full_x[s], par);
            tc_fence_after();
            mma_issue_chunk<F16, H>(d, cv.stages + (size_t)s * G::STAGE_BYTES, kc == 0);
            umma_commit(&ctl->empty[s]);
          }
          umma_commit(&ctl->acc_full[ph]);
        }
      }
    }
    __syncwarp();
  } else {
    if (lane == 0) {
      uint32_t gc = 0;
      for (int it = 0; it < n_my; ++it) {
        tma_role<H>(ctl, cv.stages, g.W3hi, g.W3lo, gc, C1);
        tma_role<H>(ctl, cv.stages, g.W4hi, g.W4lo, gc, C2);
      }
    }
    __syncwarp();
  }
  tc_end(ctl, warp);
}

// =====================================================================================================
// fused node block (CTA pairs, 3xFP16): everything between the two edge kernels of an equivariant block in one launch.
//   phase 1   hid = SiLU(W3 [h | agg/norm] + b3)            (egnn_new.py:48-58, K = 2H)   -> accumulator 0
//   phase 2   h  <- h + W4 hid + b4, agg re-armed                                          -> accumulator 1
//   phase 3   P   = Wq h + bq for every live H-wide column tile of the merged first layers (this block's coordinate MLPs |
//             the next block's edge MLP, DESIGN §2.4)                                      -> accumulators alternate
// A CTA pair owns 2 x 128 node rows (tcgen05 cta_group::2, M = 256; each CTA keeps its own rows).  The A operand of phases 2
// and 3 never leaves the SM: the epilogue warps write SiLU(hid) resp. the new h, already split and swizzled, into the
// resident A slots (K = H = 4 chunks of 32 KB), so h is converted to the 3xFP16 operand format ONCE per block instead of once
// per column tile (the separate merged GEMM rebuilt its A operand for each of its 4-6 column tiles, and its producers, not the
// tensor pipe, bounded it).  Phase 1 streams its 8 A chunks through the same slots.  Each CTA streams only its half of the
// weight columns (B split along N): 32 KB per k-chunk and CTA.
// Barriers: full_a / epi_done / w_peer live in the leader (cluster rank 0), whose MMA thread issues for both CTAs; the peer's
// warps arrive through the cluster address space; e0 / e3 / empty_w / acc_full are multicast commits.  A slot is written four
// times per item (phase-1 chunks 0..3, chunks 4..7, hid, new h): full_a completes once per write.
// A parity wait can only tell "the phase I expect" from "the next one", so every waiter follows its barrier phase by phase:
// the producers' second write waits for e0 (phase-1 chunk 0..3 read), their first write of the NEXT item for e3 (last
// phase-3 read), one completion per item each; the epilogue's writes are ordered by acc_full (all MMAs of the phase done).
// =====================================================================================================
// x / d from the reciprocal and one residual correction: q = x r; q += (x - q d) r.  Correctly rounded except for results within
// ~2^-46 relative of a rounding boundary (the IEEE division it replaces was 20 % of the producers' instructions); finite inputs only.
__device__ __forceinline__ float div_by(float x, float d, float r) { const float q = x * r; return fmaf(fmaf(-q, d, x), r, q); }

struct TcBlockArgs {
  float* h; int ldh;                          // [M][H], updated in place
  float* agg; int ldagg; float div;           // raw receiver sums: A2 of phase 1 (divided by div), zeroed by phase 2
  const int32_t* deg;                         // != nullptr ('mean' aggregation): row m is divided by max(deg[m], 1) instead
  const float *W3hi, *W3lo, *W4hi, *W4lo;     // node_mlp images
  const float *Wqhi, *Wqlo;                   // merged first-layer images, [Nn/H][H/64][H x 128 B]
  const float *b3, *b4, *bq;
  float inv3, inv4, invq, s4;                 // 1 / weight scale per image (powers of two); s4 = 1 / inv4
  float* P; int ldp; int Nn;
  int M; int dead_mt; int dead_nt;            // column tiles < dead_nt are not needed for row tiles >= dead_mt
};
struct BlockControl {
  uint64_t full_a[4], e0[4], e3[4];
  uint64_t pre_done;                          // leader: the phase-2 accumulator holds (h + b4) * s4 in both CTAs (count 2 * EPI_WARPS)
  uint64_t full_w[2], w_peer[2], empty_w[2];
  uint64_t acc_full[2], epi_done[2];
  uint32_t tmem_base, pad;
};
static_assert(sizeof(BlockControl) <= kControlBytes, "BlockControl grew");
template <int H> constexpr size_t block_smem_bytes() {
  return 1024 + (size_t)(H / TKC16) * 2 * A_CHUNK_BYTES + 2 * (size_t)(H * 128) + kControlBytes + sizeof(float) * EPI_WARPS * 32 * GEMM_T_STRIDE;
}

template <int H>
__global__ void __launch_bounds__(TC_THREADS, 1) tc_node_block_kernel(TcBlockArgs g) {
  using G = Geo<H>;
  constexpr int C1 = 2 * H / TKC16, C2 = H / TKC16;      // k-chunks of phase 1; of phase 2 and of one column tile of phase 3
  constexpr int NSLOT = C2;                                 // resident A slots (K = H)
  constexpr int SLOT_BYTES = 2 * A_CHUNK_BYTES;             // hi | lo
  constexpr int HB = (H / 2) * 128;                         // one k-chunk of this CTA's weight-column half (hi or lo)
  constexpr int WST_BYTES = 2 * HB;
  constexpr uint32_t IDESC = (1u << 4) | ((uint32_t)(H >> 3) << 17) | ((uint32_t)((2 * TM) >> 4) << 24);   // F16 x F16 -> F32, N = H, M = 256
  static_assert(C1 == 2 * NSLOT && NSLOT <= 4, "slot ring");
  extern __shared__ uint8_t smem_raw[];
  char* const slots = reinterpret_cast<char*>(smem_raw) + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);
  char* const wst = slots + NSLOT * SLOT_BYTES;
  BlockControl* ctl = reinterpret_cast<BlockControl*>(wst + 2 * WST_BYTES);
  float* const Tall = reinterpret_cast<float*>(reinterpret_cast<char*>(ctl) + kControlBytes);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int rank = (int)cluster_ctarank(), pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int ntm = (g.M + TM - 1) / TM, nmp = (ntm + 1) / 2, ntn = g.Nn / H;

  pdl_trigger();
  if (threadIdx.x == 0) {
    for (int k = 0; k < 4; ++k) { mbar_init(&ctl->full_a[k], 2 * PROD_WARPS); mbar_init(&ctl->e0[k], 1); mbar_init(&ctl->e3[k], 1); }
    for (int k = 0; k < 2; ++k) {
      mbar_init(&ctl->full_w[k], 1); mbar_init(&ctl->w_peer[k], 1); mbar_init(&ctl->empty_w[k], 1);
      mbar_init(&ctl->acc_full[k], 1); mbar_init(&ctl->epi_done[k], 2 * EPI_WARPS);
    }
    mbar_init(&ctl->pre_done, 2 * EPI_WARPS);
    fence_barrier_init();
  }
  __syncthreads();
  if (warp == MMA_WARP) tmem_alloc2(&ctl->tmem_base, 512);
  tc_fence_before();
  cluster_sync_all();
  tc_fence_after();
  auto kernel_end = [&]() {
    tc_fence_before();
    cluster_sync_all();
    if (warp == MMA_WARP) tmem_dealloc2(ctl->tmem_base, 512);
  };
  pdl_wait();
  const int n_items = pair < nmp ? (nmp - pair + npairs - 1) / npairs : 0;
  if (n_items == 0) { kernel_end(); return; }
  auto item_mp = [&](int it) { return pair + it * npairs; };
  // first live column tile of an item: both row tiles of the pair must lie in the dead region for a column tile to be skipped
  auto item_nt0 = [&](int it) { return (g.dead_nt > 0 && 2 * item_mp(it) >= g.dead_mt) ? g.dead_nt : 0; };
  const uint32_t l_full_a = leader_addr(&ctl->full_a[0]), l_epi_done = leader_addr(&ctl->epi_done[0]), l_w_peer = leader_addr(&ctl->w_peer[0]);
  const uint32_t l_pre_done = leader_addr(&ctl->pre_done);
  auto arrive_n = [&](uint32_t addr, uint32_t n) { asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0], %1;" ::"r"(addr), "r"(n) : "memory"); };

  if (warp < EPI_WARPS) {
    // ---------------------------------------------------------------------------------------------- epilogue warps
    float* T = Tall + warp * (32 * GEMM_T_STRIDE);
    const int tr = lane >> 3, tc4 = (lane & 7) * 4;
    const uint32_t tbase = ctl->tmem_base + ((uint32_t)(warp * 32) << 16);
    const int myrow = warp * 32 + lane;
    uint32_t u = 0;                              // accumulator uses so far (use u: accumulator u & 1, phase (u >> 1) & 1)
    for (int it = 0; it < n_items; ++it) {
      const int m0 = (2 * item_mp(it) + rank) * TM;
      // ---- while phase 1 runs: the residual goes INTO the phase-2 accumulator, (h + b4) * s4 (s4 a power of two: exact), and
      // the phase-2 MMAs accumulate on top of it.  The phase-2 epilogue then needs no global load before it can hand the new h
      // to phase 3 (it used to wait an L2 round trip per 32 columns, 20 k cycles per item on the MMA thread's critical path).
      // Row-per-thread loads: 32 rows x 16 bytes per instruction, each row's 128-byte line reused by the next 7 loads.
      {
        const uint32_t taddr = tbase + (uint32_t)(((u + 1) & 1) * ACC_STRIDE);      // free: this warp drained its previous use
        const int row = m0 + myrow;
        const float* hr = g.h + (size_t)row * g.ldh;
        const f32x2 sp = pk2(g.s4, g.s4);
#pragma unroll 1
        for (int cb = 0; cb < H / 32; ++cb) {
          float v[32];
#pragma unroll
          for (int p8 = 0; p8 < 8; ++p8) {
            const float4 x = row < g.M ? *reinterpret_cast<const float4*>(hr + cb * 32 + 4 * p8) : make_float4(0.f, 0.f, 0.f, 0.f);
            const float4 bb = __ldg(reinterpret_cast<const float4*>(g.b4 + cb * 32 + 4 * p8));
            upk2(mul2(add2(pk2(x.x, x.y), pk2(bb.x, bb.y)), sp), v[4 * p8], v[4 * p8 + 1]);
            upk2(mul2(add2(pk2(x.z, x.w), pk2(bb.z, bb.w)), sp), v[4 * p8 + 2], v[4 * p8 + 3]);
          }
          tmem_st32(taddr + cb * 32, v);
        }
        tmem_wait_st();
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(l_pre_done);
      }
      // ---- phase-1 epilogue = producer of the phase-2 A operand: SiLU(acc * inv3 + b3) -> slots (third write of a slot)
      {
        mbar_wait(&ctl->acc_full[u & 1], (u >> 1) & 1);
        tc_fence_after();
        const uint32_t taddr = tbase + (uint32_t)((u & 1) * ACC_STRIDE);
        const f32x2 ip = pk2(g.inv3, g.inv3);
#pragma unroll 1
        for (int cb = 0; cb < H / 32; ++cb) {
          const int kc = cb >> 1;
          char* st = slots + (size_t)kc * SLOT_BYTES;
          float v[32];
          tmem_ld32(taddr + cb * 32, v);
#pragma unroll
          for (int p8 = 0; p8 < 8; ++p8) {
            const float4 bb = __ldg(reinterpret_cast<const float4*>(g.b3 + cb * 32 + 4 * p8));
            f32x2 x01 = fma2(pk2(v[4 * p8], v[4 * p8 + 1]), ip, pk2(bb.x, bb.y));
            f32x2 x23 = fma2(pk2(v[4 * p8 + 2], v[4 * p8 + 3]), ip, pk2(bb.z, bb.w));
            silu4q(x01, x23);
            float4 x;
            upk2(x01, x.x, x.y); upk2(x23, x.z, x.w);
            store_piece<true>(st, myrow, cb & 1, p8, x);
          }
          if (cb & 1) {
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) arrive_n(l_full_a + 8u * (uint32_t)kc, PROD_WARPS / EPI_WARPS);
          }
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(l_epi_done + 8u * (u & 1));
        ++u;
      }
      // ---- phase-2 epilogue: new h = acc * inv4 (the accumulator started from (h + b4) * s4).  First the phase-3 A operand
      // (fourth write of a slot; phase 3 starts as soon as all four slots are handed over), then the global side: h in place,
      // aggregate re-armed, each 32x32 block through the per-warp buffer so that 8 lanes cover 128 contiguous bytes of a row.
      {
        mbar_wait(&ctl->acc_full[u & 1], (u >> 1) & 1);
        tc_fence_after();
        const uint32_t taddr = tbase + (uint32_t)((u & 1) * ACC_STRIDE);
        const f32x2 ip = pk2(g.inv4, g.inv4);
#pragma unroll 1
        for (int cb = 0; cb < H / 32; ++cb) {
          const int kc = cb >> 1;
          char* st = slots + (size_t)kc * SLOT_BYTES;
          float v[32];
          tmem_ld32(taddr + cb * 32, v);
#pragma unroll
          for (int p8 = 0; p8 < 8; ++p8) {
            float4 x;
            upk2(mul2(pk2(v[4 * p8], v[4 * p8 + 1]), ip), x.x, x.y); upk2(mul2(pk2(v[4 * p8 + 2], v[4 * p8 + 3]), ip), x.z, x.w);
            store_piece<true>(st, myrow, cb & 1, p8, x);
          }
          if (cb & 1) {
            fence_proxy_async();
            __syncwarp();
            if (lane == 0) arrive_n(l_full_a + 8u * (uint32_t)kc, PROD_WARPS / EPI_WARPS);
          }
        }
#pragma unroll 1
        for (int cb = 0; cb < H / 32; ++cb) {
          const int n = cb * 32 + tc4;
          float v[32];
          tmem_ld32(taddr + cb * 32, v);
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(T + lane * GEMM_T_STRIDE + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          __syncwarp();
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rl = 4 * i + tr;
            const int row = m0 + warp * 32 + rl;
            const float4 x = *reinterpret_cast<const float4*>(T + rl * GEMM_T_STRIDE + tc4);
            float4 o;
            upk2(mul2(pk2(x.x, x.y), ip), o.x, o.y); upk2(mul2(pk2(x.z, x.w), ip), o.z, o.w);
            if (row < g.M) {
              *reinterpret_cast<float4*>(g.h + (size_t)row * g.ldh + n) = o;
              *reinterpret_cast<float4*>(g.agg + (size_t)row * g.ldagg + n) = make_float4(0.f, 0.f, 0.f, 0.f);
            }
          }
          __syncwarp();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(l_epi_done + 8u * (u & 1));
        ++u;
      }
      // ---- phase-3 epilogues: P[:, column tile] = acc * invq + bq
      for (int nt = item_nt0(it); nt < ntn; ++nt) {
        mbar_wait(&ctl->acc_full[u & 1], (u >> 1) & 1);
        tc_fence_after();
        const uint32_t taddr = tbase + (uint32_t)((u & 1) * ACC_STRIDE);
        const f32x2 ip = pk2(g.invq, g.invq);
#pragma unroll 1
        for (int cb = 0; cb < H / 32; ++cb) {
          const int n = nt * H + cb * 32 + tc4;
          const float4 bias = __ldg(reinterpret_cast<const float4*>(g.bq + n));
          float v[32];
          tmem_ld32(taddr + cb * 32, v);
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(T + lane * GEMM_T_STRIDE + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          __syncwarp();
          const f32x2 b01 = pk2(bias.x, bias.y), b23 = pk2(bias.z, bias.w);
#pragma unroll
          for (int i = 0; i < 8; ++i) {
            const int rl = 4 * i + tr;
            const int row = m0 + warp * 32 + rl;
            const float4 x = *reinterpret_cast<const float4*>(T + rl * GEMM_T_STRIDE + tc4);
            float4 o;
            upk2(fma2(pk2(x.x, x.y), ip, b01), o.x, o.y); upk2(fma2(pk2(x.z, x.w), ip, b23), o.z, o.w);
            if (row < g.M) *reinterpret_cast<float4*>(g.P + (size_t)row * g.ldp + n) = o;
          }
          __syncwarp();
        }
        tc_fence_before();
        __syncwarp();
        if (lane == 0) mbar_arrive_cluster(l_epi_done + 8u * (u & 1));
        ++u;
      }
    }
  } else if (warp < MMA_WARP) {
    // ---------------------------------------------------------------------------------------------- producers: phase-1 A chunks
    // [h | agg / norm] rows of this CTA's tile, 64 k per chunk, two register sets (loads two chunks ahead, issued after the
    // proxy fence: see tc_node_gemm_kernel)
    const int ptid = threadIdx.x - EPI_WARPS * 32;
    const int pw = ptid >> 5, sr = lane >> 3, pc = lane & 7;
    const int total = n_items * C1;
    const float rdiv = __frcp_rn(g.div);
    auto load_chunk = [&](int j, float4 (&buf)[2][4]) {
      const int it = j / C1, kc = j - it * C1;
      const int m0 = (2 * item_mp(it) + rank) * TM;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const int k = (kc * 2 + hh) * TKC + 4 * pc;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int m = m0 + 16 * pw + 4 * sr + i;
          float4 x = make_float4(0.f, 0.f, 0.f, 0.f);
          if (m < g.M) x = k < H ? *reinterpret_cast<const float4*>(g.h + (size_t)m * g.ldh + k)
                                    : *reinterpret_cast<const float4*>(g.agg + (size_t)m * g.ldagg + (k - H));
          buf[hh][i] = x;
        }
      }
    };
    auto stage_chunk = [&](int j, float4 (&buf)[2][4]) {
      const int it = j / C1, kc = j - it * C1;
      const int slot = kc % NSLOT;
      if (kc >= NSLOT) mbar_wait(&ctl->e0[slot], (uint32_t)it & 1u);            // second write of the slot: phase-1 chunk kc - NSLOT was read
      else if (it > 0) mbar_wait(&ctl->e3[slot], (uint32_t)(it - 1) & 1u);     // first write: the previous item's phase 3 is done with it
      char* st = slots + (size_t)slot * SLOT_BYTES;
#pragma unroll
      for (int hh = 0; hh < 2; ++hh) {
        const bool second = (kc * 2 + hh) * TKC + 4 * pc >= H;          // aggregate columns: exact division by the normalisation
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          float4 x = buf[hh][i];
          if (second) {
            float dv = g.div, rv = rdiv;
            if (g.deg) { const int m = (2 * item_mp(it) + rank) * TM + 16 * pw + 4 * sr + i; dv = (float)max(m < g.M ? g.deg[m] : 1, 1); rv = __frcp_rn(dv); }
            x.x = div_by(x.x, dv, rv); x.y = div_by(x.y, dv, rv); x.z = div_by(x.z, dv, rv); x.w = div_by(x.w, dv, rv);
          }
          store_piece<true>(st, 16 * pw + 4 * sr + i, hh, pc, x);
        }
      }
      fence_proxy_async();
      __syncwarp();
      if (lane == 0) mbar_arrive_cluster(l_full_a + 8u * (uint32_t)slot);
      if (j + 2 < total) load_chunk(j + 2, buf);
    };
    float4 bufA[2][4], bufB[2][4];
    load_chunk(0, bufA);
    if (total > 1) load_chunk(1, bufB);
    for (int j = 0; j < total; j += 2) {
      stage_chunk(j, bufA);
      if (j + 1 < total) stage_chunk(j + 1, bufB);
    }
  } else if (warp == MMA_WARP) {
    if (lane == 0 && rank == 0) {
      // -------------------------------------------------------------------------------------------- MMA issuer (leader)
      const uint32_t tmem = ctl->tmem_base;
      uint32_t gw = 0, u = 0;
      // cycle accounting (instrumented library, flag 512): g_tc_prof[48 + 4 * phase + {0: wait A, 1: wait W, 2: wait peer's W, 3: issue}],
      // [60] accumulator waits, [61] items, [62] whole loop
      const bool bprof = (tc_debug() & 512) != 0;
      long long w_a[3] = {0, 0, 0}, w_w[3] = {0, 0, 0}, w_p[3] = {0, 0, 0}, w_i[3] = {0, 0, 0}, w_acc = 0;
      int ph = 0;
      const long long b0 = bprof ? tc_clock() : 0;
      auto chunk = [&](uint32_t d, int slot, uint32_t a_parity, bool wait_a, bool first, uint64_t* release_a) {
        const int s = gw & 1;
        const uint32_t par = (gw >> 1) & 1;
        long long q0 = 0, q1 = 0, q2 = 0, q3 = 0;
        if (bprof) q0 = tc_clock();
        if (wait_a) mbar_wait_cluster(&ctl->full_a[slot], a_parity);
        if (bprof) q1 = tc_clock();
        mbar_wait(&ctl->full_w[s], par);
        if (bprof) q2 = tc_clock();
        mbar_wait_cluster(&ctl->w_peer[s], par);
        if (bprof) { q3 = tc_clock(); w_a[ph] += q1 - q0; w_w[ph] += q2 - q1; w_p[ph] += q3 - q2; }
        tc_fence_after();
        const uint32_t xhi = smem_u32(slots + (size_t)slot * SLOT_BYTES), xlo = xhi + A_CHUNK_BYTES;
        const uint32_t whi = smem_u32(wst + (size_t)s * WST_BYTES), wlo = whi + HB;
#pragma unroll
        for (int ks = 0; ks < 4; ++ks) {
          const uint32_t ko = ks * 32;
          umma_f16_2cta(d, umma_desc_sw128(xlo + ko), umma_desc_sw128(whi + ko), IDESC, (first && ks == 0) ? 0u : 1u);
          umma_f16_2cta(d, umma_desc_sw128(xhi + ko), umma_desc_sw128(wlo + ko), IDESC, 1u);
          umma_f16_2cta(d, umma_desc_sw128(xhi + ko), umma_desc_sw128(whi + ko), IDESC, 1u);
        }
        umma_commit_2cta(&ctl->empty_w[s]);
        if (release_a) umma_commit_2cta(release_a);
        if (bprof) w_i[ph] += tc_clock() - q3;
        ++gw;
      };
      auto begin_use = [&]() {
        const long long q0 = bprof ? tc_clock() : 0;
        mbar_wait_cluster(&ctl->epi_done[u & 1], ((u >> 1) & 1) ^ 1);     // accumulator drained by both CTAs' epilogue warps
        if (bprof) w_acc += tc_clock() - q0;
        tc_fence_after();
        return tmem + (uint32_t)((u & 1) * ACC_STRIDE);
      };
      auto end_use = [&]() { umma_commit_2cta(&ctl->acc_full[u & 1]); ++u; };
      for (int it = 0; it < n_items; ++it) {
        const uint32_t fa = (uint32_t)it * 4u;      // full_a completions before this item (4 slot writes per item): write k has parity (fa + k) & 1
        ph = 0;
        uint32_t d = begin_use();
        for (int kc = 0; kc < C1; ++kc) chunk(d, kc % NSLOT, (fa + (kc < NSLOT ? 0u : 1u)) & 1u, true, kc == 0, kc < NSLOT ? &ctl->e0[kc] : nullptr);     // slot writes 1, 2
        end_use();
        ph = 1;
        d = begin_use();
        mbar_wait_cluster(&ctl->pre_done, (uint32_t)it & 1u);          // the accumulator holds the residual in both CTAs
        tc_fence_after();
        for (int kc = 0; kc < C2; ++kc) chunk(d, kc, (fa + 2u) & 1u, true, false, nullptr);       // slot write 3 (hid); accumulates onto the residual
        end_use();
        const int nt0 = item_nt0(it);
        ph = 2;
        for (int nt = nt0; nt < ntn; ++nt) {
          d = begin_use();
          for (int kc = 0; kc < C2; ++kc) chunk(d, kc, (fa + 3u) & 1u, nt == nt0, kc == 0, nt == ntn - 1 ? &ctl->e3[kc] : nullptr);   // slot write 4 (new h)
          end_use();
        }
      }
      if (bprof) {
        for (int k = 0; k < 3; ++k) {
          atomicAdd(&g_tc_prof[48 + 4 * k + 0], (unsigned long long)w_a[k]); atomicAdd(&g_tc_prof[48 + 4 * k + 1], (unsigned long long)w_w[k]);
          atomicAdd(&g_tc_prof[48 + 4 * k + 2], (unsigned long long)w_p[k]); atomicAdd(&g_tc_prof[48 + 4 * k + 3], (unsigned long long)w_i[k]);
        }
        atomicAdd(&g_tc_prof[60], (unsigned long long)w_acc); atomicAdd(&g_tc_prof[61], (unsigned long long)n_items);
        atomicAdd(&g_tc_prof[62], (unsigned long long)(tc_clock() - b0));
      }
    } else if (lane == 0) {
      // peer CTA: forward "my weight half of chunk gw has landed" to the leader
      uint32_t total = 0;
      for (int it = 0; it < n_items; ++it) total += C1 + C2 + (uint32_t)(ntn - item_nt0(it)) * C2;
      for (uint32_t gw = 0; gw < total; ++gw) {
        mbar_wait(&ctl->full_w[gw & 1], (gw >> 1) & 1);
        mbar_arrive_cluster(l_w_peer + 8u * (gw & 1));
      }
    }
    __syncwarp();
  } else {
    if (lane == 0) {
      // -------------------------------------------------------------------------------------------- weight stream (both CTAs)
      uint32_t gw = 0;
      auto load = [&](const float* hi, const float* lo, int kc) {
        const int s = gw & 1;
        mbar_wait(&ctl->empty_w[s], ((gw >> 1) & 1) ^ 1);
        char* dst = wst + (size_t)s * WST_BYTES;
        mbar_arrive_expect_tx(&ctl->full_w[s], WST_BYTES);
        bulk_g2s(dst, hi + (size_t)kc * G::B_CHUNK_FLOATS + (size_t)rank * (HB / 4), HB, &ctl->full_w[s]);
        bulk_g2s(dst + HB, lo + (size_t)kc * G::B_CHUNK_FLOATS + (size_t)rank * (HB / 4), HB, &ctl->full_w[s]);
        ++gw;
      };
      for (int it = 0; it < n_items; ++it) {
        for (int kc = 0; kc < C1; ++kc) load(g.W3hi, g.W3lo, kc);
        for (int kc = 0; kc < C2; ++kc) load(g.W4hi, g.W4lo, kc);
        for (int nt = item_nt0(it); nt < ntn; ++nt)
          for (int kc = 0; kc < C2; ++kc) load(g.Wqhi + (size_t)nt * C2 * G::B_CHUNK_FLOATS, g.Wqlo + (size_t)nt * C2 * G::B_CHUNK_FLOATS, kc);
      }
    }
    __syncwarp();
  }
  kernel_end();
}

// =====================================================================================================
// edge kernels
// =====================================================================================================
constexpr int kE1Unroll = 2, kE2Unroll = 2;   // unroll factors of the epilogue's pass-1 and pass-2 loops
constexpr int EPI_T_STRIDE = 36;          // 16-byte aligned rows: conflict-free row-wise STS.128 and column-wise LDS.32
constexpr int NSCAL = 3;                   // scalar buffer sets (the j-th tile of a CTA uses set j % NSCAL)
constexpr int SCAL_WARPS = 2;              // warps 14, 15 of the edge kernels: per-edge scalars one tile ahead of the producers
constexpr int EDGE_THREADS = TC_THREADS + SCAL_WARPS * 32;   // 512

template <int H>
struct EdgeExtra {            // shared memory after Control
  float vec[2][3 * H];     // per MLP: wr, wr0, b2   (the edge-type table tb stays in global/L1)
  float wa[H];                // attention weight (GCL) or w3 (coord)
  float gate4[EPI_WARPS][32]; // GCL pass 2: attention gates of the warp's 32 rows (read back per 4-row chunk)
  float d2[NSCAL][TM], d0[NSCAL][TM];       // per-edge scalars: NSCAL sets so the scalar warps run a full tile ahead of the
  int row[NSCAL][TM], col[NSCAL][TM], type[NSCAL][TM];   // producers while the epilogue still reads the set of the tile before
  union {
    float T[EPI_WARPS][32 * EPI_T_STRIDE];                     // GCL: per-warp transpose buffer
    struct { float dir[NSCAL][3][TM]; float T4[EPI_WARPS][32 * 4]; } c;   // coord: direction of this MLP + small transpose buffer
  } u;
};

struct TcEdgeArgs {
  const float* P; int ldp;
  const float4* x; const float4* cent; const int32_t* gid;
  const int32_t* vrow_ptr; const int32_t* vmap; int n_rows;   // virtual rows [0, vrow_ptr[n_rows]): vmap[v] = edge index or -1 (pad)
  const int32_t *erow, *ecol; const float* ed0; int NL;
  int nm;                                    // MLPs per edge tile: 1 (GCL, reflection-equivariant coord) or 2 (coord + cross)
  const float* W2hi[2]; const float* W2lo[2];   // [8][8192] images
  const float* wr[2]; const float* wr0[2]; const float* tb[2]; const float* b2[2];
  const float* wa; const float* ba;          // GCL attention (nullptr: none) / coord: wa = w3
  float norm_constant, coords_range; int use_tanh;
  float* agg;                                // GCL: [N][H] raw sums
  float4* xagg;                              // coord: [N] raw sums of trans
  float inv_scale[2];                        // 3xFP16: 1 / (X_SCALE * W2 scale) per MLP; 1 for 3xTF32
  int32_t* status;
};

// per-edge scalars of edge tile v0/TM for MLP m (thread pr handles virtual row v0 + pr), written by the scalar warps
template <bool COORD, int H>
__device__ __forceinline__ void edge_scalars(const TcEdgeArgs& a, EdgeExtra<H>* ex, int par, int pr, int v0, int V, int m) {
  const int vr = v0 + pr;
  const int e = vr < V ? a.vmap[vr] : -1;
  int r = -1, c = 0, ty = 0; float d2 = 0.f, d0 = 0.f;
  float dir[3] = {0.f, 0.f, 0.f};
  if (e >= 0) {
    r = a.erow[e]; c = a.ecol[e]; d0 = a.ed0[e];
    const float4 xi = a.x[r], xj = a.x[c];
    const float dx = xi.x - xj.x, dy = xi.y - xj.y, dz = xi.z - xj.z;
    d2 = dx * dx + dy * dy + dz * dz;
    ty = (r < a.NL) == (c < a.NL) ? (r < a.NL ? 1 : 2) : 0;
    if (COORD) {
      if (m == 0) {                                                     // egnn_new.py:300-301 (coord2diff)
        const float den = sqrtf(d2 + 1e-8f) + a.norm_constant;
        dir[0] = dx / den; dir[1] = dy / den; dir[2] = dz / den;
      } else {                                                          // egnn_new.py:312-315 (coord2cross)
        const float4 mu = a.cent[a.gid[r]];
        const float ax = xi.x - mu.x, ay = xi.y - mu.y, az = xi.z - mu.z;
        const float bx = xj.x - mu.x, by = xj.y - mu.y, bz = xj.z - mu.z;
        const float cx = ay * bz - az * by, cy = az * bx - ax * bz, cz = ax * by - ay * bx;
        const float cn = sqrtf(cx * cx + cy * cy + cz * cz) + a.norm_constant;
        dir[0] = cx / cn; dir[1] = cy / cn; dir[2] = cz / cn;
      }
    }
  }
  ex->row[par][pr] = r; ex->col[par][pr] = c; ex->d2[par][pr] = d2; ex->d0[par][pr] = d0; ex->type[par][pr] = ty;
  if (COORD) {
#pragma unroll
    for (int k = 0; k < 3; ++k) ex->u.c.dir[par][k][pr] = dir[k];
  }
}

// Work unit = virtual tile v = edge_tile * nm + m (the m-th MLP over 128 virtual edge rows).  The coordinate update is a sum
// of independent terms per MLP (egnn_new.py:100-109: trans = diff * f(phi) + cross * f(phi_x)), so the two MLPs of an edge tile
// are independent units that add into the same receiver sums: units, not edge tiles, are dealt round-robin to the CTAs (610 edge
// tiles on 148 CTAs would leave 21 % of the machine idle in the last wave; 1220 units leave 9 %).  The j-th unit of a CTA uses
// scalar set j % NSCAL and accumulator j & 1.
//
// PAIR = true (3xFP16 only): the kernel runs as 74 CTA pairs (cluster of 2, tcgen05 cta_group::2).  A pair works on two edge
// tiles at a time (M = 256: each CTA produces, and post-processes, its own 128 rows) and on ONE MLP for the whole launch, whose
// second-layer weights stay in shared memory: each CTA holds the hi and lo images of its half of the H output columns (B is
// split along N between the two CTAs: 128 KB per CTA at H = 256), loaded once before the first tile.  Against PAIR = false
// this removes the per-tile weight stream (256 KB of bulk copies into shared memory per tile and SM) and a third of the tensor
// core's operand reads (per MMA and CTA: A 4 KB + half of B 4 KB instead of 4 + 8) from the L1 data pipe, the busiest unit of
// these kernels (profiles/r2b_edge_ncu.txt).  The leader CTA's MMA thread issues for both CTAs; the peer's producers and
// epilogue warps arrive on the leader's full_x / epi_done barriers through the cluster address space, the commits are multicast.
template <int H, bool PAIR>
struct EdgeGeo {
  static constexpr int STAGE_BYTES = PAIR ? 2 * A_CHUNK_BYTES : Geo<H>::STAGE_BYTES;      // PAIR: the ring holds A chunks only
  static constexpr int HB = (H / 2) * 128;                                                // one k-chunk of this CTA's weight half (hi or lo)
  static constexpr int W_BYTES = PAIR ? (H / TKC16) * 2 * HB : 0;                         // resident weight half: chunks x (hi | lo)
  static constexpr uint32_t IDESC_F16_2CTA = (1u << 4) | ((uint32_t)(H >> 3) << 17) | ((uint32_t)((2 * TM) >> 4) << 24);   // D=F32, A=B=F16, N=H, M=256
};
template <int H, bool PAIR> constexpr size_t edge_smem_base() { return 1024 + (size_t)NSTAGE * EdgeGeo<H, PAIR>::STAGE_BYTES + EdgeGeo<H, PAIR>::W_BYTES + kControlBytes; }

template <bool COORD, bool F16, int H, bool TB, bool PAIR>
__global__ void __launch_bounds__(EDGE_THREADS, 1) tc_edge_kernel(TcEdgeArgs a) {
  static_assert(!PAIR || F16, "the CTA-pair kernel keeps 3xFP16 weight halves resident; 3xTF32 images do not fit");
  using G = Geo<H>;
  using EG = EdgeGeo<H, PAIR>;
  constexpr int TN = H;
  extern __shared__ uint8_t smem_raw[];
  Carve cv;
  {
    const uint32_t base = smem_u32(smem_raw);
    cv.stages = reinterpret_cast<char*>(smem_raw) + ((1024u - (base & 1023u)) & 1023u);
    cv.ctl = reinterpret_cast<Control*>(cv.stages + NSTAGE * EG::STAGE_BYTES + EG::W_BYTES);
    cv.extra = reinterpret_cast<char*>(cv.ctl) + kControlBytes;
  }
  char* const wres = cv.stages + NSTAGE * EG::STAGE_BYTES;      // PAIR: resident weight half, [chunk][hi | lo][H/2 rows x 128 B]
  Control* ctl = cv.ctl;
  EdgeExtra<H>* ex = reinterpret_cast<EdgeExtra<H>*>(cv.extra);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int nm = a.nm;
  constexpr int halves = H / TKC;           // 32-k production steps per unit
  constexpr int HPC = F16 ? 2 : 1;             // production steps per pipeline chunk (stage)
  constexpr int chunks = halves / HPC;
  const int rank = PAIR ? (int)cluster_ctarank() : 0;          // 0 = leader
  // PAIR: pair p of npairs works on MLP p % nm for the whole launch (its weights stay resident) and on the tile pairs
  // p / nm, p / nm + npairs / nm, ...; this CTA takes tile 2 * pair_unit + rank (a tile beyond the end is all padding)
  const int pair = blockIdx.x >> 1, npairs = gridDim.x >> 1;
  const int m_pair = PAIR ? pair % nm : 0, pu0 = PAIR ? pair / nm : 0, pustride = PAIR ? npairs / nm : 1;

  pdl_trigger();
  for (int i = threadIdx.x; i < H; i += EDGE_THREADS) {
    for (int m = 0; m < nm; ++m) {
      float* v = ex->vec[m];
      v[i] = a.wr[m][i]; v[H + i] = a.wr0[m][i]; v[2 * H + i] = a.b2[m][i];
    }
    ex->wa[i] = a.wa ? a.wa[i] : 0.f;
  }
  if constexpr (PAIR) {
    if (threadIdx.x == 0) {
      for (int s = 0; s < NSTAGE; ++s) { mbar_init(&ctl->full_x[s], 2 * PROD_WARPS); mbar_init(&ctl->full_w[s], 1); mbar_init(&ctl->empty[s], 1); }
      for (int k = 0; k < 2; ++k) { mbar_init(&ctl->acc_full[k], 1); mbar_init(&ctl->epi_done[k], 2 * EPI_WARPS); }
      for (int k = 0; k < 3; ++k) { mbar_init(&ctl->scal_full[k], SCAL_WARPS); mbar_init(&ctl->scal_empty[k], EPI_WARPS); }
      mbar_init(&ctl->w_full, 1); mbar_init(&ctl->w_ready, 2);
      fence_barrier_init();
    }
    __syncthreads();
    if (warp == MMA_WARP) tmem_alloc2(&ctl->tmem_base, 512);
    if (warp == TMA_WARP && lane == 0) {
      // the resident weight half: constant data, requested before the dependency wait so it overlaps the predecessor's tail
      mbar_arrive_expect_tx(&ctl->w_full, EG::W_BYTES);
      const float* hi = a.W2hi[m_pair] + (size_t)rank * (EG::HB / 4);
      const float* lo = a.W2lo[m_pair] + (size_t)rank * (EG::HB / 4);
      for (int kc = 0; kc < chunks; ++kc) {
        bulk_g2s(wres + (size_t)kc * 2 * EG::HB, hi + (size_t)kc * G::B_CHUNK_FLOATS, EG::HB, &ctl->w_full);
        bulk_g2s(wres + (size_t)kc * 2 * EG::HB + EG::HB, lo + (size_t)kc * G::B_CHUNK_FLOATS, EG::HB, &ctl->w_full);
      }
    }
    __syncwarp();
    tc_fence_before();
    cluster_sync_all();         // both CTAs' barriers are initialised before anyone arrives remotely; publishes the vectors
    tc_fence_after();
  } else {
    tc_begin(ctl, warp, SCAL_WARPS);        // contains the __syncthreads that publishes the vectors
  }
  auto kernel_end = [&]() {
    if constexpr (PAIR) {
      tc_fence_before();
      cluster_sync_all();       // the peer may still arrive on this CTA's barriers / the leader's MMAs read the peer's shared memory
      if (warp == MMA_WARP) tmem_dealloc2(ctl->tmem_base, 512);
    } else {
      tc_end(ctl, warp);
    }
  };
  pdl_wait();                 // everything above touches only kernel arguments and constant weights
  const int E = a.vrow_ptr[a.n_rows];          // virtual rows: every receiver's edges start at a multiple of kRowChunk
  const int n_tiles_e = (E + TM - 1) / TM;
  const int n_units = PAIR ? (n_tiles_e + 1) / 2 : n_tiles_e * nm;      // PAIR: tile pairs (of this pair's MLP)
  const int u0 = PAIR ? pu0 : (int)blockIdx.x, ustride = PAIR ? pustride : (int)gridDim.x;
  const int n_my = (u0 < n_units) ? (n_units - u0 + ustride - 1) / ustride : 0;
  if (n_my == 0) {
    if (PAIR && warp == TMA_WARP && lane == 0) mbar_wait(&ctl->w_full, 0);      // no shared memory may be freed under a bulk copy in flight
    __syncwarp();
    kernel_end();
    return;
  }
  auto unit_tile = [&](int j, int& m) {
    const int v = u0 + j * ustride;
    if constexpr (PAIR) { m = m_pair; return 2 * v + rank; }
    else { const int t = v / nm; m = v - t * nm; return t; }
  };
  // arrivals that the (leader's) MMA thread waits for
  const uint32_t l_full_x = PAIR ? leader_addr(&ctl->full_x[0]) : 0u, l_epi_done = PAIR ? leader_addr(&ctl->epi_done[0]) : 0u;
  auto arrive_full_x = [&](int s) { if constexpr (PAIR) mbar_arrive_cluster(l_full_x + 8u * (uint32_t)s); else mbar_arrive(&ctl->full_x[s]); };
  auto arrive_epi_done = [&](int k) { if constexpr (PAIR) mbar_arrive_cluster(l_epi_done + 8u * (uint32_t)k); else mbar_arrive(&ctl->epi_done[k]); };

  if (warp < EPI_WARPS) {
    // ------------------------------------------------------------------------------------------ epilogue
    const bool has_att = (!COORD) && a.wa != nullptr;
    const float ba = has_att ? a.ba[0] : 0.f;
    float* T = COORD ? ex->u.c.T4[warp] : ex->u.T[warp];
    const long long ep0 = (!COORD && (tc_debug() & 512) && warp == 0 && lane == 0) ? tc_clock() : 0;
    for (int j = 0; j < n_my; ++j) {
      int m;
      unit_tile(j, m);
      const int par = j % NSCAL, acc = j & 1;
      const uint32_t sph = (uint32_t)(j / NSCAL) & 1u;          // phase of this use of scalar set `par`
      const bool prof_on = !COORD && (tc_debug() & 512) && warp == 0 && lane == 0;     // cycle accounting: GCL kernel only
      long long c0 = 0, c1 = 0, c2 = 0, c3 = 0;
      if (prof_on) c0 = tc_clock();
      mbar_wait(&ctl->scal_full[par], sph);
      mbar_wait(&ctl->acc_full[acc], (j >> 1) & 1);
      tc_fence_after();
      if (prof_on) c1 = tc_clock();
      const uint32_t taddr = ctl->tmem_base + ((uint32_t)(warp * 32) << 16) + (uint32_t)(acc * ACC_STRIDE);
      const float* b2 = ex->vec[m] + 2 * H;
      const float inv = a.inv_scale[m];
      const int myrow = ex->row[par][warp * 32 + lane];
      if (tc_debug() & 4) {
        tc_fence_before(); __syncwarp();
        if (lane == 0) { arrive_epi_done(acc); mbar_arrive(&ctl->scal_empty[par]); }
        continue;
      }
      // pass 1: m = SiLU(acc + b2); s = wa . m   (GCL: attention logit; coord: phi, wa = w3)
      f32x2 s01 = pk2(0.f, 0.f), s23 = s01;      // four independent partial dot products
      const int edbg = tc_debug();
#pragma unroll kE1Unroll
      for (int cb = 0; cb < TN / 32; ++cb) {
        float v[32];
        tmem_ld32(taddr + cb * 32, v);
        if (!(edbg & 32))
#pragma unroll
        for (int q = 0; q < 8; ++q) {
          const float4 bb = *reinterpret_cast<const float4*>(b2 + cb * 32 + 4 * q);
          const float4 ww = *reinterpret_cast<const float4*>(ex->wa + cb * 32 + 4 * q);
          f32x2 a01, a23;
          if (F16) {
            const f32x2 ip = pk2(inv, inv);
            a01 = fma2(pk2(v[4 * q], v[4 * q + 1]), ip, pk2(bb.x, bb.y));
            a23 = fma2(pk2(v[4 * q + 2], v[4 * q + 3]), ip, pk2(bb.z, bb.w));
          } else {
            a01 = add2(pk2(v[4 * q], v[4 * q + 1]), pk2(bb.x, bb.y));
            a23 = add2(pk2(v[4 * q + 2], v[4 * q + 3]), pk2(bb.z, bb.w));
          }
          silu4q(a01, a23);
          upk2(a01, v[4 * q], v[4 * q + 1]); upk2(a23, v[4 * q + 2], v[4 * q + 3]);
          s01 = fma2(a01, pk2(ww.x, ww.y), s01); s23 = fma2(a23, pk2(ww.z, ww.w), s23);
        }
        if (!COORD && !(edbg & 2048)) tmem_st32(taddr + cb * 32, v);
      }
      float s0, s1, s2, s3;
      upk2(s01, s0, s1); upk2(s23, s2, s3);
      const float s = (s0 + s1) + (s2 + s3);
      if (prof_on) c2 = tc_clock();
      if (!COORD) {
        tmem_wait_st();
        const float gate = myrow >= 0 ? (has_att ? sigmoid_f(s + ba) : 1.0f) : 0.f;    // pad rows share a chunk with real rows: weight 0
        // Receiver segments start at multiples of kRowChunk rows (virtual edge order), so every chunk of 4 rows belongs to one
        // receiver (or is padding): no segment search.  Pass 2 works per 32-column block: the activated messages go row-wise
        // (STS.128, unscaled) into the per-warp buffer; lane (k = lane / 4, g = lane % 4) then owns chunk k x columns
        // {4g..4g+3, 16+4g..16+4g+3}: 8 LDS.128 (4 rows x 2 pieces, conflict-free: the quarter-warp's rows are 4 x 36 words
        // apart), the gate-weighted 4-row sums as 16 FFMA2, two 16-byte RED (red.global.add.v4.f32) into the receiver's row.
        // A chunk of padding only (tile tail) has gate 0 on all rows: its sums are exactly 0 and are added to row 0.
        static_assert(kRowChunk == 4, "chunk sums below assume 4-row chunks");
        float* G4 = ex->gate4[warp];
        G4[lane] = gate;
        __syncwarp();
        // lane (rg = lane / 8, cg = lane % 8) owns the chunk PAIR of rows 8 rg .. 8 rg + 7 x columns 4 cg .. 4 cg + 3 of the block:
        // 8 LDS.128 (one row each; the quarter-warp reads 128 contiguous bytes of a row), the two gate-weighted chunk sums,
        // and ONE 16-byte RED when both chunks belong to the same receiver (3 of 4 pairs at ~24 edges per receiver; a chunk of
        // padding has gates 0 and merges with anything), else two: ~35 % fewer atomics to L2 than one per chunk.
        const int rg = lane >> 3, cg = lane & 7;
        const float4 ga4 = *reinterpret_cast<const float4*>(G4 + 8 * rg), gb4 = *reinterpret_cast<const float4*>(G4 + 8 * rg + 4);
        const f32x2 g0 = pk2(ga4.x, ga4.x), g1 = pk2(ga4.y, ga4.y), g2 = pk2(ga4.z, ga4.z), g3 = pk2(ga4.w, ga4.w);
        const f32x2 g4 = pk2(gb4.x, gb4.x), g5 = pk2(gb4.y, gb4.y), g6 = pk2(gb4.z, gb4.z), g7 = pk2(gb4.w, gb4.w);
        const int cr0 = ex->row[par][warp * 32 + 8 * rg], cr1 = ex->row[par][warp * 32 + 8 * rg + 4];
        const bool merge = cr1 < 0 || cr1 == cr0;
        float* const dstA = a.agg + (size_t)max(cr0, 0) * H + 4 * cg;
        float* const dstB = a.agg + (size_t)max(cr1, 0) * H + 4 * cg;
        const float* const tp = T + (8 * rg) * EPI_T_STRIDE + 4 * cg;
#pragma unroll kE2Unroll
        for (int cb = 0; cb < ((edbg & 16) ? 0 : TN / 32); ++cb) {
          float v[32];
          tmem_ld32(taddr + cb * 32, v);
#pragma unroll
          for (int q = 0; q < 8; ++q)
            *reinterpret_cast<float4*>(T + lane * EPI_T_STRIDE + 4 * q) = make_float4(v[4 * q], v[4 * q + 1], v[4 * q + 2], v[4 * q + 3]);
          __syncwarp();
          if (!(edbg & 1024)) {
            const float4 x0 = *reinterpret_cast<const float4*>(tp), x1 = *reinterpret_cast<const float4*>(tp + EPI_T_STRIDE);
            const float4 x2 = *reinterpret_cast<const float4*>(tp + 2 * EPI_T_STRIDE), x3 = *reinterpret_cast<const float4*>(tp + 3 * EPI_T_STRIDE);
            const float4 x4 = *reinterpret_cast<const float4*>(tp + 4 * EPI_T_STRIDE), x5 = *reinterpret_cast<const float4*>(tp + 5 * EPI_T_STRIDE);
            const float4 x6 = *reinterpret_cast<const float4*>(tp + 6 * EPI_T_STRIDE), x7 = *reinterpret_cast<const float4*>(tp + 7 * EPI_T_STRIDE);
            f32x2 a01 = add2(fma2(g1, pk2(x1.x, x1.y), mul2(g0, pk2(x0.x, x0.y))), fma2(g3, pk2(x3.x, x3.y), mul2(g2, pk2(x2.x, x2.y))));
            f32x2 a23 = add2(fma2(g1, pk2(x1.z, x1.w), mul2(g0, pk2(x0.z, x0.w))), fma2(g3, pk2(x3.z, x3.w), mul2(g2, pk2(x2.z, x2.w))));
            const f32x2 b01 = add2(fma2(g5, pk2(x5.x, x5.y), mul2(g4, pk2(x4.x, x4.y))), fma2(g7, pk2(x7.x, x7.y), mul2(g6, pk2(x6.x, x6.y))));
            const f32x2 b23 = add2(fma2(g5, pk2(x5.z, x5.w), mul2(g4, pk2(x4.z, x4.w))), fma2(g7, pk2(x7.z, x7.w), mul2(g6, pk2(x6.z, x6.w))));
            if (merge) { a01 = add2(a01, b01); a23 = add2(a23, b23); }
            float o0, o1, o2, o3;
            upk2(a01, o0, o1); upk2(a23, o2, o3);
            asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dstA + cb * 32), "f"(o0), "f"(o1), "f"(o2), "f"(o3) : "memory");
            if (!merge) {
              upk2(b01, o0, o1); upk2(b23, o2, o3);
              asm volatile("red.global.add.v4.f32 [%0], {%1, %2, %3, %4};" ::"l"(dstB + cb * 32), "f"(o0), "f"(o1), "f"(o2), "f"(o3) : "memory");
            }
          }
          __syncwarp();
        }
      } else {
        // coord: s = phi_m for this edge row; this unit's term of trans (egnn_new.py:100-109)
        const int r = warp * 32 + lane;
        float tr[3];
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const float d = ex->u.c.dir[par][k][r];
          float t;
          if (m == 0) t = a.use_tanh ? (d * tanhf(s)) * a.coords_range : d * s;       // coord_diff * tanh(phi) * range
          else t = d * (a.use_tanh ? tanhf(s) * a.coords_range : s);                     // coord_cross * (tanh(phi_x) * range)
          tr[k] = myrow >= 0 ? t : 0.f;
        }
        // 4-row chunks belong to one receiver: lane = (chunk k, component) sums 4 rows and issues one RED
        T[lane * 4 + 0] = tr[0]; T[lane * 4 + 1] = tr[1]; T[lane * 4 + 2] = tr[2];
        __syncwarp();
        {
          const int k = lane >> 2, comp = lane & 3;
          const int crow = ex->row[par][warp * 32 + 4 * k];
          if (comp < 3 && crow >= 0) {
            const float sum = (T[(4 * k) * 4 + comp] + T[(4 * k + 1) * 4 + comp]) + (T[(4 * k + 2) * 4 + comp] + T[(4 * k + 3) * 4 + comp]);
            atomicAdd(reinterpret_cast<float*>(a.xagg) + (size_t)crow * 4 + comp, sum);
          }
        }
        __syncwarp();
      }
      if (prof_on) {
        c3 = tc_clock();
        atomicAdd(&g_tc_prof[0], (unsigned long long)(c1 - c0));   // epilogue: waiting for scalars/accumulator
        atomicAdd(&g_tc_prof[1], (unsigned long long)(c2 - c1));   // pass 1
        atomicAdd(&g_tc_prof[2], (unsigned long long)(c3 - c2));   // pass 2 (GCL) / trans + chunk sums (coord)
        atomicAdd(&g_tc_prof[3], 1ull);                            // units
      }
      tc_fence_before();
      __syncwarp();
      if (lane == 0) {
        arrive_epi_done(acc);
        mbar_arrive(&ctl->scal_empty[par]);
      }
    }
    if (!COORD && (tc_debug() & 512) && warp == 0 && lane == 0) {
      atomicAdd(&g_tc_prof[14], (unsigned long long)(tc_clock() - ep0));     // epilogue warp 0: whole loop of this CTA
      atomicAdd(&g_tc_prof[15], 1ull);
    }
  } else if (warp < MMA_WARP) {
    // ------------------------------------------------------------------------------------------ producers
    // Thread mapping (coalesced gathers): producer warp pw owns tile rows [16 pw, 16 pw + 16); lane = (sub-row sr, piece pc):
    // 8 lanes cover one row's contiguous 128 bytes (32 k-values), one LDG.128 instruction covers 4 rows = 4 L1 wavefronts.
    // A thread handles the 4-row chunk 16 pw + 4 sr + {0..3} x 4 k per 32-k half.  The chunk is one receiver (item 6 of DESIGN
    // §2: segments are padded to 4 rows), so the receiver operand P[recv] is ONE load per half, not four; the four sender rows
    // differ.  Within a half the two rows of a half-warp differ in bit 2 of the row index, so their 64-byte pieces land in
    // different halves of the 128B-swizzled row and the operand STS.64 are bank-conflict free.
    //
    // Load scheduling around the proxy fence: fence.proxy.async (one per pipeline chunk, before the arrive) waits for every
    // outstanding load of the thread, so a gather issued shortly before it delays the hand-off to the MMA thread by an L2
    // round trip.  Gathers are therefore issued (i) for the second half of a chunk: row by row while the first half is being
    // computed (they are consumed before the fence), (ii) for the first half of the NEXT chunk: into a second register set at
    // the start of the current chunk's last half — a full half (~1 k cycles) before the fence, i.e. complete when it executes,
    // (iii) across a unit boundary: right after the fence.
    const int ptid = threadIdx.x - EPI_WARPS * 32;
    const int pw = ptid >> 5, sr = lane >> 3, pc = lane & 7;
    const int dbg = tc_debug();
    const bool pprof = !COORD && (dbg & 512) && ptid == 0;
    uint32_t gc = 0;
    const int r0 = 16 * pw + 4 * sr;           // first of this thread's four tile rows
    // Everything that does not change from chunk to chunk is computed once: the swizzled byte offsets of the thread's four
    // operand rows (the second 32-k half of a 3xFP16 chunk sits 64 bytes further in the swizzled row: offset ^ 64), and, per
    // unit, the five 64-bit row pointers of the gathers.  With the chunk loop unrolled every gather is `pointer + immediate`
    // and every operand store `stage + register offset` (the address arithmetic was ~40 % of the loop's instructions).
    uint32_t so[4];
#pragma unroll
    for (int i = 0; i < 4; ++i) so[i] = F16 ? sw128_offset(r0 + i, pc >> 1) + (uint32_t)(pc & 1) * 8u : sw128_offset(r0 + i, pc);
    float pd2[4], pd0[4];
    const float* const Pt = a.P + 4 * pc;      // this thread's 16-byte piece of a P row
    const float* pr = Pt;                      // receiver row of the thread's 4-row chunk (this unit's MLP block)
    const float* ps[4] = {Pt, Pt, Pt, Pt};     // the four sender rows
    int pty[4] = {0, 0, 0, 0};
    const int soff = nm * H;                   // sender block follows the nm receiver blocks
    float4 GA[2], GB[2][4];                    // two gather register sets: chunk kc computes from set kc & 1 while the other one fills
    auto setup_ptrs = [&](int j) {             // row pointers of unit j (gathers); returns its MLP index
      int m;
      unit_tile(j, m);
      const int par = j % NSCAL;
      mbar_wait(&ctl->scal_full[par], (uint32_t)(j / NSCAL) & 1u);
      const int moff = m * H;                  // column offset of the unit's MLP inside the receiver / sender blocks
      pr = Pt + (size_t)max(ex->row[par][r0], 0) * a.ldp + moff;
#pragma unroll
      for (int i = 0; i < 4; ++i) ps[i] = Pt + (size_t)ex->col[par][r0 + i] * a.ldp + (soff + moff);
      return m;
    };
    auto setup_scal = [&](int j) {             // per-row scalars of unit j (after setup_ptrs(j): the set has arrived)
      const int par = j % NSCAL;
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        pd2[i] = ex->d2[par][r0 + i]; pd0[i] = ex->d0[par][r0 + i];
        if (TB) pty[i] = ex->type[par][r0 + i] * H;
      }
    };
    const bool no_gather = (dbg & 64) != 0;        // instrumented builds only: operands from registers instead of L2
    auto ld4 = [&](const float* p) { return no_gather ? make_float4(0.1f, -0.2f, 0.3f, 0.05f) : *reinterpret_cast<const float4*>(p); };
    auto issue = [&](int hf, float4& xa, float4 (&xb)[4]) {
      xa = ld4(pr + hf * TKC);
#pragma unroll
      for (int i = 0; i < 4; ++i) xb[i] = ld4(ps[i] + hf * TKC);
    };
    long long t0 = 0, t1 = 0, t2 = 0, acc_wait = 0, acc_comp = 0, acc_fence = 0;
    const long long pp0 = pprof ? tc_clock() : 0;
    int m = setup_ptrs(0);
    setup_scal(0);
    issue(0, GA[0], GB[0]);
    for (int j = 0; j < n_my; ++j) {
      const float* wr = ex->vec[m] + 4 * pc; const float* wr0 = wr + H;
      const float* tbm = TB ? a.tb[m] + 4 * pc : nullptr;
#pragma unroll
      for (int kc = 0; kc < chunks; ++kc) {
        const int s = gc & 1;
        char* st = cv.stages + (size_t)s * EG::STAGE_BYTES;
        if (pprof) t0 = tc_clock();
        mbar_wait(&ctl->empty[s], ((gc >> 1) & 1) ^ 1);      // stage released by the MMAs that read it two chunks ago
        if (pprof) { t1 = tc_clock(); acc_wait += t1 - t0; }
        float4& ga = GA[kc & 1];                             // (static indices: the chunk loop is unrolled, no register copies)
        float4 (&gb)[4] = GB[kc & 1];
#pragma unroll
        for (int h = 0; h < HPC; ++h) {
          const int hf = kc * HPC + h;
          const bool last_half = (h == HPC - 1);
          if (last_half && kc + 1 < chunks && !(dbg & 2)) issue(hf + 1, GA[(kc & 1) ^ 1], GB[(kc & 1) ^ 1]);          // (ii)
          if (!(dbg & 2)) {
            const float4 r4 = *reinterpret_cast<const float4*>(wr + hf * TKC);
            const float4 r04 = *reinterpret_cast<const float4*>(wr0 + hf * TKC);
            const f32x2 a01 = pk2(ga.x, ga.y), a23 = pk2(ga.z, ga.w);
            if (!last_half) ga = ld4(pr + (hf + 1) * TKC);        // (i)
#pragma unroll
            for (int i = 0; i < 4; ++i) {
              const f32x2 d2p = pk2(pd2[i], pd2[i]), d0p = pk2(pd0[i], pd0[i]);
              f32x2 u01 = fma2(d0p, pk2(r04.x, r04.y), fma2(d2p, pk2(r4.x, r4.y), add2(a01, pk2(gb[i].x, gb[i].y))));
              f32x2 u23 = fma2(d0p, pk2(r04.z, r04.w), fma2(d2p, pk2(r4.z, r4.w), add2(a23, pk2(gb[i].z, gb[i].w))));
              if (!last_half) gb[i] = ld4(ps[i] + (hf + 1) * TKC);   // (i): registers of row i are free
              if (TB) {
                const float4 t4 = *reinterpret_cast<const float4*>(tbm + pty[i] + hf * TKC);
                u01 = add2(u01, pk2(t4.x, t4.y)); u23 = add2(u23, pk2(t4.z, t4.w));
              }
              if (!(dbg & 128)) silu4q(u01, u23);      // 128: instrumented builds only
              store_pair<F16>(st + (F16 && (hf & 1) ? (so[i] ^ 64u) : so[i]), u01, u23);
            }
          }
        }
        if (pprof) { t2 = tc_clock(); acc_comp += t2 - t1; }
        fence_proxy_async();
        __syncwarp();
        if (lane == 0) arrive_full_x(s);
        ++gc;
        if (pprof) acc_fence += tc_clock() - t2;
      }
      if (j + 1 < n_my) {                                                                      // (iii)
        m = setup_ptrs(j + 1);
        if (!(dbg & 2)) issue(0, GA[0], GB[0]);
        setup_scal(j + 1);
      }
      if (pprof) {
        atomicAdd(&g_tc_prof[9], (unsigned long long)acc_comp);    // gather wait + pre-activation + SiLU + split + swizzled stores
        atomicAdd(&g_tc_prof[10], (unsigned long long)acc_wait);   // waiting for the stage to be released by the MMAs
        atomicAdd(&g_tc_prof[12], (unsigned long long)acc_fence);  // fence.proxy.async + arrive
        atomicAdd(&g_tc_prof[13], 1ull);
        acc_comp = acc_wait = acc_fence = 0;
      }
    }
    if (pprof) {
      atomicAdd(&g_tc_prof[24], (unsigned long long)(tc_clock() - pp0));     // producer thread 0: whole loop of this CTA
      atomicAdd(&g_tc_prof[25], 1ull);
    }
  } else if (warp == MMA_WARP) {
    if constexpr (PAIR) {
      if (lane == 0 && rank == 0) {
        // the leader issues for the pair: per tile pair and chunk 4 k-steps x 3 split products, M = 256, operands at the same
        // shared-memory offsets in both CTAs (A: ring stage; B: resident weight half, chunk kc)
        const uint32_t tmem = ctl->tmem_base;
        mbar_wait_cluster(&ctl->w_ready, 0);
        uint32_t g = 0;
        for (int j = 0; j < n_my; ++j) {
          const int k = j & 1;
          mbar_wait_cluster(&ctl->epi_done[k], ((j >> 1) & 1) ^ 1);      // accumulator drained by both CTAs' epilogues
          tc_fence_after();
          const uint32_t d = tmem + (uint32_t)(k * ACC_STRIDE);
#pragma unroll 1
          for (int kc = 0; kc < chunks; ++kc, ++g) {
            const int s = g & 1;
            mbar_wait_cluster(&ctl->full_x[s], (g >> 1) & 1);            // both CTAs' producers filled stage s
            tc_fence_after();
            const uint32_t xhi = smem_u32(cv.stages + (size_t)s * EG::STAGE_BYTES), xlo = xhi + A_CHUNK_BYTES;
            const uint32_t whi = smem_u32(wres + (size_t)kc * 2 * EG::HB), wlo = whi + EG::HB;
#pragma unroll
            for (int ks = 0; ks < 4; ++ks) {
              const uint32_t ko = ks * 32;
              umma_f16_2cta(d, umma_desc_sw128(xlo + ko), umma_desc_sw128(whi + ko), EG::IDESC_F16_2CTA, (kc == 0 && ks == 0) ? 0u : 1u);
              umma_f16_2cta(d, umma_desc_sw128(xhi + ko), umma_desc_sw128(wlo + ko), EG::IDESC_F16_2CTA, 1u);
              umma_f16_2cta(d, umma_desc_sw128(xhi + ko), umma_desc_sw128(whi + ko), EG::IDESC_F16_2CTA, 1u);
            }
            umma_commit_2cta(&ctl->empty[s]);         // stage reusable in both CTAs once these MMAs have read it
          }
          umma_commit_2cta(&ctl->acc_full[k]);        // both CTAs' accumulators complete
        }
      }
    } else {
      if (lane == 0) mma_role<F16, H>(ctl, cv.stages, n_my, chunks, COORD ? 2 : 1);
    }
    __syncwarp();
  } else if (warp == TMA_WARP) {
    if constexpr (PAIR) {
      if (lane == 0) {
        mbar_wait(&ctl->w_full, 0);                   // this CTA's weight half has landed
        mbar_arrive_cluster(leader_addr(&ctl->w_ready));
      }
    } else {
      if (lane == 0) {
        uint32_t gc = 0;
        for (int j = 0; j < n_my; ++j) {
          int m;
          unit_tile(j, m);
          tma_role<H>(ctl, cv.stages, a.W2hi[m], a.W2lo[m], gc, chunks);
        }
      }
    }
    __syncwarp();
  } else {
    // ------------------------------------------------------------------------------------------ scalar warps
    // 64 threads, two edges each: erow/ecol -> x[r], x[c] (-> centroid) is a chain of dependent global loads; running it
    // one unit ahead (NSCAL buffer sets) keeps it off the producers' critical path.
    const int st = threadIdx.x - (TMA_WARP + 1) * 32;
    for (int j = 0; j < n_my; ++j) {
      const int par = j % NSCAL;
      int m;
      const int e0 = unit_tile(j, m) * TM;
      mbar_wait(&ctl->scal_empty[par], ((uint32_t)(j / NSCAL) & 1u) ^ 1u);   // epilogue finished the unit that last used this set
      edge_scalars<COORD, H>(a, ex, par, st, e0, E, m);
      edge_scalars<COORD, H>(a, ex, par, st + SCAL_WARPS * 32, e0, E, m);
      __syncwarp();
      if (lane == 0) mbar_arrive(&ctl->scal_full[par]);
    }
  }
  kernel_end();
}

// =====================================================================================================
// launchers
// =====================================================================================================
template <int H> static size_t gemm_smem_bytes() { return tc_smem_base<H>() + sizeof(float) * EPI_WARPS * 32 * GEMM_T_STRIDE; }
template <int H, bool PAIR> static size_t edge_smem_bytes() {
  static_assert(edge_smem_base<H, PAIR>() + sizeof(EdgeExtra<H>) <= 232448, "edge kernel exceeds the 227 KB of shared memory per CTA");
  return edge_smem_base<H, PAIR>() + sizeof(EdgeExtra<H>);
}
// Kernel-form selection (dsb_set_kernel_variants): bit 0 = CTA-pair weight-stationary edge kernels, bit 1 = fused node block
// kernel.  3xTF32 always uses the single-CTA kernels.
int g_kernel_variants = [] {
  int v = 3;
  const char* e = getenv("DSB_EDGE_PAIR"); if (e && e[0] == '0') v &= ~1;
  e = getenv("DSB_NODE_BLOCK"); if (e && e[0] == '0') v &= ~2;
  return v;
}();
static bool edge_pair_enabled() { return (g_kernel_variants & 1) != 0; }

bool tc_width_supported(int H) { return H == 128 || H == 192 || H == 256; }

// run `fn.template operator()<H>()` for the run-time width
template <typename Fn>
static int dispatch_width(int H, Fn&& fn) {
  switch (H) {
    case 128: return fn.template operator()<128>();
    case 192: return fn.template operator()<192>();
    case 256: return fn.template operator()<256>();
    default: set_error("tensor-core kernels exist for hidden_nf 128, 192, 256 (got %d)", H); return DSB_ERR_UNSUPPORTED_CONFIG;
  }
}

int configure_tc_kernels(int H) {
  return dispatch_width(H, [&]<int W>() -> int {
    const int gs = (int)gemm_smem_bytes<W>(), es = (int)edge_smem_bytes<W, false>(), ep = (int)edge_smem_bytes<W, true>();
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_node_mlp_kernel<false, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, gs));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_node_mlp_kernel<true, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, gs));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_node_gemm_kernel<false, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, gs));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_node_gemm_kernel<true, W>, cudaFuncAttributeMaxDynamicSharedMemorySize, gs));
    static_assert(block_smem_bytes<W>() <= 232448, "node block kernel exceeds shared memory");
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_node_block_kernel<W>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)block_smem_bytes<W>()));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_edge_kernel<false, false, W, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, es));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_edge_kernel<false, false, W, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, es));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_edge_kernel<false, true, W, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, es));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_edge_kernel<false, true, W, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, es));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_edge_kernel<true, false, W, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, es));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_edge_kernel<true, false, W, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, es));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_edge_kernel<true, true, W, false, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, es));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_edge_kernel<true, true, W, true, false>, cudaFuncAttributeMaxDynamicSharedMemorySize, es));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_edge_kernel<false, true, W, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ep));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_edge_kernel<false, true, W, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ep));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_edge_kernel<true, true, W, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ep));
    DSB_CUDA_OK(cudaFuncSetAttribute(tc_edge_kernel<true, true, W, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, ep));
    return 0;
  });
}

int launch_tc_node_gemm(const dsb_dynamics* d, const GemmArgs& g, const TcImage& w, bool f16, int32_t* status, cudaStream_t s) {
  if (g.M == 0) return 0;
  const int TN = d->cfg.hidden_nf;
  if (g.A2 || g.K2 || !g.bias || g.R || g.act || g.Z) {
    set_error("tc_node_gemm computes C = A W + bias only (no second operand, activation, residual or zeroing)");
    return DSB_ERR_INVALID_ARGUMENT;
  }
  if ((g.Nn % TN) || (g.K1 % TKC16) || (g.lda1 % 4) || (g.ldc % 4)) {
    set_error("tc_node_gemm: unsupported shape K=%d Nn=%d", g.K1, g.Nn);
    return DSB_ERR_INVALID_ARGUMENT;
  }
  TcGemmArgs a;
  a.A = g.A1; a.lda = g.lda1; a.K = g.K1;
  a.Bhi = f16 ? w.h_hi : w.t_hi; a.Blo = f16 ? w.h_lo : w.t_lo;
  a.dead_nt = g.dead_cols / TN; a.dead_mt = a.dead_nt > 0 ? (g.dead_rows_from + TM - 1) / TM : 0;
  a.bias = g.bias; a.C = g.C; a.ldc = g.ldc; a.M = g.M; a.Nn = g.Nn;
  a.inv_scale = f16 ? w.h_inv : 1.0f; a.status = status;
  const int ntn_ = g.Nn / TN, ntm_ = (g.M + TM - 1) / TM;
  const int dmt_ = a.dead_nt > 0 ? (a.dead_mt < ntm_ ? a.dead_mt : ntm_) : ntm_;
  const int n_tiles = dmt_ * ntn_ + (ntm_ - dmt_) * (ntn_ - a.dead_nt);
  const int grid = n_tiles < d->num_sms ? n_tiles : d->num_sms;
  return dispatch_width(TN, [&]<int W>() -> int {
    DSB_CUDA_OK(launch_k(f16 ? tc_node_gemm_kernel<true, W> : tc_node_gemm_kernel<false, W>, grid, TC_THREADS, gemm_smem_bytes<W>(), s, a));
    return 0;
  });
}

int launch_tc_node_mlp(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, const GclW& w, bool f16, int32_t* status, cudaStream_t s) {
  if (dm.N == 0) return 0;
  TcMlpArgs a = {};
  const int H = d->cfg.hidden_nf;
  a.h = ws.h; a.ldh = H; a.agg = ws.agg; a.ldagg = H; a.div = d->cfg.normalization_factor;
  a.deg = d->cfg.aggregation_mean ? ws.deg : nullptr;
  a.W3hi = f16 ? w.iW3.h_hi : w.iW3.t_hi; a.W3lo = f16 ? w.iW3.h_lo : w.iW3.t_lo;
  a.W4hi = f16 ? w.iW4.h_hi : w.iW4.t_hi; a.W4lo = f16 ? w.iW4.h_lo : w.iW4.t_lo;
  a.b3 = w.b3; a.b4 = w.b4;
  a.inv3 = f16 ? w.iW3.h_inv : 1.0f; a.inv4 = f16 ? w.iW4.h_inv : 1.0f;
  a.hout = ws.h; a.zero = ws.agg; a.M = dm.N; a.status = status;
  const int ntm = (dm.N + TM - 1) / TM;
  const int grid = ntm < d->num_sms ? ntm : d->num_sms;
  return dispatch_width(H, [&]<int W>() -> int {
    DSB_CUDA_OK(launch_k(f16 ? tc_node_mlp_kernel<true, W> : tc_node_mlp_kernel<false, W>, grid, TC_THREADS, gemm_smem_bytes<W>(), s, a));
    return 0;
  });
}

// node_model of GCL `w` followed by the merged first-layer GEMM `q` of the same block (nullptr: none), one launch
bool tc_node_block_available(int H, bool f16) {
  return (g_kernel_variants & 2) && f16 && tc_width_supported(H);
}
int launch_tc_node_block(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, const GclW& w, const EquivW& q, float* P, int ldp,
                         int dead_rows_from, int dead_cols, cudaStream_t s) {
  if (dm.N == 0) return 0;
  const int H = d->cfg.hidden_nf;
  TcBlockArgs a = {};
  a.h = ws.h; a.ldh = H; a.agg = ws.agg; a.ldagg = H; a.div = d->cfg.normalization_factor;
  a.deg = d->cfg.aggregation_mean ? ws.deg : nullptr;
  a.W3hi = w.iW3.h_hi; a.W3lo = w.iW3.h_lo; a.W4hi = w.iW4.h_hi; a.W4lo = w.iW4.h_lo;
  a.Wqhi = q.iW1.h_hi; a.Wqlo = q.iW1.h_lo;
  a.b3 = w.b3; a.b4 = w.b4; a.bq = q.b1;
  a.inv3 = w.iW3.h_inv; a.inv4 = w.iW4.h_inv; a.invq = q.iW1.h_inv; a.s4 = 1.0f / w.iW4.h_inv;
  a.P = P; a.ldp = ldp; a.Nn = q.nq + q.np; a.M = dm.N;
  a.dead_nt = dead_cols / H; a.dead_mt = a.dead_nt > 0 ? (dead_rows_from + TM - 1) / TM : 0;
  if (a.Nn % H) { set_error("tc_node_block: %d output columns are not a multiple of hidden_nf", a.Nn); return DSB_ERR_INVALID_ARGUMENT; }
  const int ntm = (dm.N + TM - 1) / TM, nmp = (ntm + 1) / 2, hw = d->num_sms / 2;
  const int grid = 2 * (nmp < hw ? nmp : hw);
  return dispatch_width(H, [&]<int W>() -> int {
    DSB_CUDA_OK(launch_k_pair(tc_node_block_kernel<W>, grid, TC_THREADS, block_smem_bytes<W>(), s, a));
    return 0;
  });
}

int launch_tc_edge_gcl(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, const GclW& w, const float4* x, PView pv, bool f16,
                       int32_t* status, cudaStream_t s) {
  TcEdgeArgs a = {};
  a.P = pv.P; a.ldp = pv.ldp; a.x = x; a.cent = ws.cent; a.gid = ws.gid; a.vrow_ptr = ws.vrow_ptr; a.vmap = ws.vmap; a.n_rows = dm.N;
  a.erow = ws.erow; a.ecol = ws.ecol; a.ed0 = ws.ed0; a.NL = dm.NL; a.nm = 1;
  a.W2hi[0] = f16 ? w.iW2.h_hi : w.iW2.t_hi; a.W2lo[0] = f16 ? w.iW2.h_lo : w.iW2.t_lo;
  a.inv_scale[0] = f16 ? w.iW2.h_inv : 1.0f; a.inv_scale[1] = 1.0f;
  a.wr[0] = w.wr; a.wr0[0] = w.wr0; a.tb[0] = w.tb; a.b2[0] = w.b2;
  a.wa = w.wa; a.ba = w.ba; a.agg = ws.agg; a.status = status;
  return dispatch_width(d->cfg.hidden_nf, [&]<int W>() -> int {
    if (f16 && edge_pair_enabled() && d->num_sms >= 2) {
      DSB_CUDA_OK(launch_k_pair(w.tb ? tc_edge_kernel<false, true, W, true, true> : tc_edge_kernel<false, true, W, false, true>,
                                d->num_sms & ~1, EDGE_THREADS, edge_smem_bytes<W, true>(), s, a));
      return 0;
    }
    auto kern = w.tb ? (f16 ? tc_edge_kernel<false, true, W, true, false> : tc_edge_kernel<false, false, W, true, false>)
                     : (f16 ? tc_edge_kernel<false, true, W, false, false> : tc_edge_kernel<false, false, W, false, false>);
    DSB_CUDA_OK(launch_k(kern, d->num_sms, EDGE_THREADS, edge_smem_bytes<W, false>(), s, a));
    return 0;
  });
}

int launch_tc_edge_coord(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, const EquivW& w, const float4* x, PView pv, bool f16,
                         int32_t* status, cudaStream_t s) {
  const dsb_config& c = d->cfg;
  TcEdgeArgs a = {};
  a.nm = c.reflection_equivariant ? 1 : 2;
  a.P = pv.P; a.ldp = pv.ldp; a.x = x; a.cent = ws.cent; a.gid = ws.gid; a.vrow_ptr = ws.vrow_ptr; a.vmap = ws.vmap; a.n_rows = dm.n_coord_rows;
  a.erow = ws.erow; a.ecol = ws.ecol; a.ed0 = ws.ed0; a.NL = dm.NL;
  a.inv_scale[0] = a.inv_scale[1] = 1.0f;
  for (int m = 0; m < a.nm; ++m) {
    a.W2hi[m] = f16 ? w.iW2[m].h_hi : w.iW2[m].t_hi; a.W2lo[m] = f16 ? w.iW2[m].h_lo : w.iW2[m].t_lo;
    a.inv_scale[m] = f16 ? w.iW2[m].h_inv : 1.0f;
    a.wr[m] = w.wr[m]; a.wr0[m] = w.wr0[m]; a.tb[m] = w.tb[m]; a.b2[m] = w.b2[m];
  }
  a.wa = w.w3; a.ba = nullptr;
  a.norm_constant = c.norm_constant; a.coords_range = c.coords_range; a.use_tanh = c.tanh; a.xagg = ws.xagg; a.status = status;
  return dispatch_width(c.hidden_nf, [&]<int W>() -> int {
    const int npairs = d->num_sms / 2;
    if (f16 && edge_pair_enabled() && npairs >= a.nm && npairs % a.nm == 0) {       // every pair keeps ONE MLP's weights resident
      DSB_CUDA_OK(launch_k_pair(w.tb[0] ? tc_edge_kernel<true, true, W, true, true> : tc_edge_kernel<true, true, W, false, true>,
                                2 * npairs, EDGE_THREADS, edge_smem_bytes<W, true>(), s, a));
      return 0;
    }
    auto kern = w.tb[0] ? (f16 ? tc_edge_kernel<true, true, W, true, false> : tc_edge_kernel<true, false, W, true, false>)
                        : (f16 ? tc_edge_kernel<true, true, W, false, false> : tc_edge_kernel<true, false, W, false, false>);
    DSB_CUDA_OK(launch_k(kern, d->num_sms, EDGE_THREADS, edge_smem_bytes<W, false>(), s, a));
    return 0;
  });
}

}  // namespace dsb
