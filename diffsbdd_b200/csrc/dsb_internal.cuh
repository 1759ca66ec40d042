// Internal declarations shared by the translation units of libdiffsbdd_b200.so (sm_100a only).
#pragma once
#include <cstring>

#include <cuda_runtime.h>
#include <stdint.h>
#include <stdio.h>

#include "../../include/diffsbdd_b200.h"

namespace dsb {

constexpr int kMaxSub = 4;      // inv_sublayers supported per block
constexpr int kMaxLayers = 16;

// tensor-core operand images of one weight matrix B[n][k] (hidden_nf H in {128,192,256}; all nullptr otherwise), n-tiles H wide:
//   t_*: TF32 hi/lo split, [Nn/H][K/32][H rows x 128 B SWIZZLE_128B]
//   h_*: FP16 hi/lo split of w * h_scale, [Nn/H][K/64][H rows x 128 B]; h_inv = 1 / h_scale undoes the
//        weight scale and the activation scale in the epilogue (both powers of two: exact)
struct TcImage {
  const float *t_hi, *t_lo;
  const float *h_hi, *h_lo;
  float h_inv;
};

// ---- packed weights (device pointers into one blob; all GEMM operands k-major: W[k][n]) -------------
struct GclW {            // one GCL (reference egnn_new.py:6-66)
  const float* W1ab;     // [H][2H]  cols 0..H-1: edge_mlp.0.weight[:, 0:H]^T (receiver h_i), H..2H-1: [:, H:2H]^T (sender h_j)
  const float* b1ab;     // [2H]     (edge_mlp.0.bias | 0)
  const float* wr;       // [H]      edge_mlp.0.weight[:, 2H]   (coefficient of current d^2)
  const float* wr0;      // [H]      edge_mlp.0.weight[:, 2H+1] (coefficient of input-geometry d^2)
  const float* tb;       // [3][H]   edge_mlp.0.weight[:, 2H+2:] @ edge_embedding[type]  (nullptr without embedding)
  const float* W2;       // [H][H]   edge_mlp.2.weight^T
  const float* b2;       // [H]
  const float* wa;       // [H]      att_mlp.0.weight (nullptr without attention)
  const float* ba;       // [1]
  const float* W3;       // [2H][H]  node_mlp.0.weight^T (rows 0..H-1 multiply h, H..2H-1 multiply agg)
  const float* b3;       // [H]
  const float* W4;       // [H][H]   node_mlp.2.weight^T
  const float* b4;       // [H]
  TcImage iW1ab, iW2, iW3, iW4;   // Nn x K = 2H x H, H x H, H x 2H, H x H
};

struct EquivW {          // EquivariantUpdate (reference egnn_new.py:69-132); index 0 = coord_mlp, 1 = cross_product_mlp
  const float* W1;       // [H][nm*2H] receiver block (coord recv | cross recv) then sender block (coord send | cross send)
  const float* b1;       // [nm*2H]    (bias coord | bias cross | 0 | 0)
  const float* wr[2];
  const float* wr0[2];
  const float* tb[2];
  const float* W2[2];    // [H][H]
  const float* b2[2];    // [H]
  const float* w3;       // [H] shared bias-free last layer (egnn_new.py:78)
  TcImage iW1;                      // Nn = nm*2H (+2H), K = H
  TcImage iW2[2];                   // Nn = H, K = H
  // The first-layer GEMM of this block's coordinate MLPs is merged with the first-layer GEMM of the NEXT block's first
  // GCL (both consume the same h): W1/b1/iW1 hold [receiver block | sender block | next W1a | next W1b] (nq + np columns).
  int nq;                           // nm*2H
  int np;                           // 2H if a next GCL exists, else 0
};

struct PackedWeights {
  // encoders / decoders keep the reference [out][in] layout (tiny)
  const float *aenc0_w, *aenc0_b, *aenc2_w, *aenc2_b;
  const float *renc0_w, *renc0_b, *renc2_w, *renc2_b;
  const float *adec0_w, *adec0_b, *adec2_w, *adec2_b;
  const float *rdec0_w, *rdec0_b, *rdec2_w, *rdec2_b;
  // folded affine pairs (index 0 = atoms, 1 = residues):
  //   pre_wT [2F+1][H]  = (embedding.W[:, :J] @ encoder.2.W)^T, last row = embedding.W[:, J] (time column)
  //   pre_b  [H]        = embedding.b + embedding.W[:, :J] @ encoder.2.b
  //   dec_w  [2F][H]    = decoder.0.W @ embedding_out.W[:J, :]
  //   dec_b  [2F]       = decoder.0.b + decoder.0.W @ embedding_out.b[:J]
  const float *pre_wT[2], *pre_b[2], *dec_w[2], *dec_b[2];
  GclW gcl[kMaxLayers][kMaxSub];
  EquivW eq[kMaxLayers];
};

constexpr int kRowChunk = 4;     // rows of one receiver start at multiples of this in the padded (virtual) edge order

// ---- workspace carve-up ---------------------------------------------------------------------------
struct Workspace {
  int32_t *lig_off, *poc_off;   // [B+1]
  int32_t *gid;                 // [N]
  float4 *xbuf[3];              // [N] (x,y,z,0): input, ping, pong
  float4 *cent;                 // [B]
  float4 *xagg;                 // [N] raw segment sums of trans
  float4 *velmean;              // [B]
  float *h, *hT, *agg, *P;      // [N][H], [N][H] (hidden layer of the fp32 node MLP), [N][H], [N][6H] (Q block of the current layer | P block of the next GCL)
  int32_t *deg, *row_ptr;       // [N], [N+1]
  int32_t *vrow_ptr, *vmap;     // [N+1], [Ecap + 3N]: receiver segments padded to multiples of kRowChunk rows (tensor-core edge kernels)
  int32_t *erow, *ecol;         // [Ecap]
  float *ed0;                   // [Ecap]
  size_t bytes;
};

struct Dims {
  int NL, NP, N, B;
  int64_t Ecap;
  int n_coord_rows;   // rows whose coordinates move: NL (conditional) or N (joint)
};

}  // namespace dsb

namespace dsb {
// kernel classes for the optional per-class CUDA-event timing (dsb_dynamics_set_profiling)
enum KClass { KC_SETUP = 0, KC_NODE_GEMM = 1, KC_MEMSET = 2, KC_EDGE_GCL = 3, KC_EDGE_COORD = 4,
              KC_COORD_FINISH = 5, KC_POST = 6, KC_COUNT = 7 };
constexpr int kMaxProfEvents = 512;
}

struct dsb_dynamics {
  dsb_config cfg;
  dsb::PackedWeights w;
  float* blob = nullptr;
  size_t blob_floats = 0;
  int num_sms = 148;
  int math_mode = 0;         // bitmask: 1 node GEMMs, 2 edge_gcl, 4 edge_coord on tcgen05 (H in {128,192,256}); 8: 3xFP16 split instead of 3xTF32
  int last_launches = 0;     // kernels only
  int last_memsets = 0;
  // profiling
  int prof_enabled = 0;
  cudaEvent_t* prof_ev = nullptr;      // [2 * kMaxProfEvents]
  int prof_cls[dsb::kMaxProfEvents];
  int prof_n = 0;
  double prof_ms[dsb::KC_COUNT] = {0, 0, 0, 0, 0, 0, 0};
  long long prof_cnt[dsb::KC_COUNT] = {0, 0, 0, 0, 0, 0, 0};
};

namespace dsb {

void set_error(const char* fmt, ...);

#define DSB_CUDA_OK(expr)                                                                   \
  do {                                                                                      \
    cudaError_t _e = (expr);                                                                \
    if (_e != cudaSuccess) {                                                                \
      dsb::set_error("%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
      return DSB_ERR_CUDA;                                                                  \
    }                                                                                       \
  } while (0)

// ---- programmatic dependent launch (PDL) ---------------------------------------------------------------
// With g_pdl != 0 the forward's kernels are launched with cudaLaunchAttributeProgrammaticStreamSerialization:
// every such kernel triggers its dependents at entry (pdl_trigger) and executes griddepcontrol.wait (pdl_wait)
// before its first access to global memory a predecessor may have touched, so a kernel's launch latency and
// prologue (barrier init, TMEM allocation, constant-vector staging) overlap the predecessor's tail.  Both
// instructions are no-ops for a kernel launched without the attribute.
extern int g_pdl;
extern int g_kernel_variants;      // dsb_set_kernel_variants (dsb_tc.cu)
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[1];
  if (g_pdl) {
    at[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
  }
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
// the same for a kernel that runs as clusters of two CTAs (CTA pairs on one TPC: tcgen05 cta_group::2); grid must be even
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k_pair(void (*kern)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t s, Args... args) {
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = s;
  cudaLaunchAttribute at[2];
  at[0].id = cudaLaunchAttributeClusterDimension;
  at[0].val.clusterDim.x = 2; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
  cfg.attrs = at; cfg.numAttrs = 1;
  if (g_pdl) {
    at[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    at[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.numAttrs = 2;
  }
  return cudaLaunchKernelEx(&cfg, kern, static_cast<KArgs>(args)...);
}
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;"); }
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
#endif

// ---- launchers implemented in dsb_node.cu ----------------------------------------------------------
struct GemmArgs {
  const float* A1; int lda1; int K1;
  const float* A2; int lda2; int K2; float div2;   // columns K1..K1+K2-1 come from A2 / div2 (exact division)
  const float* W; int ldw;                          // k-major [K1+K2][ldw]
  const float* bias;                                // [Nn] or nullptr
  const float* R; int ldr;                          // residual (added after bias) or nullptr
  float* C; int ldc;
  int M; int Nn; int act;                           // act: 0 none, 1 SiLU
  float* Z; int ldz;                                // optional: Z[m][n] = 0 for every output element (re-arms the aggregate)
  int dead_rows_from; int dead_cols;                // output block rows >= dead_rows_from x cols < dead_cols is not needed (skipped)
  const int32_t* deg2;                              // != nullptr ('mean' aggregation): row m of A2 is divided by max(deg2[m], 1) instead of div2
};
int launch_node_gemm(const GemmArgs& a, cudaStream_t s);
int configure_node_kernels();

int launch_plan(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, const int64_t* mask_atoms,
                const int64_t* mask_residues, cudaStream_t s);
int launch_prep(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, const float* xh_atoms,
                const float* xh_residues, const float* t, int64_t t_numel, const int64_t* mask_atoms,
                const int64_t* mask_residues, bool coords_only, cudaStream_t s);
int launch_edges(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, int32_t* status, cudaStream_t s);
int launch_coord_finish(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, const float4* x_old,
                        float4* x_new, bool apply_update, cudaStream_t s);
int launch_post(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, const float4* x_final,
                float* out_atoms, float* out_residues, int32_t* status, cudaStream_t s);

// ---- launchers implemented in dsb_edge.cu ----------------------------------------------------------
struct PView { const float* P; int ldp; };           // where an edge kernel finds its factorised first-layer outputs
int launch_edge_gcl(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, const GclW& w,
                    const float4* x, PView pv, cudaStream_t s);
int launch_edge_coord(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, const EquivW& w,
                      const float4* x, PView pv, cudaStream_t s);
int configure_edge_kernels(int H);

// ---- tensor-core path (dsb_tc.cu) --------------------------------------------------------------------
void launch_pack_b_image(float* hi, float* lo, const float* src, int lds, int scol, int n_rows, int n_dst_off, int K, int tn);
void launch_pack_b_image_f16(float* hi, float* lo, const float* src, int lds, int scol, int n_rows, int n_dst_off, int K, float scale, int tn);
void launch_absmax(const float* src, int lds, int scol, int n_rows, int K, unsigned* out);
int configure_tc_kernels(int H);
bool tc_width_supported(int H);     // hidden_nf values with tensor-core kernels (128, 192, 256)
int launch_tc_node_gemm(const dsb_dynamics* d, const GemmArgs& g, const TcImage& w, bool f16, int32_t* status, cudaStream_t s);   // C = A1 W + bias only
int launch_tc_node_mlp(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, const GclW& w, bool f16, int32_t* status, cudaStream_t s);
bool tc_node_block_available(int H, bool f16);
int launch_tc_node_block(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, const GclW& w, const EquivW& q, float* P, int ldp,
                         int dead_rows_from, int dead_cols, cudaStream_t s);
int launch_tc_edge_gcl(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, const GclW& w, const float4* x, PView pv, bool f16,
                       int32_t* status, cudaStream_t s);
int launch_tc_edge_coord(const dsb_dynamics* d, const Dims& dm, const Workspace& ws, const EquivW& w, const float4* x, PView pv, bool f16,
                         int32_t* status, cudaStream_t s);

// ---- device math helpers ----------------------------------------------------------------------------
// SiLU / sigmoid as FMUL, MUFU.EX2, FADD, MUFU.RCP, FMUL (ex2.approx / rcp.approx, ~2 ulp each): relative error
// ~3e-7 + |x|*6e-8 from the exponent scaling, i.e. at the fp32 noise floor of the reference itself (SURVEY.md §4).
// The libdevice forms (__expf/__fdividef) add range fix-ups (FSETP + 2 FMUL each) that double the instruction count
// of the hot loops for inputs that never occur here (|pre-activation| > 87).
__device__ __forceinline__ float ex2_approx(float x) { float y; asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float rcp_approx(float x) { float y; asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x)); return y; }
__device__ __forceinline__ float silu_f(float x) { return x * rcp_approx(1.0f + ex2_approx(x * -1.4426950408889634f)); }
__device__ __forceinline__ float sigmoid_f(float x) { return rcp_approx(1.0f + ex2_approx(x * -1.4426950408889634f)); }


// Packed fp32x2 arithmetic (FFMA2 / FADD2 / FMUL2 on sm_100a): the same IEEE operations as two scalar instructions, one
// issue slot.  A pair is carried in a 64-bit register pair (u64); scalar operands broadcast for free in SASS.
typedef unsigned long long f32x2;
__device__ __forceinline__ f32x2 pk2(float a, float b) { f32x2 r; asm("mov.b64 %0, {%1, %2};" : "=l"(r) : "f"(a), "f"(b)); return r; }
__device__ __forceinline__ void upk2(f32x2 v, float& a, float& b) { asm("mov.b64 {%0, %1}, %2;" : "=f"(a), "=f"(b) : "l"(v)); }
__device__ __forceinline__ f32x2 fma2(f32x2 a, f32x2 b, f32x2 c) { f32x2 r; asm("fma.rn.f32x2 %0, %1, %2, %3;" : "=l"(r) : "l"(a), "l"(b), "l"(c)); return r; }
__device__ __forceinline__ f32x2 add2(f32x2 a, f32x2 b) { f32x2 r; asm("add.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
__device__ __forceinline__ f32x2 mul2(f32x2 a, f32x2 b) { f32x2 r; asm("mul.rn.f32x2 %0, %1, %2;" : "=l"(r) : "l"(a), "l"(b)); return r; }
// silu_f on a pair: bit-identical to two silu_f calls (same operations in the same order)
__device__ __forceinline__ f32x2 silu2(f32x2 u) {
  float a, b;
  upk2(mul2(u, pk2(-1.4426950408889634f, -1.4426950408889634f)), a, b);
  upk2(add2(pk2(ex2_approx(a), ex2_approx(b)), pk2(1.0f, 1.0f)), a, b);
  return mul2(u, pk2(rcp_approx(a), rcp_approx(b)));
}

// SiLU of four values with ONE reciprocal instead of four: the 16-lane XU pipe (MUFU: 8 issue cycles per warp instruction
// and sub-partition) is the busiest pipe of the edge kernels (2 SiLU per edge element = 4 MUFU), the FMA pipe is not.
// With d_i = 1 + 2^{t_i}: r = 1 / (d_0 d_1 d_2 d_3), 1/d_0 = r (d_1 d_3) d_2 ... arranged on pairs:
//   p = d01 * d23 = (d_0 d_2, d_1 d_3);  r = 1 / (p.x p.y);  (r p.y, r p.x) = (1/(d_0 d_2), 1/(d_1 d_3));  times d23 -> 1/d01,
//   times d01 -> 1/d23.  5 MUFU per 4 values.  Exponent argument clamped to 31 (four factors below 2^31 + 1 cannot overflow;
// pre-activation >= -21.5, where |SiLU(x)| < 1e-8 and the clamp changes it by < 5e-9).  Relative error ~6e-7.
__device__ __forceinline__ void silu4q(f32x2& u01, f32x2& u23) {
  const f32x2 c = pk2(-1.4426950408889634f, -1.4426950408889634f), one = pk2(1.0f, 1.0f);
  float t0, t1, t2, t3;
  upk2(mul2(u01, c), t0, t1); upk2(mul2(u23, c), t2, t3);
  const f32x2 d01 = add2(pk2(ex2_approx(fminf(t0, 31.f)), ex2_approx(fminf(t1, 31.f))), one);
  const f32x2 d23 = add2(pk2(ex2_approx(fminf(t2, 31.f)), ex2_approx(fminf(t3, 31.f))), one);
  const f32x2 w01 = mul2(u01, d23), w23 = mul2(u23, d01);      // independent of the reciprocal: one multiply after it, not two
  float p0, p1;
  upk2(mul2(d01, d23), p0, p1);
  const float r = rcp_approx(p0 * p1);
  const f32x2 rr = mul2(pk2(r, r), pk2(p1, p0));  // (1 / (d0 d2), 1 / (d1 d3)); broadcast and swapped pair are operand modifiers
  u01 = mul2(w01, rr);
  u23 = mul2(w23, rr);
}

__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
  unsigned s = (unsigned)__cvta_generic_to_shared(smem_dst);
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;\n" ::"r"(s), "l"(gmem_src));
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;\n" ::); }
__device__ __forceinline__ void cp_async_wait_all() { asm volatile("cp.async.wait_group 0;\n" ::); }

}  // namespace dsb
