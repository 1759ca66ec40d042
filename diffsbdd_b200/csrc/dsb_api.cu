// C ABI of libdiffsbdd_b200.so: parameter table, weight packing, workspace carve-up, forward
// orchestration (include/diffsbdd_b200.h).  Host logic only + tiny packing kernels.
#include <math.h>
#include <stdarg.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <string>
#include <vector>

#include "dsb_internal.cuh"

namespace dsb {

static int pdl_from_env() { const char* e = getenv("DSB_PDL"); return e ? (atoi(e) != 0) : 1; }
int g_pdl = pdl_from_env();

static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

// ---- parameter table (reference state_dict order of diffsbdd_b200/synthetic.py::state_dict_spec) -------
struct ParamInfo { std::string name; int64_t numel; int rows, cols; };

static int validate(const dsb_config* c) {
  if (!c) { set_error("null config"); return DSB_ERR_INVALID_ARGUMENT; }
  if (c->n_dims != 3) { set_error("n_dims must be 3"); return DSB_ERR_UNSUPPORTED_CONFIG; }
  if (c->hidden_nf != 64 && c->hidden_nf != 128 && c->hidden_nf != 192 && c->hidden_nf != 256) {
    set_error("hidden_nf=%d unsupported (64,128,192,256)", c->hidden_nf); return DSB_ERR_UNSUPPORTED_CONFIG;
  }
  if (c->n_layers < 1 || c->n_layers > kMaxLayers || c->inv_sublayers < 1 || c->inv_sublayers > kMaxSub) {
    set_error("n_layers/inv_sublayers out of range"); return DSB_ERR_UNSUPPORTED_CONFIG;
  }
  if (c->atom_nf < 1 || c->residue_nf < 1 || c->joint_nf < 1 || c->atom_nf > 64 || c->residue_nf > 64 ||
      c->joint_nf > 1024 || c->edge_embedding_dim < 0 || c->edge_embedding_dim > 64) {
    set_error("feature sizes out of range"); return DSB_ERR_UNSUPPORTED_CONFIG;
  }
  if (!(c->normalization_factor > 0.f)) { set_error("normalization_factor must be > 0"); return DSB_ERR_INVALID_ARGUMENT; }
  return 0;
}

static std::vector<ParamInfo> param_table(const dsb_config& c) {
  std::vector<ParamInfo> v;
  const int A = c.atom_nf, R = c.residue_nf, J = c.joint_nf, H = c.hidden_nf;
  const int Din = J + (c.condition_time ? 1 : 0), F = (c.sin_embedding ? 24 : 2) + c.edge_embedding_dim;      // egnn_new.py:203-210
  auto lin = [&](const std::string& p, int out_f, int in_f, bool bias = true) {
    v.push_back({p + ".weight", (int64_t)out_f * in_f, out_f, in_f});
    if (bias) v.push_back({p + ".bias", out_f, out_f, 1});
  };
  lin("atom_encoder.0", 2 * A, A); lin("atom_encoder.2", J, 2 * A);
  lin("atom_decoder.0", 2 * A, J); lin("atom_decoder.2", A, 2 * A);
  lin("residue_encoder.0", 2 * R, R); lin("residue_encoder.2", J, 2 * R);
  lin("residue_decoder.0", 2 * R, J); lin("residue_decoder.2", R, 2 * R);
  if (c.edge_embedding_dim > 0) v.push_back({"edge_embedding.weight", (int64_t)3 * c.edge_embedding_dim, 3, c.edge_embedding_dim});
  lin("egnn.embedding", H, Din); lin("egnn.embedding_out", Din, H);
  for (int k = 0; k < c.n_layers; ++k) {
    const std::string b = "egnn.e_block_" + std::to_string(k);
    for (int s = 0; s < c.inv_sublayers; ++s) {
      const std::string g = b + ".gcl_" + std::to_string(s);
      lin(g + ".edge_mlp.0", H, 2 * H + F); lin(g + ".edge_mlp.2", H, H);
      lin(g + ".node_mlp.0", H, 2 * H); lin(g + ".node_mlp.2", H, H);
      if (c.attention) lin(g + ".att_mlp.0", 1, H);
    }
    const std::string q = b + ".gcl_equiv";
    lin(q + ".coord_mlp.0", H, 2 * H + F); lin(q + ".coord_mlp.2", H, H); lin(q + ".coord_mlp.4", 1, H, false);
    if (!c.reflection_equivariant) { lin(q + ".cross_product_mlp.0", H, 2 * H + F); lin(q + ".cross_product_mlp.2", H, H); }
  }
  return v;
}

// ---- packing kernels -----------------------------------------------------------------------------------
// dst[k*ldd + dcol + n] = src[n*lds + scol + k]   for n < N, k < K
__global__ void pack_T_kernel(float* dst, int ldd, int dcol, const float* src, int lds, int scol, int N, int K) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (int64_t)N * K) return;
  const int n = (int)(idx / K), k = (int)(idx - (int64_t)n * K);
  dst[(size_t)k * ldd + dcol + n] = src[(size_t)n * lds + scol + k];
}
__global__ void pack_copy_kernel(float* dst, const float* src, int64_t n) {
  const int64_t idx = (int64_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx < n) dst[idx] = src[idx];
}
// tb[t][n] = sum_e W1[n][scol + e] * emb[t][e]
__global__ void pack_tb_kernel(float* dst, const float* w1, int lds, int scol, const float* emb, int De, int H) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= 3 * H) return;
  const int t = idx / H, n = idx - t * H;
  float acc = 0.f;
  for (int e = 0; e < De; ++e) acc = fmaf(w1[(size_t)n * lds + scol + e], emb[t * De + e], acc);
  dst[idx] = acc;
}

// folded affine pairs, accumulated in fp64 and rounded once (see PackedWeights)
// dst[k*H + c] = sum_j embW[c*Din + j] * enc2W[j*F2 + k]  (k < F2);  dst[F2*H + c] = embW[c*Din + J] when Din > J
__global__ void pack_pre_kernel(float* dst, float* dst_b, const float* embW, const float* embB, const float* enc2W,
                                const float* enc2B, int H, int J, int Din, int F2) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  const int K = F2 + (Din > J ? 1 : 0);
  if (idx >= (K + 1) * H) return;
  const int k = idx / H, c = idx - k * H;
  if (k < F2) {
    double acc = 0.0;
    for (int j = 0; j < J; ++j) acc += (double)embW[(size_t)c * Din + j] * (double)enc2W[(size_t)j * F2 + k];
    dst[idx] = (float)acc;
  } else if (k < K) {
    dst[idx] = embW[(size_t)c * Din + J];
  } else {
    double acc = (double)embB[c];
    for (int j = 0; j < J; ++j) acc += (double)embW[(size_t)c * Din + j] * (double)enc2B[j];
    dst_b[c] = (float)acc;
  }
}
// dst[o*H + k] = sum_j dec0W[o*J + j] * outW[j*H + k];  dst_b[o] = dec0B[o] + sum_j dec0W[o*J + j] * outB[j]
__global__ void pack_dec_kernel(float* dst, float* dst_b, const float* dec0W, const float* dec0B, const float* outW,
                                const float* outB, int H, int J, int F2) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= F2 * (H + 1)) return;
  const int o = idx / (H + 1), k = idx - o * (H + 1);
  if (k < H) {
    double acc = 0.0;
    for (int j = 0; j < J; ++j) acc += (double)dec0W[(size_t)o * J + j] * (double)outW[(size_t)j * H + k];
    dst[(size_t)o * H + k] = (float)acc;
  } else {
    double acc = (double)dec0B[o];
    for (int j = 0; j < J; ++j) acc += (double)dec0W[(size_t)o * J + j] * (double)outB[j];
    dst_b[o] = (float)acc;
  }
}

struct Packer {
  float* blob; size_t used = 0; bool dry;
  explicit Packer(float* b) : blob(b), dry(b == nullptr) {}
  float* alloc(size_t n) { size_t o = used; used += (n + 63) & ~size_t(63); return dry ? nullptr : blob + o; }
  const float* T(const float* src, int lds, int scol, int N, int K, float* dst, int ldd, int dcol) {
    if (!dry) { int64_t tot = (int64_t)N * K; pack_T_kernel<<<(unsigned)((tot + 255) / 256), 256>>>(dst, ldd, dcol, src, lds, scol, N, K); }
    return dst;
  }
  // tensor-core operand images of one B[Nn][K] matrix assembled from `nblk` row blocks of the reference weights
  // (src, lds, scol, n_rows, n_dst_off).  Builds the TF32 and the FP16 split images; the FP16 scale is the power of two
  // that puts max|w| into [4096, 8192) so that the low part of every non-tiny weight is a normal fp16.
  struct Blk { const float* src; int lds, scol, n_rows, n_dst_off; };
  unsigned* d_absmax = nullptr;
  int tn = 256;                    // n-tile width of the images = hidden_nf
  void image(TcImage* img, int Nn, int K, const Blk* blk, int nblk) {
    const size_t nt = (size_t)Nn * K;            // floats per TF32 image (hi or lo): [Nn/tn][K/32][tn x 32]
    const size_t nh = (size_t)Nn * K / 2;        // 32-bit words per FP16 image:       [Nn/tn][K/64][tn x 64 halfs]
    float* thi = alloc(nt); float* tlo = alloc(nt); float* hhi = alloc(nh); float* hlo = alloc(nh);
    img->t_hi = thi; img->t_lo = tlo; img->h_hi = hhi; img->h_lo = hlo; img->h_inv = 1.0f;
    if (dry) return;
    if (!d_absmax) cudaMalloc(&d_absmax, sizeof(unsigned));
    cudaMemset(d_absmax, 0, sizeof(unsigned));
    for (int i = 0; i < nblk; ++i) launch_absmax(blk[i].src, blk[i].lds, blk[i].scol, blk[i].n_rows, K, d_absmax);
    unsigned bits = 0;
    cudaMemcpy(&bits, d_absmax, sizeof(unsigned), cudaMemcpyDeviceToHost);
    float amax; memcpy(&amax, &bits, sizeof(float));
    float scale = 1.0f;
    if (amax > 0.f && amax < 3.0e38f) { int e; frexpf(amax, &e); scale = ldexpf(1.0f, 13 - e); }   // amax*scale in [4096, 8192)
    img->h_inv = 1.0f / scale;     // activation scale X_SCALE is 1
    for (int i = 0; i < nblk; ++i) {
      launch_pack_b_image(thi, tlo, blk[i].src, blk[i].lds, blk[i].scol, blk[i].n_rows, blk[i].n_dst_off, K, tn);
      launch_pack_b_image_f16(hhi, hlo, blk[i].src, blk[i].lds, blk[i].scol, blk[i].n_rows, blk[i].n_dst_off, K, scale, tn);
    }
  }
  const float* copy(const float* src, int64_t n) {
    float* d = alloc(n);
    if (!dry) pack_copy_kernel<<<(unsigned)((n + 255) / 256), 256>>>(d, src, n);
    return d;
  }
};

static int pack_weights(dsb_dynamics* d, const float* const* params, const std::vector<ParamInfo>& tab, bool dry,
                        size_t* floats_out) {
  const dsb_config& c = d->cfg;
  const int H = c.hidden_nf, J = c.joint_nf, Din = J + (c.condition_time ? 1 : 0), De = c.edge_embedding_dim;
  const int NS = c.sin_embedding ? 12 : 1;         // radial features per distance: d^2, or its 12 sinusoids (egnn_new.py:282-293)
  const int F = 2 * NS + De, ld1 = 2 * H + F;
  std::map<std::string, int> index;
  for (size_t i = 0; i < tab.size(); ++i) index[tab[i].name] = (int)i;
  auto P = [&](const std::string& n) -> const float* { return dry ? nullptr : params[index.at(n)]; };
  auto numel = [&](const std::string& n) { return tab[index.at(n)].numel; };
  Packer pk(dry ? nullptr : d->blob);
  pk.tn = H;
  const bool tc = tc_width_supported(H);
  PackedWeights& w = d->w;
  auto cp = [&](const std::string& n) { return pk.copy(P(n), numel(n)); };

  w.aenc0_w = cp("atom_encoder.0.weight"); w.aenc0_b = cp("atom_encoder.0.bias");
  w.renc0_w = cp("residue_encoder.0.weight"); w.renc0_b = cp("residue_encoder.0.bias");
  w.adec2_w = cp("atom_decoder.2.weight"); w.adec2_b = cp("atom_decoder.2.bias");
  w.rdec2_w = cp("residue_decoder.2.weight"); w.rdec2_b = cp("residue_decoder.2.bias");
  for (int ty = 0; ty < 2; ++ty) {
    const std::string enc = ty == 0 ? "atom_encoder" : "residue_encoder", dec = ty == 0 ? "atom_decoder" : "residue_decoder";
    const int F2 = 2 * (ty == 0 ? c.atom_nf : c.residue_nf), K = F2 + (Din > J ? 1 : 0);
    float* pw = pk.alloc((size_t)K * H); float* pb = pk.alloc(H);
    float* dw = pk.alloc((size_t)F2 * H); float* db = pk.alloc(F2);
    if (!dry) {
      pack_pre_kernel<<<((K + 1) * H + 255) / 256, 256>>>(pw, pb, P("egnn.embedding.weight"), P("egnn.embedding.bias"),
                                                            P(enc + ".2.weight"), P(enc + ".2.bias"), H, J, Din, F2);
      pack_dec_kernel<<<(F2 * (H + 1) + 255) / 256, 256>>>(dw, db, P(dec + ".0.weight"), P(dec + ".0.bias"),
                                                            P("egnn.embedding_out.weight"), P("egnn.embedding_out.bias"), H, J, F2);
    }
    w.pre_wT[ty] = pw; w.pre_b[ty] = pb; w.dec_w[ty] = dw; w.dec_b[ty] = db;
  }
  const float* emb = De > 0 ? P("edge_embedding.weight") : nullptr;

  auto first_layer = [&](const std::string& pre, float* W1dst, int ldd, int dcol_recv, int dcol_send, float* b1dst,
                         const float** wr, const float** wr0, const float** tb) {
    const float* W1 = P(pre + ".weight");
    pk.T(W1, ld1, 0, H, H, W1dst, ldd, dcol_recv);     // receiver part  (h[row], egnn_new.py:35/99)
    pk.T(W1, ld1, H, H, H, W1dst, ldd, dcol_send);     // sender part    (h[col])
    if (!dry) pack_copy_kernel<<<(H + 255) / 256, 256>>>(b1dst + dcol_recv, P(pre + ".bias"), H);
    float* r = pk.alloc((size_t)NS * H); pk.T(W1, ld1, 2 * H, H, NS, r, H, 0); *wr = r;                 // [NS][H]: current geometry
    float* r0 = pk.alloc((size_t)NS * H); pk.T(W1, ld1, 2 * H + NS, H, NS, r0, H, 0); *wr0 = r0;      // [NS][H]: input geometry
    if (De > 0) {
      float* t = pk.alloc((size_t)3 * H);
      if (!dry) pack_tb_kernel<<<(3 * H + 255) / 256, 256>>>(t, W1, ld1, 2 * H + 2 * NS, emb, De, H);
      *tb = t;
    } else {
      *tb = nullptr;
    }
  };

  for (int k = 0; k < c.n_layers; ++k) {
    const std::string b = "egnn.e_block_" + std::to_string(k);
    for (int s = 0; s < c.inv_sublayers; ++s) {
      const std::string g = b + ".gcl_" + std::to_string(s);
      GclW& G = w.gcl[k][s];
      float* W1 = pk.alloc((size_t)H * 2 * H); float* b1 = pk.alloc(2 * H);
      first_layer(g + ".edge_mlp.0", W1, 2 * H, 0, H, b1, &G.wr, &G.wr0, &G.tb);
      G.W1ab = W1; G.b1ab = b1;
      { float* t = pk.alloc((size_t)H * H); G.W2 = pk.T(P(g + ".edge_mlp.2.weight"), H, 0, H, H, t, H, 0); }
      G.b2 = cp(g + ".edge_mlp.2.bias");
      if (c.attention) { G.wa = cp(g + ".att_mlp.0.weight"); G.ba = cp(g + ".att_mlp.0.bias"); }
      else { G.wa = nullptr; G.ba = nullptr; }
      { float* t = pk.alloc((size_t)2 * H * H); G.W3 = pk.T(P(g + ".node_mlp.0.weight"), 2 * H, 0, H, 2 * H, t, H, 0); }
      G.b3 = cp(g + ".node_mlp.0.bias");
      { float* t = pk.alloc((size_t)H * H); G.W4 = pk.T(P(g + ".node_mlp.2.weight"), H, 0, H, H, t, H, 0); }
      G.b4 = cp(g + ".node_mlp.2.bias");
      G.iW1ab = G.iW2 = G.iW3 = G.iW4 = TcImage{nullptr, nullptr, nullptr, nullptr, 1.0f};
      if (tc) {
        const float* W1 = P(g + ".edge_mlp.0.weight");
        Packer::Blk b1[2] = {{W1, ld1, 0, H, 0}, {W1, ld1, H, H, H}};     // receiver part -> columns 0..H-1, sender -> H..2H-1
        pk.image(&G.iW1ab, 2 * H, H, b1, 2);
        Packer::Blk b2 = {P(g + ".edge_mlp.2.weight"), H, 0, H, 0};
        pk.image(&G.iW2, H, H, &b2, 1);
        Packer::Blk b3 = {P(g + ".node_mlp.0.weight"), 2 * H, 0, H, 0};
        pk.image(&G.iW3, H, 2 * H, &b3, 1);
        Packer::Blk b4 = {P(g + ".node_mlp.2.weight"), H, 0, H, 0};
        pk.image(&G.iW4, H, H, &b4, 1);
      }
    }
    const std::string q = b + ".gcl_equiv";
    EquivW& Q = w.eq[k];
    const int nm = c.reflection_equivariant ? 1 : 2;
    Q.nq = nm * 2 * H;
    Q.np = (k + 1 < c.n_layers) ? 2 * H : 0;          // merged with the next block's first GCL (same input h)
    const int ldm = Q.nq + Q.np;
    float* W1 = pk.alloc((size_t)H * ldm); float* b1 = pk.alloc((size_t)ldm);
    const char* names[2] = {".coord_mlp", ".cross_product_mlp"};
    for (int m = 0; m < 2; ++m) {
      if (m < nm) {
        first_layer(q + names[m] + ".0", W1, ldm, m * H, nm * H + m * H, b1, &Q.wr[m], &Q.wr0[m], &Q.tb[m]);
        float* t = pk.alloc((size_t)H * H);
        Q.W2[m] = pk.T(P(q + names[m] + ".2.weight"), H, 0, H, H, t, H, 0);
        Q.b2[m] = cp(q + names[m] + ".2.bias");
      } else {
        Q.wr[m] = Q.wr0[m] = Q.tb[m] = Q.W2[m] = Q.b2[m] = nullptr;
      }
    }
    const std::string gnext = "egnn.e_block_" + std::to_string(k + 1) + ".gcl_0.edge_mlp.0";
    if (Q.np) {
      const float* Wn = P(gnext + ".weight");
      pk.T(Wn, ld1, 0, H, H, W1, ldm, Q.nq);           // next GCL: receiver part
      pk.T(Wn, ld1, H, H, H, W1, ldm, Q.nq + H);       //           sender part
      if (!dry) pack_copy_kernel<<<(H + 255) / 256, 256>>>(b1 + Q.nq, P(gnext + ".bias"), H);
    }
    Q.W1 = W1; Q.b1 = b1;
    Q.w3 = cp(q + ".coord_mlp.4.weight");
    Q.iW1 = Q.iW2[0] = Q.iW2[1] = TcImage{nullptr, nullptr, nullptr, nullptr, 1.0f};
    if (tc) {
      Packer::Blk blk[6];
      int nb = 0;
      for (int m = 0; m < nm; ++m) {
        const float* W = P(q + names[m] + ".0.weight");
        blk[nb++] = {W, ld1, 0, H, m * H};                    // receiver block
        blk[nb++] = {W, ld1, H, H, nm * H + m * H};           // sender block
        Packer::Blk b2 = {P(q + names[m] + ".2.weight"), H, 0, H, 0};
        pk.image(&Q.iW2[m], H, H, &b2, 1);
      }
      if (Q.np) {
        const float* Wn = P(gnext + ".weight");
        blk[nb++] = {Wn, ld1, 0, H, Q.nq};
        blk[nb++] = {Wn, ld1, H, H, Q.nq + H};
      }
      pk.image(&Q.iW1, Q.nq + Q.np, H, blk, nb);
    }
  }
  if (pk.d_absmax) cudaFree(pk.d_absmax);
  *floats_out = pk.used;
  return 0;
}

// ---- workspace --------------------------------------------------------------------------------------------
static Workspace carve(const dsb_config& c, int64_t NL, int64_t NP, int64_t B, int64_t Ecap, void* base) {
  Workspace ws;
  const int64_t N = NL + NP;
  const int H = c.hidden_nf;
  size_t off = 0;
  auto take = [&](size_t bytes) { size_t o = off; off += (bytes + 255) & ~size_t(255); return base ? (char*)base + o : (char*)nullptr; };
  ws.lig_off = (int32_t*)take(sizeof(int32_t) * (B + 2));
  ws.poc_off = (int32_t*)take(sizeof(int32_t) * (B + 2));
  ws.gid = (int32_t*)take(sizeof(int32_t) * (N + 1));
  for (int i = 0; i < 3; ++i) ws.xbuf[i] = (float4*)take(sizeof(float4) * (N + 1));
  ws.cent = (float4*)take(sizeof(float4) * (B + 1));
  ws.xagg = (float4*)take(sizeof(float4) * (N + 1));
  ws.velmean = (float4*)take(sizeof(float4) * (B + 1));
  ws.h = (float*)take(sizeof(float) * (size_t)(N + 1) * H);
  ws.hT = (float*)take(sizeof(float) * (size_t)(N + 1) * H);
  ws.agg = (float*)take(sizeof(float) * (size_t)(N + 1) * H);
  ws.P = (float*)take(sizeof(float) * (size_t)(N + 1) * 6 * H);
  ws.deg = (int32_t*)take(sizeof(int32_t) * (N + 1));
  ws.row_ptr = (int32_t*)take(sizeof(int32_t) * (N + 2));
  ws.vrow_ptr = (int32_t*)take(sizeof(int32_t) * (N + 2));
  ws.vmap = (int32_t*)take(sizeof(int32_t) * (size_t)(Ecap + (kRowChunk - 1) * N + 1));
  ws.erow = (int32_t*)take(sizeof(int32_t) * (size_t)(Ecap + 1));
  ws.ecol = (int32_t*)take(sizeof(int32_t) * (size_t)(Ecap + 1));
  ws.ed0 = (float*)take(sizeof(float) * (size_t)(Ecap + 1));
  ws.bytes = off;
  return ws;
}

static int check_sizes(int64_t NL, int64_t NP, int64_t B, int64_t Ecap) {
  if (NL < 0 || NP < 0 || B < 0 || Ecap < 0 || NL + NP > (int64_t)1 << 30 || Ecap > ((int64_t)1 << 31) - 256) {
    set_error("sizes out of range (n_atoms=%lld n_residues=%lld n_graphs=%lld edge_capacity=%lld)", (long long)NL,
              (long long)NP, (long long)B, (long long)Ecap);
    return DSB_ERR_INVALID_ARGUMENT;
  }
  return 0;
}

// ---- fused DDPM ligand update --------------------------------------------------------------------------
__device__ __forceinline__ int lb64(const int64_t* a, int n, int64_t v) {
  int lo = 0, hi = n;
  while (lo < hi) { int mid = (lo + hi) >> 1; if (a[mid] < v) lo = mid + 1; else hi = mid; }
  return lo;
}

// z/z_out and pocket/pocket_out may alias (in-place use is part of the contract): no __restrict__ on those pairs.
__global__ void __launch_bounds__(128) ddpm_update_kernel(const float* z, const float* __restrict__ eps,
                                                           const float* __restrict__ noise, const float* __restrict__ coef,
                                                           const int64_t* __restrict__ mask_atoms, const int64_t* __restrict__ mask_res,
                                                           const float* pocket, int NL, int NP, int A, int R,
                                                           float* z_out, float* pocket_out) {
  const int g = blockIdx.x;
  const int l0 = lb64(mask_atoms, NL, g), l1 = lb64(mask_atoms, NL, (int64_t)g + 1);
  const int p0 = lb64(mask_res, NP, g), p1 = lb64(mask_res, NP, (int64_t)g + 1);
  const int D = 3 + A, DR = 3 + R;
  const float alpha = coef[g * 3 + 0], cb = coef[g * 3 + 1], sigma = coef[g * 3 + 2];
  float s[3] = {0.f, 0.f, 0.f};
  for (int idx = l0 * D + threadIdx.x; idx < l1 * D; idx += blockDim.x) {
    const float mu = z[idx] / alpha - cb * eps[idx];          // conditional_model.py:451-453
    const float v = mu + sigma * noise[idx];                   // conditional_model.py:151
    z_out[idx] = v;
    const int c = idx % D;
    if (c < 3) s[c] += v;
  }
  __shared__ float red[3][4];
  __shared__ float com[3];
#pragma unroll
  for (int k = 0; k < 3; ++k)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s[k] += __shfl_xor_sync(0xffffffffu, s[k], o);
  if ((threadIdx.x & 31) == 0) { red[0][threadIdx.x >> 5] = s[0]; red[1][threadIdx.x >> 5] = s[1]; red[2][threadIdx.x >> 5] = s[2]; }
  __syncthreads();
  if (threadIdx.x < 3) {
    const float cnt = (l1 - l0) > 0 ? (float)(l1 - l0) : 1.f;
    com[threadIdx.x] = (red[threadIdx.x][0] + red[threadIdx.x][1] + red[threadIdx.x][2] + red[threadIdx.x][3]) / cnt;
  }
  __syncthreads();
  for (int i = l0 + threadIdx.x; i < l1; i += blockDim.x) {     // conditional_model.py:694
    z_out[(size_t)i * D + 0] -= com[0]; z_out[(size_t)i * D + 1] -= com[1]; z_out[(size_t)i * D + 2] -= com[2];
  }
  for (int idx = p0 * DR + threadIdx.x; idx < p1 * DR; idx += blockDim.x) {   // conditional_model.py:695
    const int c = idx % DR;
    const float v = pocket[idx];
    pocket_out[idx] = c < 3 ? v - com[c] : v;
  }
}


// ---- fused RePaint iteration of ConditionalDDPM.inpaint (conditional_model.py:636-666) -------------------------------
// sum of `nv` (<= 9) per-thread values over a 128-thread block; result valid in every thread.  `red` is [9][4] shared floats.
__device__ __forceinline__ void block_sum(float* v, int nv, float (*red)[4]) {
  for (int k = 0; k < nv; ++k)
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) v[k] += __shfl_xor_sync(0xffffffffu, v[k], o);
  __syncthreads();                      // previous use of `red` is complete
  if ((threadIdx.x & 31) == 0) for (int k = 0; k < nv; ++k) red[k][threadIdx.x >> 5] = v[k];
  __syncthreads();
  for (int k = 0; k < nv; ++k) v[k] = (red[k][0] + red[k][1]) + (red[k][2] + red[k][3]);
}

// One block per graph.  On entry z = z_unknown (the reverse step's output), pocket = the pocket that step left.  In place:
//   known part noised to level s around the pocket's current COM, ligand-COM removed (noised_representation, :162-183),
//   COM of the fixed atoms aligned noised -> denoised (:645-656), blend (:659), optional re-noising step
//   z_t ~ q(z_t | z_s) with its own COM removal (sample_p_zt_given_zs, :420-430, :662-666).
// Every per-element fp32 operation is the one the torch ops of the eager loop perform, in the same order; only the
// per-graph means are summed in a different order.
__global__ void __launch_bounds__(128) ddpm_inpaint_kernel(float* z, float* pocket, const float* __restrict__ known,
                                                            const float* __restrict__ com_pocket0, const float* __restrict__ fixed,
                                                            const float* __restrict__ noise1, const float* __restrict__ noise2,
                                                            const float* __restrict__ coef, const int64_t* __restrict__ mask_atoms,
                                                            const int64_t* __restrict__ mask_res, int NL, int NP, int A, int R) {
  const int g = blockIdx.x;
  const int l0 = lb64(mask_atoms, NL, g), l1 = lb64(mask_atoms, NL, (int64_t)g + 1);
  const int p0 = lb64(mask_res, NP, g), p1 = lb64(mask_res, NP, (int64_t)g + 1);
  const int D = 3 + A, DR = 3 + R;
  const float alpha_s = coef[g * 4 + 0], sigma_s = coef[g * 4 + 1], alpha_ts = coef[g * 4 + 2], sigma_ts = coef[g * 4 + 3];
  __shared__ float red[9][4];
  const float nl = (l1 - l0) > 0 ? (float)(l1 - l0) : 1.f, np_ = (p1 - p0) > 0 ? (float)(p1 - p0) : 1.f;

  // pocket COM now vs. at the start: the known ligand follows the pocket (:636-640)
  float v[9];
  v[0] = v[1] = v[2] = 0.f;
  for (int i = p0 + threadIdx.x; i < p1; i += blockDim.x) {
    v[0] += pocket[(size_t)i * DR + 0]; v[1] += pocket[(size_t)i * DR + 1]; v[2] += pocket[(size_t)i * DR + 2];
  }
  block_sum(v, 3, red);
  float shift[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) shift[c] = v[c] / np_ - com_pocket0[g * 3 + c];

  auto zk_raw = [&](int idx, int c) {       // alpha_s * xh_known + sigma_s * eps   (:176)
    const float xk = c < 3 ? known[idx] + shift[c] : known[idx];
    return alpha_s * xk + sigma_s * noise1[idx];
  };
  // ligand COM of the noised known part (:180-182)
  v[0] = v[1] = v[2] = 0.f;
  for (int idx = l0 * D + threadIdx.x; idx < l1 * D; idx += blockDim.x) {
    const int c = idx % D;
    if (c < 3) v[c] += zk_raw(idx, c);
  }
  block_sum(v, 3, red);
  float comk[3] = {v[0] / nl, v[1] / nl, v[2] / nl};
  // COM of the fixed atoms: noised vs. denoised (:648-652)
  for (int k = 0; k < 7; ++k) v[k] = 0.f;
  for (int idx = l0 * D + threadIdx.x; idx < l1 * D; idx += blockDim.x) {
    const int c = idx % D, i = idx / D;
    if (c < 3 && fixed[i] != 0.f) { v[c] += zk_raw(idx, c) - comk[c]; v[3 + c] += z[idx]; if (c == 0) v[6] += 1.f; }
  }
  block_sum(v, 7, red);
  const float nf = v[6] > 0.f ? v[6] : 1.f;
  float dx[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) dx[c] = v[3 + c] / nf - v[c] / nf;
  // blend (+ re-noise)
  float s2[3] = {0.f, 0.f, 0.f};
  for (int idx = l0 * D + threadIdx.x; idx < l1 * D; idx += blockDim.x) {
    const int c = idx % D, i = idx / D;
    float zk = zk_raw(idx, c);
    if (c < 3) zk = (zk - comk[c]) + dx[c];
    const float f = fixed[i];
    float o = zk * f + z[idx] * (1.f - f);                        // :659
    if (noise2) { o = alpha_ts * o + sigma_ts * noise2[idx]; if (c < 3) s2[c] += o; }
    z[idx] = o;
  }
  float com2[3] = {0.f, 0.f, 0.f};
  if (noise2) {
    block_sum(s2, 3, red);
#pragma unroll
    for (int c = 0; c < 3; ++c) com2[c] = s2[c] / nl;
    __syncthreads();
    for (int i = l0 + threadIdx.x; i < l1; i += blockDim.x) {
      z[(size_t)i * D + 0] -= com2[0]; z[(size_t)i * D + 1] -= com2[1]; z[(size_t)i * D + 2] -= com2[2];
    }
  }
  for (int idx = p0 * DR + threadIdx.x; idx < p1 * DR; idx += blockDim.x) {
    const int c = idx % DR;
    if (c < 3) {
      float q = (pocket[idx] - comk[c]) + dx[c];
      if (noise2) q -= com2[c];
      pocket[idx] = q;
    }
  }
}


// ---- joint model (EnVariationalDiffusion): fused reverse update and fused RePaint iteration ---------------------------
// Node n of graph g: ligand rows [l0, l1) of the ligand tensors, pocket rows [p0, p1) of the pocket tensors.  The position
// noise nx is ONE tensor [NL + NP, 3] (ligand rows first), as sample_center_gravity_zero_gaussian_batch draws it
// (en_diffusion.py:559-578); its per-graph mean over ligand+pocket nodes is removed before use (en_diffusion.py:940-944).
struct JointSpan { int l0, l1, p0, p1; float n; };
__device__ __forceinline__ JointSpan joint_span(const int64_t* mask_atoms, const int64_t* mask_res, int NL, int NP, int g) {
  JointSpan s;
  s.l0 = lb64(mask_atoms, NL, g); s.l1 = lb64(mask_atoms, NL, (int64_t)g + 1);
  s.p0 = lb64(mask_res, NP, g); s.p1 = lb64(mask_res, NP, (int64_t)g + 1);
  const int cnt = (s.l1 - s.l0) + (s.p1 - s.p0);
  s.n = cnt > 0 ? (float)cnt : 1.f;
  return s;
}
// per-graph mean of the position noise rows
__device__ __forceinline__ void joint_noise_mean(const float* nx, const JointSpan& sp, int NL, float (*red)[4], float* mean) {
  float v[3] = {0.f, 0.f, 0.f};
  for (int i = sp.l0 + threadIdx.x; i < sp.l1; i += blockDim.x) { v[0] += nx[i * 3]; v[1] += nx[i * 3 + 1]; v[2] += nx[i * 3 + 2]; }
  for (int i = sp.p0 + threadIdx.x; i < sp.p1; i += blockDim.x) {
    const size_t r = (size_t)(NL + i) * 3; v[0] += nx[r]; v[1] += nx[r + 1]; v[2] += nx[r + 2];
  }
  block_sum(v, 3, red);
  mean[0] = v[0] / sp.n; mean[1] = v[1] / sp.n; mean[2] = v[2] / sp.n;
}

// EnVariationalDiffusion.sample_p_zs_given_zt without the denoiser call (en_diffusion.py:503-557):
//   mu = z / alpha_ts - coef * eps_hat ; z' = mu + sigma * eps (eps.x COM-free over ligand+pocket) ; joint COM of z'.x removed.
__global__ void __launch_bounds__(128) ddpm_joint_update_kernel(float* z_lig, float* z_poc, const float* __restrict__ eps_lig,
                                                                 const float* __restrict__ eps_poc, const float* __restrict__ nx,
                                                                 const float* __restrict__ nhl, const float* __restrict__ nhp,
                                                                 const float* __restrict__ coef, const int64_t* __restrict__ mask_atoms,
                                                                 const int64_t* __restrict__ mask_res, int NL, int NP, int A, int R) {
  const int g = blockIdx.x;
  const JointSpan sp = joint_span(mask_atoms, mask_res, NL, NP, g);
  const int D = 3 + A, DR = 3 + R;
  const float alpha = coef[g * 3 + 0], cb = coef[g * 3 + 1], sigma = coef[g * 3 + 2];
  __shared__ float red[9][4];
  float nm[3];
  joint_noise_mean(nx, sp, NL, red, nm);
  float s[3] = {0.f, 0.f, 0.f};
  for (int idx = sp.l0 * D + threadIdx.x; idx < sp.l1 * D; idx += blockDim.x) {
    const int c = idx % D, i = idx / D;
    const float e = c < 3 ? nx[(size_t)i * 3 + c] - nm[c] : nhl[(size_t)i * A + (c - 3)];
    const float v = (z_lig[idx] / alpha - cb * eps_lig[idx]) + sigma * e;
    z_lig[idx] = v;
    if (c < 3) s[c] += v;
  }
  for (int idx = sp.p0 * DR + threadIdx.x; idx < sp.p1 * DR; idx += blockDim.x) {
    const int c = idx % DR, i = idx / DR;
    const float e = c < 3 ? nx[(size_t)(NL + i) * 3 + c] - nm[c] : nhp[(size_t)i * R + (c - 3)];
    const float v = (z_poc[idx] / alpha - cb * eps_poc[idx]) + sigma * e;
    z_poc[idx] = v;
    if (c < 3) s[c] += v;
  }
  block_sum(s, 3, red);
  const float m0 = s[0] / sp.n, m1 = s[1] / sp.n, m2 = s[2] / sp.n;
  __syncthreads();
  for (int i = sp.l0 + threadIdx.x; i < sp.l1; i += blockDim.x) {
    z_lig[(size_t)i * D] -= m0; z_lig[(size_t)i * D + 1] -= m1; z_lig[(size_t)i * D + 2] -= m2;
  }
  for (int i = sp.p0 + threadIdx.x; i < sp.p1; i += blockDim.x) {
    z_poc[(size_t)i * DR] -= m0; z_poc[(size_t)i * DR + 1] -= m1; z_poc[(size_t)i * DR + 2] -= m2;
  }
}

// One RePaint iteration of EnVariationalDiffusion.inpaint after the reverse step (en_diffusion.py:741-807), in place on
// (z_lig, z_poc) = the denoised "unknown" sample:
//   z_known = alpha_s xh0 + sigma_s eps1 (eps1.x COM-free)                                  (noised_representation, :302-317)
//   shift   = COM_fixed(z_unknown) - COM_fixed(z_known) over the fixed ligand+pocket nodes ; z_known.x += shift   (:751-772)
//   z       = z_known * fixed + z_unknown * (1 - fixed)                                       (:774-775)
//   if nx3: z = alpha_ts z + sigma_ts eps3 (eps3.x COM-free), joint COM of z.x removed        (sample_p_zt_given_zs, :479-501, :790-807)
__global__ void __launch_bounds__(128) ddpm_joint_inpaint_kernel(
    float* z_lig, float* z_poc, const float* __restrict__ x0_lig, const float* __restrict__ x0_poc, const float* __restrict__ fix_lig,
    const float* __restrict__ fix_poc, const float* __restrict__ nx1, const float* __restrict__ nhl1, const float* __restrict__ nhp1,
    const float* __restrict__ nx3, const float* __restrict__ nhl3, const float* __restrict__ nhp3, const float* __restrict__ coef,
    const int64_t* __restrict__ mask_atoms, const int64_t* __restrict__ mask_res, int NL, int NP, int A, int R) {
  const int g = blockIdx.x;
  const JointSpan sp = joint_span(mask_atoms, mask_res, NL, NP, g);
  const int D = 3 + A, DR = 3 + R;
  const float alpha_s = coef[g * 4 + 0], sigma_s = coef[g * 4 + 1], alpha_ts = coef[g * 4 + 2], sigma_ts = coef[g * 4 + 3];
  __shared__ float red[9][4];
  float n1[3];
  joint_noise_mean(nx1, sp, NL, red, n1);
  auto zk_lig = [&](int idx, int c, int i) {
    const float e = c < 3 ? nx1[(size_t)i * 3 + c] - n1[c] : nhl1[(size_t)i * A + (c - 3)];
    return alpha_s * x0_lig[idx] + sigma_s * e;
  };
  auto zk_poc = [&](int idx, int c, int i) {
    const float e = c < 3 ? nx1[(size_t)(NL + i) * 3 + c] - n1[c] : nhp1[(size_t)i * R + (c - 3)];
    return alpha_s * x0_poc[idx] + sigma_s * e;
  };
  // COM of the fixed nodes: denoised vs. noised
  float v[7] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int idx = sp.l0 * D + threadIdx.x; idx < sp.l1 * D; idx += blockDim.x) {
    const int c = idx % D, i = idx / D;
    if (c < 3 && fix_lig[i] != 0.f) { v[c] += z_lig[idx]; v[3 + c] += zk_lig(idx, c, i); if (c == 0) v[6] += 1.f; }
  }
  for (int idx = sp.p0 * DR + threadIdx.x; idx < sp.p1 * DR; idx += blockDim.x) {
    const int c = idx % DR, i = idx / DR;
    if (c < 3 && fix_poc[i] != 0.f) { v[c] += z_poc[idx]; v[3 + c] += zk_poc(idx, c, i); if (c == 0) v[6] += 1.f; }
  }
  block_sum(v, 7, red);
  const float nf = v[6] > 0.f ? v[6] : 1.f;
  float shift[3];
#pragma unroll
  for (int c = 0; c < 3; ++c) shift[c] = v[c] / nf - v[3 + c] / nf;
  float n3[3] = {0.f, 0.f, 0.f};
  if (nx3) joint_noise_mean(nx3, sp, NL, red, n3);
  float s[3] = {0.f, 0.f, 0.f};
  for (int idx = sp.l0 * D + threadIdx.x; idx < sp.l1 * D; idx += blockDim.x) {
    const int c = idx % D, i = idx / D;
    float zk = zk_lig(idx, c, i);
    if (c < 3) zk += shift[c];
    const float f = fix_lig[i];
    float o = zk * f + z_lig[idx] * (1.f - f);
    if (nx3) {
      const float e = c < 3 ? nx3[(size_t)i * 3 + c] - n3[c] : nhl3[(size_t)i * A + (c - 3)];
      o = alpha_ts * o + sigma_ts * e;
      if (c < 3) s[c] += o;
    }
    z_lig[idx] = o;
  }
  for (int idx = sp.p0 * DR + threadIdx.x; idx < sp.p1 * DR; idx += blockDim.x) {
    const int c = idx % DR, i = idx / DR;
    float zk = zk_poc(idx, c, i);
    if (c < 3) zk += shift[c];
    const float f = fix_poc[i];
    float o = zk * f + z_poc[idx] * (1.f - f);
    if (nx3) {
      const float e = c < 3 ? nx3[(size_t)(NL + i) * 3 + c] - n3[c] : nhp3[(size_t)i * R + (c - 3)];
      o = alpha_ts * o + sigma_ts * e;
      if (c < 3) s[c] += o;
    }
    z_poc[idx] = o;
  }
  if (nx3) {
    block_sum(s, 3, red);
    const float m0 = s[0] / sp.n, m1 = s[1] / sp.n, m2 = s[2] / sp.n;
    __syncthreads();
    for (int i = sp.l0 + threadIdx.x; i < sp.l1; i += blockDim.x) {
      z_lig[(size_t)i * D] -= m0; z_lig[(size_t)i * D + 1] -= m1; z_lig[(size_t)i * D + 2] -= m2;
    }
    for (int i = sp.p0 + threadIdx.x; i < sp.p1; i += blockDim.x) {
      z_poc[(size_t)i * DR] -= m0; z_poc[(size_t)i * DR + 1] -= m1; z_poc[(size_t)i * DR + 2] -= m2;
    }
  }
}

}  // namespace dsb

using namespace dsb;

extern "C" {

const char* dsb_last_error(void) { return g_err; }
const char* dsb_version(void) { return "diffsbdd_b200 0.3 (sm_100a: tcgen05 3xFP16 CTA-pair edge kernels and fused node block kernel, 3xTF32 single-CTA kernels, fp32 FFMA kernels)"; }

int dsb_param_count(const dsb_config* cfg) {
  if (int e = validate(cfg)) return e;
  return (int)param_table(*cfg).size();
}

int64_t dsb_param_name(const dsb_config* cfg, int i, char* buf, size_t buflen) {
  if (int e = validate(cfg)) return e;
  auto tab = param_table(*cfg);
  if (i < 0 || i >= (int)tab.size() || !buf || buflen == 0) { set_error("param index out of range"); return DSB_ERR_INVALID_ARGUMENT; }
  snprintf(buf, buflen, "%s", tab[i].name.c_str());
  return tab[i].numel;
}

int dsb_dynamics_create(const dsb_config* cfg, const float* const* params, int n_params, dsb_dynamics** out) {
  if (!out) { set_error("null out"); return DSB_ERR_INVALID_ARGUMENT; }
  *out = nullptr;
  if (int e = validate(cfg)) return e;
  auto tab = param_table(*cfg);
  if (!params || n_params != (int)tab.size()) { set_error("expected %d parameters, got %d", (int)tab.size(), n_params); return DSB_ERR_INVALID_ARGUMENT; }
  for (int i = 0; i < n_params; ++i)
    if (!params[i]) { set_error("parameter %d (%s) is null", i, tab[i].name.c_str()); return DSB_ERR_INVALID_ARGUMENT; }
  dsb_dynamics* d = new dsb_dynamics();
  d->cfg = *cfg;
  size_t floats = 0;
  pack_weights(d, params, tab, /*dry=*/true, &floats);
  d->blob_floats = floats;
  cudaError_t ce = cudaMalloc(&d->blob, floats * sizeof(float));
  if (ce != cudaSuccess) { set_error("cudaMalloc(%zu) failed: %s", floats * sizeof(float), cudaGetErrorString(ce)); delete d; return DSB_ERR_CUDA; }
  cudaMemset(d->blob, 0, floats * sizeof(float));
  pack_weights(d, params, tab, /*dry=*/false, &floats);
  ce = cudaDeviceSynchronize();
  if (ce == cudaSuccess) ce = cudaGetLastError();
  if (ce != cudaSuccess) { set_error("weight packing failed: %s", cudaGetErrorString(ce)); cudaFree(d->blob); delete d; return DSB_ERR_CUDA; }
  int dev = 0; cudaGetDevice(&dev);
  cudaDeviceGetAttribute(&d->num_sms, cudaDevAttrMultiProcessorCount, dev);
  if (int e = configure_node_kernels()) { cudaFree(d->blob); delete d; return e; }
  if (int e = configure_edge_kernels(cfg->hidden_nf)) { cudaFree(d->blob); delete d; return e; }
  if (tc_width_supported(cfg->hidden_nf)) { if (int e = configure_tc_kernels(cfg->hidden_nf)) { cudaFree(d->blob); delete d; return e; } }
  *out = d;
  return 0;
}

void dsb_dynamics_destroy(dsb_dynamics* dyn) {
  if (!dyn) return;
  cudaDeviceSynchronize();
  cudaFree(dyn->blob);
  if (dyn->prof_ev) { for (int i = 0; i < 2 * kMaxProfEvents; ++i) cudaEventDestroy(dyn->prof_ev[i]); delete[] dyn->prof_ev; }
  delete dyn;
}

int64_t dsb_edge_capacity(const int64_t* n_lig, const int64_t* n_pocket, int n_graphs) {
  int64_t tot = 0;
  for (int g = 0; g < n_graphs; ++g) { const int64_t n = n_lig[g] + n_pocket[g]; tot += n * n; }
  return tot;
}

size_t dsb_dynamics_workspace_bytes(const dsb_dynamics* dyn, int64_t n_atoms, int64_t n_residues, int64_t n_graphs,
                                    int64_t edge_capacity) {
  if (!dyn || check_sizes(n_atoms, n_residues, n_graphs, edge_capacity)) return 0;
  return carve(dyn->cfg, n_atoms, n_residues, n_graphs, edge_capacity, nullptr).bytes + 256;
}

static int setup(dsb_dynamics* dyn, int64_t n_atoms, int64_t n_residues, int64_t n_graphs, int64_t edge_capacity,
                 void* workspace, size_t workspace_bytes, Dims* dm, Workspace* ws) {
  if (!dyn) { set_error("null handle"); return DSB_ERR_INVALID_ARGUMENT; }
  if (int e = check_sizes(n_atoms, n_residues, n_graphs, edge_capacity)) return e;
  if (!workspace) { set_error("null workspace"); return DSB_ERR_INVALID_ARGUMENT; }
  char* base = (char*)(((uintptr_t)workspace + 255) & ~(uintptr_t)255);
  *ws = carve(dyn->cfg, n_atoms, n_residues, n_graphs, edge_capacity, base);
  if ((size_t)(base - (char*)workspace) + ws->bytes > workspace_bytes) {
    set_error("workspace too small: need %zu bytes, got %zu", ws->bytes + 256, workspace_bytes);
    return DSB_ERR_WORKSPACE_TOO_SMALL;
  }
  dm->NL = (int)n_atoms; dm->NP = (int)n_residues; dm->N = (int)(n_atoms + n_residues); dm->B = (int)n_graphs;
  dm->Ecap = edge_capacity;
  dm->n_coord_rows = dyn->cfg.update_pocket_coords ? dm->N : dm->NL;
  return 0;
}

int dsb_dynamics_edges(dsb_dynamics* dyn, const float* xh_atoms, const float* xh_residues, const int64_t* mask_atoms,
                       const int64_t* mask_residues, int64_t n_atoms, int64_t n_residues, int64_t n_graphs,
                       int64_t edge_capacity, int32_t* rows, int32_t* cols, int32_t* n_edges, void* workspace,
                       size_t workspace_bytes, void* stream) {
  Dims dm; Workspace ws;
  if (int e = setup(dyn, n_atoms, n_residues, n_graphs, edge_capacity, workspace, workspace_bytes, &dm, &ws)) return e;
  cudaStream_t s = (cudaStream_t)stream;
  if (dm.N == 0) { DSB_CUDA_OK(cudaMemsetAsync(n_edges, 0, sizeof(int32_t), s)); return 0; }
  if (int e = launch_plan(dyn, dm, ws, mask_atoms, mask_residues, s)) return e;
  if (int e = launch_prep(dyn, dm, ws, xh_atoms, xh_residues, nullptr, 0, mask_atoms, mask_residues, true, s)) return e;
  ws.erow = rows; ws.ecol = cols;
  if (int e = launch_edges(dyn, dm, ws, nullptr, s)) return e;
  DSB_CUDA_OK(cudaMemcpyAsync(n_edges, ws.row_ptr + dm.N, sizeof(int32_t), cudaMemcpyDeviceToDevice, s));
  return 0;
}

int dsb_dynamics_forward(dsb_dynamics* dyn, const float* xh_atoms, const float* xh_residues, const float* t,
                         int64_t t_numel, const int64_t* mask_atoms, const int64_t* mask_residues, int64_t n_atoms,
                         int64_t n_residues, int64_t n_graphs, int64_t edge_capacity, float* out_atoms,
                         float* out_residues, void* workspace, size_t workspace_bytes, int32_t* status, void* stream) {
  Dims dm; Workspace ws;
  if (int e = setup(dyn, n_atoms, n_residues, n_graphs, edge_capacity, workspace, workspace_bytes, &dm, &ws)) return e;
  const dsb_config& c = dyn->cfg;
  if (c.condition_time && !(t_numel == 1 || t_numel == n_graphs)) {
    set_error("t must have 1 or n_graphs=%lld elements, got %lld", (long long)n_graphs, (long long)t_numel);
    return DSB_ERR_INVALID_ARGUMENT;
  }
  if (!status || (!out_atoms && n_atoms) || (!out_residues && n_residues)) { set_error("null output/status"); return DSB_ERR_INVALID_ARGUMENT; }
  cudaStream_t s = (cudaStream_t)stream;
  int launches = 0, memsets = 0;
  dyn->last_launches = 0; dyn->last_memsets = 0;
  if (dm.N == 0) return 0;
  const int H = c.hidden_nf;
  const int nm = c.reflection_equivariant ? 1 : 2;
  const size_t hbytes = sizeof(float) * (size_t)dm.N * H;

  // optional per-class timing with CUDA events on the launch stream (never during stream capture)
  bool prof = dyn->prof_enabled != 0;
  if (prof) {
    cudaStreamCaptureStatus cs = cudaStreamCaptureStatusNone;
    cudaStreamIsCapturing(s, &cs);
    if (cs != cudaStreamCaptureStatusNone) prof = false;
  }
  if (prof && dyn->prof_n > 0) {        // drain the previous forward's intervals into the accumulators
    for (int i = 0; i < dyn->prof_n; ++i) {
      float ms = 0.f;
      if (cudaEventSynchronize(dyn->prof_ev[2 * i + 1]) == cudaSuccess &&
          cudaEventElapsedTime(&ms, dyn->prof_ev[2 * i], dyn->prof_ev[2 * i + 1]) == cudaSuccess) {
        dyn->prof_ms[dyn->prof_cls[i]] += ms; dyn->prof_cnt[dyn->prof_cls[i]] += 1;
      }
    }
  }
  if (prof) dyn->prof_n = 0;
  int cur_cls = -1;
  auto mark = [&](int cls) {            // closes the open interval and opens one of class `cls` (-1: just close)
    if (!prof) return;
    if (cur_cls >= 0) { cudaEventRecord(dyn->prof_ev[2 * dyn->prof_n + 1], s); dyn->prof_cls[dyn->prof_n] = cur_cls; dyn->prof_n++; }
    cur_cls = -1;
    if (cls >= 0 && dyn->prof_n < kMaxProfEvents) { cudaEventRecord(dyn->prof_ev[2 * dyn->prof_n], s); cur_cls = cls; }
  };
#define DSB_TRY(expr) do { if (int e_ = (expr)) return e_; } while (0)
  const int mm = (tc_width_supported(H) && !c.sin_embedding) ? dyn->math_mode : 0;      // sin_embedding: fp32 FFMA kernels only
  const bool f16 = (mm & 8) != 0;
  auto gemm = [&](const GemmArgs& ga, const TcImage& img) -> int {
    return ((mm & 1) && img.t_hi) ? launch_tc_node_gemm(dyn, ga, img, f16, status, s) : launch_node_gemm(ga, s);
  };

  mark(KC_SETUP);
  DSB_TRY(launch_plan(dyn, dm, ws, mask_atoms, mask_residues, s)); launches += 1;
  DSB_TRY(launch_prep(dyn, dm, ws, xh_atoms, xh_residues, t, t_numel, mask_atoms, mask_residues, false, s)); launches += 1;
  DSB_TRY(launch_edges(dyn, dm, ws, status, s)); launches += 3;
  const float4* xcur = ws.xbuf[0];
  if (nm == 2) { mark(KC_COORD_FINISH); DSB_TRY(launch_coord_finish(dyn, dm, ws, xcur, nullptr, false, s)); launches += 1; }

  // the aggregates are zeroed once here; afterwards each consumer re-arms them (node GEMM g3 zeroes agg, coord_finish zeroes xagg)
  mark(KC_MEMSET);
  DSB_CUDA_OK(cudaMemsetAsync(ws.agg, 0, hbytes, s));
  DSB_CUDA_OK(cudaMemsetAsync(ws.xagg, 0, sizeof(float4) * (size_t)dm.N, s));
  memsets += 2;
  // P buffer columns: [0, nq) = coordinate first layer of the current block (receiver block | sender block),
  // [nq, nq + 2H) = edge first layer (receiver | sender) of the GCL that runs next.
  const int nq = nm * 2 * H, ldP = nq + 2 * H, nrecv = nm * H;
  const PView pv_gcl = {ws.P + nq, ldP}, pv_coord = {ws.P, ldP};
  const bool conditional = dm.n_coord_rows < dm.N;
  for (int l = 0; l < c.n_layers; ++l) {
    bool fused_block = false;
    for (int sub = 0; sub < c.inv_sublayers; ++sub) {
      const GclW& G = dyn->w.gcl[l][sub];
      if (!(sub == 0 && l > 0)) {      // otherwise produced by the previous block's merged GEMM
        mark(KC_NODE_GEMM);
        GemmArgs g1 = {ws.h, H, H, nullptr, 0, 0, 1.f, G.W1ab, 2 * H, G.b1ab, nullptr, 0, ws.P + nq, ldP, dm.N, 2 * H, 0, nullptr, 0, 0, 0};
        DSB_TRY(gemm(g1, G.iW1ab));
        launches += 1;
      }
      mark(KC_EDGE_GCL);
      DSB_TRY((mm & 2) ? launch_tc_edge_gcl(dyn, dm, ws, G, xcur, pv_gcl, f16, status, s) : launch_edge_gcl(dyn, dm, ws, G, xcur, pv_gcl, s));
      // node_model: h + W4 SiLU(W3 [h | agg/norm] + b3) + b4   (egnn_new.py:48-58)
      mark(KC_NODE_GEMM);
      const EquivW& Qb = dyn->w.eq[l];
      if ((mm & 1) && sub == c.inv_sublayers - 1 && tc_node_block_available(H, f16)) {
        // node_model and the merged first-layer GEMM of this block in one CTA-pair kernel (h converted to operand format once)
        DSB_TRY(launch_tc_node_block(dyn, dm, ws, G, Qb, ws.P, ldP, conditional ? dm.n_coord_rows : 0, conditional ? nrecv : 0, s));
        launches += 2;      // GCL edge kernel + block kernel
        fused_block = true;
      } else if (mm & 1) {
        DSB_TRY(launch_tc_node_mlp(dyn, dm, ws, G, f16, status, s));        // both layers in one kernel, hidden stays on chip
        launches += 2;
      } else {
        GemmArgs g2 = {ws.h, H, H, ws.agg, H, H, c.normalization_factor, G.W3, H, G.b3, nullptr, 0, ws.hT, H, dm.N, H, 1, nullptr, 0, 0, 0,
                       c.aggregation_mean ? ws.deg : nullptr};
        DSB_TRY(launch_node_gemm(g2, s));
        GemmArgs g3 = {ws.hT, H, H, nullptr, 0, 0, 1.f, G.W4, H, G.b4, ws.h, H, ws.h, H, dm.N, H, 0, ws.agg, H, 0, 0};
        DSB_TRY(launch_node_gemm(g3, s));
        launches += 3;
      }
    }
    // one GEMM for everything that consumes the updated h: this block's coord/cross first layers and the next block's
    // edge first layer.  In conditional mode the receiver-side coord columns are needed for ligand rows only.
    const EquivW& Q = dyn->w.eq[l];
    mark(KC_NODE_GEMM);
    if (!fused_block) {
    GemmArgs g4 = {ws.h, H, H, nullptr, 0, 0, 1.f, Q.W1, Q.nq + Q.np, Q.b1, nullptr, 0, ws.P, ldP, dm.N, Q.nq + Q.np, 0, nullptr, 0,
                   conditional ? dm.n_coord_rows : 0, conditional ? nrecv : 0};
    DSB_TRY(gemm(g4, Q.iW1));
    }
    mark(KC_EDGE_COORD);
    DSB_TRY((mm & 4) ? launch_tc_edge_coord(dyn, dm, ws, Q, xcur, pv_coord, f16, status, s) : launch_edge_coord(dyn, dm, ws, Q, xcur, pv_coord, s));
    float4* xnext = ws.xbuf[1 + (l & 1)];
    mark(KC_COORD_FINISH);
    DSB_TRY(launch_coord_finish(dyn, dm, ws, xcur, xnext, true, s));
    xcur = xnext;
    launches += fused_block ? 2 : 3;      // (merged GEMM,) coordinate edge kernel, finish
  }
  mark(KC_POST);
  DSB_TRY(launch_post(dyn, dm, ws, xcur, out_atoms, out_residues, status, s));
  mark(-1);
#undef DSB_TRY
  launches += 1 + (c.update_pocket_coords ? 1 : 0);
  dyn->last_launches = launches;
  dyn->last_memsets = memsets;
  return 0;
}

int dsb_set_programmatic_launch(int enable) {
  const int old = dsb::g_pdl;
  if (enable >= 0) dsb::g_pdl = enable != 0;
  return old;
}

int dsb_set_kernel_variants(int variants) {
  const int old = dsb::g_kernel_variants;
  if (variants >= 0) dsb::g_kernel_variants = variants & 3;
  return old;
}

int dsb_dynamics_set_math_mode(dsb_dynamics* dyn, int mode) {
  if (!dyn) { set_error("null handle"); return DSB_ERR_INVALID_ARGUMENT; }
  if (mode < 0 || mode > 15) { set_error("math mode must be a bitmask in [0,15]"); return DSB_ERR_INVALID_ARGUMENT; }
  if (mode != 0 && dyn->cfg.sin_embedding) { set_error("sin_embedding is built in the fp32 FFMA kernels only (math mode 0)"); return DSB_ERR_UNSUPPORTED_CONFIG; }
  if (mode != 0 && !tc_width_supported(dyn->cfg.hidden_nf)) { set_error("the tcgen05 kernels are built for hidden_nf 128, 192 and 256 only"); return DSB_ERR_UNSUPPORTED_CONFIG; }
  dyn->math_mode = mode;
  return 0;
}

int dsb_dynamics_set_profiling(dsb_dynamics* dyn, int enabled) {
  if (!dyn) { set_error("null handle"); return DSB_ERR_INVALID_ARGUMENT; }
  if (enabled && !dyn->prof_ev) {
    dyn->prof_ev = new cudaEvent_t[2 * kMaxProfEvents];
    for (int i = 0; i < 2 * kMaxProfEvents; ++i) DSB_CUDA_OK(cudaEventCreate(&dyn->prof_ev[i]));
  }
  dyn->prof_enabled = enabled ? 1 : 0;
  dyn->prof_n = 0;
  return 0;
}

int dsb_dynamics_collect_profile(dsb_dynamics* dyn, double* ms_by_class, int64_t* count_by_class, int reset) {
  if (!dyn || !ms_by_class || !count_by_class) { set_error("null argument"); return DSB_ERR_INVALID_ARGUMENT; }
  for (int i = 0; i < dyn->prof_n; ++i) {
    DSB_CUDA_OK(cudaEventSynchronize(dyn->prof_ev[2 * i + 1]));
    float ms = 0.f;
    DSB_CUDA_OK(cudaEventElapsedTime(&ms, dyn->prof_ev[2 * i], dyn->prof_ev[2 * i + 1]));
    dyn->prof_ms[dyn->prof_cls[i]] += ms;
    dyn->prof_cnt[dyn->prof_cls[i]] += 1;
  }
  dyn->prof_n = 0;
  for (int k = 0; k < KC_COUNT; ++k) { ms_by_class[k] = dyn->prof_ms[k]; count_by_class[k] = dyn->prof_cnt[k]; }
  if (reset) for (int k = 0; k < KC_COUNT; ++k) { dyn->prof_ms[k] = 0; dyn->prof_cnt[k] = 0; }
  return 0;
}

int dsb_dynamics_last_launch_count(const dsb_dynamics* dyn) { return dyn ? dyn->last_launches : 0; }

int dsb_ddpm_ligand_update(const float* z_lig, const float* eps_hat, const float* noise, const float* coef,
                           const int64_t* mask_atoms, const int64_t* mask_residues, const float* xh_pocket,
                           int64_t n_atoms, int64_t n_residues, int64_t n_graphs, int32_t atom_nf, int32_t residue_nf,
                           float* z_out, float* xh_pocket_out, void* stream) {
  if (n_graphs <= 0) return 0;
  if (!z_lig || !eps_hat || !noise || !coef || !mask_atoms || !mask_residues || !xh_pocket || !z_out || !xh_pocket_out) {
    set_error("null pointer"); return DSB_ERR_INVALID_ARGUMENT;
  }
  ddpm_update_kernel<<<(unsigned)n_graphs, 128, 0, (cudaStream_t)stream>>>(z_lig, eps_hat, noise, coef, mask_atoms, mask_residues,
                                                                          xh_pocket, (int)n_atoms, (int)n_residues, atom_nf,
                                                                          residue_nf, z_out, xh_pocket_out);
  DSB_CUDA_OK(cudaGetLastError());
  return 0;
}

int dsb_ddpm_inpaint_update(float* z_lig, float* xh_pocket, const float* xh_known, const float* com_pocket0,
                            const float* lig_fixed, const float* noise_known, const float* noise_renoise, const float* coef,
                            const int64_t* mask_atoms, const int64_t* mask_residues, int64_t n_atoms, int64_t n_residues,
                            int64_t n_graphs, int32_t atom_nf, int32_t residue_nf, void* stream) {
  if (n_graphs <= 0) return 0;
  if (!z_lig || !xh_pocket || !xh_known || !com_pocket0 || !lig_fixed || !noise_known || !coef || !mask_atoms || !mask_residues) {
    set_error("null pointer"); return DSB_ERR_INVALID_ARGUMENT;
  }
  ddpm_inpaint_kernel<<<(unsigned)n_graphs, 128, 0, (cudaStream_t)stream>>>(z_lig, xh_pocket, xh_known, com_pocket0, lig_fixed,
                                                                           noise_known, noise_renoise, coef, mask_atoms,
                                                                           mask_residues, (int)n_atoms, (int)n_residues, atom_nf,
                                                                           residue_nf);
  DSB_CUDA_OK(cudaGetLastError());
  return 0;
}

int dsb_ddpm_joint_update(float* z_lig, float* z_pocket, const float* eps_lig, const float* eps_pocket, const float* noise_x,
                          const float* noise_h_lig, const float* noise_h_pocket, const float* coef, const int64_t* mask_atoms,
                          const int64_t* mask_residues, int64_t n_atoms, int64_t n_residues, int64_t n_graphs, int32_t atom_nf,
                          int32_t residue_nf, void* stream) {
  if (n_graphs <= 0) return 0;
  if (!z_lig || !z_pocket || !eps_lig || !eps_pocket || !noise_x || !noise_h_lig || !noise_h_pocket || !coef || !mask_atoms || !mask_residues) {
    set_error("null pointer"); return DSB_ERR_INVALID_ARGUMENT;
  }
  ddpm_joint_update_kernel<<<(unsigned)n_graphs, 128, 0, (cudaStream_t)stream>>>(z_lig, z_pocket, eps_lig, eps_pocket, noise_x, noise_h_lig,
                                                                                noise_h_pocket, coef, mask_atoms, mask_residues,
                                                                                (int)n_atoms, (int)n_residues, atom_nf, residue_nf);
  DSB_CUDA_OK(cudaGetLastError());
  return 0;
}

int dsb_ddpm_joint_inpaint_update(float* z_lig, float* z_pocket, const float* xh0_lig, const float* xh0_pocket,
                                  const float* lig_fixed, const float* pocket_fixed, const float* noise_x, const float* noise_h_lig,
                                  const float* noise_h_pocket, const float* renoise_x, const float* renoise_h_lig,
                                  const float* renoise_h_pocket, const float* coef, const int64_t* mask_atoms,
                                  const int64_t* mask_residues, int64_t n_atoms, int64_t n_residues, int64_t n_graphs,
                                  int32_t atom_nf, int32_t residue_nf, void* stream) {
  if (n_graphs <= 0) return 0;
  if (!z_lig || !z_pocket || !xh0_lig || !xh0_pocket || !lig_fixed || !pocket_fixed || !noise_x || !noise_h_lig || !noise_h_pocket ||
      !coef || !mask_atoms || !mask_residues || (renoise_x && (!renoise_h_lig || !renoise_h_pocket))) {
    set_error("null pointer"); return DSB_ERR_INVALID_ARGUMENT;
  }
  ddpm_joint_inpaint_kernel<<<(unsigned)n_graphs, 128, 0, (cudaStream_t)stream>>>(
      z_lig, z_pocket, xh0_lig, xh0_pocket, lig_fixed, pocket_fixed, noise_x, noise_h_lig, noise_h_pocket, renoise_x, renoise_h_lig,
      renoise_h_pocket, coef, mask_atoms, mask_residues, (int)n_atoms, (int)n_residues, atom_nf, residue_nf);
  DSB_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // extern "C"
