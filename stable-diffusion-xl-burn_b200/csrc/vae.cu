// Latent decoder / encoder front end of libsdxl_b200.so (C ABI: sdxl_vae_*). See engine_core.h for the shared machinery.
#include "engine_core.h"

// ================================================================================================
// Latent decoder (SURVEY.md §8(f) rank 1): LatentDecoder::{decode_latent, latent_to_image}
//   Autoencoder::decode_latent      src/model/autoencoder/mod.rs:66-69
//   Decoder::forward                src/model/autoencoder/mod.rs:202-216
//   Mid / ResnetBlock / ConvSelfAttentionBlock / DecoderBlock
//                                   src/model/autoencoder/mod.rs:436-452, 507-524, 548-586, 298-324
//   LatentDecoder                   src/model/stablediffusion/mod.rs:199-237, 263-266
// Same machinery as the UNet: weights re-laid-out once on the device, a flat launch plan replayed as a CUDA graph.
// All convolutions and the attention contractions run on the tcgen05 implicit-GEMM kernel with f16 operands and f32
// accumulation; the residual stream, GroupNorm statistics, the score matrix and the softmax are f32 (the reference
// runs this module in f32 end to end; tests/test_vae_gpu.py states the resulting tolerance).
// The attention block is single-head with d = C (512): scores are materialised (f32 [T,T] per image, 1.07 GB at
// 1024^2), soft-maxed by rows into f16 probabilities and multiplied with V by a second GEMM.
// ================================================================================================
struct VRes {
  Norm n1, n2;
  Conv c1, c2;  // c2 carries the fused nin_shortcut 1x1 segment when Cin != Cout
  int Cin = 0, Cout = 0;
  bool has_skip = false;
};
struct VBlock {
  VRes r[3];
  bool up = false;
  Conv upc;
  int Cout = 0;
};
struct sdxl_vae {
  sdxl_ctx* ctx = nullptr;
  sdxl_vae_cfg cfg{};
  Arena warena;
  float* pq_w = nullptr;   // [Cl, Cl] f32
  float* pq_b = nullptr;
  float* cin_w = nullptr;  // [C0][3][3][Cl] f32
  float* cin_b = nullptr;
  int C0 = 0;
  VRes mid1, mid2;
  Norm attn_norm;
  Lin aq, ak, av, aproj;
  std::vector<VBlock> blocks;
  Norm norm_out;
  Conv conv_out;  // O padded to 4
  // encoder half (optional)
  bool has_enc = false;
  float* ecin_w = nullptr;  // [EC0][3][3][3] f32
  float* ecin_b = nullptr;
  int EC0 = 0;
  struct EBlock { VRes r[2]; bool down = false; Conv downc; int Cout = 0; };
  std::vector<EBlock> eblocks;
  VRes emid1, emid2;
  Norm eattn_norm;
  Lin eq, ek, ev, eproj;
  Norm enorm_out;
  Conv econv_out;           // Cm -> enc_z_channels
  float* qc_w = nullptr;    // quant_conv [Cz][Cz] f32
  float* qc_b = nullptr;
  std::unique_ptr<Plan> enc_plan;
  float* enc_z = nullptr;        // [B, hw, Cz] f32 NHWC (conv_out output)
  float* enc_lat = nullptr;      // [B, Cl, hw] f32 NCHW staging
  uint8_t* enc_u8 = nullptr;     // [B, HW, 3] staging for host u8 input
  std::unique_ptr<Plan> plan;
  float* img_nhwc = nullptr;     // [B, 64hw, 4] f32 (decoder output, first 3 channels valid)
  float* out_f32 = nullptr;      // [B, 3, 8h, 8w] staging for host reads
  uint8_t* out_u8 = nullptr;     // [B, 8h, 8w, 3]
};

static Lin lin_from_conv1x1(const Conv& cv) {
  Lin L;
  L.w = cv.w; L.b = cv.b; L.K = cv.I; L.Kpad = cv.Ipad; L.N = cv.O;
  return L;
}
static VRes load_vres(Loader& L, const std::string& path, int Cin, int Cout) {
  VRes r;
  r.Cin = Cin; r.Cout = Cout; r.has_skip = (Cin != Cout);
  r.n1 = L.norm(path + "/norm1", Cin);
  r.c1 = L.conv(path + "/conv1", Cin, Cout, 3);
  r.n2 = L.norm(path + "/norm2", Cout);
  if (r.has_skip) r.c2 = L.conv(path + "/conv2", Cout, Cout, 3, path + "/nin_shortcut", Cin);
  else r.c2 = L.conv(path + "/conv2", Cout, Cout, 3);
  return r;
}
static int build_vae(sdxl_vae* v, const PackView& pv, Arena& A) {
  sdxl_ctx* c = v->ctx;
  const sdxl_vae_cfg& g = v->cfg;
  Loader L{nullptr, c, &pv, &A, c->stream};
  const int Cl = g.latent_channels;
  v->blocks.clear();
  v->C0 = g.block_in[0];
  // post_quant_conv: OIHW [Cl,Cl,1,1] f16 -> f32 [Cl][Cl]
  {
    const PackEntry* e = L.need("post_quant_conv/weight", 4);
    if (!e) return L.err;
    if ((int)e->shape[0] != Cl || (int)e->shape[1] != Cl || e->shape[2] != 1 || e->shape[3] != 1) return fail(c, 4301, "post_quant_conv/weight bad shape");
    v->pq_w = A.get<float>((size_t)Cl * Cl);
    if (!v->pq_w) return fail(c, 4005, "weight arena exhausted");
    if (!A.measure) { int r = cast_f16_to_f32_launch(c->stream, L.ptr(e), (size_t)Cl * Cl, v->pq_w); if (r) return fail(c, r, "post_quant cast failed"); }
    v->pq_b = L.vec_f32("post_quant_conv/bias", Cl);
    if (L.err) return L.err;
  }
  // decoder/conv_in: OIHW f16 -> [O][kh][kw][I] f32 (CUDA-core kernel, exact f32 like the reference)
  {
    const PackEntry* e = L.need("decoder/conv_in/weight", 4);
    if (!e) return L.err;
    if ((int)e->shape[0] != v->C0 || (int)e->shape[1] != Cl || e->shape[2] != 3 || e->shape[3] != 3) return fail(c, 4302, "decoder/conv_in/weight bad shape");
    const size_t n = (size_t)v->C0 * 9 * Cl;
    __half* tmp = A.get<__half>(n);
    v->cin_w = A.get<float>(n);
    if (!tmp || !v->cin_w) return fail(c, 4005, "weight arena exhausted");
    if (!A.measure) {
      int r = repack_conv_launch(c->stream, L.ptr(e), v->C0, Cl, 3, 3, tmp, 9 * Cl, 0, Cl);
      if (!r) r = cast_f16_to_f32_launch(c->stream, tmp, n, v->cin_w);
      if (r) return fail(c, r, "decoder conv_in repack failed");
    }
    v->cin_b = L.vec_f32("decoder/conv_in/bias", v->C0);
    if (L.err) return L.err;
  }
  const int Cm = v->C0;
  v->mid1 = load_vres(L, "decoder/mid/block_1", Cm, Cm);
  v->attn_norm = L.norm("decoder/mid/attn/norm", Cm);
  v->aq = lin_from_conv1x1(L.conv("decoder/mid/attn/q", Cm, Cm, 1));
  v->ak = lin_from_conv1x1(L.conv("decoder/mid/attn/k", Cm, Cm, 1));
  v->av = lin_from_conv1x1(L.conv("decoder/mid/attn/v", Cm, Cm, 1));
  v->aproj = lin_from_conv1x1(L.conv("decoder/mid/attn/proj_out", Cm, Cm, 1));
  v->mid2 = load_vres(L, "decoder/mid/block_2", Cm, Cm);
  if (L.err) return L.err;
  for (int i = 0; i < g.n_blocks && !L.err; ++i) {
    VBlock b;
    const std::string bp = "decoder/blocks/" + std::to_string(i);
    const int ci = g.block_in[i], co = g.block_out[i];
    b.Cout = co;
    b.r[0] = load_vres(L, bp + "/res1", ci, co);
    b.r[1] = load_vres(L, bp + "/res2", co, co);
    b.r[2] = load_vres(L, bp + "/res3", co, co);
    b.up = (i != g.n_blocks - 1);
    if (b.up) b.upc = L.upconv(bp + "/upsampler", co, co);
    v->blocks.push_back(b);
  }
  if (L.err) return L.err;
  const int Cf = g.block_out[g.n_blocks - 1];
  v->norm_out = L.norm("decoder/norm_out", Cf);
  v->conv_out = L.conv("decoder/conv_out", Cf, 3, 3, "", 0, 4);
  if (L.err) return L.err;
  // ---- encoder half (autoencoder/load.rs:82-116)
  v->has_enc = g.n_enc_blocks > 0;
  v->eblocks.clear();
  if (v->has_enc) {
    v->EC0 = g.enc_in[0];
    const PackEntry* e = L.need("encoder/conv_in/weight", 4);
    if (!e) return L.err;
    if ((int)e->shape[0] != v->EC0 || e->shape[1] != 3 || e->shape[2] != 3 || e->shape[3] != 3) return fail(c, 4320, "encoder/conv_in/weight bad shape");
    const size_t n = (size_t)v->EC0 * 27;
    __half* tmp = A.get<__half>(n);
    v->ecin_w = A.get<float>(n);
    if (!tmp || !v->ecin_w) return fail(c, 4005, "weight arena exhausted");
    if (!A.measure) {
      int r = repack_conv_launch(c->stream, L.ptr(e), v->EC0, 3, 3, 3, tmp, 27, 0, 3);
      if (!r) r = cast_f16_to_f32_launch(c->stream, tmp, n, v->ecin_w);
      if (r) return fail(c, r, "encoder conv_in repack failed");
    }
    v->ecin_b = L.vec_f32("encoder/conv_in/bias", v->EC0);
    for (int i = 0; i < g.n_enc_blocks && !L.err; ++i) {
      sdxl_vae::EBlock b;
      const std::string bp = "encoder/blocks/" + std::to_string(i);
      const int ci = g.enc_in[i], co = g.enc_out[i];
      b.Cout = co;
      b.r[0] = load_vres(L, bp + "/res1", ci, co);
      b.r[1] = load_vres(L, bp + "/res2", co, co);
      b.down = (i != g.n_enc_blocks - 1);
      if (b.down) b.downc = L.conv(bp + "/downsampler/conv", co, co, 3);
      v->eblocks.push_back(b);
    }
    if (L.err) return L.err;
    const int Ce = g.enc_out[g.n_enc_blocks - 1], Cz = g.enc_z_channels;
    v->emid1 = load_vres(L, "encoder/mid/block_1", Ce, Ce);
    v->eattn_norm = L.norm("encoder/mid/attn/norm", Ce);
    v->eq = lin_from_conv1x1(L.conv("encoder/mid/attn/q", Ce, Ce, 1));
    v->ek = lin_from_conv1x1(L.conv("encoder/mid/attn/k", Ce, Ce, 1));
    v->ev = lin_from_conv1x1(L.conv("encoder/mid/attn/v", Ce, Ce, 1));
    v->eproj = lin_from_conv1x1(L.conv("encoder/mid/attn/proj_out", Ce, Ce, 1));
    v->emid2 = load_vres(L, "encoder/mid/block_2", Ce, Ce);
    v->enorm_out = L.norm("encoder/norm_out", Ce);
    v->econv_out = L.conv("encoder/conv_out", Ce, Cz, 3);
    if (L.err) return L.err;
    const PackEntry* q = L.need("quant_conv/weight", 4);
    if (!q) return L.err;
    if ((int)q->shape[0] != Cz || (int)q->shape[1] != Cz || q->shape[2] != 1 || q->shape[3] != 1) return fail(c, 4321, "quant_conv/weight bad shape");
    v->qc_w = A.get<float>((size_t)Cz * Cz);
    if (!v->qc_w) return fail(c, 4005, "weight arena exhausted");
    if (!A.measure) { int r = cast_f16_to_f32_launch(c->stream, L.ptr(q), (size_t)Cz * Cz, v->qc_w); if (r) return fail(c, r, "quant_conv cast failed"); }
    v->qc_b = L.vec_f32("quant_conv/bias", Cz);
  }
  return L.err;
}

extern "C" void sdxl_vae_destroy(sdxl_vae* v) {
  if (!v) return;
  cudaStreamSynchronize(v->ctx->stream);
  v->plan.reset();
  v->enc_plan.reset();
  v->warena.release();
  delete v;
}

extern "C" int sdxl_vae_load(sdxl_ctx* c, const sdxl_vae_cfg* cfg, const void* pack, size_t bytes, int pack_on_device,
                             sdxl_vae** out) {
  if (!c || !cfg || !pack || !out) return fail(c, -1, "sdxl_vae_load: null argument");
  *out = nullptr;
  if (cfg->n_blocks < 1 || cfg->n_blocks > SDXL_MAX_LEVELS) return fail(c, 4310, "bad n_blocks");
  if (cfg->latent_channels < 1 || cfg->latent_channels > 8) return fail(c, 4311, "latent_channels must be 1..8");
  if (cfg->n_group != 32) return fail(c, 4312, "n_group must be 32 (got %d)", cfg->n_group);
  if (!(cfg->scale_factor > 0)) return fail(c, 4313, "scale_factor must be positive");
  for (int i = 0; i < cfg->n_blocks; ++i) {
    if (cfg->block_in[i] % 64 || cfg->block_out[i] % 64) return fail(c, 4314, "decoder widths must be multiples of 64");
    if (i && cfg->block_in[i] != cfg->block_out[i - 1]) return fail(c, 4315, "block_in[%d] != block_out[%d]", i, i - 1);
  }
  if (cfg->n_enc_blocks < 0 || cfg->n_enc_blocks > SDXL_MAX_LEVELS) return fail(c, 4316, "bad n_enc_blocks");
  for (int i = 0; i < cfg->n_enc_blocks; ++i) {
    if (cfg->enc_in[i] % 64 || cfg->enc_out[i] % 64) return fail(c, 4317, "encoder widths must be multiples of 64");
    if (i && cfg->enc_in[i] != cfg->enc_out[i - 1]) return fail(c, 4318, "enc_in[%d] != enc_out[%d]", i, i - 1);
  }
  if (cfg->n_enc_blocks && (cfg->enc_z_channels < cfg->latent_channels || cfg->enc_z_channels > 16 || cfg->enc_z_channels % 4))
    return fail(c, 4319, "enc_z_channels must be a multiple of 4 in [latent_channels, 16]");
  CU(c, cudaSetDevice(c->device));
  std::unique_ptr<sdxl_vae> v(new sdxl_vae());
  v->ctx = c;
  v->cfg = *cfg;
  PackView pv;
  std::vector<uint8_t> table;
  int r = parse_pack(c, pack, bytes, pack_on_device, pv, table);
  if (r) return r;
  void* dev_pack = nullptr;
  if (pack_on_device) {
    pv.dev = (const uint8_t*)pack;
  } else {
    CU(c, cudaMalloc(&dev_pack, bytes));
    cudaError_t e = cudaMemcpyAsync(dev_pack, pack, bytes, cudaMemcpyHostToDevice, c->stream);
    if (e != cudaSuccess) { cudaFree(dev_pack); return fail(c, (int)e, "pack upload failed"); }
    pv.dev = (const uint8_t*)dev_pack;
  }
  Arena meas;
  meas.measure = true;
  r = build_vae(v.get(), pv, meas);
  if (!r && v->warena.init(meas.off + (1 << 20))) r = fail(c, 4203, "cannot allocate %zu bytes for weights", meas.off);
  if (!r) r = build_vae(v.get(), pv, v->warena);
  cudaError_t se = cudaStreamSynchronize(c->stream);
  if (dev_pack) cudaFree(dev_pack);
  if (!r && se != cudaSuccess) r = fail(c, (int)se, "weight re-layout failed: %s", cudaGetErrorString(se));
  if (r) { v->warena.release(); return r; }
  *out = v.release();
  return 0;
}

// Shared pieces of the encoder / decoder plans: ping-pong f32 stream buffers + scratch, ResnetBlock and the mid attention.
struct VaeStage {
  PlanBuilder& B;
  Plan* P;
  int Bn;
  int H = 0, W = 0;
  float* xb[2] = {nullptr, nullptr};
  int cur = 0;
  __half* s_gn1 = nullptr; __half* s_raw = nullptr; float* s_h = nullptr; __half* s_gn2 = nullptr;
  // attention scratch
  __half* q16 = nullptr; __half* k16 = nullptr; __half* v16 = nullptr; __half* vT = nullptr; __half* ao = nullptr;
  float* S = nullptr; __half* Pm = nullptr;

  void alloc(size_t max_x, size_t max_in, size_t max_out, int T, int Cm) {
    xb[0] = B.buf<float>(Bn * max_x);
    xb[1] = B.buf<float>(Bn * max_x);
    s_gn1 = B.buf<__half>(Bn * max_in);
    s_raw = B.buf<__half>(Bn * max_in);
    s_h = B.buf<float>(Bn * max_out);
    s_gn2 = B.buf<__half>(Bn * max_out);
    q16 = B.buf<__half>((size_t)Bn * T * Cm);
    k16 = B.buf<__half>((size_t)Bn * T * Cm);
    v16 = B.buf<__half>((size_t)Bn * T * Cm);
    vT = B.buf<__half>((size_t)T * Cm);
    ao = B.buf<__half>((size_t)Bn * T * Cm);
    S = B.buf<float>((size_t)T * T);
    Pm = B.buf<__half>((size_t)T * T);
  }
  float* x() const { return xb[cur]; }
  float* other() const { return xb[cur ^ 1]; }
  void flip() { cur ^= 1; }

  // ResnetBlock::forward (autoencoder/mod.rs:507-524)
  void vres(const VRes& r) {
    const int HW = H * W;
    B.gn(x(), r.Cin, nullptr, 0, HW, r.n1, 1, s_gn1, r.has_skip ? s_raw : nullptr);
    ActView a1{s_gn1, Bn, H, W, r.Cin};
    B.conv3(a1, nullptr, r.c1, s_h, r.c1.b, 0, nullptr);
    B.gn(s_h, r.Cout, nullptr, 0, HW, r.n2, 1, s_gn2, nullptr);
    ActView a2{s_gn2, Bn, H, W, r.Cout};
    if (r.has_skip) {
      ActView sk{s_raw, Bn, H, W, r.Cin};
      B.conv3(a2, &sk, r.c2, other(), r.c2.b, 0, nullptr);  // nin_shortcut(x) + h as one GEMM (autoencoder/mod.rs:519-523)
    } else {
      B.conv3(a2, nullptr, r.c2, other(), r.c2.b, 0, x());
    }
    flip();
  }
  // ConvSelfAttentionBlock::forward (autoencoder/mod.rs:548-586): single head, d = C, scores materialised per image
  void attn(const Norm& norm, const Lin& aq, const Lin& ak, const Lin& av, const Lin& aproj) {
    const int T = H * W, Cm = aq.K, M = Bn * T;
    B.gn(x(), Cm, nullptr, 0, T, norm, 0, s_gn1, nullptr);
    B.linear(s_gn1, M, aq, IGEMM_LINEAR, q16, 0, Cm, nullptr, 0);
    B.linear(s_gn1, M, ak, IGEMM_LINEAR, k16, 0, Cm, nullptr, 0);
    B.linear(s_gn1, M, av, IGEMM_LINEAR, v16, 0, Cm, nullptr, 0);
    for (int b = 0; b < Bn && !B.err; ++b) {
      const size_t o = (size_t)b * T * Cm;
      B.attn_single_head(q16 + o, k16 + o, v16 + o, T, Cm, S, Pm, vT, ao + o);
    }
    B.linear(ao, M, aproj, IGEMM_LINEAR, other(), 1, Cm, x(), Cm);  // x + proj_out(attn)
    flip();
  }
};

// Builds the op list of Decoder::forward at batch B, latent h x w.
static int build_vae_plan(sdxl_vae* v, Plan* P, Arena* A) {
  sdxl_ctx* c = v->ctx;
  const sdxl_vae_cfg& g = v->cfg;
  PlanBuilder B{c, P, A, P->Bf};
  P->ops.clear();
  P->flops = 0;
  const int Bn = P->Bf, Cl = g.latent_channels;
  VaeStage st{B, P, Bn};
  st.H = P->h; st.W = P->w;
  if ((st.H * st.W) % 64) return fail(c, 5101, "latent %dx%d: h*w must be a multiple of 64", st.H, st.W);

  // buffer maxima over the stages
  size_t max_x = (size_t)st.H * st.W * v->C0, max_in = max_x, max_out = max_x, max_up = 0;
  {
    int hh = st.H, ww = st.W;
    for (const VBlock& b : v->blocks) {
      for (int k = 0; k < 3; ++k) {
        max_in = std::max(max_in, (size_t)hh * ww * b.r[k].Cin);
        max_out = std::max(max_out, (size_t)hh * ww * b.r[k].Cout);
      }
      if (b.up) { max_up = std::max(max_up, (size_t)hh * ww * b.Cout); hh *= 2; ww *= 2; }
      max_x = std::max(max_x, (size_t)hh * ww * b.Cout);
    }
    max_in = std::max(max_in, max_x);  // norm_out operand
  }
  P->x_in = B.buf<float>((size_t)Bn * Cl * st.H * st.W);
  float* pq_out = B.buf<float>((size_t)Bn * Cl * st.H * st.W);
  B.gn_partial = B.buf<float>(gn_scratch_floats(Bn, 32));
  if (B.gn_partial && !A->measure && gn_scratch_init(c->stream, B.gn_partial, Bn, 32)) return fail(c, 5007, "GroupNorm scratch init failed");
  st.alloc(max_x, max_in, max_out, st.H * st.W, v->C0);
  __half* s_up = max_up ? B.buf<__half>(Bn * max_up) : nullptr;
  if (B.err) return B.err;

  // post_quant_conv(latent / scale_factor), conv_in
  {
    Op op{};
    op.kind = OP_PQ;
    op.pq = {P->x_in, Bn, Cl, st.H * st.W, v->pq_w, v->pq_b, (float)(1.0 / g.scale_factor), pq_out};
    P->ops.push_back(op);
    P->flops += 2.0 * Bn * st.H * st.W * (double)Cl * Cl;
  }
  {
    Op op{};
    op.kind = OP_CONV_IN;
    op.ci = {pq_out, Bn, Bn, Cl, st.H, st.W, v->cin_w, v->cin_b, v->C0, st.x()};
    P->ops.push_back(op);
    P->flops += 2.0 * Bn * st.H * st.W * 9.0 * Cl * v->C0;
  }
  // mid: ResnetBlock, ConvSelfAttentionBlock, ResnetBlock
  st.vres(v->mid1);
  st.attn(v->attn_norm, v->aq, v->ak, v->av, v->aproj);
  st.vres(v->mid2);
  // up blocks
  for (const VBlock& b : v->blocks) {
    if (B.err) break;
    for (int k = 0; k < 3; ++k) st.vres(b.r[k]);
    if (b.up) {
      // nearest-2x then 3x3 conv (autoencoder/mod.rs:311-319), as four 2x2 phase convolutions of the source image
      B.upconv(st.x(), Bn, st.H, st.W, b.upc, s_up, st.other());
      st.H *= 2; st.W *= 2;
      st.flip();
    }
  }
  if (B.err) return B.err;
  // head: GN -> SiLU -> conv 3x3 to RGB (autoencoder/mod.rs:213-214); N padded to 4
  const int Cf = g.block_out[g.n_blocks - 1];
  const int H = st.H, W = st.W;
  B.gn(st.x(), Cf, nullptr, 0, H * W, v->norm_out, 1, st.s_gn1, nullptr);
  v->img_nhwc = B.buf<float>((size_t)Bn * H * W * 4);
  {
    ActView a{st.s_gn1, Bn, H, W, Cf};
    std::vector<IgemmSeg> segs;
    for (int kh = 0; kh < 3; ++kh)
      for (int kw = 0; kw < 3; ++kw) segs.push_back({0, (int16_t)(kw - 1), (int16_t)(kh - 1), 0, v->conv_out.Ipad / 64});
    B.igemm(a, nullptr, segs, v->conv_out.w, 4, v->conv_out.Ktot, H, W, Bn, IGEMM_LINEAR, 0, v->img_nhwc, 1, 4, v->conv_out.b, 0,
            nullptr, 0);
    B.add_flops(2.0 * Bn * H * W * 9.0 * Cf * 3);
  }
  v->out_f32 = B.buf<float>((size_t)Bn * 3 * H * W);
  v->out_u8 = B.buf<uint8_t>((size_t)Bn * 3 * H * W);
  return B.err;
}

// Builds the op list of Encoder::forward (autoencoder/mod.rs:128-144) + quant_conv at batch B, image H x W.
static int build_vae_enc_plan(sdxl_vae* v, Plan* P, Arena* A) {
  sdxl_ctx* c = v->ctx;
  const sdxl_vae_cfg& g = v->cfg;
  PlanBuilder B{c, P, A, P->Bf};
  P->ops.clear();
  P->flops = 0;
  const int Bn = P->Bf, nb = g.n_enc_blocks;
  VaeStage st{B, P, Bn};
  st.H = P->h; st.W = P->w;
  const int down = 1 << (nb - 1);
  if (st.H % down || st.W % down) return fail(c, 5102, "image %dx%d not divisible by %d", st.H, st.W, down);
  const int hl = st.H / down, wl = st.W / down;
  if ((hl * wl) % 64) return fail(c, 5103, "image %dx%d: (H/%d)*(W/%d) must be a multiple of 64", st.H, st.W, down, down);
  size_t max_x = (size_t)st.H * st.W * v->EC0, max_in = 0, max_out = 0, max_ph = 0;
  {
    int hh = st.H, ww = st.W;
    for (const auto& b : v->eblocks) {
      for (int k = 0; k < 2; ++k) {
        max_in = std::max(max_in, (size_t)hh * ww * b.r[k].Cin);
        max_out = std::max(max_out, (size_t)hh * ww * b.r[k].Cout);
        max_x = std::max(max_x, (size_t)hh * ww * b.r[k].Cout);
      }
      if (b.down) { max_ph = std::max(max_ph, (size_t)hh * ww * b.Cout); hh /= 2; ww /= 2; }
    }
    max_in = std::max(max_in, max_x);
  }
  const int Ce = g.enc_out[nb - 1], Cz = g.enc_z_channels, Cl = g.latent_channels;
  P->x_in = B.buf<float>((size_t)Bn * 3 * st.H * st.W);
  v->enc_u8 = B.buf<uint8_t>((size_t)Bn * 3 * st.H * st.W);
  B.gn_partial = B.buf<float>(gn_scratch_floats(Bn, 32));
  if (B.gn_partial && !A->measure && gn_scratch_init(c->stream, B.gn_partial, Bn, 32)) return fail(c, 5007, "GroupNorm scratch init failed");
  st.alloc(max_x, max_in, max_out, hl * wl, Ce);
  __half* s_ph = max_ph ? B.buf<__half>(Bn * max_ph) : nullptr;
  v->enc_z = B.buf<float>((size_t)Bn * hl * wl * Cz);
  v->enc_lat = B.buf<float>((size_t)Bn * Cl * hl * wl);
  if (B.err) return B.err;
  {
    Op op{};
    op.kind = OP_CONV_IN;
    op.ci = {P->x_in, Bn, Bn, 3, st.H, st.W, v->ecin_w, v->ecin_b, v->EC0, st.x()};
    P->ops.push_back(op);
    P->flops += 2.0 * Bn * st.H * st.W * 27.0 * v->EC0;
  }
  for (const auto& b : v->eblocks) {
    if (B.err) break;
    st.vres(b.r[0]);
    st.vres(b.r[1]);
    if (b.down) {
      // PaddedConv2d(3x3, stride 2, padding (left 0, right 1, top 0, bottom 1)), autoencoder/mod.rs:326-407
      B.padded_conv_s2(st.x(), Bn, st.H, st.W, b.downc, s_ph, st.other());
      st.flip();
      st.H /= 2; st.W /= 2;
    }
  }
  if (B.err) return B.err;
  st.vres(v->emid1);
  st.attn(v->eattn_norm, v->eq, v->ek, v->ev, v->eproj);
  st.vres(v->emid2);
  B.gn(st.x(), Ce, nullptr, 0, st.H * st.W, v->enorm_out, 1, st.s_gn1, nullptr);
  {
    ActView a{st.s_gn1, Bn, st.H, st.W, Ce};
    B.conv3(a, nullptr, v->econv_out, v->enc_z, v->econv_out.b, 0, nullptr);
  }
  P->flops += 2.0 * Bn * st.H * st.W * (double)Cz * Cz;  // quant_conv (all Cz outputs in the reference)
  return B.err;
}

static int vae_encode_run(sdxl_vae* v, int Bn, int H, int W, const float* image, const uint8_t* rgb, int on_host, float* latent_out) {
  sdxl_ctx* c = v->ctx;
  if (!v->has_enc) return fail(c, 5104, "this sdxl_vae was loaded without the encoder half (n_enc_blocks = 0)");
  if (!latent_out || (!image && !rgb)) return fail(c, -1, "null argument");
  if (Bn < 1 || H < 1 || W < 1) return fail(c, 5100, "bad encode shape B=%d H=%d W=%d", Bn, H, W);
  CU(c, cudaSetDevice(c->device));
  if (!v->enc_plan || v->enc_plan->Bf != Bn || v->enc_plan->h != H || v->enc_plan->w != W) {
    CU(c, cudaStreamSynchronize(c->stream));
    v->enc_plan.reset(new Plan());
    Plan* P = v->enc_plan.get();
    P->Bf = Bn; P->Bx = Bn; P->h = H; P->w = W;
    Arena meas;
    meas.measure = true;
    int r = build_vae_enc_plan(v, P, &meas);
    if (!r && P->arena.init(meas.off + (1 << 20))) r = fail(c, 5011, "cannot allocate %zu bytes of workspace", meas.off);
    if (!r) r = build_vae_enc_plan(v, P, &P->arena);
    if (r) { v->enc_plan.reset(); return r; }
  }
  Plan* P = v->enc_plan.get();
  const size_t npix = (size_t)Bn * H * W;
  if (image) {
    CU(c, cudaMemcpyAsync(P->x_in, image, npix * 3 * sizeof(float), on_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, c->stream));
  } else {
    const uint8_t* src = rgb;
    if (on_host) {
      CU(c, cudaMemcpyAsync(v->enc_u8, rgb, npix * 3, cudaMemcpyHostToDevice, c->stream));
      src = v->enc_u8;
    }
    KL(c, image_from_u8_launch(c->stream, src, Bn, (long)H * W, P->x_in));
  }
  int r = run_plan_ops(c, P);
  if (r) return r;
  const int down = 1 << (v->cfg.n_enc_blocks - 1);
  const long hw = (long)(H / down) * (W / down);
  float* dst = on_host ? v->enc_lat : latent_out;
  KL(c, quant_out_launch(c->stream, v->enc_z, Bn, v->cfg.enc_z_channels, v->cfg.latent_channels, hw, v->qc_w, v->qc_b,
                         (float)v->cfg.scale_factor, dst));
  if (on_host) {
    CU(c, cudaMemcpyAsync(latent_out, dst, (size_t)Bn * v->cfg.latent_channels * hw * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
  }
  return 0;
}
extern "C" int sdxl_vae_encode_image(sdxl_vae* v, int Bn, int H, int W, const float* image, int on_host, float* latent_out) {
  if (!v || !image) return fail(v ? v->ctx : nullptr, -1, "sdxl_vae_encode_image: null argument");
  return vae_encode_run(v, Bn, H, W, image, nullptr, on_host, latent_out);
}
extern "C" int sdxl_vae_image_to_latent(sdxl_vae* v, int Bn, int H, int W, const uint8_t* rgb, int on_host, float* latent_out) {
  if (!v || !rgb) return fail(v ? v->ctx : nullptr, -1, "sdxl_vae_image_to_latent: null argument");
  return vae_encode_run(v, Bn, H, W, nullptr, rgb, on_host, latent_out);
}
extern "C" double sdxl_vae_encode_plan_flops(const sdxl_vae* v) { return (v && v->enc_plan) ? v->enc_plan->flops : 0.0; }

static int vae_ensure_plan(sdxl_vae* v, int Bn, int h, int w) {
  sdxl_ctx* c = v->ctx;
  if (Bn < 1 || h < 1 || w < 1) return fail(c, 5100, "bad decode shape B=%d h=%d w=%d", Bn, h, w);
  if (v->plan && v->plan->Bf == Bn && v->plan->h == h && v->plan->w == w) return 0;
  CU(c, cudaStreamSynchronize(c->stream));
  v->plan.reset(new Plan());
  Plan* P = v->plan.get();
  P->Bf = Bn; P->Bx = Bn; P->h = h; P->w = w;
  Arena meas;
  meas.measure = true;
  int r = build_vae_plan(v, P, &meas);
  if (r) { v->plan.reset(); return r; }
  if (P->arena.init(meas.off + (1 << 20))) { v->plan.reset(); return fail(c, 5011, "cannot allocate %zu bytes of workspace", meas.off); }
  r = build_vae_plan(v, P, &P->arena);
  if (r) { v->plan.reset(); return r; }
  return 0;
}

static int vae_run(sdxl_vae* v, int Bn, int h, int w, const float* latent, int on_host) {
  sdxl_ctx* c = v->ctx;
  if (!latent) return fail(c, -1, "null latent");
  CU(c, cudaSetDevice(c->device));
  int r = vae_ensure_plan(v, Bn, h, w);
  if (r) return r;
  Plan* P = v->plan.get();
  const size_t n = (size_t)Bn * v->cfg.latent_channels * h * w;
  CU(c, cudaMemcpyAsync(P->x_in, latent, n * sizeof(float), on_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, c->stream));
  return run_plan_ops(c, P);
}

extern "C" int sdxl_vae_decode_latent(sdxl_vae* v, int Bn, int h, int w, const float* latent, int on_host, float* image_out) {
  if (!v || !image_out) return fail(v ? v->ctx : nullptr, -1, "sdxl_vae_decode_latent: null argument");
  sdxl_ctx* c = v->ctx;
  int r = vae_run(v, Bn, h, w, latent, on_host);
  if (r) return r;
  const int up = 1 << (v->cfg.n_blocks - 1);
  const int HW = h * up * w * up;
  float* dst = on_host ? v->out_f32 : image_out;
  KL(c, nhwc_to_nchw_f32_launch(c->stream, v->img_nhwc, Bn, HW, 3, 4, dst));
  if (on_host) {
    CU(c, cudaMemcpyAsync(image_out, dst, (size_t)Bn * 3 * HW * sizeof(float), cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
  }
  return 0;
}
extern "C" int sdxl_vae_latent_to_image(sdxl_vae* v, int Bn, int h, int w, const float* latent, int on_host, uint8_t* rgb_out) {
  if (!v || !rgb_out) return fail(v ? v->ctx : nullptr, -1, "sdxl_vae_latent_to_image: null argument");
  sdxl_ctx* c = v->ctx;
  int r = vae_run(v, Bn, h, w, latent, on_host);
  if (r) return r;
  const int up = 1 << (v->cfg.n_blocks - 1);
  const long npix = (long)Bn * h * up * w * up;
  uint8_t* dst = on_host ? v->out_u8 : rgb_out;
  KL(c, image_u8_launch(c->stream, v->img_nhwc, npix, 4, dst));
  if (on_host) {
    CU(c, cudaMemcpyAsync(rgb_out, dst, (size_t)npix * 3, cudaMemcpyDeviceToHost, c->stream));
    CU(c, cudaStreamSynchronize(c->stream));
  }
  return 0;
}
extern "C" double sdxl_vae_plan_flops(const sdxl_vae* v) { return (v && v->plan) ? v->plan->flops : 0.0; }
extern "C" int sdxl_vae_profile_plan(sdxl_vae* v, double* ms_by_kind, double* flops_by_kind, int* launches_by_kind) {
  if (!v || !v->plan) return -1;
  return profile_plan_impl(v->ctx, v->plan.get(), ms_by_kind, flops_by_kind, launches_by_kind);
}
extern "C" int sdxl_vae_profile_dump(sdxl_vae* v, const char* path) {
  if (!v || !v->plan || !path) return -1;
  return profile_dump_impl(v->ctx, v->plan.get(), path);
}


