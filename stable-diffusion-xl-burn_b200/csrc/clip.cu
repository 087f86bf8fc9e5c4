// Text-encoder front end of libsdxl_b200.so (C ABI: sdxl_clip_*). See engine_core.h for the shared machinery.
#include "engine_core.h"

// ================================================================================================
// Text encoders of the Embedder (SURVEY.md §8(f) rank 2): CLIP::{forward_hidden, forward_hidden_pooled}
//   CLIP / ResidualDecoderAttentionBlock / MultiHeadSelfAttention / MLP / QuickGELU
//                                   src/model/clip/mod.rs:82-147, 176-182, 228-245, 289-305, 315-319
//   weight names                    src/model/clip/load.rs:15-115
// 77-token sequences: Linear layers on the tcgen05 GEMM (one M tile), causal attention / activation / embedding on
// small CUDA-core kernels (clip_kernels.cu). Residual stream f32, GEMM operands f16 (the reference runs f32).
// ================================================================================================
struct CBlock {
  Norm attn_ln, mlp_ln;
  Lin qkv, out, fc1, fc2;
};
struct sdxl_clip {
  sdxl_ctx* ctx = nullptr;
  sdxl_clip_cfg cfg{};
  Arena warena;
  __half* tok_emb = nullptr;
  __half* pos_emb = nullptr;
  std::vector<CBlock> blocks;
  Norm ln_final;
  Lin proj;
  bool has_proj = false;
  // plan (keyed by batch, number of blocks run, captured hidden index, pooled)
  std::unique_ptr<Plan> plan;
  int pB = 0, p_nrun = 0, p_hidden = -1, p_pooled = 0;
  int* tokens_dev = nullptr;
  int* eot_dev = nullptr;
  int* err_dev = nullptr;
  float* hidden = nullptr;   // [B*T, C] result of forward_hidden / h_out
  float* pooled = nullptr;   // [B, embed_dim]
};

static int build_clip(sdxl_clip* m, const PackView& pv, Arena& A) {
  sdxl_ctx* c = m->ctx;
  const sdxl_clip_cfg& g = m->cfg;
  Loader L{nullptr, c, &pv, &A, c->stream};
  const int C = g.n_state;
  m->blocks.clear();
  auto table = [&](const std::string& name, int rows, __half*& dst) {
    const PackEntry* e = L.need(name, 2);
    if (!e) return;
    if ((int)e->shape[0] != rows || (int)e->shape[1] != C) { L.err = fail(c, 4401, "weight pack: '%s' is [%llu,%llu], expected [%d,%d]", name.c_str(), (unsigned long long)e->shape[0], (unsigned long long)e->shape[1], rows, C); return; }
    dst = A.get<__half>((size_t)rows * C);
    if (!dst) { L.err = fail(c, 4005, "weight arena exhausted"); return; }
    if (!A.measure && cudaMemcpyAsync(dst, L.ptr(e), (size_t)rows * C * sizeof(__half), cudaMemcpyDeviceToDevice, c->stream) != cudaSuccess)
      L.err = fail(c, 4402, "embedding copy failed");
  };
  table("token_embedding/weight", g.n_vocab, m->tok_emb);
  table("position_embedding/weight", g.n_ctx, m->pos_emb);
  if (L.err) return L.err;
  const int Cpad = Loader::pad64(C);
  for (int i = 0; i < g.n_layer && !L.err; ++i) {
    const std::string bp = "blocks/" + std::to_string(i);
    CBlock b;
    b.attn_ln = L.norm(bp + "/attn_ln", C);
    b.mlp_ln = L.norm(bp + "/mlp_ln", C);
    // fused q/k/v projection (clip/mod.rs:229-231: three Linears with bias on the same input)
    b.qkv.K = C; b.qkv.Kpad = Cpad; b.qkv.N = 3 * C;
    b.qkv.w = A.get<__half>((size_t)3 * C * Cpad);
    b.qkv.b = A.get<float>((size_t)3 * C);
    if (!b.qkv.w || !b.qkv.b) { L.err = fail(c, 4005, "weight arena exhausted"); break; }
    const char* names[3] = {"query", "key", "value"};
    for (int j = 0; j < 3 && !L.err; ++j) {
      const std::string lp = bp + "/attn/" + names[j];
      L.lin_into(lp, b.qkv.w, Cpad, j * C, C, C, 0);
      const PackEntry* be = L.need(lp + "/bias", 1);
      if (!be) break;
      if ((int)be->shape[0] != C) { L.err = fail(c, 4403, "weight pack: '%s/bias' mis-sized", lp.c_str()); break; }
      if (!A.measure) { int r = bias_to_f32_launch(c->stream, L.ptr(be), C, b.qkv.b + j * C, 0, 0); if (r) L.err = fail(c, r, "bias_to_f32 failed"); }
    }
    b.out = L.linear(bp + "/attn/out", C, C, true);
    b.fc1 = L.linear(bp + "/mlp/fc1", C, 4 * C, true);
    b.fc2 = L.linear(bp + "/mlp/fc2", 4 * C, C, true);
    m->blocks.push_back(b);
  }
  if (L.err) return L.err;
  m->ln_final = L.norm("layer_norm", C);
  m->has_proj = pv.find("text_projection") != nullptr;
  if (m->has_proj) {
    const PackEntry* e = L.need("text_projection", 2);
    if (!e) return L.err;
    if ((int)e->shape[0] != C || (int)e->shape[1] != g.embed_dim) return fail(c, 4404, "text_projection is [%llu,%llu], expected [%d,%d]", (unsigned long long)e->shape[0], (unsigned long long)e->shape[1], C, g.embed_dim);
    Lin& P = m->proj;
    P.K = C; P.Kpad = Cpad; P.N = g.embed_dim;
    P.w = A.get<__half>((size_t)g.embed_dim * Cpad);
    if (!P.w) return fail(c, 4005, "weight arena exhausted");
    if (!A.measure) { int r = transpose_linear_launch(c->stream, L.ptr(e), C, g.embed_dim, P.w, Cpad, 0, 0); if (r) return fail(c, r, "text_projection re-layout failed"); }
  }
  return L.err;
}

extern "C" void sdxl_clip_destroy(sdxl_clip* m) {
  if (!m) return;
  cudaStreamSynchronize(m->ctx->stream);
  m->plan.reset();
  m->warena.release();
  if (m->tokens_dev) cudaFree(m->tokens_dev);
  delete m;
}

extern "C" int sdxl_clip_load(sdxl_ctx* c, const sdxl_clip_cfg* cfg, const void* pack, size_t bytes, int pack_on_device, sdxl_clip** out) {
  if (!c || !cfg || !pack || !out) return fail(c, -1, "sdxl_clip_load: null argument");
  *out = nullptr;
  if (cfg->n_head < 1 || cfg->n_state != cfg->n_head * 64) return fail(c, 4410, "text encoder head dim must be 64 (n_state=%d, n_head=%d)", cfg->n_state, cfg->n_head);
  if (cfg->n_ctx < 1 || cfg->n_ctx > 1024 || cfg->n_layer < 1 || cfg->n_vocab < 1 || cfg->embed_dim < 1) return fail(c, 4411, "bad text encoder config");
  CU(c, cudaSetDevice(c->device));
  std::unique_ptr<sdxl_clip> m(new sdxl_clip());
  m->ctx = c;
  m->cfg = *cfg;
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
  r = build_clip(m.get(), pv, meas);
  if (!r && m->warena.init(meas.off + (1 << 20))) r = fail(c, 4203, "cannot allocate %zu bytes for weights", meas.off);
  if (!r) r = build_clip(m.get(), pv, m->warena);
  cudaError_t se = cudaStreamSynchronize(c->stream);
  if (dev_pack) cudaFree(dev_pack);
  if (!r && se != cudaSuccess) r = fail(c, (int)se, "weight re-layout failed: %s", cudaGetErrorString(se));
  if (!r && cudaMalloc((void**)&m->tokens_dev, (size_t)(64 * cfg->n_ctx + 64 + 16) * sizeof(int)) != cudaSuccess) r = fail(c, 4412, "cudaMalloc failed");
  if (r) { m->warena.release(); return r; }
  m->eot_dev = m->tokens_dev + 64 * cfg->n_ctx;
  m->err_dev = m->eot_dev + 64;
  *out = m.release();
  return 0;
}

// n_run blocks are executed; when capture >= 0 the stream entering block `capture` is preserved as the hidden output.
static int build_clip_plan(sdxl_clip* m, Plan* P, Arena* A, int n_run, int capture, int pooled) {
  sdxl_ctx* c = m->ctx;
  const sdxl_clip_cfg& g = m->cfg;
  PlanBuilder B{c, P, A, P->Bf};
  P->ops.clear();
  P->flops = 0;
  const int Bn = P->Bf, T = g.n_ctx, C = g.n_state, M = Bn * T;
  float* xa = B.buf<float>((size_t)M * C);
  float* xb = B.buf<float>((size_t)M * C);
  __half* a16 = B.buf<__half>((size_t)M * C);
  __half* qkv16 = B.buf<__half>((size_t)M * 3 * C);
  __half* ao16 = B.buf<__half>((size_t)M * C);
  float* h32 = B.buf<float>((size_t)M * 4 * C);
  __half* h16 = B.buf<__half>((size_t)M * 4 * C);
  float* pin = B.buf<float>((size_t)Bn * C);
  m->pooled = B.buf<float>((size_t)Bn * g.embed_dim);
  if (B.err) return B.err;
  {
    Op op{};
    op.kind = OP_EMBED;
    op.em = {m->tokens_dev, M, T, C, g.n_vocab, m->tok_emb, m->pos_emb, xa, m->err_dev};
    P->ops.push_back(op);
  }
  float* x = xa;
  m->hidden = nullptr;
  for (int i = 0; i < n_run && !B.err; ++i) {
    const CBlock& b = m->blocks[i];
    float* xn = x;
    if (i == capture) {  // keep the input of this block: write the updated stream into the other buffer
      m->hidden = x;
      xn = (x == xa) ? xb : xa;
    }
    // x = x + attn(attn_ln(x), causal mask)    (clip/mod.rs:177-179)
    B.ln(x, b.attn_ln, M, a16);
    B.linear(a16, M, b.qkv, IGEMM_LINEAR, qkv16, 0, 3 * C, nullptr, 0);
    B.attn_small(qkv16, 3 * C, 0, qkv16, 3 * C, C, 2 * C, T, T, g.n_head, nullptr, 1, ao16, C);
    B.linear(ao16, M, b.out, IGEMM_LINEAR, xn, 1, C, x, C);
    // x = x + mlp(mlp_ln(x))
    B.ln(xn, b.mlp_ln, M, a16);
    B.linear(a16, M, b.fc1, IGEMM_LINEAR, h32, 1, 4 * C, nullptr, 0);
    {
      Op op{};
      op.kind = OP_ACT;
      op.ac = {h32, (size_t)M * 4 * C, g.quick_gelu ? 1 : 0, h16};
      P->ops.push_back(op);
    }
    B.linear(h16, M, b.fc2, IGEMM_LINEAR, xn, 1, C, xn, C);
    x = xn;
  }
  if (capture < 0 || capture >= n_run) m->hidden = x;
  if (pooled && !B.err) {
    // features of the end-of-text position: layer_norm(x)[b, argmax(tokens[b])] (@ text_projection)   (clip/mod.rs:130-141)
    Op op{};
    op.kind = OP_LN_GATHER;
    op.lg = {x, m->eot_dev, Bn, T, C, m->ln_final.g, m->ln_final.b, m->ln_final.eps, m->has_proj ? pin : m->pooled};
    P->ops.push_back(op);
    if (m->has_proj) B.gemv(pin, C, Bn, m->proj, nullptr, 0, 0, 0, m->pooled, g.embed_dim);
  }
  return B.err;
}

static int clip_run(sdxl_clip* m, int Bn, const int32_t* tokens_host, int n_run, int capture, int pooled) {
  sdxl_ctx* c = m->ctx;
  const sdxl_clip_cfg& g = m->cfg;
  if (!tokens_host) return fail(c, -1, "null tokens");
  if (Bn < 1 || Bn > 64) return fail(c, 5201, "text encoder batch must be 1..64 (got %d)", Bn);
  if (n_run < 0 || n_run > g.n_layer) return fail(c, 5202, "hidden_idx %d out of range (n_layer %d)", n_run, g.n_layer);
  CU(c, cudaSetDevice(c->device));
  if (!m->plan || m->pB != Bn || m->p_nrun != n_run || m->p_hidden != capture || m->p_pooled != pooled) {
    CU(c, cudaStreamSynchronize(c->stream));
    m->plan.reset(new Plan());
    Plan* P = m->plan.get();
    P->Bf = Bn; P->Bx = Bn;
    Arena meas;
    meas.measure = true;
    int r = build_clip_plan(m, P, &meas, n_run, capture, pooled);
    if (!r && P->arena.init(meas.off + (1 << 20))) r = fail(c, 5011, "cannot allocate %zu bytes of workspace", meas.off);
    if (!r) r = build_clip_plan(m, P, &P->arena, n_run, capture, pooled);
    if (r) { m->plan.reset(); return r; }
    m->pB = Bn; m->p_nrun = n_run; m->p_hidden = capture; m->p_pooled = pooled;
  }
  // eot_indices = tokens.argmax(1): first position of the largest id (clip/mod.rs:130)
  std::vector<int> meta(64 + 1, 0);
  for (int b = 0; b < Bn; ++b) {
    int best = 0;
    for (int t = 1; t < g.n_ctx; ++t)
      if (tokens_host[b * g.n_ctx + t] > tokens_host[b * g.n_ctx + best]) best = t;
    meta[b] = best;
  }
  CU(c, cudaMemcpyAsync(m->tokens_dev, tokens_host, (size_t)Bn * g.n_ctx * sizeof(int), cudaMemcpyHostToDevice, c->stream));
  CU(c, cudaMemcpyAsync(m->eot_dev, meta.data(), 65 * sizeof(int), cudaMemcpyHostToDevice, c->stream));  // also clears err_dev
  CU(c, cudaStreamSynchronize(c->stream));  // meta / tokens_host are pageable host memory
  int r = run_plan_ops(c, m->plan.get());
  if (r) return r;
  int err = 0;
  CU(c, cudaMemcpyAsync(&err, m->err_dev, sizeof(int), cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  if (err) return fail(c, 5203, "token id outside [0, %d) (the reference's embedding lookup panics)", g.n_vocab);
  return 0;
}

static int clip_copy_out(sdxl_clip* m, const float* src, size_t n, float* dst, int on_host) {
  sdxl_ctx* c = m->ctx;
  if (!dst) return 0;
  CU(c, cudaMemcpyAsync(dst, src, n * sizeof(float), on_host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, c->stream));
  if (on_host) CU(c, cudaStreamSynchronize(c->stream));
  return 0;
}

extern "C" int sdxl_clip_forward_hidden(sdxl_clip* m, int Bn, const int32_t* tokens_host, int hidden_idx, float* hidden_out, int out_on_host) {
  if (!m || !hidden_out) return fail(m ? m->ctx : nullptr, -1, "sdxl_clip_forward_hidden: null argument");
  int r = clip_run(m, Bn, tokens_host, hidden_idx, -1, 0);
  if (r) return r;
  return clip_copy_out(m, m->hidden, (size_t)Bn * m->cfg.n_ctx * m->cfg.n_state, hidden_out, out_on_host);
}
extern "C" int sdxl_clip_forward_hidden_pooled(sdxl_clip* m, int Bn, const int32_t* tokens_host, int hidden_idx, float* hidden_out,
                                               float* pooled_out, int out_on_host) {
  if (!m || !hidden_out || !pooled_out) return fail(m ? m->ctx : nullptr, -1, "sdxl_clip_forward_hidden_pooled: null argument");
  if (hidden_idx < 0 || hidden_idx >= m->cfg.n_layer) return fail(m->ctx, 5204, "hidden_idx %d out of range: the reference returns an uninitialised tensor there (clip/mod.rs:120-126)", hidden_idx);
  int r = clip_run(m, Bn, tokens_host, m->cfg.n_layer, hidden_idx, 1);
  if (r) return r;
  r = clip_copy_out(m, m->hidden, (size_t)Bn * m->cfg.n_ctx * m->cfg.n_state, hidden_out, out_on_host);
  if (r) return r;
  return clip_copy_out(m, m->pooled, (size_t)Bn * (m->has_proj ? m->cfg.embed_dim : m->cfg.n_state), pooled_out, out_on_host);
}
extern "C" double sdxl_clip_plan_flops(const sdxl_clip* m) { return (m && m->plan) ? m->plan->flops : 0.0; }

