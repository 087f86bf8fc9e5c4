// UNet / sampler front end of libsdxl_b200.so: context entry points, the UNet weight loader (re-layout on device), the
// UNet launch plan, the DDIM/CFG sampler loop and the operator-level entry points of include/sdxl_b200.h. The shared
// machinery (arena, pack parsing, launch plan, CUDA-graph replay) is in engine_core.h; the latent decoder / encoder is
// vae.cu, the text encoders clip.cu, the tokenizers tokenizer.cpp. No torch, no cuBLAS/cuDNN: every device op is one of
// this library's own sm_100a kernels.
//
// Structure mirrored from the reference (file:line relative to the reference root):
//   UNet::forward               src/model/unet/mod.rs:449-493
//   UNetConfig::init (blocks)   src/model/unet/mod.rs:72-430
//   ResBlock / SpatialTransformer / TransformerBlock / MHA / GEGLU
//                               src/model/unet/mod.rs:1082-1106, 820-845, 885-891, 1005-1023, 942-956
//   Diffuser::{sample_latent, sample_latent_with_inpainting, refine_latent, diffuse_latent*,
//              forward_diffuser, get_alpha}
//                               src/model/stablediffusion/mod.rs:317-541
#include "engine_core.h"

// ================================================================================================
// context
// ================================================================================================
extern "C" int sdxl_ctx_create(int device, void* cuda_stream, sdxl_ctx** out) {
  if (!out) return -1;
  *out = nullptr;
  int n = 0;
  if (cudaGetDeviceCount(&n) != cudaSuccess || n <= 0 || device >= n) {
    fprintf(stderr, "sdxl_b200: no CUDA device %d (this library has no CPU fallback)\n", device);
    return -2;
  }
  cudaDeviceProp prop;
  if (cudaGetDeviceProperties(&prop, device) != cudaSuccess) return -3;
  if (prop.major != 10) {
    fprintf(stderr, "sdxl_b200: device %d is sm_%d%d; this library contains sm_100a code only\n", device,
            prop.major, prop.minor);
    return -4;
  }
  if (cudaSetDevice(device) != cudaSuccess) return -5;
  sdxl_ctx* c = new sdxl_ctx();
  c->device = device;
  c->num_sms = prop.multiProcessorCount;
  if (cuda_stream) {
    c->stream = (cudaStream_t)cuda_stream;
  } else {
    if (cudaStreamCreateWithFlags(&c->stream, cudaStreamNonBlocking) != cudaSuccess) {
      delete c;
      return -6;
    }
    c->own_stream = true;
  }
  *out = c;
  return 0;
}
extern "C" void sdxl_ctx_destroy(sdxl_ctx* c) {
  if (!c) return;
  cudaStreamSynchronize(c->stream);
  if (c->own_stream) cudaStreamDestroy(c->stream);
  delete c;
}
extern "C" const char* sdxl_last_error(const sdxl_ctx* c) { return c ? c->err.c_str() : "null ctx"; }
extern "C" int sdxl_ctx_synchronize(sdxl_ctx* c) {
  CU(c, cudaStreamSynchronize(c->stream));
  return 0;
}
extern "C" uint64_t sdxl_ctx_launch_count(const sdxl_ctx* c) { return c ? c->launches : 0; }

// ================================================================================================
// model
// ================================================================================================
struct TBlock {
  Norm n1, n2, n3;
  Lin qkv, out1;      // self-attention (fused [3C, C])
  Lin q2, kv2, out2;  // cross-attention (kv fused [2C, ctx])
  Lin ff1, ff2;
};
struct STrans { Norm norm; Lin proj_in, proj_out; std::vector<TBlock> blocks; int C = 0, n_head = 0; };
struct Res {
  Norm n_in, n_out;
  Conv conv_in, conv_out;  // conv_out carries the fused skip 1x1 segment when Cin != Cout
  int Cin = 0, Cout = 0, temb_off = 0;
  bool has_skip = false;
};
enum BlockType { BT_CONV, BT_RES, BT_DOWN, BT_REST, BT_RESTU, BT_RESU };
struct Block {
  BlockType type = BT_RES;
  Res res;
  STrans st;
  Conv conv;  // BT_CONV (unused: first conv has its own path), BT_DOWN, upsample conv
  int Cout = 0;
};

struct Plan;
struct Sampler;

struct sdxl_unet {
  sdxl_ctx* ctx = nullptr;
  sdxl_unet_cfg cfg{};
  Arena warena;  // re-laid-out weights
  // embeddings
  Lin t1, t2, l1, l2;      // time / label MLPs
  Lin temb_all;            // concatenated lin_embed of every ResBlock [sumC, 4mc], bias folded with conv_in bias
  float* conv0_w = nullptr;  // first conv [mc][3][3][4] f32
  float* conv0_b = nullptr;
  std::vector<Block> in_blocks, out_blocks;
  Res mid_res1, mid_res2;
  STrans mid_st;
  Norm norm_out;
  Conv conv_out;
  __half* conv_out_w2 = nullptr;   // [O, 2*Ktot] = [W | W]: head conv on the hi/lo-split activation
  std::vector<double> alphas;  // host copy (f16-stored values widened)
  int n_tblocks = 0;
  // conditioning state
  Arena carena;
  int condB = 0, n_ctx = 0, ctx_pitch = 0;
  __half* ctx16 = nullptr;     // [B*n_ctx, ctx_pitch]
  float* y32 = nullptr;        // [B, adm]
  float* lab1 = nullptr;       // [B, 4mc]
  float* label_emb = nullptr;  // [B, 4mc]
  std::vector<__half*> kv;     // per transformer block [B*n_ctx, 2C]
  std::vector<int> kvC;
  uint64_t cond_version = 0;
  // plan
  std::unique_ptr<Plan> plan;
  std::unique_ptr<Sampler> sampler;
  int* t_dev = nullptr;
  int* t_pinned = nullptr;
  int t_slot = 0;              // ring position in t_pinned (per model: independent contexts never share it)
};


static int geglu_bn_for(int n_out /*4C*/) {
  for (int hb = 128; hb >= 32; hb >>= 1)
    if (n_out % hb == 0) return 2 * hb;
  return 0;
}

// temb bookkeeping while building: list of (lin_embed path, Cout, conv_in bias) in block order
struct TembItem { std::string path; int Cout; float* conv_bias; };

static Res load_res(Loader& L, const std::string& path, int Cin, int Cout, int temb_dim, std::vector<TembItem>& tembs, int& temb_total) {
  Res r;
  r.Cin = Cin; r.Cout = Cout; r.has_skip = (Cin != Cout);
  r.n_in = L.norm(path + "/norm_in", Cin);
  r.conv_in = L.conv(path + "/conv_in", Cin, Cout, 3);
  r.n_out = L.norm(path + "/norm_out", Cout);
  if (r.has_skip) r.conv_out = L.conv(path + "/conv_out", Cout, Cout, 3, path + "/skip_connection", Cin);
  else r.conv_out = L.conv(path + "/conv_out", Cout, Cout, 3);
  r.temb_off = temb_total;
  tembs.push_back({path + "/lin_embed", Cout, r.conv_in.b});
  temb_total += Cout;
  (void)temb_dim;
  return r;
}

static STrans load_st(Loader& L, const std::string& path, int C, int ctx_dim, int n_head, int depth) {
  STrans s;
  s.C = C; s.n_head = n_head;
  s.norm = L.norm(path + "/norm", C);
  s.proj_in = L.linear(path + "/proj_in", C, C, true);
  s.proj_out = L.linear(path + "/proj_out", C, C, true);
  const int ctx_pad = Loader::pad64(ctx_dim);
  const int Cpad = Loader::pad64(C);
  for (int j = 0; j < depth && !L.err; ++j) {
    const std::string bp = path + "/transformer_" + std::to_string(j);
    TBlock b;
    b.n1 = L.norm(bp + "/norm1", C);
    b.n2 = L.norm(bp + "/norm2", C);
    b.n3 = L.norm(bp + "/norm3", C);
    // fused QKV for self-attention (reference unet/mod.rs:1009-1011: three bias-free Linears on x)
    b.qkv.K = C; b.qkv.Kpad = Cpad; b.qkv.N = 3 * C;
    b.qkv.w = L.A->get<__half>((size_t)3 * C * Cpad);
    if (!b.qkv.w) { L.err = fail(L.c, 4005, "weight arena exhausted"); break; }
    L.lin_into(bp + "/attn1/query", b.qkv.w, Cpad, 0, C, C, 0);
    L.lin_into(bp + "/attn1/key", b.qkv.w, Cpad, C, C, C, 0);
    L.lin_into(bp + "/attn1/value", b.qkv.w, Cpad, 2 * C, C, C, 0);
    b.out1 = L.linear(bp + "/attn1/out", C, C, true);
    b.q2 = L.linear(bp + "/attn2/query", C, C, false);
    b.kv2.K = ctx_dim; b.kv2.Kpad = ctx_pad; b.kv2.N = 2 * C;
    b.kv2.w = L.A->get<__half>((size_t)2 * C * ctx_pad);
    if (!b.kv2.w) { L.err = fail(L.c, 4005, "weight arena exhausted"); break; }
    L.lin_into(bp + "/attn2/key", b.kv2.w, ctx_pad, 0, ctx_dim, C, 0);
    L.lin_into(bp + "/attn2/value", b.kv2.w, ctx_pad, C, ctx_dim, C, 0);
    b.out2 = L.linear(bp + "/attn2/out", C, C, true);
    const int gbn = geglu_bn_for(4 * C);
    if (!gbn) { L.err = fail(L.c, 4009, "GEGLU width %d not tileable", 4 * C); break; }
    b.ff1 = L.linear(bp + "/mlp/geglu/proj", C, 8 * C, true, gbn);
    b.ff2 = L.linear(bp + "/mlp/lin", 4 * C, C, true);
    s.blocks.push_back(b);
  }
  return s;
}

// Builds every layer (in measure mode only sizes are accumulated).
static int build_model(sdxl_unet* u, const PackView& pv, Arena& A) {
  sdxl_ctx* c = u->ctx;
  const sdxl_unet_cfg& g = u->cfg;
  Loader L{u, c, &pv, &A, c->stream};
  const int mc = g.model_channels, ted = 4 * mc;
  u->in_blocks.clear();
  u->out_blocks.clear();
  std::vector<TembItem> tembs;
  int temb_total = 0;
  auto n_head = [&](int ch) { return ch / g.n_head_channels; };

  u->t1 = L.linear("lin1_time_embed", mc, ted, true);
  u->t2 = L.linear("lin2_time_embed", ted, ted, true);
  u->l1 = L.linear("lin1_label_embed", g.adm_in_channels, ted, true);
  u->l2 = L.linear("lin2_label_embed", ted, ted, true);
  if (L.err) return L.err;

  // first conv: OIHW f16 -> [O][kh][kw][I] f32 (CUDA-core kernel)
  {
    const PackEntry* e = L.need("input_blocks/0/weight", 4);
    if (!e) return L.err;
    if ((int)e->shape[0] != mc || (int)e->shape[1] != g.in_channels || e->shape[2] != 3 || e->shape[3] != 3)
      return fail(c, 4010, "input_blocks/0/weight bad shape");
    const size_t n = (size_t)mc * 9 * g.in_channels;
    __half* tmp = A.get<__half>(n);
    u->conv0_w = A.get<float>(n);
    if (!tmp || !u->conv0_w) return fail(c, 4005, "weight arena exhausted");
    if (!A.measure) {
      int r = repack_conv_launch(c->stream, L.ptr(e), mc, g.in_channels, 3, 3, tmp, 9 * g.in_channels, 0, g.in_channels);
      if (!r) r = cast_f16_to_f32_launch(c->stream, tmp, n, u->conv0_w);
      if (r) return fail(c, r, "conv0 repack failed");
    }
    u->conv0_b = L.vec_f32("input_blocks/0/bias", mc);
    if (L.err) return L.err;
  }
  {
    Block b0; b0.type = BT_CONV; b0.Cout = mc;
    u->in_blocks.push_back(b0);
  }
  // input blocks (reference unet/mod.rs:121-173)
  int idx = 1;
  for (int level = 0; level < g.n_levels && !L.err; ++level) {
    const int cin = g.channel_mults[level > 0 ? level - 1 : 0] * mc;
    const int cout = g.channel_mults[level] * mc;
    const bool tr = (level == 1 || level == 2);
    for (int k = 0; k < 2; ++k) {
      Block b;
      const std::string bp = "input_blocks/" + std::to_string(idx++);
      b.Cout = cout;
      if (!tr) {
        b.type = BT_RES;
        b.res = load_res(L, bp, k == 0 ? cin : cout, cout, ted, tembs, temb_total);
      } else {
        b.type = BT_REST;
        b.res = load_res(L, bp + "/res", k == 0 ? cin : cout, cout, ted, tembs, temb_total);
        b.st = load_st(L, bp + "/transformer", cout, g.context_dim, n_head(cout), g.transformer_depths[level]);
      }
      u->in_blocks.push_back(std::move(b));
    }
    if (level != g.n_levels - 1) {
      Block b;
      b.type = BT_DOWN;
      b.Cout = cout;
      b.conv = L.conv("input_blocks/" + std::to_string(idx++), cout, cout, 3);
      u->in_blocks.push_back(std::move(b));
    }
  }
  if (L.err) return L.err;
  // middle (reference unet/mod.rs:238-248)
  {
    const int cm = g.channel_mults[g.n_levels - 1] * mc;
    u->mid_res1 = load_res(L, "middle_block/res1", cm, cm, ted, tembs, temb_total);
    u->mid_st = load_st(L, "middle_block/transformer", cm, g.context_dim, n_head(cm), g.transformer_depths[g.n_levels - 1]);
    u->mid_res2 = load_res(L, "middle_block/res2", cm, cm, ted, tembs, temb_total);
  }
  if (L.err) return L.err;
  // output blocks (reference unet/mod.rs:250-328)
  idx = 0;
  for (int level = g.n_levels - 1; level >= 0 && !L.err; --level) {
    const int next_level = (level != g.n_levels - 1) ? level + 1 : level;
    const int cout = g.channel_mults[level] * mc;
    const int cin1 = g.channel_mults[next_level] * mc + cout;
    const int cin2 = 2 * cout;
    const int cin3 = cout + g.channel_mults[level > 0 ? level - 1 : 0] * mc;
    const bool tr = (level == 1 || level == 2);
    const int cins[3] = {cin1, cin2, cin3};
    for (int k = 0; k < 3; ++k) {
      Block b;
      const std::string bp = "output_blocks/" + std::to_string(idx++);
      b.Cout = cout;
      const bool up = (k == 2) && (tr || level != 0);
      if (!tr) {
        b.type = up ? BT_RESU : BT_RES;
        b.res = load_res(L, up ? bp + "/res" : bp, cins[k], cout, ted, tembs, temb_total);
      } else {
        b.type = up ? BT_RESTU : BT_REST;
        b.res = load_res(L, bp + "/res", cins[k], cout, ted, tembs, temb_total);
        b.st = load_st(L, bp + "/transformer", cout, g.context_dim, n_head(cout), g.transformer_depths[level]);
      }
      if (up) b.conv = L.upconv(bp + "/upsample/conv", cout, cout);
      u->out_blocks.push_back(std::move(b));
    }
  }
  if (L.err) return L.err;
  u->norm_out = L.norm("norm_out", mc);
  u->conv_out = L.conv("conv_out", mc, g.out_channels, 3);
  if (L.err) return L.err;
  // The head conv is the one GEMM whose operand-rounding error reaches eps undamped (every other layer's is averaged by what
  // follows), so its activation operand is split hi + lo (two f16 tensors, ~22 bits): same weights twice along K.
  u->conv_out_w2 = L.dup_k(u->conv_out);
  if (L.err) return L.err;

  // concatenated lin_embed matrix (one GEMV per forward for all ResBlocks); bias += conv_in bias
  {
    Lin& T = u->temb_all;
    T.K = ted; T.Kpad = Loader::pad64(ted); T.N = temb_total;
    T.w = A.get<__half>((size_t)temb_total * T.Kpad);
    T.b = A.get<float>(temb_total);
    if (!T.w || !T.b) return fail(c, 4005, "weight arena exhausted");
    int off = 0;
    for (auto& it : tembs) {
      if (L.lin_into(it.path, T.w, T.Kpad, off, ted, it.Cout, 0)) return L.err;
      const PackEntry* e = L.need(it.path + "/bias", 1);
      if (!e) return L.err;
      if (!A.measure) {
        int r = bias_to_f32_launch(c->stream, L.ptr(e), it.Cout, T.b + off, 0, 0);
        // fold the conv_in bias: h = conv_in(..) + b_conv + lin_embed(..)   (unet/mod.rs:1086-1092)
        if (!r) r = vec_add_f32_launch(c->stream, T.b + off, it.conv_bias, it.Cout);
        if (r) return fail(c, r, "temb bias failed");
      }
      off += it.Cout;
    }
  }
  // count transformer blocks (for the hoisted K/V buffers)
  int nt = 0;
  for (auto& b : u->in_blocks) nt += (int)b.st.blocks.size();
  nt += (int)u->mid_st.blocks.size();
  for (auto& b : u->out_blocks) nt += (int)b.st.blocks.size();
  u->n_tblocks = nt;
  return 0;
}

// ================================================================================================
// load
// ================================================================================================

extern "C" void sdxl_unet_destroy(sdxl_unet* u);

static int unet_load_impl(sdxl_ctx* c, const sdxl_unet_cfg* cfg, const void* pack, size_t bytes, int pack_on_device, sdxl_unet** out);

extern "C" int sdxl_unet_load(sdxl_ctx* c, const sdxl_unet_cfg* cfg, const void* pack, size_t bytes, int pack_on_device,
                              sdxl_unet** out) {
  return unet_load_impl(c, cfg, pack, bytes, pack_on_device, out);
}

// ---- NCCL, resolved at run time (no link-time dependency: the library must load on machines without it) ----
#include <dlfcn.h>
namespace {
typedef int (*PFN_ncclBroadcast)(const void*, void*, size_t, int /*ncclDataType_t*/, int, void* /*ncclComm_t*/, cudaStream_t);
typedef const char* (*PFN_ncclGetErrorString)(int);
struct NcclApi { PFN_ncclBroadcast bcast = nullptr; PFN_ncclGetErrorString errstr = nullptr; bool tried = false; };
NcclApi& nccl_api() {
  static NcclApi api;
  if (!api.tried) {
    api.tried = true;
    void* h = dlopen("libnccl.so.2", RTLD_NOW | RTLD_NOLOAD);   // the copy the host application (e.g. torch) already loaded
    if (!h && getenv("SDXL_B200_NCCL_LIB")) h = dlopen(getenv("SDXL_B200_NCCL_LIB"), RTLD_NOW);
    if (!h) h = dlopen("libnccl.so.2", RTLD_NOW);
    if (h) {
      api.bcast = (PFN_ncclBroadcast)dlsym(h, "ncclBroadcast");
      api.errstr = (PFN_ncclGetErrorString)dlsym(h, "ncclGetErrorString");
    }
  }
  return api;
}
}  // namespace

extern "C" int sdxl_unet_load_broadcast(sdxl_ctx* c, const sdxl_unet_cfg* cfg, const void* pack, size_t bytes, int pack_on_device,
                                        void* nccl_comm, int rank, int root, sdxl_unet** out) {
  if (!c || !cfg || !out) return fail(c, -1, "sdxl_unet_load_broadcast: null argument");
  *out = nullptr;
  if (!nccl_comm) return fail(c, 4300, "sdxl_unet_load_broadcast: null NCCL communicator");
  if (rank == root && (!pack || !bytes)) return fail(c, 4301, "sdxl_unet_load_broadcast: the root rank must pass the weight pack");
  NcclApi& N = nccl_api();
  if (!N.bcast) return fail(c, 4302, "sdxl_unet_load_broadcast: libnccl.so.2 not found (set SDXL_B200_NCCL_LIB)");
  CU(c, cudaSetDevice(c->device));
  const int ncclUint8 = 1;
  // 1. the size, so that non-root ranks can allocate
  unsigned long long* dsz = nullptr;
  CU(c, cudaMalloc((void**)&dsz, 8));
  unsigned long long hsz = rank == root ? (unsigned long long)bytes : 0ull;
  cudaError_t e = cudaMemcpyAsync(dsz, &hsz, 8, cudaMemcpyHostToDevice, c->stream);
  int nr = e == cudaSuccess ? N.bcast(dsz, dsz, 8, ncclUint8, root, nccl_comm, c->stream) : 0;
  if (e == cudaSuccess && !nr) e = cudaMemcpyAsync(&hsz, dsz, 8, cudaMemcpyDeviceToHost, c->stream);
  if (e == cudaSuccess && !nr) e = cudaStreamSynchronize(c->stream);
  cudaFree(dsz);
  if (nr) return fail(c, 4303, "ncclBroadcast (pack size) failed: %s", N.errstr ? N.errstr(nr) : "?");
  if (e != cudaSuccess) return fail(c, (int)e, "pack size broadcast failed: %s", cudaGetErrorString(e));
  if (hsz < sizeof(PackHeader)) return fail(c, 4304, "broadcast pack size %llu is not a weight pack", hsz);
  // 2. the pack itself: one flat message
  uint8_t* dpack = nullptr;
  CU(c, cudaMalloc((void**)&dpack, (size_t)hsz));
  if (rank == root)
    e = cudaMemcpyAsync(dpack, pack, (size_t)hsz, pack_on_device ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice, c->stream);
  if (e == cudaSuccess) nr = N.bcast(dpack, dpack, (size_t)hsz, ncclUint8, root, nccl_comm, c->stream);
  if (e == cudaSuccess && !nr) e = cudaStreamSynchronize(c->stream);
  int r = 0;
  if (nr) r = fail(c, 4303, "ncclBroadcast (pack) failed: %s", N.errstr ? N.errstr(nr) : "?");
  else if (e != cudaSuccess) r = fail(c, (int)e, "pack broadcast failed: %s", cudaGetErrorString(e));
  else r = unet_load_impl(c, cfg, dpack, (size_t)hsz, 1, out);
  cudaFree(dpack);
  return r;
}

static int unet_load_impl(sdxl_ctx* c, const sdxl_unet_cfg* cfg, const void* pack, size_t bytes, int pack_on_device, sdxl_unet** out) {
  if (!c || !cfg || !pack || !out) return fail(c, -1, "sdxl_unet_load: null argument");
  *out = nullptr;
  if (cfg->n_head_channels != 64) return fail(c, 4200, "n_head_channels must be 64 (got %d)", cfg->n_head_channels);
  if (cfg->n_levels < 1 || cfg->n_levels > SDXL_MAX_LEVELS) return fail(c, 4201, "bad n_levels");
  if (cfg->in_channels > 8 || cfg->model_channels % 32) return fail(c, 4202, "unsupported channel config");
  CU(c, cudaSetDevice(c->device));
  std::unique_ptr<sdxl_unet> u(new sdxl_unet());
  u->ctx = c;
  u->cfg = *cfg;
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
  // pass 1: measure, pass 2: build
  Arena meas;
  meas.measure = true;
  r = build_model(u.get(), pv, meas);
  if (!r) {
    if (u->warena.init(meas.off + (1 << 20))) r = fail(c, 4203, "cannot allocate %zu bytes for weights", meas.off);
  }
  if (!r) r = build_model(u.get(), pv, u->warena);
  // alphas_cumprod: f16-stored in the reference's record (HalfPrecisionSettings), read as f64 (mod.rs:485-492)
  if (!r) {
    const PackEntry* e = pv.find("alphas_cumprod");
    if (!e || e->ndim != 1 || e->dtype != 0) r = fail(c, 4204, "weight pack: missing f16 'alphas_cumprod'");
    else {
      std::vector<uint16_t> raw(e->shape[0]);
      cudaError_t ce = cudaMemcpyAsync(raw.data(), pv.dev + e->offset, raw.size() * 2, cudaMemcpyDeviceToHost, c->stream);
      if (ce == cudaSuccess) ce = cudaStreamSynchronize(c->stream);
      if (ce != cudaSuccess) r = fail(c, (int)ce, "alphas download failed");
      else {
        u->alphas.resize(raw.size());
        for (size_t i = 0; i < raw.size(); ++i) {
          __half_raw hr;
          hr.x = raw[i];
          u->alphas[i] = (double)__half2float(__half(hr));
        }
      }
    }
  }
  cudaError_t se = cudaStreamSynchronize(c->stream);
  if (dev_pack) cudaFree(dev_pack);
  if (!r && se != cudaSuccess) r = fail(c, (int)se, "weight re-layout failed: %s", cudaGetErrorString(se));
  if (r) return r;
  CU(c, cudaMalloc((void**)&u->t_dev, 64));
  CU(c, cudaMallocHost((void**)&u->t_pinned, 4096 * sizeof(int)));
  *out = u.release();
  return 0;
}

// ================================================================================================
// launch plan
// ================================================================================================
// UNet-specific plan pieces on top of the generic PlanBuilder (engine_core.h)
struct UNetPlanBuilder : PlanBuilder {
  sdxl_unet* u = nullptr;
  int kv_index = 0;

  // ---- ResBlock (reference unet/mod.rs:1082-1106) ----
  float* resblock(const Res& r, const float* xa, int Ca, const float* xb, int Cb, int H, int W, const float* temb_all,
                  int temb_total, __half* s_gn1, __half* s_raw, float* s_h, __half* s_gn2) {
    const int HW = H * W;
    float* out = buf<float>((size_t)Bf * HW * r.Cout);
    gn(xa, Ca, xb, Cb, HW, r.n_in, 1, s_gn1, r.has_skip ? s_raw : nullptr);
    ActView a1{s_gn1, Bf, H, W, r.Cin};
    // h = conv_in(silu(gn(x))) + b + lin_embed(silu(emb))[:, :, None, None]   (bias folded into temb_all)
    conv3(a1, nullptr, r.conv_in, s_h, temb_all + r.temb_off, temb_total, nullptr);
    gn(s_h, r.Cout, nullptr, 0, HW, r.n_out, 1, s_gn2, nullptr);
    ActView a2{s_gn2, Bf, H, W, r.Cout};
    if (r.has_skip) {
      ActView sk{s_raw, Bf, H, W, r.Cin};
      conv3(a2, &sk, r.conv_out, out, r.conv_out.b, 0, nullptr);  // skip 1x1 conv fused as a K segment
    } else {
      conv3(a2, nullptr, r.conv_out, out, r.conv_out.b, 0, xa);   // identity residual in the epilogue
    }
    return out;
  }

  // ---- SpatialTransformer (reference unet/mod.rs:820-845, 885-891, 1005-1023) ----
  float* strans(const STrans& s, const float* x, int H, int W, __half* s_a16, float* s_tok, __half* s_qkv, __half* s_ao,
                __half* s_q, __half* s_ff) {
    const int T = H * W, M = Bf * T, C = s.C;
    float* out = buf<float>((size_t)M * C);
    const float sl2e = (float)(1.4426950408889634 / sqrt(64.0));
    gn(x, C, nullptr, 0, T, s.norm, 0, s_a16, nullptr);
    linear(s_a16, M, s.proj_in, IGEMM_LINEAR, s_tok, 1, C, nullptr, 0);
    for (const TBlock& b : s.blocks) {
      // x = x + attn1(norm1(x))
      ln(s_tok, b.n1, M, s_a16);
      linear(s_a16, M, b.qkv, IGEMM_LINEAR, s_qkv, 0, 3 * C, nullptr, 0);
      attn(s_qkv, 3 * C, 0, s_qkv, 3 * C, C, 2 * C, T, T, s.n_head, s_ao, C, sl2e);
      linear(s_ao, M, b.out1, IGEMM_LINEAR, s_tok, 1, C, s_tok, C);
      // x = x + attn2(norm2(x), context)   (K/V hoisted to set_conditioning)
      ln(s_tok, b.n2, M, s_a16);
      linear(s_a16, M, b.q2, IGEMM_LINEAR, s_q, 0, C, nullptr, 0);
      const __half* kvp = A->measure ? nullptr : u->kv[kv_index];
      attn(s_q, C, 0, kvp, 2 * C, 0, C, T, u->n_ctx, s.n_head, s_ao, C, sl2e);
      P->flops += 2.0 * Bf * u->n_ctx * (double)b.kv2.K * b.kv2.N;  // hoisted K/V projections (algorithmic work)
      kv_index++;
      linear(s_ao, M, b.out2, IGEMM_LINEAR, s_tok, 1, C, s_tok, C);
      // x = x + mlp(norm3(x))
      ln(s_tok, b.n3, M, s_a16);
      linear(s_a16, M, b.ff1, IGEMM_GEGLU, s_ff, 0, 4 * C, nullptr, 0);
      // the last block's stream only feeds proj_out: its residual add writes the f16 operand directly (no f32 copy, no cast launch)
      if (&b == &s.blocks.back()) linear(s_ff, M, b.ff2, IGEMM_LINEAR, s_a16, 0, C, s_tok, C);
      else linear(s_ff, M, b.ff2, IGEMM_LINEAR, s_tok, 1, C, s_tok, C);
    }
    if (s.blocks.empty() && !err) {   // no block to fold the cast into
      Op op{};
      op.kind = OP_CAST16;
      op.cs = {s_tok, (size_t)M * C, s_a16};
      P->ops.push_back(op);
    }
    // proj_out(tokens) + x_in
    linear(s_a16, M, s.proj_out, IGEMM_LINEAR, out, 1, C, x, C);
    return out;
  }
};



// Builds the op list for UNet::forward (reference unet/mod.rs:449-493) at batch Bf, latent h x w.
static int build_plan_ops(sdxl_unet* u, Plan* P, Arena* A) {
  sdxl_ctx* c = u->ctx;
  const sdxl_unet_cfg& g = u->cfg;
  UNetPlanBuilder B{{c, P, A, P->Bf}, u};
  P->ops.clear();
  P->block_names.clear();
  P->flops = 0;
  const int Bf = P->Bf, mc = g.model_channels, ted = 4 * mc;
  const int temb_total = u->temb_all.N;
  const int levels = g.n_levels;
  if ((P->h % (1 << (levels - 1))) || (P->w % (1 << (levels - 1)))) return fail(c, 5003, "latent %dx%d not divisible by %d", P->h, P->w, 1 << (levels - 1));

  P->x_in = B.buf<float>((size_t)P->Bx * g.in_channels * P->h * P->w);
  P->eps_ld = g.out_channels;
  P->eps = B.buf<float>((size_t)Bf * P->h * P->w * P->eps_ld);
  B.gn_partial = B.buf<float>(gn_scratch_floats(Bf, 32));
  if (B.gn_partial && !A->measure && gn_scratch_init(c->stream, B.gn_partial, Bf, 32)) return fail(c, 5007, "GroupNorm scratch init failed");
  float* te = B.buf<float>(mc);
  float* t1 = B.buf<float>(ted);
  float* semb = B.buf<float>((size_t)Bf * ted);
  float* temb_all = B.buf<float>((size_t)Bf * temb_total);

  // maxima for the shared scratch buffers
  size_t max_pixC_cat = 0, max_pixC = 0, max_tokC = 0, max_tok = 0;
  {
    int H = P->h, W = P->w;
    auto upd = [&](const Res& r, int hh, int ww) {
      max_pixC_cat = std::max(max_pixC_cat, (size_t)hh * ww * r.Cin);
      max_pixC = std::max(max_pixC, (size_t)hh * ww * r.Cout);
    };
    for (auto& b : u->in_blocks) {
      if (b.type == BT_RES || b.type == BT_REST) upd(b.res, H, W);
      if (b.type == BT_REST) { max_tokC = std::max(max_tokC, (size_t)H * W * b.st.C); max_tok = std::max(max_tok, (size_t)H * W); }
      if (b.type == BT_DOWN) { H /= 2; W /= 2; }
    }
    upd(u->mid_res1, H, W);
    upd(u->mid_res2, H, W);
    max_tokC = std::max(max_tokC, (size_t)H * W * u->mid_st.C);
    max_tok = std::max(max_tok, (size_t)H * W);
    for (auto& b : u->out_blocks) {
      upd(b.res, H, W);
      if (b.type == BT_REST || b.type == BT_RESTU) { max_tokC = std::max(max_tokC, (size_t)H * W * b.st.C); max_tok = std::max(max_tok, (size_t)H * W); }
      if (b.type == BT_RESTU || b.type == BT_RESU) { H *= 2; W *= 2; }
    }
  }
  __half* s_gn1 = B.buf<__half>(Bf * max_pixC_cat);
  __half* s_raw = B.buf<__half>(Bf * max_pixC_cat);
  float* s_h = B.buf<float>(Bf * max_pixC);
  __half* s_gn2 = B.buf<__half>(Bf * max_pixC);
  __half* s_a16 = B.buf<__half>(Bf * max_tokC);
  float* s_tok = B.buf<float>(Bf * max_tokC);
  __half* s_qkv = B.buf<__half>(Bf * max_tokC * 3);
  __half* s_ao = B.buf<__half>(Bf * max_tokC);
  __half* s_q = B.buf<__half>(Bf * max_tokC);
  __half* s_ff = B.buf<__half>(Bf * max_tokC * 4);
  if (B.err) return B.err;

  // --- embeddings (unet/mod.rs:458-468): emb = time_mlp(temb(t)) + label_emb; only SiLU(emb) is consumed
  {
    Op op{};
    op.kind = OP_TEMB;
    op.te = {u->t_dev, 1, mc, te};
    P->ops.push_back(op);
  }
  B.gemv(te, 0, 1, u->t1, nullptr, 0, 0, 1, t1, 0);
  B.gemv(t1, 0, Bf, u->t2, u->label_emb, ted, 0, 1, semb, ted);
  B.gemv(semb, ted, Bf, u->temb_all, nullptr, 0, 0, 0, temb_all, temb_total);

  // --- input blocks
  struct Saved { float* p; int C, H, W; };
  std::vector<Saved> saved;
  int H = P->h, W = P->w;
  float* x = B.buf<float>((size_t)Bf * H * W * mc);
  int Cx = mc;
  {
    Op op{};
    op.kind = OP_CONV_IN;
    op.ci = {P->x_in, P->Bx, Bf, g.in_channels, H, W, u->conv0_w, u->conv0_b, mc, x};
    P->ops.push_back(op);
    P->flops += 2.0 * Bf * H * W * 9.0 * g.in_channels * mc;
  }
  saved.push_back({x, Cx, H, W});
  for (size_t i = 1; i < u->in_blocks.size() && !B.err; ++i) {
    const Block& b = u->in_blocks[i];
    B.begin_block("input_blocks/" + std::to_string(i));
    if (b.type == BT_RES || b.type == BT_REST) {
      x = B.resblock(b.res, x, Cx, nullptr, 0, H, W, temb_all, temb_total, s_gn1, s_raw, s_h, s_gn2);
      Cx = b.res.Cout;
      if (b.type == BT_REST) x = B.strans(b.st, x, H, W, s_a16, s_tok, s_qkv, s_ao, s_q, s_ff);
    } else if (b.type == BT_DOWN) {
      // 3x3 stride 2 pad 1 (unet/mod.rs:760-774) on phase-split input: tap kh -> (phase, offset)
      __half* ph = B.buf<__half>((size_t)Bf * H * W * Cx);
      Op op{};
      op.kind = OP_PHASE;
      op.rs = {x, Bf, H, W, Cx, ph};
      P->ops.push_back(op);
      const int H2 = H / 2, W2 = W / 2;
      ActView a{ph, 4 * Bf, H2, W2, Cx};
      std::vector<IgemmSeg> segs;
      for (int kh = 0; kh < 3; ++kh)
        for (int kw = 0; kw < 3; ++kw) {
          const int phh = (kh == 1) ? 0 : 1, pw = (kw == 1) ? 0 : 1;
          const int dh = (kh == 0) ? -1 : 0, dw = (kw == 0) ? -1 : 0;
          segs.push_back({0, (int16_t)dw, (int16_t)dh, (int16_t)((phh * 2 + pw) * Bf), b.conv.Ipad / 64});
        }
      float* y = B.buf<float>((size_t)Bf * H2 * W2 * Cx);
      B.igemm(a, nullptr, segs, b.conv.w, b.conv.O, b.conv.Ktot, H2, W2, Bf, IGEMM_LINEAR, 0, y, 1, b.conv.O, b.conv.b, 0, nullptr, 0);
      B.add_flops(2.0 * Bf * H2 * W2 * 9.0 * Cx * b.conv.O);
      x = y; H = H2; W = W2;
    }
    B.end_block();
    saved.push_back({x, Cx, H, W});
  }
  // --- middle
  B.begin_block("middle_block");
  x = B.resblock(u->mid_res1, x, Cx, nullptr, 0, H, W, temb_all, temb_total, s_gn1, s_raw, s_h, s_gn2);
  x = B.strans(u->mid_st, x, H, W, s_a16, s_tok, s_qkv, s_ao, s_q, s_ff);
  x = B.resblock(u->mid_res2, x, Cx, nullptr, 0, H, W, temb_all, temb_total, s_gn1, s_raw, s_h, s_gn2);
  B.end_block();
  // --- output blocks: cat([x, saved.pop()], channel) is never materialised (GN + skip conv read both)
  for (size_t i = 0; i < u->out_blocks.size() && !B.err; ++i) {
    const Block& b = u->out_blocks[i];
    if (saved.empty()) return fail(c, 5004, "skip stack underflow");
    Saved sk = saved.back();
    saved.pop_back();
    if (sk.H != H || sk.W != W || Cx + sk.C != b.res.Cin) return fail(c, 5005, "skip shape mismatch at output block %zu", i);
    B.begin_block("output_blocks/" + std::to_string(i));
    x = B.resblock(b.res, x, Cx, sk.p, sk.C, H, W, temb_all, temb_total, s_gn1, s_raw, s_h, s_gn2);
    Cx = b.res.Cout;
    if (b.type == BT_REST || b.type == BT_RESTU) x = B.strans(b.st, x, H, W, s_a16, s_tok, s_qkv, s_ao, s_q, s_ff);
    if (b.type == BT_RESTU || b.type == BT_RESU) {
      // nearest-2x then 3x3 conv (unet/mod.rs:742-751), as four 2x2 phase convolutions of the source image
      __half* x16 = B.buf<__half>((size_t)Bf * H * W * Cx);
      float* y = B.buf<float>((size_t)Bf * 4 * H * W * Cx);
      B.upconv(x, Bf, H, W, b.conv, x16, y);
      H *= 2; W *= 2;
      x = y;
    }
    B.end_block();
  }
  if (B.err) return B.err;
  B.begin_block("norm_out+conv_out");
  // --- head: GN -> SiLU -> conv 3x3 (unet/mod.rs:488-490), hi/lo split (s_raw holds the rounding residue of the activation)
  B.head_hilo(x, Cx, H, W, u->norm_out, u->conv_out, u->conv_out_w2, s_gn1, s_raw, P->eps, P->eps_ld);
  B.end_block();
  return B.err;
}

static int ensure_plan(sdxl_unet* u, int Bf, int Bx, int h, int w) {
  sdxl_ctx* c = u->ctx;
  if (u->condB != Bf) return fail(c, 5010, "conditioning is set for batch %d but forward batch is %d (call sdxl_unet_set_conditioning first)", u->condB, Bf);
  if (u->plan && u->plan->Bf == Bf && u->plan->Bx == Bx && u->plan->h == h && u->plan->w == w && u->plan->cond_version == u->cond_version)
    return 0;
  CU(c, cudaStreamSynchronize(c->stream));
  u->plan.reset(new Plan());
  Plan* P = u->plan.get();
  P->Bf = Bf; P->Bx = Bx; P->h = h; P->w = w; P->cond_version = u->cond_version;
  Arena meas;
  meas.measure = true;
  int r = build_plan_ops(u, P, &meas);
  if (r) { u->plan.reset(); return r; }
  if (P->arena.init(meas.off + (1 << 20))) { u->plan.reset(); return fail(c, 5011, "cannot allocate %zu bytes of workspace", meas.off); }
  r = build_plan_ops(u, P, &P->arena);
  if (r) { u->plan.reset(); return r; }
  return 0;
}

static int run_plan(sdxl_unet* u) { return run_plan_ops(u->ctx, u->plan.get()); }

static int set_t(sdxl_unet* u, int t) {
  sdxl_ctx* c = u->ctx;
  const int slot = u->t_slot = (u->t_slot + 1) % 4096;
  u->t_pinned[slot] = t;
  CU(c, cudaMemcpyAsync(u->t_dev, &u->t_pinned[slot], sizeof(int), cudaMemcpyHostToDevice, c->stream));
  return 0;
}

// ================================================================================================
// conditioning (step-invariant work hoisted out of UNet::forward)
// ================================================================================================
static int set_conditioning_dev(sdxl_unet* u, int B, int n_ctx, const __half* context_dev, const __half* y_dev) {
  sdxl_ctx* c = u->ctx;
  const sdxl_unet_cfg& g = u->cfg;
  const int ted = 4 * g.model_channels;
  if (B < 1 || n_ctx < 1) return fail(c, 5100, "bad conditioning shape");
  if (u->condB != B || u->n_ctx != n_ctx) {
    CU(c, cudaStreamSynchronize(c->stream));
    u->plan.reset();
    // collect transformer blocks
    std::vector<const TBlock*> tbs;
    for (auto& b : u->in_blocks) for (auto& t : b.st.blocks) tbs.push_back(&t);
    for (auto& t : u->mid_st.blocks) tbs.push_back(&t);
    for (auto& b : u->out_blocks) for (auto& t : b.st.blocks) tbs.push_back(&t);
    u->ctx_pitch = (g.context_dim + 7) / 8 * 8;
    size_t need = 0;
    auto al = [&](size_t b) { need = ((need + 1023) & ~size_t(1023)) + b; };
    al((size_t)B * n_ctx * u->ctx_pitch * 2);
    al((size_t)B * g.adm_in_channels * 4);
    al((size_t)B * ted * 4);
    al((size_t)B * ted * 4);
    for (auto* t : tbs) al((size_t)B * n_ctx * t->kv2.N * 2);
    if (u->carena.init(need + (1 << 16))) return fail(c, 5101, "cannot allocate conditioning buffers");
    u->ctx16 = u->carena.get<__half>((size_t)B * n_ctx * u->ctx_pitch);
    u->y32 = u->carena.get<float>((size_t)B * g.adm_in_channels);
    u->lab1 = u->carena.get<float>((size_t)B * ted);
    u->label_emb = u->carena.get<float>((size_t)B * ted);
    u->kv.clear();
    u->kvC.clear();
    for (auto* t : tbs) {
      u->kv.push_back(u->carena.get<__half>((size_t)B * n_ctx * t->kv2.N));
      u->kvC.push_back(t->kv2.N / 2);
    }
    u->condB = B;
    u->n_ctx = n_ctx;
    CU(c, cudaMemsetAsync(u->ctx16, 0, (size_t)B * n_ctx * u->ctx_pitch * 2, c->stream));
  }
  u->cond_version++;
  if (u->plan) u->plan->cond_version = u->cond_version;  // buffers unchanged: plan stays valid
  CU(c, cudaMemcpy2DAsync(u->ctx16, (size_t)u->ctx_pitch * 2, context_dev, (size_t)g.context_dim * 2, (size_t)g.context_dim * 2,
                          (size_t)B * n_ctx, cudaMemcpyDeviceToDevice, c->stream));
  KL(c, cast_f16_to_f32_launch(c->stream, y_dev, (size_t)B * g.adm_in_channels, u->y32));
  // label_emb = lin2(SiLU(lin1(y)))   (unet/mod.rs:464-466)
  for (int b0 = 0; b0 < B; b0 += 8) {
    const int nb = B - b0 < 8 ? B - b0 : 8;
    KL(c, gemv_launch(c->stream, u->y32 + (size_t)b0 * g.adm_in_channels, g.adm_in_channels, nb, g.adm_in_channels, u->l1.w,
                      u->l1.Kpad, u->l1.b, nullptr, 0, ted, 0, 1, u->lab1 + (size_t)b0 * ted, ted));
    KL(c, gemv_launch(c->stream, u->lab1 + (size_t)b0 * ted, ted, nb, u->l2.K, u->l2.w, u->l2.Kpad, u->l2.b, nullptr, 0, ted, 0, 0,
                      u->label_emb + (size_t)b0 * ted, ted));
  }
  // K/V projections of the context for every cross-attention (unet/mod.rs:1010-1011)
  {
    std::vector<const TBlock*> tbs;
    for (auto& b : u->in_blocks) for (auto& t : b.st.blocks) tbs.push_back(&t);
    for (auto& t : u->mid_st.blocks) tbs.push_back(&t);
    for (auto& b : u->out_blocks) for (auto& t : b.st.blocks) tbs.push_back(&t);
    const int M = B * n_ctx;
    for (size_t i = 0; i < tbs.size(); ++i) {
      const Lin& L = tbs[i]->kv2;
      IgemmParams p{};
      p.nseg = 1;
      p.seg[0] = {0, 0, 0, 0, L.Kpad / 64};
      p.out = u->kv[i]; p.out_f32 = 0; p.ldo = L.N;
      IgemmOperands o{u->ctx16, 1, 1, M, g.context_dim, u->ctx_pitch, nullptr, 0, 0, 0, 0, 0, L.w, L.N, L.Kpad};
      int r = igemm_configure(p, o, M, 1, 1, IGEMM_LINEAR, 0);
      if (r) return fail(c, r, "igemm configuration failed (kv projection)");
      KL(c, igemm_launch(c->stream, p));
    }
  }
  return 0;
}

extern "C" int sdxl_unet_set_conditioning(sdxl_unet* u, int B, int n_ctx, const sdxl_half* context, const sdxl_half* y) {
  if (!u || !context || !y) return -1;
  CU(u->ctx, cudaSetDevice(u->ctx->device));
  return set_conditioning_dev(u, B, n_ctx, (const __half*)context, (const __half*)y);
}

// ================================================================================================
// UNet::forward
// ================================================================================================
extern "C" int sdxl_unet_forward(sdxl_unet* u, int B, int h, int w, const sdxl_half* x, int32_t t_host, sdxl_half* eps_out) {
  if (!u || !x || !eps_out) return -1;
  sdxl_ctx* c = u->ctx;
  CU(c, cudaSetDevice(c->device));
  int r = ensure_plan(u, B, B, h, w);
  if (r) return r;
  Plan* P = u->plan.get();
  KL(c, cast_f16_to_f32_launch(c->stream, (const __half*)x, (size_t)B * u->cfg.in_channels * h * w, P->x_in));
  if ((r = set_t(u, t_host))) return r;
  if ((r = run_plan(u))) return r;
  KL(c, nhwc_to_nchw_f16_launch(c->stream, P->eps, B, h * w, u->cfg.out_channels, P->eps_ld, (__half*)eps_out));
  return 0;
}
extern "C" int sdxl_unet_forward_f32(sdxl_unet* u, int B, int h, int w, const float* x, int32_t t_host, float* eps_out) {
  if (!u || !x || !eps_out) return -1;
  sdxl_ctx* c = u->ctx;
  CU(c, cudaSetDevice(c->device));
  int r = ensure_plan(u, B, B, h, w);
  if (r) return r;
  Plan* P = u->plan.get();
  CU(c, cudaMemcpyAsync(P->x_in, x, (size_t)B * u->cfg.in_channels * h * w * sizeof(float), cudaMemcpyDeviceToDevice, c->stream));
  if ((r = set_t(u, t_host))) return r;
  if ((r = run_plan(u))) return r;
  KL(c, nhwc_to_nchw_f32_launch(c->stream, P->eps, B, h * w, u->cfg.out_channels, P->eps_ld, eps_out));
  return 0;
}
// Per-kernel-kind device time of one plan execution, measured with CUDA events on the ctx stream
// (eager launches, one event pair per op). kinds: see OpKind. Arrays must hold 16 entries.
extern "C" int sdxl_unet_profile_plan(sdxl_unet* u, double* ms_by_kind, double* flops_by_kind, int* launches_by_kind) {
  if (!u || !u->plan) return -1;
  return profile_plan_impl(u->ctx, u->plan.get(), ms_by_kind, flops_by_kind, launches_by_kind);
}
// Per-op dump of one eager plan execution (CUDA-event time per launch) as CSV: analysis aid for profiles/.
extern "C" int sdxl_unet_profile_dump(sdxl_unet* u, const char* path) {
  if (!u || !u->plan || !path) return -1;
  return profile_dump_impl(u->ctx, u->plan.get(), path);
}
extern "C" double sdxl_unet_alpha(const sdxl_unet* u, int i) {
  if (!u || i < 0 || i >= (int)u->alphas.size()) return NAN;
  return u->alphas[i];
}
// algorithmic FLOPs of the current plan (debug / bench helper, not in the public header)
extern "C" double sdxl_unet_plan_flops(const sdxl_unet* u) { return (u && u->plan) ? u->plan->flops : 0.0; }
extern "C" int sdxl_unet_plan_num_ops(const sdxl_unet* u) { return (u && u->plan) ? (int)u->plan->ops.size() : 0; }
// FLOPs the plan's tensor-core launches actually execute (see Op::flops_exec): excludes the hoisted K/V projections (not in
// the plan), counts the phase-decomposed upsample convs at 4/9 of the algorithmic figure, includes channel / key padding.
extern "C" double sdxl_unet_plan_flops_executed(const sdxl_unet* u) {
  if (!u || !u->plan) return 0.0;
  double f = 0;
  for (const Op& o : u->plan->ops) f += o.flops_exec;
  return f;
}

// ================================================================================================
// sampler (Diffuser)
// ================================================================================================
struct Sampler {
  int Bimg = 0, nfwd = 1, h = 0, w = 0, n_ctx = 0;
  float guidance = 1.f;
  float* noise = nullptr;  // scratch [Bimg,4,h,w]
  float* ref = nullptr;
  uint8_t* mask = nullptr;
  __half* cond_ctx = nullptr;  // staged [nfwd*Bimg, n_ctx, ctx]
  __half* cond_y = nullptr;
  float* host_stage = nullptr;  // pinned
  size_t latent_elems = 0;
  Arena arena;
  ~Sampler() {
    arena.release();
    if (host_stage) cudaFreeHost(host_stage);
  }
};

// Uploads/assembles the batched conditioning: rows [0,Bimg) conditional, rows [Bimg,2*Bimg) the
// unconditional context repeated (reference stablediffusion/mod.rs:506-537).
static int sampler_begin(sdxl_unet* u, const sdxl_conditioning* cond, double guidance) {
  sdxl_ctx* c = u->ctx;
  const sdxl_unet_cfg& g = u->cfg;
  if (!cond) return fail(c, 5200, "null conditioning");
  const int Bimg = cond->n_batch, n_ctx = cond->n_ctx;
  const int h = cond->resolution[0] / 8, w = cond->resolution[1] / 8;
  const int nfwd = g.is_refiner ? 1 : 2;
  const sdxl_half* ctx_c = g.is_refiner ? cond->context_open_clip : cond->context_full;
  const sdxl_half* ctx_u = g.is_refiner ? cond->unconditional_context_open_clip : cond->unconditional_context_full;
  const sdxl_half* y_c = g.is_refiner ? cond->channel_context_refiner : cond->channel_context;
  const sdxl_half* y_u = g.is_refiner ? cond->unconditional_channel_context_refiner : cond->unconditional_channel_context;
  if (!ctx_c || !y_c || (nfwd == 2 && (!ctx_u || !y_u))) return fail(c, 5201, "conditioning tensors for this model are null");
  if (Bimg < 1 || h < 1 || w < 1) return fail(c, 5202, "bad conditioning batch/resolution");
  Sampler* S = u->sampler.get();
  const size_t lat = (size_t)Bimg * g.in_channels * h * w;
  if (n_ctx < 1) return fail(c, 5202, "bad conditioning context length");
  if (!S || S->Bimg != Bimg || S->h != h || S->w != w || S->nfwd != nfwd || S->n_ctx != n_ctx) {   // staging buffers are sized by all five
    CU(c, cudaStreamSynchronize(c->stream));
    u->sampler.reset(new Sampler());
    S = u->sampler.get();
    S->Bimg = Bimg; S->nfwd = nfwd; S->h = h; S->w = w; S->n_ctx = n_ctx; S->latent_elems = lat;
    const size_t ctx_elems = (size_t)nfwd * Bimg * n_ctx * g.context_dim;
    const size_t y_elems = (size_t)nfwd * Bimg * g.adm_in_channels;
    if (S->arena.init(lat * 4 * 2 + lat + ctx_elems * 2 + y_elems * 2 + (1 << 16))) return fail(c, 5203, "cannot allocate sampler buffers");
    S->noise = S->arena.get<float>(lat);
    S->ref = S->arena.get<float>(lat);
    S->mask = S->arena.get<uint8_t>(lat);
    S->cond_ctx = S->arena.get<__half>(ctx_elems);
    S->cond_y = S->arena.get<__half>(y_elems);
    CU(c, cudaMallocHost((void**)&S->host_stage, lat * sizeof(float)));
  }
  S->guidance = (float)guidance;
  const cudaMemcpyKind kind = cond->on_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  const size_t ctx_row = (size_t)n_ctx * g.context_dim * 2, y_row = (size_t)g.adm_in_channels * 2;
  CU(c, cudaMemcpyAsync(S->cond_ctx, ctx_c, ctx_row * Bimg, kind, c->stream));
  CU(c, cudaMemcpyAsync(S->cond_y, y_c, y_row * Bimg, kind, c->stream));
  if (nfwd == 2)
    for (int b = 0; b < Bimg; ++b) {  // unsqueeze().repeat(0, n_batch)
      CU(c, cudaMemcpyAsync((uint8_t*)S->cond_ctx + ctx_row * (Bimg + b), ctx_u, ctx_row, kind, c->stream));
      CU(c, cudaMemcpyAsync((uint8_t*)S->cond_y + y_row * (Bimg + b), y_u, y_row, kind, c->stream));
    }
  int r = set_conditioning_dev(u, nfwd * Bimg, n_ctx, S->cond_ctx, S->cond_y);
  if (r) return r;
  return ensure_plan(u, nfwd * Bimg, Bimg, h, w);
}

// one loop-body iteration (reference stablediffusion/mod.rs:406-429)
static int sampler_step(sdxl_unet* u, int t, int t_prev) {
  sdxl_ctx* c = u->ctx;
  Sampler* S = u->sampler.get();
  Plan* P = u->plan.get();
  if (!S || !P) return fail(c, 5210, "sampler not initialised (call sdxl_sampler_begin)");
  if (t < 0 || t >= (int)u->alphas.size() || t_prev >= (int)u->alphas.size()) return fail(c, 5211, "timestep out of range");
  const double a = u->alphas[t];
  const double ap = t_prev >= 0 ? u->alphas[t_prev] : 1.0;
  int r = set_t(u, t);
  if (r) return r;
  if ((r = run_plan(u))) return r;
  KL(c, cfg_ddim_launch(c->stream, P->eps, P->eps_ld, S->Bimg, u->cfg.in_channels, S->h * S->w, S->nfwd == 2, S->guidance,
                        (float)sqrt(a), (float)sqrt(1.0 - a), (float)sqrt(ap), (float)sqrt(1.0 - ap), P->x_in, nullptr));
  return 0;
}

extern "C" int sdxl_sampler_begin(sdxl_unet* u, const sdxl_conditioning* cond, double guidance_scale) {
  if (!u) return -1;
  CU(u->ctx, cudaSetDevice(u->ctx->device));
  return sampler_begin(u, cond, guidance_scale);
}
extern "C" int sdxl_sampler_step(sdxl_unet* u, int t, int t_prev) {
  if (!u) return -1;
  CU(u->ctx, cudaSetDevice(u->ctx->device));
  return sampler_step(u, t, t_prev);
}
extern "C" int sdxl_sampler_set_latent(sdxl_unet* u, const float* latent, int on_host) {
  if (!u || !u->sampler || !u->plan) return -1;
  sdxl_ctx* c = u->ctx;
  CU(c, cudaSetDevice(c->device));
  CU(c, cudaMemcpyAsync(u->plan->x_in, latent, u->sampler->latent_elems * 4, on_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice, c->stream));
  if (on_host) CU(c, cudaStreamSynchronize(c->stream));
  return 0;
}
extern "C" int sdxl_sampler_get_latent(sdxl_unet* u, float* latent, int on_host) {
  if (!u || !u->sampler || !u->plan) return -1;
  sdxl_ctx* c = u->ctx;
  CU(c, cudaSetDevice(c->device));
  CU(c, cudaMemcpyAsync(latent, u->plan->x_in, u->sampler->latent_elems * 4, on_host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, c->stream));
  if (on_host) CU(c, cudaStreamSynchronize(c->stream));
  return 0;
}
extern "C" int sdxl_sampler_step_host(sdxl_unet* u, int t, int t_prev, float* latent_host) {
  if (!u || !u->sampler || !u->plan || !latent_host) return -1;
  sdxl_ctx* c = u->ctx;
  CU(c, cudaSetDevice(c->device));
  Sampler* S = u->sampler.get();
  const size_t bytes = S->latent_elems * 4;
  memcpy(S->host_stage, latent_host, bytes);  // caller memory may be pageable: stage through pinned
  CU(c, cudaMemcpyAsync(u->plan->x_in, S->host_stage, bytes, cudaMemcpyHostToDevice, c->stream));
  int r = sampler_step(u, t, t_prev);
  if (r) return r;
  CU(c, cudaMemcpyAsync(S->host_stage, u->plan->x_in, bytes, cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  memcpy(latent_host, S->host_stage, bytes);
  return 0;
}
extern "C" int sdxl_randn(sdxl_ctx* c, float* out, size_t n, uint64_t seed, uint64_t subsequence) {
  if (!c || !out) return -1;
  CU(c, cudaSetDevice(c->device));
  KL(c, randn_launch(c->stream, out, n, seed, subsequence));
  return 0;
}

extern "C" int sdxl_sample_latent(sdxl_unet* u, const sdxl_conditioning* cond, double guidance_scale, int n_steps,
                                  int step_start, const float* init_latent, const float* noise, int n_noise, uint64_t seed,
                                  const float* inpaint_ref, const uint8_t* inpaint_mask, float* latent_out) {
  if (!u || !cond || !latent_out) return -1;
  sdxl_ctx* c = u->ctx;
  CU(c, cudaSetDevice(c->device));
  const int total = u->cfg.n_steps;
  if (n_steps < 1 || n_steps > total) return fail(c, 5220, "n_steps must be in [1,%d]", total);
  if (step_start < 0 || step_start >= total) return fail(c, 5221, "bad step_start");
  if ((inpaint_ref == nullptr) != (inpaint_mask == nullptr)) return fail(c, 5222, "inpaint_ref and inpaint_mask must be given together");
  if (step_start > 0 && !init_latent) return fail(c, 5223, "refine (step_start>0) needs init_latent");
  int r = sampler_begin(u, cond, guidance_scale);
  if (r) return r;
  Sampler* S = u->sampler.get();
  Plan* P = u->plan.get();
  const size_t lat = S->latent_elems, bytes = lat * 4;
  const cudaMemcpyKind in_kind = cond->on_host ? cudaMemcpyHostToDevice : cudaMemcpyDeviceToDevice;
  const int step_size = total / n_steps;      // mod.rs:400
  const int t_begin = total - step_start;     // mod.rs:404
  int noise_used = 0;
  uint64_t subseq = 0;
  auto next_noise = [&](float* dst) -> int {  // injected noise first, then the seeded stream
    if (noise && noise_used < n_noise) {
      CU(c, cudaMemcpyAsync(dst, noise + (size_t)noise_used * lat, bytes, in_kind, c->stream));
      noise_used++;
      return 0;
    }
    KL(c, randn_launch(c->stream, dst, lat, seed, subseq++));
    return 0;
  };
  // initial latent
  if (init_latent) CU(c, cudaMemcpyAsync(P->x_in, init_latent, bytes, in_kind, c->stream));
  else if ((r = next_noise(P->x_in))) return r;
  if (step_start > 0) {
    // refine_latent entry (mod.rs:363-367): x = x*sqrt(a_t0) + noise*sqrt(1-a_t0), t0 = n_steps_total - step_start
    const double a0 = u->alphas[t_begin];
    if ((r = next_noise(S->noise))) return r;
    KL(c, axpby_launch(c->stream, P->x_in, S->noise, lat, (float)sqrt(a0), (float)sqrt(1.0 - a0)));
  }
  if (inpaint_ref) {
    CU(c, cudaMemcpyAsync(S->ref, inpaint_ref, bytes, in_kind, c->stream));
    CU(c, cudaMemcpyAsync(S->mask, inpaint_mask, lat, in_kind, c->stream));
  }
  // for t in (0..t_begin).rev().step_by(step_size)   (mod.rs:406, 452)
  for (int t = t_begin - 1; t >= 0; t -= step_size) {
    const int t_prev = (t >= step_size) ? t - step_size : -1;
    if (inpaint_ref) {
      const double a = u->alphas[t];
      if ((r = next_noise(S->noise))) return r;
      KL(c, inpaint_blend_launch(c->stream, P->x_in, S->ref, S->noise, S->mask, lat, S->nfwd, (float)sqrt(a), (float)sqrt(1.0 - a), nullptr));
    }
    if ((r = sampler_step(u, t, t_prev))) return r;
  }
  CU(c, cudaMemcpyAsync(latent_out, P->x_in, bytes, cond->on_host ? cudaMemcpyDeviceToHost : cudaMemcpyDeviceToDevice, c->stream));
  if (cond->on_host) CU(c, cudaStreamSynchronize(c->stream));
  return 0;
}

// ================================================================================================
// inpainting mask of the `sample` front end (reference src/bin/sample/main.rs:144-190)
// ================================================================================================
// Crop window in PIXELS -> Bool mask [1, n_channels, h/8... ] in latent coordinates: pixel coordinates are divided by
// scale = image height / latent height (integer division, main.rs:164-169), ones inside [top,bottom) x [left,right), zero padding
// outside, inverted by crop_out (main.rs:183-187). mask = 1 keeps the GENERATED latent (mask_where, stablediffusion/mod.rs:465).
// A negative bound means "not given" (the reference's Option defaults: 0 / image extent). Host memory, [n_channels, lat_h, lat_w].
extern "C" int sdxl_make_inpaint_mask(int img_w, int img_h, int lat_w, int lat_h, int crop_left, int crop_right, int crop_top,
                                      int crop_bottom, int crop_out, int n_channels, uint8_t* mask_out_host) {
  if (!mask_out_host || img_w <= 0 || img_h <= 0 || lat_w <= 0 || lat_h <= 0 || n_channels <= 0 || lat_h > img_h) return -1;
  const int l = crop_left < 0 ? 0 : crop_left, r = crop_right < 0 ? img_w : crop_right;
  const int t = crop_top < 0 ? 0 : crop_top, b = crop_bottom < 0 ? img_h : crop_bottom;
  // the reference asserts `right <= w && bottom <= h && left < right || top < bottom` (operator precedence makes it weaker than
  // intended); here every condition must hold
  if (r > img_w || b > img_h || l >= r || t >= b) return 5500;
  const int scale = img_h / lat_h;
  if (scale <= 0) return 5501;
  const int cl = l / scale, cr = r / scale, ct = t / scale, cb = b / scale;
  if (cr > lat_w || cb > lat_h) return 5502;
  for (int c = 0; c < n_channels; ++c)
    for (int y = 0; y < lat_h; ++y)
      for (int x = 0; x < lat_w; ++x) {
        const bool inside = y >= ct && y < cb && x >= cl && x < cr;
        mask_out_host[((size_t)c * lat_h + y) * lat_w + x] = (uint8_t)(inside != (crop_out != 0));
      }
  return 0;
}

extern "C" void sdxl_unet_destroy(sdxl_unet* u) {
  if (!u) return;
  cudaStreamSynchronize(u->ctx->stream);
  u->plan.reset();
  u->sampler.reset();
  u->warena.release();
  u->carena.release();
  if (u->t_dev) cudaFree(u->t_dev);
  if (u->t_pinned) cudaFreeHost(u->t_pinned);
  delete u;
}

// ================================================================================================
// operator-level entry points
// ================================================================================================

extern "C" int sdxl_qkv_attention(sdxl_ctx* c, const sdxl_half* q, const sdxl_half* k, const sdxl_half* v, const sdxl_half* mask,
                                  int B, int T, int S, int C, int n_head, sdxl_half* out) {
  if (!c || !q || !k || !v || !out) return -1;
  if (n_head < 1 || C != n_head * 64) return fail(c, 5301, "sdxl_qkv_attention: head dim must be 64 (C=%d, n_head=%d)", C, n_head);
  if (mask) {
    // additive [T,S] mask (the text encoders' causal mask, clip/mod.rs:88): short sequences, CUDA-core kernel
    KL(c, attention_small_launch(c->stream, (const __half*)q, C, 0, (const __half*)k, (const __half*)v, C, 0, 0, B, T, S, n_head,
                                 (const __half*)mask, 0, (__half*)out, C));
    return 0;
  }
  AttnParams p{};
  p.T = T; p.S = S; p.n_head = n_head; p.B = B;
  p.q_col0 = p.k_col0 = p.v_col0 = 0;
  p.out = (__half*)out; p.ldo = C;
  p.scale_log2e = (float)(1.4426950408889634 / sqrt(64.0));
  int r = make_tmap_rows(&p.tmQ, (const __half*)q, T, B, C, C);
  if (!r) r = make_tmap_rows(&p.tmK, (const __half*)k, S, B, C, C);
  if (!r) r = make_tmap_rows(&p.tmV, (const __half*)v, S, B, C, C);
  if (r) return fail(c, r, "tensor map creation failed");
  KL(c, attention_launch(c->stream, p));
  return 0;
}

extern "C" int sdxl_op_linear(sdxl_ctx* c, const sdxl_half* x, const sdxl_half* w, const sdxl_half* bias, const float* residual,
                              int M, int K, int N, int geglu, int out_f16, void* out) {
  if (!c || !x || !w || !out) return -1;
  if (K % 8) return fail(c, 5310, "sdxl_op_linear: K must be a multiple of 8");
  TmpBufs T(c->stream);
  const int Kpad = (K + 63) / 64 * 64;
  int gbn = 0;
  if (geglu) {
    gbn = geglu_bn_for(N / 2);
    if (!gbn || (N & 1)) return fail(c, 5311, "sdxl_op_linear: GEGLU width not tileable");
  }
  __half* wt = (__half*)T.get((size_t)N * Kpad * 2);
  float* b32 = bias ? (float*)T.get((size_t)N * 4) : nullptr;
  if (!wt || (bias && !b32)) return fail(c, 5312, "temporary allocation failed");
  KL(c, transpose_linear_launch(c->stream, (const __half*)w, K, N, wt, Kpad, 0, gbn));
  if (bias) KL(c, bias_to_f32_launch(c->stream, (const __half*)bias, N, b32, gbn, 0));
  IgemmParams p{};
  p.nseg = 1;
  p.seg[0] = {0, 0, 0, 0, Kpad / 64};
  p.out = out;
  p.out_f32 = geglu ? 0 : !out_f16;
  p.ldo = geglu ? N / 2 : N;
  p.bias = b32; p.bias_bstride = 0;
  p.res = geglu ? nullptr : residual; p.ldr = N;
  IgemmOperands o{(const __half*)x, 1, 1, M, K, K, nullptr, 0, 0, 0, 0, 0, wt, N, Kpad};
  int r = igemm_configure(p, o, M, 1, 1, geglu ? IGEMM_GEGLU : IGEMM_LINEAR, gbn);
  if (r) return fail(c, r, "igemm configuration failed");
  KL(c, igemm_launch(c->stream, p));
  return 0;
}

extern "C" int sdxl_op_conv2d(sdxl_ctx* c, const float* x, const sdxl_half* w, const sdxl_half* bias, int B, int H, int W, int Cin,
                              int Cout, int ksize, int stride, int upsample, float* out) {
  if (!c || !x || !w || !out) return -1;
  if ((ksize != 1 && ksize != 3) || (stride != 1 && stride != 2) || (stride == 2 && (upsample || ksize != 3)))
    return fail(c, 5320, "sdxl_op_conv2d: unsupported ksize/stride/upsample combination");
  if (Cin % 8) return fail(c, 5321, "sdxl_op_conv2d: Cin must be a multiple of 8");
  TmpBufs T(c->stream);
  const int Ipad = (Cin + 63) / 64 * 64, Ktot = ksize * ksize * Ipad;
  __half* wt = (__half*)T.get((size_t)Cout * Ktot * 2);
  float* b32 = bias ? (float*)T.get((size_t)Cout * 4) : nullptr;
  const int Hi = upsample ? 2 * H : H, Wi = upsample ? 2 * W : W;  // conv input extent
  __half* a16 = (__half*)T.get((size_t)B * Hi * Wi * Cin * 2);
  if (!wt || !a16 || (bias && !b32)) return fail(c, 5322, "temporary allocation failed");
  KL(c, repack_conv_launch(c->stream, (const __half*)w, Cout, Cin, ksize, ksize, wt, Ktot, 0, Ipad));
  if (bias) KL(c, bias_to_f32_launch(c->stream, (const __half*)bias, Cout, b32, 0, 0));
  IgemmParams p{};
  int Ho = Hi, Wo = Wi;
  ActView a{a16, B, Hi, Wi, Cin};
  p.nseg = 0;
  if (stride == 2) {
    if ((H & 1) || (W & 1)) return fail(c, 5323, "sdxl_op_conv2d: stride 2 needs even H, W");
    KL(c, phase_split_launch(c->stream, x, B, H, W, Cin, a16));
    Ho = H / 2; Wo = W / 2;
    a = ActView{a16, 4 * B, Ho, Wo, Cin};
    for (int kh = 0; kh < 3; ++kh)
      for (int kw = 0; kw < 3; ++kw) {
        const int ph = (kh == 1) ? 0 : 1, pw = (kw == 1) ? 0 : 1;
        p.seg[p.nseg++] = {0, (int16_t)((kw == 0) ? -1 : 0), (int16_t)((kh == 0) ? -1 : 0), (int16_t)((ph * 2 + pw) * B), Ipad / 64};
      }
  } else {
    if (upsample) KL(c, upsample2x_launch(c->stream, x, B, H, W, Cin, a16));
    else KL(c, cast_f32_to_f16_launch(c->stream, x, (size_t)B * H * W * Cin, a16));
    const int pad = ksize / 2;
    for (int kh = 0; kh < ksize; ++kh)
      for (int kw = 0; kw < ksize; ++kw) p.seg[p.nseg++] = {0, (int16_t)(kw - pad), (int16_t)(kh - pad), 0, Ipad / 64};
  }
  p.out = out; p.out_f32 = 1; p.ldo = Cout;
  p.bias = b32; p.bias_bstride = 0; p.res = nullptr; p.ldr = 0;
  IgemmOperands o{a.p, a.Bn, a.H, a.W, a.C, a.C, nullptr, 0, 0, 0, 0, 0, wt, Cout, Ktot};
  int r = igemm_configure(p, o, Wo, Ho, B, IGEMM_LINEAR, 0);
  if (r) return fail(c, r, "igemm configuration failed");
  KL(c, igemm_launch(c->stream, p));
  return 0;
}

extern "C" int sdxl_op_group_norm(sdxl_ctx* c, const float* x1, int C1, const float* x2, int C2, int B, int HW, int n_group,
                                  const float* gamma, const float* beta, float eps, int silu, sdxl_half* out) {
  if (!c || !x1 || !gamma || !beta || !out) return -1;
  TmpBufs T(c->stream);
  float* part = (float*)T.get(gn_scratch_floats(B, n_group) * 4);
  if (part && gn_scratch_init(c->stream, part, B, n_group)) return fail(c, 5007, "GroupNorm scratch init failed");
  if (!part) return fail(c, 5330, "temporary allocation failed");
  GnParams p{x1, C1, x2, x2 ? C2 : 0, B, HW, n_group, gamma, beta, eps, silu, (__half*)out, nullptr, part, 0};
  KL(c, gn_launch(c->stream, p));
  c->launches++;
  return 0;
}
extern "C" int sdxl_op_layer_norm(sdxl_ctx* c, const float* x, const float* gamma, const float* beta, float eps, int rows, int C,
                                  sdxl_half* out) {
  if (!c || !x || !gamma || !beta || !out) return -1;
  KL(c, layernorm_launch(c->stream, x, gamma, beta, eps, rows, C, (__half*)out));
  return 0;
}
extern "C" int sdxl_op_timestep_embedding(sdxl_ctx* c, const int32_t* t_host, int n, int dim, int max_period, float* out) {
  if (!c || !t_host || !out || n < 1 || (dim & 1)) return -1;
  TmpBufs T(c->stream);
  int* td = (int*)T.get((size_t)n * 4);
  if (!td) return fail(c, 5340, "temporary allocation failed");
  CU(c, cudaMemcpyAsync(td, t_host, (size_t)n * 4, cudaMemcpyHostToDevice, c->stream));
  KL(c, timestep_embedding_launch(c->stream, td, n, dim, (float)max_period, out));
  CU(c, cudaStreamSynchronize(c->stream));  // t_host is pageable caller memory
  return 0;
}

// Diagnostics: clock64 stamps of CTA 0 of one attention launch on synthetic data (tools/attn_timeline.py).
// stamps_host[3][256][4]: role 0/1 = softmax slot A/B (one warp's lane 0): {S ready, exp phase done, P handed over, item written
// back}; role 2 = MMA issuer: {P_A ready, P V_A + Q K_A issued, P_B ready, P V_B + Q K_B issued}; per key block, in clocks.
extern "C" int sdxl_dbg_attention_timeline(sdxl_ctx* c, int B, int T, int S, int n_head, long long* stamps_host) {
  if (!c || !stamps_host) return -1;
  CU(c, cudaSetDevice(c->device));
  TmpBufs Tm(c->stream);
  const int C = n_head * 64;
  __half* q = (__half*)Tm.get((size_t)B * T * C * 2);
  __half* k = (__half*)Tm.get((size_t)B * S * C * 2);
  __half* v = (__half*)Tm.get((size_t)B * S * C * 2);
  __half* o = (__half*)Tm.get((size_t)B * T * C * 2);
  long long* dbg = (long long*)Tm.get(3 * 1024 * 8);
  if (!q || !k || !v || !o || !dbg) return fail(c, 5400, "temporary allocation failed");
  CU(c, cudaMemsetAsync(q, 0, (size_t)B * T * C * 2, c->stream));
  CU(c, cudaMemsetAsync(k, 0, (size_t)B * S * C * 2, c->stream));
  CU(c, cudaMemsetAsync(v, 0, (size_t)B * S * C * 2, c->stream));
  CU(c, cudaMemsetAsync(dbg, 0, 3 * 1024 * 8, c->stream));
  AttnParams p{};
  p.T = T; p.S = S; p.n_head = n_head; p.B = B;
  p.out = o; p.ldo = C;
  p.scale_log2e = (float)(1.4426950408889634 / sqrt(64.0));
  int r = make_tmap_rows(&p.tmQ, q, T, B, C, C);
  if (!r) r = make_tmap_rows(&p.tmK, k, S, B, C, C);
  if (!r) r = make_tmap_rows(&p.tmV, v, S, B, C, C);
  if (r) return fail(c, r, "tensor map creation failed");
  for (int i = 0; i < 3; ++i) KL(c, attention_launch(c->stream, p));
  p.dbg = dbg;
  KL(c, attention_launch(c->stream, p));
  CU(c, cudaMemcpyAsync(stamps_host, dbg, 3 * 1024 * 8, cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  return 0;
}

// Diagnostics: in-kernel timeline (%globaltimer, ns) of CTA 0 of one igemm launch on a synthetic [M,K]x[K,N] problem.
// stamps_host[0..6] = prologue done, dependencies resolved, first operands landed, first accumulator complete,
// first epilogue done, producer done, all roles done; stamps_host[7] = CUDA-event duration of the launch in ns.
// Launch ramp / drain of back-to-back launches of one GEMM (programmatic dependent launch, eager): every CTA stamps its entry, the end of
// its prologue, the moment its dependencies are resolved and its exit. out_host: n_launch x 8 = {first, last} x {entry, prologue done,
// dependencies resolved, exit} in ns relative to the first entry of launch 0; out_host[n_launch * 8] = grid size.
extern "C" int sdxl_dbg_igemm_gaps(sdxl_ctx* c, int M, int K, int N, int with_residual, int n_launch, int64_t* out_host) {
  if (!c || !out_host || n_launch < 1 || n_launch > 16) return -1;
  TmpBufs T(c->stream);
  const int Kpad = (K + 63) / 64 * 64;
  __half* x = (__half*)T.get((size_t)M * K * 2);
  __half* w = (__half*)T.get((size_t)N * Kpad * 2);
  float* bias = (float*)T.get((size_t)N * 4);
  float* res = (float*)T.get((size_t)M * N * 4);
  void* out = T.get((size_t)M * N * 4);
  const size_t per = 256 * 8;   // stamps per launch (grid <= 256 CTAs)
  unsigned long long* dbg = (unsigned long long*)T.get((size_t)n_launch * per * 8);
  if (!x || !w || !bias || !res || !out || !dbg) return fail(c, 5400, "temporary allocation failed");
  CU(c, cudaMemsetAsync(x, 0, (size_t)M * K * 2, c->stream));
  CU(c, cudaMemsetAsync(w, 0, (size_t)N * Kpad * 2, c->stream));
  CU(c, cudaMemsetAsync(bias, 0, (size_t)N * 4, c->stream));
  CU(c, cudaMemsetAsync(res, 0, (size_t)M * N * 4, c->stream));
  CU(c, cudaMemsetAsync(dbg, 0, (size_t)n_launch * per * 8, c->stream));
  IgemmParams p{};
  p.nseg = 1;
  p.seg[0] = {0, 0, 0, 0, Kpad / 64};
  p.out = out; p.out_f32 = 1; p.ldo = N;
  p.bias = bias; p.bias_bstride = 0;
  p.res = with_residual ? res : nullptr; p.ldr = N;
  IgemmOperands o{x, 1, 1, M, K, K, nullptr, 0, 0, 0, 0, 0, w, N, Kpad};
  int r = igemm_configure(p, o, M, 1, 1, IGEMM_LINEAR, 0);
  if (r) return fail(c, r, "igemm configuration failed");
  if (!p.pair) return fail(c, 5401, "sdxl_dbg_igemm_gaps: shape does not use the 2-CTA kernel");
  for (int i = 0; i < 3; ++i) KL(c, igemm_launch(c->stream, p));
  for (int i = 0; i < n_launch; ++i) {
    p.dbg_all = dbg + (size_t)i * per;
    KL(c, igemm_launch(c->stream, p));
  }
  std::vector<unsigned long long> h((size_t)n_launch * per);
  CU(c, cudaMemcpyAsync(h.data(), dbg, h.size() * 8, cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  int grid = 0;
  while (grid < 256 && h[(size_t)grid * 8] != 0) ++grid;
  const unsigned long long t0 = [&] { unsigned long long m = ~0ull; for (int b = 0; b < grid; ++b) m = std::min(m, h[(size_t)b * 8]); return m; }();
  for (int i = 0; i < n_launch; ++i)
    for (int k = 0; k < 8; ++k) {
      unsigned long long lo = ~0ull, hi = 0;
      for (int b = 0; b < grid; ++b) {
        const unsigned long long v = h[(size_t)i * per + (size_t)b * 8 + k];
        lo = std::min(lo, v); hi = std::max(hi, v);
      }
      out_host[i * 16 + 2 * k] = (int64_t)(lo - t0);
      out_host[i * 16 + 2 * k + 1] = (int64_t)(hi - t0);
    }
  out_host[n_launch * 16] = grid;
  return 0;
}

extern "C" int sdxl_dbg_igemm_timeline(sdxl_ctx* c, int M, int K, int N, int geglu, int with_residual, uint64_t* stamps_host) {
  if (!c || !stamps_host) return -1;
  TmpBufs T(c->stream);
  const int Kpad = (K + 63) / 64 * 64;
  int gbn = geglu ? geglu_bn_for(N / 2) : 0;
  __half* x = (__half*)T.get((size_t)M * K * 2);
  __half* w = (__half*)T.get((size_t)N * Kpad * 2);
  float* bias = (float*)T.get((size_t)N * 4);
  float* res = (float*)T.get((size_t)M * N * 4);
  void* out = T.get((size_t)M * N * 4);
  unsigned long long* dbg = (unsigned long long*)T.get(16 * 8);
  if (!x || !w || !bias || !res || !out || !dbg) return fail(c, 5400, "temporary allocation failed");
  CU(c, cudaMemsetAsync(x, 0, (size_t)M * K * 2, c->stream));
  CU(c, cudaMemsetAsync(w, 0, (size_t)N * Kpad * 2, c->stream));
  CU(c, cudaMemsetAsync(bias, 0, (size_t)N * 4, c->stream));
  CU(c, cudaMemsetAsync(res, 0, (size_t)M * N * 4, c->stream));
  CU(c, cudaMemsetAsync(dbg, 0, 128, c->stream));
  IgemmParams p{};
  p.nseg = 1;
  p.seg[0] = {0, 0, 0, 0, Kpad / 64};
  p.out = out; p.out_f32 = geglu ? 0 : 1; p.ldo = geglu ? N / 2 : N;
  p.bias = bias; p.bias_bstride = 0;
  p.res = (geglu || !with_residual) ? nullptr : res; p.ldr = N;
  IgemmOperands o{x, 1, 1, M, K, K, nullptr, 0, 0, 0, 0, 0, w, N, Kpad};
  int r = igemm_configure(p, o, M, 1, 1, geglu ? IGEMM_GEGLU : IGEMM_LINEAR, gbn);
  if (r) return fail(c, r, "igemm configuration failed");
  cudaEvent_t e0, e1;
  CU(c, cudaEventCreate(&e0));
  CU(c, cudaEventCreate(&e1));
  if (getenv("SDXL_B200_DBG_MODE")) p.dbg_mode = atoi(getenv("SDXL_B200_DBG_MODE"));
  if (getenv("SDXL_B200_DBG_NST")) p.nstages = atoi(getenv("SDXL_B200_DBG_NST"));
  for (int i = 0; i < 3; ++i) KL(c, igemm_launch(c->stream, p));
  p.dbg = dbg;
  CU(c, cudaEventRecord(e0, c->stream));
  KL(c, igemm_launch(c->stream, p));
  CU(c, cudaEventRecord(e1, c->stream));
  unsigned long long hostbuf[16];
  CU(c, cudaMemcpyAsync(hostbuf, dbg, 128, cudaMemcpyDeviceToHost, c->stream));
  CU(c, cudaStreamSynchronize(c->stream));
  float ms = 0;
  cudaEventElapsedTime(&ms, e0, e1);
  for (int i = 0; i < 7; ++i) stamps_host[i] = hostbuf[i];
  fprintf(stderr, "  epi block0: tmem_ld %llu ns, st.shared+sync %llu ns, phase2 %llu ns (since acc ready: %llu)\n",
          hostbuf[10] - hostbuf[9], hostbuf[11] - hostbuf[10], hostbuf[12] - hostbuf[11], hostbuf[9] - hostbuf[3]);
  stamps_host[7] = (uint64_t)(ms * 1e6);
  stamps_host[8] = (uint64_t)p.BN | ((uint64_t)p.pair << 16) | ((uint64_t)p.CM << 20) | ((uint64_t)p.CN << 24) | ((uint64_t)p.nstages << 28);
  cudaEventDestroy(e0);
  cudaEventDestroy(e1);
  return 0;
}

// ================================================================================================
// Diagnostics: the plans' own launch builders on caller data (tests/test_plan_kernels_gpu.py)
// ================================================================================================
// Builds a scratch plan the way the UNet / VAE / CLIP plans are built: a measure pass sizes one arena for the weights
// (re-laid out from `pack` by the Loader helpers) and the plan's scratch, the real pass loads and records the ops, and the
// plan's op executor runs them once (eager). `body(L, B)` loads its weights and records its ops; it runs in both passes.
template <typename F>
static int run_scratch_plan(sdxl_ctx* c, const void* pack, size_t pack_bytes, int Bf, int32_t* cfg_out, int cfg_cap, F body) {
  CU(c, cudaSetDevice(c->device));
  PackView pv;
  std::vector<uint8_t> table;
  TmpBufs T(c->stream);
  if (pack) {
    int r = parse_pack(c, pack, pack_bytes, 0, pv, table);
    if (r) return r;
    uint8_t* dev = (uint8_t*)T.get(pack_bytes);
    if (!dev) return fail(c, 5410, "temporary allocation failed");
    CU(c, cudaMemcpyAsync(dev, pack, pack_bytes, cudaMemcpyHostToDevice, c->stream));
    pv.dev = dev;
  }
  Plan P;
  P.Bf = P.Bx = Bf;
  Arena meas;
  meas.measure = true;
  for (int pass = 0; pass < 2; ++pass) {
    Arena* A = pass ? &P.arena : &meas;
    if (pass && P.arena.init(meas.off + (1 << 20))) return fail(c, 5411, "cannot allocate %zu bytes of workspace", meas.off);
    P.ops.clear();
    Loader L{nullptr, c, &pv, A, c->stream};
    PlanBuilder B{c, &P, A, Bf};
    B.gn_partial = B.buf<float>(gn_scratch_floats(Bf, 32));
    if (pass && B.gn_partial && gn_scratch_init(c->stream, B.gn_partial, Bf, 32)) return fail(c, 5007, "GroupNorm scratch init failed");
    body(L, B);
    if (L.err) return L.err;
    if (B.err) return B.err;
  }
  int r = run_plan_ops(c, &P);
  if (r) return r;
  CU(c, cudaStreamSynchronize(c->stream));
  // the configuration every igemm launch ran with (after igemm_launch's own adjustments)
  int n = 0;
  for (const Op& op : P.ops) {
    if (op.kind != OP_IGEMM) continue;
    if (cfg_out && n < cfg_cap) {
      const IgemmParams& g = op.ig;
      const int32_t v[SDXL_DBG_CFG_FIELDS] = {g.pair, g.CM, g.CN, g.a_split_dim, g.BN, g.nstages, g.epi_tma, g.epi_box_bytes};
      memcpy(cfg_out + (size_t)n * SDXL_DBG_CFG_FIELDS, v, sizeof v);
    }
    ++n;
  }
  for (int i = n; cfg_out && i < cfg_cap; ++i)
    for (int j = 0; j < SDXL_DBG_CFG_FIELDS; ++j) cfg_out[(size_t)i * SDXL_DBG_CFG_FIELDS + j] = -1;
  return 0;
}

extern "C" int sdxl_dbg_plan_gemm(sdxl_ctx* c, int kind, const void* pack, size_t pack_bytes, int B, int H, int W, int Cin,
                                  int Cout, int C2, const void* x, const void* x2, const float* bias_rows, int bias_ld,
                                  int bias_off, const float* residual, void* out, int ldo, int32_t* cfg_out, int cfg_cap) {
  if (!c || !pack || !x || !out || B < 1 || H < 1 || W < 1) return fail(c, -1, "sdxl_dbg_plan_gemm: bad argument");
  switch (kind) {
    case SDXL_DBG_CONV3:
      return run_scratch_plan(c, pack, pack_bytes, B, cfg_out, cfg_cap, [&](Loader& L, PlanBuilder& P) {
        const Conv cv = C2 ? L.conv("conv", Cin, Cout, 3, "skip", C2) : L.conv("conv", Cin, Cout, 3);
        if (L.err) return;
        ActView a{(const __half*)x, B, H, W, Cin}, sk{(const __half*)x2, B, H, W, C2};
        P.conv3(a, C2 ? &sk : nullptr, cv, (float*)out, bias_rows ? bias_rows + bias_off : cv.b, bias_rows ? bias_ld : 0, residual);
      });
    case SDXL_DBG_UPCONV:
      return run_scratch_plan(c, pack, pack_bytes, B, cfg_out, cfg_cap, [&](Loader& L, PlanBuilder& P) {
        const Conv cv = L.upconv("conv", Cin, Cout);
        __half* x16 = P.buf<__half>((size_t)B * H * W * Cin);
        if (!L.err) P.upconv((const float*)x, B, H, W, cv, x16, (float*)out);
      });
    case SDXL_DBG_HEAD_HILO:
      return run_scratch_plan(c, pack, pack_bytes, B, cfg_out, cfg_cap, [&](Loader& L, PlanBuilder& P) {
        const Norm n = L.norm("norm", Cin);
        const Conv cv = L.conv("conv", Cin, Cout, 3);
        __half* w2 = L.dup_k(cv);
        __half* y = P.buf<__half>((size_t)B * H * W * Cin);
        __half* y_lo = P.buf<__half>((size_t)B * H * W * Cin);
        if (!L.err) P.head_hilo((const float*)x, Cin, H, W, n, cv, w2, y, y_lo, (float*)out, ldo);
      });
    case SDXL_DBG_PADDED_S2:
      if ((H & 1) || (W & 1)) return fail(c, 5412, "sdxl_dbg_plan_gemm: PaddedConv2d needs even H, W");
      return run_scratch_plan(c, pack, pack_bytes, B, cfg_out, cfg_cap, [&](Loader& L, PlanBuilder& P) {
        const Conv cv = L.conv("conv", Cin, Cout, 3);
        __half* ph = P.buf<__half>((size_t)B * H * W * Cin);
        if (!L.err) P.padded_conv_s2((const float*)x, B, H, W, cv, ph, (float*)out);
      });
    case SDXL_DBG_LINEAR:
    case SDXL_DBG_LINEAR_F16:
    case SDXL_DBG_GEGLU:
      return run_scratch_plan(c, pack, pack_bytes, 1, cfg_out, cfg_cap, [&](Loader& L, PlanBuilder& P) {
        const bool geglu = kind == SDXL_DBG_GEGLU;
        const int gbn = geglu ? geglu_bn_for(Cout / 2) : 0;
        if (geglu && (!gbn || (Cout & 1))) { L.err = fail(c, 5413, "sdxl_dbg_plan_gemm: GEGLU width %d not tileable", Cout); return; }
        const Lin lin = L.linear("lin", Cin, Cout, true, gbn);
        if (!L.err)
          P.linear((const __half*)x, W, lin, geglu ? IGEMM_GEGLU : IGEMM_LINEAR, out, kind == SDXL_DBG_LINEAR, ldo,
                   geglu ? nullptr : residual, ldo);
      });
  }
  return fail(c, 5414, "sdxl_dbg_plan_gemm: unknown kind %d", kind);
}

extern "C" int sdxl_dbg_plan_group_norm(sdxl_ctx* c, const void* pack, size_t pack_bytes, const float* x1, int C1, const float* x2,
                                        int C2, int B, int HW, int silu, sdxl_half* y, sdxl_half* raw, sdxl_half* y_lo) {
  if (!c || !pack || !x1 || !y || B < 1 || HW < 1) return fail(c, -1, "sdxl_dbg_plan_group_norm: bad argument");
  return run_scratch_plan(c, pack, pack_bytes, B, nullptr, 0, [&](Loader& L, PlanBuilder& P) {
    const Norm n = L.norm("norm", C1 + (x2 ? C2 : 0));
    if (!L.err) P.gn(x1, C1, x2, x2 ? C2 : 0, HW, n, silu, (__half*)y, (__half*)raw, (__half*)y_lo);
  });
}

extern "C" int sdxl_dbg_plan_attention(sdxl_ctx* c, int small, const sdxl_half* q, int q_pitch, int q_col0, const sdxl_half* kv,
                                       int kv_pitch, int k_col0, int v_col0, int B, int T, int S, int n_head, const sdxl_half* mask,
                                       int causal, sdxl_half* out, int ldo) {
  if (!c || !q || !kv || !out || B < 1 || T < 1 || S < 1 || n_head < 1) return fail(c, -1, "sdxl_dbg_plan_attention: bad argument");
  return run_scratch_plan(c, nullptr, 0, B, nullptr, 0, [&](Loader&, PlanBuilder& P) {
    if (small)
      P.attn_small((const __half*)q, q_pitch, q_col0, (const __half*)kv, kv_pitch, k_col0, v_col0, T, S, n_head, (const __half*)mask,
                   causal, (__half*)out, ldo);
    else
      P.attn((const __half*)q, q_pitch, q_col0, (const __half*)kv, kv_pitch, k_col0, v_col0, T, S, n_head, (__half*)out, ldo,
             (float)(1.4426950408889634 / sqrt(64.0)));
  });
}

extern "C" int sdxl_dbg_plan_vae_attention(sdxl_ctx* c, const sdxl_half* q, const sdxl_half* k, const sdxl_half* v, int T, int C,
                                           float* scores, sdxl_half* probs, sdxl_half* vT, sdxl_half* out, int32_t* cfg_out,
                                           int cfg_cap) {
  if (!c || !q || !k || !v || !scores || !probs || !vT || !out) return fail(c, -1, "sdxl_dbg_plan_vae_attention: null argument");
  if (T < 64 || T % 64 || C % 64) return fail(c, 5415, "sdxl_dbg_plan_vae_attention: T and C must be multiples of 64");
  return run_scratch_plan(c, nullptr, 0, 1, cfg_out, cfg_cap, [&](Loader&, PlanBuilder& P) {
    P.attn_single_head((const __half*)q, (const __half*)k, (const __half*)v, T, C, scores, (__half*)probs, (__half*)vT, (__half*)out);
  });
}
