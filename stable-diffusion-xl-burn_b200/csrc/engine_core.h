// Internals shared by the model front ends of libsdxl_b200.so (engine.cu: UNet + sampler + op-level API, vae.cu: latent
// decoder / encoder, clip.cu: text encoders): context, device arena, weight-pack parsing and re-layout helpers, and the
// launch plan (a flat list of kernel launches with pre-built TMA descriptors, run eagerly once and then replayed as a CUDA
// graph). Everything here has internal linkage; the public boundary is include/sdxl_b200.h.
#pragma once
#include "../../include/sdxl_b200.h"
#include "kernels.h"

#include <math.h>
#include <nvtx3/nvToolsExt.h>
#include <stdarg.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>

#include <map>
#include <memory>
#include <string>
#include <vector>

using namespace sdxl;

// ================================================================================================
// context
// ================================================================================================
struct sdxl_ctx {
  int device = 0;
  cudaStream_t stream = nullptr;
  bool own_stream = false;
  int num_sms = 148;
  std::string err;
  uint64_t launches = 0;
};

static int fail(sdxl_ctx* c, int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof buf, fmt, ap);
  va_end(ap);
  if (c) c->err = buf;
  return code ? code : -1;
}
#define CU(ctx, expr)                                                                         \
  do {                                                                                        \
    cudaError_t _e = (expr);                                                                  \
    if (_e != cudaSuccess)                                                                    \
      return fail(ctx, (int)_e, "%s failed: %s (%s:%d)", #expr, cudaGetErrorString(_e), __FILE__, __LINE__); \
  } while (0)
#define KL(ctx, expr)                                                                         \
  do {                                                                                        \
    int _e = (expr);                                                                          \
    if (_e) return fail(ctx, _e, "%s failed with %d%s%s (%s:%d)", #expr, _e, _e < 1000 ? ": " : "", \
                        _e < 1000 ? cudaGetErrorString((cudaError_t)_e) : "", __FILE__, __LINE__); \
    (ctx)->launches++;                                                                        \
  } while (0)

// ================================================================================================
// device arena (bump allocator over one cudaMalloc)
// ================================================================================================
struct Arena {
  uint8_t* base = nullptr;
  size_t cap = 0, off = 0;
  bool measure = false;  // dry run: only count
  int init(size_t bytes) {
    release();
    if (cudaMalloc((void**)&base, bytes) != cudaSuccess) return 1;
    cap = bytes;
    off = 0;
    return 0;
  }
  void release() {
    if (base) cudaFree(base);
    base = nullptr;
    cap = off = 0;
  }
  void* alloc(size_t bytes) {
    const size_t a = (off + 1023) & ~size_t(1023);
    if (!measure && a + bytes > cap) return nullptr;
    off = a + bytes;
    return measure ? (void*)(uintptr_t)(0x1000 + a) : (void*)(base + a);
  }
  template <typename T>
  T* get(size_t n) { return (T*)alloc(n * sizeof(T)); }
};

// ================================================================================================
// weight pack
// ================================================================================================
#pragma pack(push, 1)
struct PackHeader {
  char magic[8];  // "SDXLPK01"
  uint32_t n_tensors;
  uint32_t reserved;
  uint64_t data_offset;
};
struct PackEntry {
  char name[120];
  uint32_t dtype;  // 0 = f16, 1 = f32
  uint32_t ndim;
  uint64_t shape[4];
  uint64_t offset;  // from pack start
  uint64_t nbytes;
};
#pragma pack(pop)

struct PackView {
  const uint8_t* dev = nullptr;  // pack bytes in device memory
  std::map<std::string, PackEntry> t;
  const PackEntry* find(const std::string& n) const {
    auto it = t.find(n);
    return it == t.end() ? nullptr : &it->second;
  }
};

// ================================================================================================
// layer records + loader
// ================================================================================================
struct Lin {
  __half* w = nullptr; float* b = nullptr; int K = 0, Kpad = 0, N = 0, geglu_bn = 0;
};
struct Conv {
  __half* w = nullptr; float* b = nullptr; int I = 0, O = 0, ks = 0, Ipad = 0, I2 = 0, I2pad = 0, Ktot = 0;
  __half* wup = nullptr;  // upconv(): four 2x2 phase kernels [4][O][4*Ipad] of a 3x3 conv that follows a nearest-2x upsample
};
struct Norm { float* g = nullptr; float* b = nullptr; int C = 0; float eps = 1e-5f; };

struct Loader {
  void* owner;  // unused by the helpers; kept so that front ends can tag a loader
  sdxl_ctx* c;
  const PackView* pv;
  Arena* A;
  cudaStream_t st;
  int err = 0;

  const PackEntry* need(const std::string& name, int ndim) {
    const PackEntry* e = pv->find(name);
    if (!e) { err = fail(c, 4001, "weight pack: missing tensor '%s'", name.c_str()); return nullptr; }
    if (e->dtype != 0) { err = fail(c, 4002, "weight pack: tensor '%s' must be f16", name.c_str()); return nullptr; }
    if ((int)e->ndim != ndim) { err = fail(c, 4003, "weight pack: tensor '%s' has ndim %u, expected %d", name.c_str(), e->ndim, ndim); return nullptr; }
    return e;
  }
  const __half* ptr(const PackEntry* e) { return (const __half*)(pv->dev + e->offset); }
  bool has(const std::string& name) { return pv->find(name) != nullptr; }

  float* vec_f32(const std::string& name, int expectN, int geglu_bn = 0) {
    const PackEntry* e = need(name, 1);
    if (!e) return nullptr;
    if ((int)e->shape[0] != expectN) { err = fail(c, 4004, "weight pack: '%s' has %llu elements, expected %d", name.c_str(), (unsigned long long)e->shape[0], expectN); return nullptr; }
    float* d = A->get<float>(expectN);
    if (!d) { err = fail(c, 4005, "weight arena exhausted"); return nullptr; }
    if (!A->measure) { int r = bias_to_f32_launch(st, ptr(e), expectN, d, geglu_bn, 0); if (r) err = fail(c, r, "bias_to_f32 failed"); }
    return d;
  }
  // Linear stored [in,out]; produce K-major [N,Kpad]. Rows may be a slice of a fused matrix.
  int lin_into(const std::string& path, __half* dst, int Kpad, int row0, int expectK, int expectN, int geglu_bn) {
    const PackEntry* e = need(path + "/weight", 2);
    if (!e) return err;
    if ((int)e->shape[0] != expectK || (int)e->shape[1] != expectN)
      return err = fail(c, 4006, "weight pack: '%s/weight' is [%llu,%llu], expected [%d,%d]", path.c_str(),
                        (unsigned long long)e->shape[0], (unsigned long long)e->shape[1], expectK, expectN);
    if (!A->measure) { int r = transpose_linear_launch(st, ptr(e), expectK, expectN, dst, Kpad, row0, geglu_bn); if (r) return err = fail(c, r, "transpose_linear failed"); }
    return 0;
  }
  static int pad64(int k) { return (k + 63) / 64 * 64; }
  Lin linear(const std::string& path, int K, int N, bool bias, int geglu_bn = 0) {
    Lin L;
    L.K = K; L.N = N; L.Kpad = pad64(K); L.geglu_bn = geglu_bn;
    L.w = A->get<__half>((size_t)N * L.Kpad);
    if (!L.w) { err = fail(c, 4005, "weight arena exhausted"); return L; }
    if (lin_into(path, L.w, L.Kpad, 0, K, N, geglu_bn)) return L;
    if (bias) L.b = vec_f32(path + "/bias", N, geglu_bn);
    return L;
  }
  // 3x3 conv applied to a nearest-2x upsampled image, stored as its four 2x2 phase convolutions on the source image
  // (2.25x fewer MACs, no upsampled copy; elementwise.cu: repack_upconv_kernel)
  Conv upconv(const std::string& path, int I, int O) {
    Conv cv;
    cv.I = I; cv.O = O; cv.ks = 3; cv.Ipad = pad64(I); cv.Ktot = 4 * cv.Ipad;
    cv.wup = A->get<__half>((size_t)4 * O * cv.Ktot);
    if (!cv.wup) { err = fail(c, 4005, "weight arena exhausted"); return cv; }
    const PackEntry* e = need(path + "/weight", 4);
    if (!e) return cv;
    if ((int)e->shape[0] != O || (int)e->shape[1] != I || e->shape[2] != 3 || e->shape[3] != 3) {
      err = fail(c, 4007, "weight pack: '%s/weight' must be [%d,%d,3,3]", path.c_str(), O, I);
      return cv;
    }
    if (!A->measure) { int r = repack_upconv_launch(st, ptr(e), O, I, cv.wup, cv.Ipad); if (r) err = fail(c, r, "repack_upconv failed"); }
    cv.b = vec_f32(path + "/bias", O);
    return cv;
  }
  Norm norm(const std::string& path, int C) {
    Norm n;
    n.C = C;
    n.g = vec_f32(path + "/weight", C);
    n.b = vec_f32(path + "/bias", C);
    return n;
  }
  // conv OIHW -> [O, ks*ks*Ipad (+ I2pad)]
  // Opad > O: the matrix (and bias) get zero rows up to Opad so the GEMM's N is a multiple of 4 (cv.O = Opad).
  Conv conv(const std::string& path, int I, int O, int ks, const std::string& skip_path = "", int I2 = 0, int Opad = 0) {
    Conv cv;
    cv.I = I; cv.O = O; cv.ks = ks; cv.Ipad = pad64(I); cv.I2 = I2; cv.I2pad = I2 ? pad64(I2) : 0;
    cv.Ktot = ks * ks * cv.Ipad + cv.I2pad;
    const int rows = Opad > O ? Opad : O;
    cv.w = A->get<__half>((size_t)rows * cv.Ktot);
    if (!cv.w) { err = fail(c, 4005, "weight arena exhausted"); return cv; }
    if (rows > O && !A->measure && cudaMemsetAsync(cv.w, 0, (size_t)rows * cv.Ktot * sizeof(__half), st) != cudaSuccess) {
      err = fail(c, 4011, "memset failed");
      return cv;
    }
    const PackEntry* e = need(path + "/weight", 4);
    if (!e) return cv;
    if ((int)e->shape[0] != O || (int)e->shape[1] != I || (int)e->shape[2] != ks || (int)e->shape[3] != ks) {
      err = fail(c, 4007, "weight pack: '%s/weight' has shape [%llu,%llu,%llu,%llu], expected [%d,%d,%d,%d]", path.c_str(),
                 (unsigned long long)e->shape[0], (unsigned long long)e->shape[1], (unsigned long long)e->shape[2],
                 (unsigned long long)e->shape[3], O, I, ks, ks);
      return cv;
    }
    if (!A->measure) { int r = repack_conv_launch(st, ptr(e), O, I, ks, ks, cv.w, cv.Ktot, 0, cv.Ipad); if (r) err = fail(c, r, "repack_conv failed"); }
    if (rows > O) {
      const PackEntry* be = need(path + "/bias", 1);
      cv.b = A->get<float>(rows);
      if (!be || !cv.b || (int)be->shape[0] != O) { if (!err) err = fail(c, 4012, "weight pack: '%s/bias' missing or mis-sized", path.c_str()); return cv; }
      if (!A->measure) {
        int r = (int)cudaMemsetAsync(cv.b, 0, rows * sizeof(float), st);
        if (!r) r = bias_to_f32_launch(st, ptr(be), O, cv.b, 0, 0);
        if (r) err = fail(c, r, "padded bias failed");
      }
      cv.O = rows;
    } else {
      cv.b = vec_f32(path + "/bias", O);
    }
    if (I2) {
      const PackEntry* s = need(skip_path + "/weight", 4);
      if (!s) return cv;
      if ((int)s->shape[0] != O || (int)s->shape[1] != I2 || s->shape[2] != 1 || s->shape[3] != 1) { err = fail(c, 4008, "weight pack: '%s/weight' bad shape", skip_path.c_str()); return cv; }
      const PackEntry* sb = need(skip_path + "/bias", 1);
      if (!sb) return cv;
      if (!A->measure) {
        int r = repack_conv_launch(st, ptr(s), O, I2, 1, 1, cv.w, cv.Ktot, ks * ks * cv.Ipad, cv.I2pad);
        if (!r) r = bias_to_f32_launch(st, ptr(sb), O, cv.b, 0, 1);
        if (r) err = fail(c, r, "skip repack failed");
      }
    }
    return cv;
  }
  // [O, 2*Ktot] = [W | W]: the weights of cv twice along K, for a conv over a hi/lo-split operand (PlanBuilder::head_hilo)
  __half* dup_k(const Conv& cv) {
    __half* w2 = A->get<__half>((size_t)cv.O * 2 * cv.Ktot);
    if (!w2) { err = fail(c, 4005, "weight arena exhausted"); return nullptr; }
    if (!A->measure)
      for (int h2 = 0; h2 < 2; ++h2) {
        cudaError_t e = cudaMemcpy2DAsync(w2 + (size_t)h2 * cv.Ktot, (size_t)2 * cv.Ktot * sizeof(__half), cv.w, (size_t)cv.Ktot * sizeof(__half),
                                          (size_t)cv.Ktot * sizeof(__half), (size_t)cv.O, cudaMemcpyDeviceToDevice, st);
        if (e != cudaSuccess) { err = fail(c, (int)e, "weight copy failed: %s", cudaGetErrorString(e)); return nullptr; }
      }
    return w2;
  }
};

static int parse_pack(sdxl_ctx* c, const void* pack, size_t bytes, int on_device, PackView& pv,
                      std::vector<uint8_t>& host_table) {
  if (bytes < sizeof(PackHeader)) return fail(c, 4100, "weight pack too small");
  PackHeader h;
  if (on_device) CU(c, cudaMemcpy(&h, pack, sizeof h, cudaMemcpyDeviceToHost));
  else memcpy(&h, pack, sizeof h);
  if (memcmp(h.magic, "SDXLPK01", 8) != 0) return fail(c, 4101, "weight pack: bad magic");
  const size_t tbytes = (size_t)h.n_tensors * sizeof(PackEntry);
  if (sizeof h + tbytes > bytes) return fail(c, 4102, "weight pack: truncated table");
  host_table.resize(tbytes);
  if (on_device) CU(c, cudaMemcpy(host_table.data(), (const uint8_t*)pack + sizeof h, tbytes, cudaMemcpyDeviceToHost));
  else memcpy(host_table.data(), (const uint8_t*)pack + sizeof h, tbytes);
  const PackEntry* e = (const PackEntry*)host_table.data();
  for (uint32_t i = 0; i < h.n_tensors; ++i) {
    if (e[i].nbytes > bytes || e[i].offset > bytes - e[i].nbytes) return fail(c, 4103, "weight pack: tensor '%.*s' out of range", 119, e[i].name);
    if (e[i].offset % 16) return fail(c, 4104, "weight pack: tensor '%.*s' not 16B aligned", 119, e[i].name);
    if (e[i].ndim > 4 || e[i].dtype > 1) return fail(c, 4105, "weight pack: tensor '%.*s' has bad rank / dtype", 119, e[i].name);
    {
      uint64_t n = 1;   // element count, overflow-checked against the byte count the entry declares
      bool ok = true;
      for (uint32_t d = 0; d < e[i].ndim && ok; ++d) {
        if (e[i].shape[d] != 0 && n > UINT64_MAX / e[i].shape[d]) ok = false;
        else n *= e[i].shape[d];
      }
      const uint64_t esz = e[i].dtype ? 4 : 2;
      if (!ok || n > UINT64_MAX / esz || n * esz != e[i].nbytes)
        return fail(c, 4106, "weight pack: tensor '%.*s' declares %llu bytes but its shape needs a different size", 119, e[i].name,
                    (unsigned long long)e[i].nbytes);
    }
    std::string name(e[i].name, strnlen(e[i].name, sizeof e[i].name));
    pv.t[name] = e[i];
  }
  return 0;
}

// ================================================================================================
// launch plan
// ================================================================================================
enum OpKind { OP_IGEMM, OP_ATTN, OP_GN, OP_LN, OP_GEMV, OP_TEMB, OP_CONV_IN, OP_UPS, OP_PHASE, OP_CAST16,
              OP_SOFTMAX, OP_TRANSPOSE, OP_PQ, OP_EMBED, OP_ATTN_SMALL, OP_ACT, OP_LN_GATHER, OP_KIND_COUNT };
// the public profile entry points take caller arrays of SDXL_PROFILE_KINDS entries (include/sdxl_b200.h)
static_assert(OP_KIND_COUNT <= SDXL_PROFILE_KINDS, "profile arrays too small for the op kinds");
static const char* const kOpNames[] = {"igemm", "attention", "group_norm", "layer_norm", "gemv", "temb", "conv_in", "upsample",
                                       "phase_split", "cast16", "softmax_rows", "transpose16", "post_quant", "embed_tokens",
                                       "attention_small", "mlp_act", "ln_gather"};
struct Op {
  OpKind kind;
  double flops = 0;  // algorithmic FLOPs of this launch (igemm / attention), 0 for HBM-bound ops
  double flops_exec = 0;  // FLOPs the launch actually issues to the tensor cores (channel / key padding in, phase-decomposed upsample convs at their real cost)
  int block = -1;    // index into Plan::block_names (NVTX range of the reference block this launch belongs to)
  IgemmParams ig;
  AttnParams at;
  GnParams gn;
  struct { const float* x; const float* g; const float* b; float eps; int rows, C; __half* y; } ln;
  struct { const float* in; int in_bstride, Bv, K; const __half* W; int ldw; const float* bias; const float* add; int add_bstride, N, in_silu, out_silu; float* out; int out_bstride; } gv;
  struct { const int* t; int n, dim; float* out; } te;
  struct { const float* x; int Bx, B, Cin, H, W; const float* w; const float* bias; int Cout; float* y; } ci;
  struct { const float* x; int B, H, W, C; __half* y; } rs;  // upsample / phase split
  struct { const float* x; size_t n; __half* y; } cs;
  struct { const float* S; size_t lds; int rows, cols; float scale; __half* P; size_t ldp; } sm;
  struct { const __half* x; size_t ldx; int rows, cols; __half* y; size_t ldy; } tr;
  struct { const float* x; int B, C, HW; const float* w; const float* bias; float inv_scale; float* y; } pq;
  struct { const int* tokens; int rows, T, C, n_vocab; const __half* tok; const __half* pos; float* x; int* err; } em;
  struct { const __half* q; int q_pitch, q_col0; const __half* k; const __half* v; int kv_pitch, k_col0, v_col0, B, T, S, n_head;
           const __half* mask; int causal; __half* out; int ldo; } as;
  struct { const float* x; size_t n; int quick; __half* y; } ac;
  struct { const float* x; const int* idx; int B, T, C; const float* g; const float* b; float eps; float* y; } lg;
};

struct Plan {
  int Bf = 0, Bx = 0, h = 0, w = 0;
  uint64_t cond_version = 0;
  Arena arena;
  std::vector<Op> ops;
  float* x_in = nullptr;  // [Bx, Cin, h, w] f32 NCHW
  float* eps = nullptr;   // [Bf, h*w, eps_ld] f32 NHWC
  int eps_ld = 4;
  cudaGraph_t graph = nullptr;
  cudaGraphExec_t gexec = nullptr;
  int runs = 0;
  double flops = 0;  // algorithmic FLOPs of one run (2*MAC over Linear/conv/attention)
  std::vector<std::string> block_names;   // reference blocks in execution order (input_blocks/3, middle_block, ...)
  ~Plan() {
    if (gexec) cudaGraphExecDestroy(gexec);
    if (graph) cudaGraphDestroy(graph);
    arena.release();
  }
};

struct ActView { const __half* p; int Bn, H, W, C; };
struct F32View { float* p; int C; };  // [Bf, HW, C]

struct PlanBuilder {
  sdxl_ctx* c;
  Plan* P;
  Arena* A;
  int Bf;
  int err = 0;
  // shared scratch
  float* gn_partial = nullptr;

  template <typename T>
  T* buf(size_t n) {
    T* p = A->get<T>(n);
    if (!p && !err) err = fail(c, 5001, "plan arena exhausted");
    return p;
  }
  void add_flops(double f) {  // attribute to the op just pushed
    if (err || P->ops.empty()) return;
    P->ops.back().flops += f;
    P->flops += f;
  }
  // generic igemm op; segs reference view a0 (map 0) / a1 (map 1)
  void igemm(const ActView& a0, const ActView* a1, const std::vector<IgemmSeg>& segs, const __half* W, int N, int Ktot,
             int outH, int outW, int outB, int mode, int geglu_bn, void* out, int out_f32, int ldo, const float* bias,
             int bias_bstride, const float* res, int ldr) {
    if (err) return;
    Op op{};
    op.kind = OP_IGEMM;
    IgemmParams& p = op.ig;
    p.nseg = (int)segs.size();
    if (p.nseg > IGEMM_MAX_SEG) { err = fail(c, 5002, "too many igemm segments"); return; }
    for (int i = 0; i < p.nseg; ++i) p.seg[i] = segs[i];
    p.out = out; p.out_f32 = out_f32; p.ldo = ldo;
    p.bias = bias; p.bias_bstride = bias_bstride;
    p.res = res; p.ldr = ldr;
    if (!A->measure) {
      IgemmOperands o{a0.p, a0.Bn, a0.H, a0.W, a0.C, a0.C, a1 ? a1->p : nullptr, a1 ? a1->Bn : 0, a1 ? a1->H : 0,
                      a1 ? a1->W : 0, a1 ? a1->C : 0, a1 ? a1->C : 0, W, N, Ktot};
      int r = igemm_configure(p, o, outW, outH, outB, mode, geglu_bn);
      if (r) { err = fail(c, r, "igemm configuration failed (N=%d K=%d)", N, Ktot); return; }
    }
    {
      double kb = 0;
      for (int i = 0; i < p.nseg; ++i) kb += p.seg[i].nkb;
      op.flops_exec = 2.0 * outB * outH * (double)outW * N * kb * 64.0;
    }
    P->ops.push_back(op);
  }
  // names the reference block the following launches belong to
  void begin_block(const std::string& name) {
    if (err) return;
    P->block_names.push_back(name);
    cur_block = (int)P->block_names.size() - 1;
    first_op_of_block = P->ops.size();
  }
  void end_block() {
    for (size_t i = first_op_of_block; i < P->ops.size(); ++i) P->ops[i].block = cur_block;
    cur_block = -1;
  }
  int cur_block = -1;
  size_t first_op_of_block = 0;
  void linear(const __half* x, int M, const Lin& L, int mode, void* out, int out_f32, int ldo, const float* res, int ldr) {
    ActView a{x, 1, 1, M, L.K};
    std::vector<IgemmSeg> segs{{0, 0, 0, 0, L.Kpad / 64}};
    igemm(a, nullptr, segs, L.w, L.N, L.Kpad, 1, M, 1, mode, L.geglu_bn, out, out_f32, ldo, L.b, 0, res, ldr);
    add_flops(2.0 * M * (double)L.K * L.N);
  }
  // nearest-2x upsample + 3x3 conv (reference unet/mod.rs:742-751, autoencoder/mod.rs:311-319) as four 2x2 convolutions of the
  // source image x [Bn,H,W,I] (f32 -> f16 copy x16), one per output parity; out is [Bn,2H,2W,O] f32. The algorithmic FLOPs
  // (9 taps on the upsampled image) are what is accounted, a quarter per launch.
  void upconv(const float* x, int Bn, int H, int W, const Conv& cv, __half* x16, float* out) {
    if (err) return;
    {
      Op op{};
      op.kind = OP_CAST16;
      op.cs = {x, (size_t)Bn * H * W * cv.I, x16};
      P->ops.push_back(op);
    }
    ActView a{x16, Bn, H, W, cv.I};
    for (int pa = 0; pa < 2; ++pa)
      for (int pb = 0; pb < 2; ++pb) {
        std::vector<IgemmSeg> segs;
        for (int th = 0; th < 2; ++th)
          for (int tw = 0; tw < 2; ++tw)
            segs.push_back({0, (int16_t)(pb == 0 ? tw - 1 : tw), (int16_t)(pa == 0 ? th - 1 : th), 0, cv.Ipad / 64});
        igemm(a, nullptr, segs, cv.wup + (size_t)(pa * 2 + pb) * cv.O * cv.Ktot, cv.O, cv.Ktot, H, W, Bn, IGEMM_LINEAR, 0, out, 1, cv.O,
              cv.b, 0, nullptr, 0);
        if (err || P->ops.empty()) return;
        IgemmParams& ig = P->ops.back().ig;
        ig.opix_row = 4 * W; ig.opix_w = 2; ig.opix_off = pa * 2 * W + pb;
        add_flops(2.0 * Bn * H * W * 9.0 * cv.I * cv.O);
      }
  }
  // 3x3 stride-1 conv (+ optional fused 1x1 skip segment on a1)
  void conv3(const ActView& a, const ActView* skip, const Conv& cv, float* out, const float* bias, int bias_bstride,
             const float* res) {
    std::vector<IgemmSeg> segs;
    for (int kh = 0; kh < 3; ++kh)
      for (int kw = 0; kw < 3; ++kw) segs.push_back({0, (int16_t)(kw - 1), (int16_t)(kh - 1), 0, cv.Ipad / 64});
    if (skip) segs.push_back({1, 0, 0, 0, cv.I2pad / 64});
    igemm(a, skip, segs, cv.w, cv.O, cv.Ktot, a.H, a.W, a.Bn, IGEMM_LINEAR, 0, out, 1, cv.O, bias, bias_bstride, res, cv.O);
    add_flops(2.0 * a.Bn * a.H * a.W * (double)cv.O * (9.0 * cv.I + cv.I2));
  }
  // PaddedConv2d (autoencoder/mod.rs:326-407): 3x3, stride 2, zero padding only past the bottom / right edge. Output (i, j) reads
  // input rows 2i..2i+2 / cols 2j..2j+2 of x [Bn,H,W,I] f32 -> phase split into ph (f16, [4, Bn, H/2, W/2, I]), tap k: phase k&1,
  // offset k>>1. out [Bn, H/2, W/2, O] f32.
  void padded_conv_s2(const float* x, int Bn, int H, int W, const Conv& cv, __half* ph, float* out) {
    if (err) return;
    Op op{};
    op.kind = OP_PHASE;
    op.rs = {x, Bn, H, W, cv.I, ph};
    P->ops.push_back(op);
    const int H2 = H / 2, W2 = W / 2;
    ActView a{ph, 4 * Bn, H2, W2, cv.I};
    std::vector<IgemmSeg> segs;
    for (int kh = 0; kh < 3; ++kh)
      for (int kw = 0; kw < 3; ++kw)
        segs.push_back({0, (int16_t)(kw >> 1), (int16_t)(kh >> 1), (int16_t)((((kh & 1) * 2) + (kw & 1)) * Bn), cv.Ipad / 64});
    igemm(a, nullptr, segs, cv.w, cv.O, cv.Ktot, H2, W2, Bn, IGEMM_LINEAR, 0, out, 1, cv.O, cv.b, 0, nullptr, 0);
    add_flops(2.0 * Bn * H2 * W2 * 9.0 * cv.I * cv.O);
  }
  // Output head GN -> SiLU -> 3x3 conv with the activation operand split hi + lo (y = f16(t), y_lo = f16(t - y)): the conv runs
  // 18 tap segments over [y | y_lo] with the weights stored twice along K (w2 = Loader::dup_k(cv)), so it sees ~22 bits of t.
  // x [Bf, HW, C] f32 -> out [Bf, HW, ldo] f32.
  void head_hilo(const float* x, int C, int H, int W, const Norm& n, const Conv& cv, const __half* w2, __half* y, __half* y_lo,
                 float* out, int ldo) {
    gn(x, C, nullptr, 0, H * W, n, 1, y, nullptr, y_lo);
    ActView a{y, Bf, H, W, C}, alo{y_lo, Bf, H, W, C};
    std::vector<IgemmSeg> segs;
    for (int part = 0; part < 2; ++part)   // K = [9 taps on hi | 9 taps on lo], weights [W | W]
      for (int kh = 0; kh < 3; ++kh)
        for (int kw = 0; kw < 3; ++kw) segs.push_back({(int16_t)part, (int16_t)(kw - 1), (int16_t)(kh - 1), 0, cv.Ipad / 64});
    igemm(a, &alo, segs, w2, cv.O, 2 * cv.Ktot, H, W, Bf, IGEMM_LINEAR, 0, out, 1, ldo, cv.b, 0, nullptr, 0);
    add_flops(2.0 * Bf * H * W * 9.0 * C * cv.O);
  }
  // Single-head attention of one image with d = Cm (autoencoder/mod.rs:572): S = q k^T (f32 [T,T]), P = softmax(S / sqrt(Cm))
  // (f16), vT = v^T, out = P vT. q, k, v, out f16 [T, Cm]; T a multiple of 64.
  void attn_single_head(const __half* q, const __half* k, const __half* v, int T, int Cm, float* S, __half* Pm, __half* vT,
                        __half* out) {
    if (err) return;
    const int Kp = Loader::pad64(Cm);
    {  // S = q k^T  (f32)
      ActView a{q, 1, 1, T, Cm};
      std::vector<IgemmSeg> segs{{0, 0, 0, 0, Kp / 64}};
      igemm(a, nullptr, segs, k, T, Kp, 1, T, 1, IGEMM_LINEAR, 0, S, 1, T, nullptr, 0, nullptr, 0);
      add_flops(2.0 * T * (double)T * Cm);
    }
    {
      Op op{};
      op.kind = OP_SOFTMAX;
      op.sm = {S, (size_t)T, T, T, (float)(1.0 / sqrt((double)Cm)), Pm, (size_t)T};
      P->ops.push_back(op);
    }
    {
      Op op{};
      op.kind = OP_TRANSPOSE;
      op.tr = {v, (size_t)Cm, T, Cm, vT, (size_t)T};
      P->ops.push_back(op);
    }
    {  // O = P v
      ActView a{Pm, 1, 1, T, T};
      std::vector<IgemmSeg> segs{{0, 0, 0, 0, T / 64}};
      igemm(a, nullptr, segs, vT, Cm, T, 1, T, 1, IGEMM_LINEAR, 0, out, 0, Cm, nullptr, 0, nullptr, 0);
      add_flops(2.0 * T * (double)T * Cm);
    }
  }
  // Multi-head attention (head dim 64) on column windows of row-major f16 matrices: q at columns q_col0.. of [Bf*T, q_pitch],
  // k / v at k_col0 / v_col0 of one [Bf*S, kv_pitch] matrix (fused QKV or KV GEMM outputs; one tensor map serves K and V).
  void attn(const __half* qm, int q_pitch, int q_col0, const __half* kvm, int kv_pitch, int k_col0, int v_col0, int T,
            int S, int n_head, __half* out, int ldo, float sl2e) {
    if (err) return;
    Op op{};
    op.kind = OP_ATTN;
    AttnParams& p = op.at;
    p.T = T; p.S = S; p.n_head = n_head; p.B = Bf;
    p.q_col0 = q_col0; p.k_col0 = k_col0; p.v_col0 = v_col0;
    p.out = out; p.ldo = ldo; p.scale_log2e = sl2e;
    if (!A->measure) {
      int r = make_tmap_rows(&p.tmQ, qm, T, Bf, q_pitch, q_pitch);
      if (!r) r = make_tmap_rows(&p.tmK, kvm, S, Bf, kv_pitch, kv_pitch);
      if (!r) p.tmV = p.tmK;
      if (r) { err = fail(c, r, "tensor map creation failed (attention)"); return; }
    }
    op.flops_exec = 4.0 * Bf * (double)((T + 127) / 128 * 128) * (double)((S + 127) / 128 * 128) * (n_head * 64);
    P->ops.push_back(op);
    add_flops(4.0 * Bf * T * (double)S * (n_head * 64));
  }
  // Masked / causal attention for short sequences (CUDA-core kernel), same column-window addressing as attn().
  void attn_small(const __half* qm, int q_pitch, int q_col0, const __half* kvm, int kv_pitch, int k_col0, int v_col0, int T, int S,
                  int n_head, const __half* mask, int causal, __half* out, int ldo) {
    if (err) return;
    Op op{};
    op.kind = OP_ATTN_SMALL;
    op.as = {qm, q_pitch, q_col0, kvm, kvm, kv_pitch, k_col0, v_col0, Bf, T, S, n_head, mask, causal, out, ldo};
    P->ops.push_back(op);
    add_flops(4.0 * Bf * T * (double)S * (n_head * 64));
  }
  void gn(const float* x1, int C1, const float* x2, int C2, int HW, const Norm& n, int silu, __half* y, __half* raw,
          __half* y_lo = nullptr) {
    if (err) return;
    Op op{};
    op.kind = OP_GN;
    op.gn = GnParams{x1, C1, x2, C2, Bf, HW, 32, n.g, n.b, n.eps, silu, y, raw, gn_partial, 0, y_lo};
    P->ops.push_back(op);
  }
  void ln(const float* x, const Norm& n, int rows, __half* y) {
    if (err) return;
    Op op{};
    op.kind = OP_LN;
    op.ln = {x, n.g, n.b, n.eps, rows, n.C, y};
    P->ops.push_back(op);
  }
  void gemv(const float* in, int in_bstride, int Bv, const Lin& L, const float* add, int add_bstride, int in_silu,
            int out_silu, float* out, int out_bstride) {
    if (err) return;
    for (int b0 = 0; b0 < Bv; b0 += 8) {
      Op op{};
      op.kind = OP_GEMV;
      const int nb = Bv - b0 < 8 ? Bv - b0 : 8;
      op.gv = {in + (size_t)b0 * in_bstride, in_bstride, nb, L.K, L.w, L.Kpad, L.b, add ? add + (size_t)b0 * add_bstride : nullptr,
               add_bstride, L.N, in_silu, out_silu, out + (size_t)b0 * out_bstride, out_bstride};
      P->ops.push_back(op);
    }
    P->flops += 2.0 * Bv * (double)L.K * L.N;
  }

};

static int exec_op(sdxl_ctx* c, Op& op) {
  cudaStream_t st = c->stream;
  switch (op.kind) {
    case OP_IGEMM: KL(c, igemm_launch(st, op.ig)); break;
    case OP_ATTN: KL(c, attention_launch(st, op.at)); break;
    case OP_GN: KL(c, gn_launch(st, op.gn)); c->launches++; break;
    case OP_LN: KL(c, layernorm_launch(st, op.ln.x, op.ln.g, op.ln.b, op.ln.eps, op.ln.rows, op.ln.C, op.ln.y)); break;
    case OP_GEMV:
      KL(c, gemv_launch(st, op.gv.in, op.gv.in_bstride, op.gv.Bv, op.gv.K, op.gv.W, op.gv.ldw, op.gv.bias, op.gv.add, op.gv.add_bstride,
                        op.gv.N, op.gv.in_silu, op.gv.out_silu, op.gv.out, op.gv.out_bstride));
      break;
    case OP_TEMB: KL(c, timestep_embedding_launch(st, op.te.t, op.te.n, op.te.dim, 10000.f, op.te.out)); break;
    case OP_CONV_IN:
      KL(c, conv_in_launch_t(st, op.ci.x, 1, op.ci.Bx, op.ci.B, op.ci.Cin, op.ci.H, op.ci.W, op.ci.w, op.ci.bias, op.ci.Cout, op.ci.y));
      break;
    case OP_UPS: KL(c, upsample2x_launch(st, op.rs.x, op.rs.B, op.rs.H, op.rs.W, op.rs.C, op.rs.y)); break;
    case OP_PHASE: KL(c, phase_split_launch(st, op.rs.x, op.rs.B, op.rs.H, op.rs.W, op.rs.C, op.rs.y)); break;
    case OP_CAST16: KL(c, cast_f32_to_f16_launch(st, op.cs.x, op.cs.n, op.cs.y)); break;
    case OP_SOFTMAX: KL(c, softmax_rows_launch(st, op.sm.S, op.sm.lds, op.sm.rows, op.sm.cols, op.sm.scale, op.sm.P, op.sm.ldp)); break;
    case OP_TRANSPOSE: KL(c, transpose_f16_launch(st, op.tr.x, op.tr.ldx, op.tr.rows, op.tr.cols, op.tr.y, op.tr.ldy)); break;
    case OP_EMBED: KL(c, embed_tokens_launch(st, op.em.tokens, op.em.rows, op.em.T, op.em.C, op.em.n_vocab, op.em.tok, op.em.pos, op.em.x, op.em.err)); break;
    case OP_ATTN_SMALL:
      KL(c, attention_small_launch(st, op.as.q, op.as.q_pitch, op.as.q_col0, op.as.k, op.as.v, op.as.kv_pitch, op.as.k_col0, op.as.v_col0,
                                   op.as.B, op.as.T, op.as.S, op.as.n_head, op.as.mask, op.as.causal, op.as.out, op.as.ldo));
      break;
    case OP_ACT: KL(c, mlp_act_launch(st, op.ac.x, op.ac.n, op.ac.quick, op.ac.y)); break;
    case OP_LN_GATHER: KL(c, ln_gather_f32_launch(st, op.lg.x, op.lg.idx, op.lg.B, op.lg.T, op.lg.C, op.lg.g, op.lg.b, op.lg.eps, op.lg.y)); break;
    case OP_PQ: KL(c, post_quant_launch(st, op.pq.x, op.pq.B, op.pq.C, op.pq.HW, op.pq.w, op.pq.bias, op.pq.inv_scale, op.pq.y)); break;
  }
  return 0;
}

static int run_plan_ops(sdxl_ctx* c, Plan* P) {
  static const bool no_graph = getenv("SDXL_B200_NO_GRAPH") != nullptr;
  if (P->gexec) {
    CU(c, cudaGraphLaunch(P->gexec, c->stream));
    c->launches += P->ops.size() + [&] { size_t g = 0; for (auto& o : P->ops) g += o.kind == OP_GN; return g; }();
    return 0;
  }
  const bool capture = !no_graph && P->runs >= 1;  // first run eager (sets func attributes), then capture
  if (capture) CU(c, cudaStreamBeginCapture(c->stream, cudaStreamCaptureModeThreadLocal));
  int r = 0;
  int open_block = -1;   // NVTX range per reference block (host side: visible in eager runs and during graph capture)
  for (auto& op : P->ops) {
    if (op.block != open_block) {
      if (open_block >= 0) nvtxRangePop();
      open_block = op.block;
      if (open_block >= 0) nvtxRangePushA(P->block_names[open_block].c_str());
    }
    r = exec_op(c, op);
    if (r) break;
  }
  if (open_block >= 0) nvtxRangePop();
  if (capture) {
    cudaGraph_t gph = nullptr;
    cudaError_t e = cudaStreamEndCapture(c->stream, &gph);
    if (r) { if (gph) cudaGraphDestroy(gph); return r; }
    if (e != cudaSuccess) return fail(c, (int)e, "graph capture failed: %s", cudaGetErrorString(e));
    P->graph = gph;
    e = cudaGraphInstantiate(&P->gexec, gph, 0);
    if (e != cudaSuccess) { P->gexec = nullptr; return fail(c, (int)e, "graph instantiate failed: %s", cudaGetErrorString(e)); }
    CU(c, cudaGraphLaunch(P->gexec, c->stream));
  }
  P->runs++;
  return r;
}

// Per-kernel-kind device time of one plan execution, measured with CUDA events on the ctx stream (eager launches, one event
// pair per op). kinds: see OpKind. Arrays must hold 16 entries.
static int profile_plan_impl(sdxl_ctx* c, Plan* P, double* ms_by_kind, double* flops_by_kind, int* launches_by_kind) {
  const size_t n = P->ops.size();
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) CU(c, cudaEventCreate(&e));
  int r = 0;
  CU(c, cudaEventRecord(ev[0], c->stream));
  for (size_t i = 0; i < n && !r; ++i) {
    r = exec_op(c, P->ops[i]);
    if (!r && cudaEventRecord(ev[i + 1], c->stream) != cudaSuccess) r = -2;
  }
  cudaError_t se = cudaStreamSynchronize(c->stream);
  for (int k = 0; k < SDXL_PROFILE_KINDS; ++k) { ms_by_kind[k] = 0; flops_by_kind[k] = 0; launches_by_kind[k] = 0; }
  if (!r && se == cudaSuccess)
    for (size_t i = 0; i < n; ++i) {
      float ms = 0;
      cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
      const int k = (int)P->ops[i].kind;
      if (k < 0 || k >= SDXL_PROFILE_KINDS) continue;
      ms_by_kind[k] += ms;
      flops_by_kind[k] += P->ops[i].flops;
      launches_by_kind[k] += (P->ops[i].kind == OP_GN) ? 2 : 1;
    }
  for (auto& e : ev) cudaEventDestroy(e);
  if (se != cudaSuccess) return fail(c, (int)se, "profile run failed: %s", cudaGetErrorString(se));
  return r;
}

// Per-op dump of one eager plan execution (CUDA-event time per launch) as CSV: analysis aid for profiles/.
static int profile_dump_impl(sdxl_ctx* c, Plan* P, const char* path) {
  const size_t n = P->ops.size();
  std::vector<cudaEvent_t> ev(n + 1);
  for (auto& e : ev) CU(c, cudaEventCreate(&e));
  int r = 0;
  CU(c, cudaEventRecord(ev[0], c->stream));
  for (size_t i = 0; i < n && !r; ++i) {
    r = exec_op(c, P->ops[i]);
    if (!r && cudaEventRecord(ev[i + 1], c->stream) != cudaSuccess) r = -2;
  }
  cudaError_t se = cudaStreamSynchronize(c->stream);
  if (!r && se == cudaSuccess) {
    FILE* f = fopen(path, "w");
    if (!f) r = fail(c, -3, "cannot open %s", path);
    else {
      fprintf(f, "op,kind,us,gflop,tflops,M_tiles,N,BN,Kblocks,T,S,heads,cluster\n");
      for (size_t i = 0; i < n; ++i) {
        float ms = 0;
        cudaEventElapsedTime(&ms, ev[i], ev[i + 1]);
        const Op& o = P->ops[i];
        int mt = 0, N = 0, BN = 0, kb = 0, T = 0, S = 0, H = 0;
        if (o.kind == OP_IGEMM) {
          mt = o.ig.tilesW * o.ig.tilesH * o.ig.tilesB; N = o.ig.N; BN = o.ig.BN;
          for (int s2 = 0; s2 < o.ig.nseg; ++s2) kb += o.ig.seg[s2].nkb;
        } else if (o.kind == OP_ATTN) { T = o.at.T; S = o.at.S; H = o.at.n_head; }
        fprintf(f, "%zu,%s,%.2f,%.3f,%.1f,%d,%d,%d,%d,%d,%d,%d,%dx%d\n", i, kOpNames[o.kind], ms * 1e3, o.flops * 1e-9,
                ms > 0 ? o.flops / (ms * 1e-3) * 1e-12 : 0.0, mt, N, BN, kb, T, S, H,
                o.kind == OP_IGEMM ? (o.ig.pair ? 9 : o.ig.CM) : 0, o.kind == OP_IGEMM ? o.ig.CN : 0);
      }
      fclose(f);
    }
  }
  for (auto& e : ev) cudaEventDestroy(e);
  if (se != cudaSuccess) return fail(c, (int)se, "profile run failed: %s", cudaGetErrorString(se));
  return r;
}

struct TmpBufs {
  std::vector<void*> p;
  cudaStream_t st;
  explicit TmpBufs(cudaStream_t s) : st(s) {}
  void* get(size_t bytes) {
    void* d = nullptr;
    if (cudaMallocAsync(&d, bytes ? bytes : 16, st) != cudaSuccess) return nullptr;
    p.push_back(d);
    return d;
  }
  ~TmpBufs() { for (void* d : p) cudaFreeAsync(d, st); }
};
