// NAR refiner (reference nn/nar.py:13-116, model.py:307-347) on the device as a handful of fused fp32 kernels:
// per stage  embed-mix + stage adapter (1 launch)  ->  6 x SSMLiteBlock (RMSNorm+GLU GEMM | dwconv+residual |
// RMSNorm+FFN1+GELU GEMM | FFN2+residual GEMM)  ->  RMSNorm+pre GEMM  ->  all heads of the stage in ONE grouped GEMM launch
// with an argmax epilogue (the logits never reach memory)  ->  argmax finish.  28 launches per stage instead of ~150
// ATen ops.  The ids must equal the reference's, so every contraction is fp32 (dense_f32.cuh).
#include <cuda_runtime.h>

#include <algorithm>
#include <cmath>
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <string>
#include <vector>

#include "../../include/sopro_b200.h"
#include "dense_f32.cuh"
#include "mimi_tc.cuh"  // tc::launch: the tcgen05 / TMEM / TMA implicit-GEMM kernel, reused for the exact split products

namespace mimi {
void set_error(const char* msg);  // ar_engine.cu: the string behind sopro_last_error()
}

namespace pstage {

int fail(int code, const char* fmt, ...) {
  char buf[1024];
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(buf, sizeof(buf), fmt, ap);
  va_end(ap);
  mimi::set_error(buf);
  return code;
}
#define PCK(call)                                                                                                       \
  do {                                                                                                                  \
    cudaError_t e__ = (call);                                                                                           \
    if (e__ != cudaSuccess)                                                                                             \
      return pstage::fail(SOPRO_ERR_CUDA, "%s failed: %s (%s:%d)", #call, cudaGetErrorString(e__), __FILE__, __LINE__); \
  } while (0)

struct FArena {
  std::vector<float> host;
  size_t add(const float* p, size_t n) {
    const size_t off = (host.size() + 63) / 64 * 64;
    host.resize(off + n);
    if (p) memcpy(host.data() + off, p, n * 4);
    return off;
  }
};

struct BlockOff {
  size_t norm_w, glu_w, glu_b, dw_w, dw_b, ffn_norm_w, w1, b1, w2, b2;
};

void add_block(FArena& A, const sopro_ssm_block_weights_t& L, int D, int k, BlockOff* o) {
  o->norm_w = A.add(L.norm_w, D);
  o->glu_w = A.add(L.glu_w, (size_t)2 * D * D);
  o->glu_b = A.add(L.glu_b, 2 * D);
  o->dw_w = A.add(L.dw_w, (size_t)D * k);
  o->dw_b = A.add(L.dw_b, D);
  o->ffn_norm_w = A.add(L.ffn_norm_w, D);
  o->w1 = A.add(L.ffn_w1, (size_t)4 * D * D);
  o->b1 = A.add(L.ffn_b1, 4 * D);
  o->w2 = A.add(L.ffn_w2, (size_t)4 * D * D);
  o->b2 = A.add(L.ffn_b2, D);
}

bool block_ok(const sopro_ssm_block_weights_t& L) {
  return L.norm_w && L.glu_w && L.glu_b && L.dw_w && L.dw_b && L.ffn_norm_w && L.ffn_w1 && L.ffn_b1 && L.ffn_w2 && L.ffn_b2;
}

// Tile edge of the tile kernel for an [M x N] output in `groups` groups: the largest of 128 / 64 / 32 that still gives
// (about) every SM a CTA -- a streaming window of ~190 rows would otherwise run on a handful of SMs.  The result does
// not depend on the choice (one fma chain over k per output, dense_f32.cuh).  GLU pairs value / gate columns inside a
// thread, which the 32-wide tile cannot: 64 is its smallest.
int tile_edge(int M, int N, int groups, int epi) {
  const int target = 120;
  for (int e : {128, 64}) {
    const long long ctas = (long long)((M + e - 1) / e) * ((N + e - 1) / e) * groups;
    if (ctas >= target) return e;
  }
  return epi == dense::EPI_GLU ? 64 : 32;
}

// C = epi(prologue(A) . W^T): picks the skinny kernel for M <= 16 rows, a tile kernel otherwise.
// groups > 1 (argmax heads): blockIdx.z = group.
int launch_dense(dense::DenseOp op, int groups, cudaStream_t st) {
  if (op.K % 16 || op.M < 1 || op.N < 1) return fail(SOPRO_ERR_INVALID, "dense: bad shape M=%d N=%d K=%d", op.M, op.N, op.K);
  if (op.M <= dense::kSkinnyRows) {
    const int ncol = op.epi == dense::EPI_GLU ? op.N / 2 : op.N;
    // about two waves of CTAs over the GPU, at least one column per warp
    int cols = std::max(8, (ncol * groups + 295) / 296);
    cols = (cols + 7) / 8 * 8;
    const int parts = (ncol + cols - 1) / cols;
    if (op.epi == dense::EPI_ARGMAX) op.parts = parts;
    const size_t smem = (size_t)dense::kSkinnyRows * op.K * 4;
    static bool attr = false;
    if (!attr) {
      PCK(cudaFuncSetAttribute(dense::dense_skinny_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 16 * 2048 * 4));
      attr = true;
    }
    if (smem > (size_t)16 * 2048 * 4) return fail(SOPRO_ERR_INVALID, "dense: K=%d too large for the skinny kernel", op.K);
    dense::dense_skinny_kernel<<<dim3(parts, 1, groups), dense::kSkinnyThreads, smem, st>>>(op, cols);
  } else {
    const int e = tile_edge(op.M, op.N, groups, op.epi);
    const dim3 grid((op.M + e - 1) / e, (op.N + e - 1) / e, groups);
    if (op.epi == dense::EPI_ARGMAX) op.parts = (int)grid.y;
    if (e == 128) dense::dense_tile_kernel<128, 128><<<grid, dense::kTileThreads, 0, st>>>(op);
    else if (e == 64) dense::dense_tile_kernel<64, 64><<<grid, dense::kTileThreads, 0, st>>>(op);
    else dense::dense_tile_kernel<32, 32><<<grid, dense::kTileThreads, 0, st>>>(op);
  }
  PCK(cudaGetLastError());
  return SOPRO_OK;
}

// argmax partial slots per row the launch above will write (must match launch_dense)
int argmax_parts(int M, int N, int groups) {
  if (M <= dense::kSkinnyRows) {
    int cols = std::max(8, (N * groups + 295) / 296);
    cols = (cols + 7) / 8 * 8;
    return (N + cols - 1) / cols;
  }
  const int e = tile_edge(M, N, groups, dense::EPI_ARGMAX);
  return (N + e - 1) / e;
}

// =================================================================================================
// Exact fp32 products on the tensor cores (row counts above the skinny kernel's).  Every fp32 operand is the exact sum
// of three bf16 terms (h + m + l: 3 x 8 mantissa bits), a product of two bf16 numbers is exact in fp32, so
//   x . w = sum over the six term pairs whose magnitude reaches fp32's last bit (mm, lh, hl, mh, hm, hh; the pairs ml, lm,
//   ll are below 2^-26 of the product)
// accumulated in fp32 in tensor memory: the same quantity the fp32 FMA kernels compute, up to the order of the fp32
// additions.  One GEMM launch does all six: the weights are stored as W6 [N][6K] (K blocks = the w term of each pair,
// built once on the host), the activations as A3 [M][3K] = [h | m | l] written by split3_rows_kernel (fused with the
// RMSNorm of the rows), and the GEMM kernel's "tap" j (mimi_tc.cuh: K block j of W against A columns tap_col[j] + ...)
// selects the x term.  M = batch x frames rows fill 128-row tiles, which is what the tensor cores need (the AR step's
// 22..86 rows per CTA do not, DESIGN.md §3).
// =================================================================================================
constexpr int kPairs = 6;
constexpr int kPairX[kPairs] = {1, 2, 0, 1, 0, 0};  // x term of pair j (0 = h, 1 = m, 2 = l), smallest products first
constexpr int kPairW[kPairs] = {1, 0, 2, 0, 1, 0};  // w term of pair j

inline uint16_t bf16_rne(float f) {
  uint32_t u;
  memcpy(&u, &f, 4);
  if ((u & 0x7fffffffu) > 0x7f800000u) return (uint16_t)((u >> 16) | 0x40);
  u += 0x7fffu + ((u >> 16) & 1u);
  return (uint16_t)(u >> 16);
}
inline float bf16_f32(uint16_t h) {
  const uint32_t u = (uint32_t)h << 16;
  float f;
  memcpy(&f, &u, 4);
  return f;
}
// W [N][K] fp32 -> W6 [N][6K] bf16 appended to `dst`; returns the element offset
size_t pack_w6(std::vector<uint16_t>& dst, const float* W, size_t N, size_t K) {
  const size_t off = (dst.size() + 63) / 64 * 64;
  dst.resize(off + N * kPairs * K);
  for (size_t n = 0; n < N; ++n)
    for (size_t k = 0; k < K; ++k) {
      const float w = W[n * K + k];
      uint16_t t[3];
      t[0] = bf16_rne(w);
      const float r1 = w - bf16_f32(t[0]);
      t[1] = bf16_rne(r1);
      t[2] = bf16_rne(r1 - bf16_f32(t[1]));
      for (int j = 0; j < kPairs; ++j) dst[off + (n * kPairs + j) * K + k] = t[kPairW[j]];
    }
  return off;
}

// rows [M][K] fp32 (optionally RMS-normalised, nn/blocks.py:32-37) -> A3 [M][3K] bf16 = [h | m | l], one warp per row
__global__ void __launch_bounds__(256) split3_rows_kernel(const float* __restrict__ x, const float* __restrict__ norm_w,
                                                          __nv_bfloat16* __restrict__ out, long long rows, int K) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* xr = x + row * K;
  float inv = 1.f;
  if (norm_w) {
    float ss = 0.f;
    for (int k = lane * 4; k < K; k += 128) {
      const float4 v = *reinterpret_cast<const float4*>(xr + k);
      ss += v.x * v.x + v.y * v.y + v.z * v.z + v.w * v.w;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
    inv = 1.0f / sqrtf(ss / (float)K + 1e-6f);
  }
  __nv_bfloat16* o = out + row * 3 * K;
  for (int k = lane * 4; k < K; k += 128) {
    float4 v = *reinterpret_cast<const float4*>(xr + k);
    if (norm_w) {
      const float4 w = __ldg(reinterpret_cast<const float4*>(norm_w + k));
      v.x = (v.x * inv) * w.x;
      v.y = (v.y * inv) * w.y;
      v.z = (v.z * inv) * w.z;
      v.w = (v.w * inv) * w.w;
    }
    const __nv_bfloat162 h0 = __floats2bfloat162_rn(v.x, v.y), h1 = __floats2bfloat162_rn(v.z, v.w);
    const float rx = v.x - __low2float(h0), ry = v.y - __high2float(h0), rz = v.z - __low2float(h1), rw = v.w - __high2float(h1);
    const __nv_bfloat162 m0 = __floats2bfloat162_rn(rx, ry), m1 = __floats2bfloat162_rn(rz, rw);
    const __nv_bfloat162 l0 = __floats2bfloat162_rn(rx - __low2float(m0), ry - __high2float(m0));
    const __nv_bfloat162 l1 = __floats2bfloat162_rn(rz - __low2float(m1), rw - __high2float(m1));
    uint2 ph, pm, pl;
    ph.x = *reinterpret_cast<const unsigned*>(&h0), ph.y = *reinterpret_cast<const unsigned*>(&h1);
    pm.x = *reinterpret_cast<const unsigned*>(&m0), pm.y = *reinterpret_cast<const unsigned*>(&m1);
    pl.x = *reinterpret_cast<const unsigned*>(&l0), pl.y = *reinterpret_cast<const unsigned*>(&l1);
    *reinterpret_cast<uint2*>(o + k) = ph;
    *reinterpret_cast<uint2*>(o + K + k) = pm;
    *reinterpret_cast<uint2*>(o + 2 * K + k) = pl;
  }
}

// GLU (nn/blocks.py:16-23) on the GEMM's [M][2D] output (bias included): h = value * sigmoid(gate)
__global__ void __launch_bounds__(256) glu_rows_kernel(const float* __restrict__ v, float* __restrict__ h, long long rows, int D) {
  const long long i = ((long long)blockIdx.x * 256 + threadIdx.x) * 4;
  if (i >= rows * D) return;
  const long long r = i / D;
  const int c = (int)(i - r * D);
  const float4 a = *reinterpret_cast<const float4*>(v + r * 2 * D + c);
  const float4 g = *reinterpret_cast<const float4*>(v + r * 2 * D + D + c);
  float4 o;
  o.x = a.x * dense::sigmoid_ref(g.x);
  o.y = a.y * dense::sigmoid_ref(g.y);
  o.z = a.z * dense::sigmoid_ref(g.z);
  o.w = a.w * dense::sigmoid_ref(g.w);
  *reinterpret_cast<float4*>(h + i) = o;
}

// first maximum (torch.argmax) of each head's V logits: one warp per (row, head)
__global__ void __launch_bounds__(256) argmax_heads_kernel(const float* __restrict__ logits, long long rows, int heads, int V,
                                                           int* __restrict__ codes, int Q) {
  const long long w = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (w >= rows * heads) return;
  const long long r = w / heads;
  const int hd = (int)(w - r * heads);
  const float* lg = logits + (r * heads + hd) * V;
  float bv = -INFINITY;
  int bi = 0x7fffffff;
  for (int c = lane * 4; c < V; c += 128) {
    const float4 q = *reinterpret_cast<const float4*>(lg + c);
    const float vv[4] = {q.x, q.y, q.z, q.w};
#pragma unroll
    for (int e = 0; e < 4; ++e)
      if (dense::before(vv[e], c + e, bv, bi)) bv = vv[e], bi = c + e;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    const float ov = __shfl_xor_sync(0xffffffffu, bv, o);
    const int oi = __shfl_xor_sync(0xffffffffu, bi, o);
    if (dense::before(ov, oi, bv, bi)) bv = ov, bi = oi;
  }
  if (lane == 0) codes[r * Q + hd] = bi;
}

// C [M][N] = epi(A . W^T + bias): A3 [M][3K] bf16 (split3_rows_kernel), W6 [N][6K] bf16 (pack_w6)
int launch_tc6(const __nv_bfloat16* A3, const uint16_t* W6, const float* bias, const float* R, float* C, long long M, int N, int K, int epi,
               cudaStream_t st) {
  tc::TcOp o{};
  o.bias = bias;
  o.R = R;
  o.out_f32 = C;
  o.c_bs = M * N;
  o.M = (int)M;
  o.N = N;
  o.K = kPairs * K;
  o.Cin = K;
  o.dil = 0;
  o.pad = 0;
  o.bias_mod = N;
  o.epi = epi;
  for (int j = 0; j < kPairs; ++j) o.tap_col[j] = kPairX[j] * K;
  if (!tc::supported(N, o.K, K)) return fail(SOPRO_ERR_INVALID, "tensor-core NAR GEMM: unsupported shape N=%d K=%d", N, K);
  const cudaError_t e = tc::launch(A3, M, W6, o, 1, st, 3 * K);
  if (e != cudaSuccess) return fail(SOPRO_ERR_CUDA, "tensor-core NAR GEMM (N=%d K=%d M=%lld): %s", N, K, M, cudaGetErrorString(e));
  return SOPRO_OK;
}

struct BlockTc {
  size_t glu, w1, w2;  // W6 element offsets
};

// one SSMLiteBlock with the three contractions on the tensor cores; a3 [M][3*4D] bf16 and v [M][4D] fp32 are scratch
int ssm_block_tc(const float* W, const BlockOff& o, const uint16_t* T, const BlockTc& t, float* x, float* h, float* v, __nv_bfloat16* a3,
                 const int* lens, int B, int Tmax, int D, int k, int dil, cudaStream_t st) {
  const long long M = (long long)B * Tmax;
  const unsigned rb = (unsigned)((M + 7) / 8);
  split3_rows_kernel<<<rb, 256, 0, st>>>(x, W + o.norm_w, a3, M, D);
  int rc = launch_tc6(a3, T + t.glu, W + o.glu_b, nullptr, v, M, 2 * D, D, tc::EPI_NONE, st);
  if (rc) return rc;
  glu_rows_kernel<<<(unsigned)((M * D / 4 + 255) / 256), 256, 0, st>>>(v, h, M, D);
  const int total = (k - 1) * dil;
  dense::dwconv_res_kernel<<<dim3(Tmax, B), 128, 0, st>>>(h, x, W + o.dw_w, W + o.dw_b, x, lens, Tmax, D, k, dil, total / 2);
  split3_rows_kernel<<<rb, 256, 0, st>>>(x, W + o.ffn_norm_w, a3, M, D);
  if ((rc = launch_tc6(a3, T + t.w1, W + o.b1, nullptr, v, M, 4 * D, D, tc::EPI_GELU, st))) return rc;
  split3_rows_kernel<<<rb, 256, 0, st>>>(v, nullptr, a3, M, 4 * D);
  if ((rc = launch_tc6(a3, T + t.w2, W + o.b2, x, x, M, D, 4 * D, tc::EPI_RES, st))) return rc;
  PCK(cudaGetLastError());
  return SOPRO_OK;
}

// one SSMLiteBlock (nn/blocks.py:143-148) over rows [B][Tmax][D], in place on x; h [M][D] and hid [M][4D] are scratch
int ssm_block(const float* W, const BlockOff& o, float* x, float* h, float* hid, const int* lens, int B, int Tmax, int D, int k, int dil,
              bool causal, cudaStream_t st) {
  const int M = B * Tmax;
  dense::DenseOp g{};
  g.A = x; g.W = W + o.glu_w; g.bias = W + o.glu_b; g.norm_w = W + o.norm_w; g.C = h; g.M = M; g.N = 2 * D; g.K = D; g.ldc = D;
  g.epi = dense::EPI_GLU;
  int rc = launch_dense(g, 1, st);
  if (rc) return rc;
  const int total = (k - 1) * dil, left = causal ? total : total / 2;
  dense::dwconv_res_kernel<<<dim3(Tmax, B), 128, 0, st>>>(h, x, W + o.dw_w, W + o.dw_b, x, lens, Tmax, D, k, dil, left);
  PCK(cudaGetLastError());
  g = dense::DenseOp{};
  g.A = x; g.W = W + o.w1; g.bias = W + o.b1; g.norm_w = W + o.ffn_norm_w; g.C = hid; g.M = M; g.N = 4 * D; g.K = D; g.ldc = 4 * D;
  g.epi = dense::EPI_GELU;
  if ((rc = launch_dense(g, 1, st))) return rc;
  g = dense::DenseOp{};
  g.A = hid; g.W = W + o.w2; g.bias = W + o.b2; g.R = x; g.C = x; g.M = M; g.N = D; g.K = 4 * D; g.ldc = D; g.epi = dense::EPI_RES;
  return launch_dense(g, 1, st);
}

// ---- NAR stage input (model.py:318-341 + nn/embeddings.py:77-112 + nn/nar.py:28-32), one warp per (b, t) row:
//   prev = sum_j w[j] * cb_embed[cb[j]*V + tok[j]]      (the codebooks decided so far, softmax weights)
//   x    = mix0 * cond + mix1 * prev
//   out  = RMSNorm(x) * (1 + tanh(g)) + tanh(b)         (stage adapter; g, b depend on the stage only)
struct EmbedMix {
  const float* cond;      // [B][cond_bs] rows of D
  long long cond_bs;
  const int* codes;       // [B][Tmax][Q] (codebooks < n_prev already decided)
  const float* emb;       // [Q*V + 1][D]
  const float* w_prev;    // [n_prev]
  const float* norm_w;    // adapter RMSNorm
  const float* mul;       // [D] 1 + tanh(g)
  const float* add;       // [D] tanh(b)
  float* out;             // [B][Tmax][D]
  float mix0, mix1;
  int Tmax, D, Q, V, n_prev;
};

__global__ void __launch_bounds__(256) nar_embed_mix_kernel(const EmbedMix p, long long rows) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const long long b = row / p.Tmax, t = row - b * p.Tmax;
  const float* c = p.cond + b * p.cond_bs + t * p.D;
  const int* tk = p.codes + row * p.Q;
  constexpr int kMaxPer = 16;  // D <= 512
  float x[kMaxPer];
  float ss = 0.f;
  int n = 0;
  for (int k = lane; k < p.D; k += 32, ++n) {
    float prev = 0.f;
    for (int j = 0; j < p.n_prev; ++j) {
      const int tok = min(max(tk[j], 0), p.V - 1);
      prev += __ldg(p.w_prev + j) * __ldg(p.emb + ((size_t)j * p.V + tok) * p.D + k);
    }
    const float v = p.mix0 * c[k] + p.mix1 * prev;
    x[n] = v;
    ss += v * v;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) ss += __shfl_xor_sync(0xffffffffu, ss, o);
  const float inv = 1.0f / sqrtf(ss / (float)p.D + 1e-6f);
  n = 0;
  for (int k = lane; k < p.D; k += 32, ++n)
    p.out[row * p.D + k] = ((x[n] * inv) * __ldg(p.norm_w + k)) * __ldg(p.mul + k) + __ldg(p.add + k);
}

// codes[b][t][0] = rvq1[b][t]
__global__ void set_first_codebook_kernel(const int* __restrict__ rvq1, int* __restrict__ codes, long long rows, int Q) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < rows) codes[i * Q] = rvq1[i];
}

}  // namespace pstage

using namespace pstage;

struct sopro_nar {
  int device = 0;
  sopro_nar_config_t cfg{};
  float* dev = nullptr;
  size_t n_floats = 0;
  BlockOff blk[SOPRO_MAX_SSM_LAYERS]{};
  size_t norm_w = 0, pre_w = 0, pre_b = 0, adapter_norm_w = 0, emb = 0;
  struct Stage {
    int first, count, n_prev;
    size_t w_prev, mul, add, head_w, head_b, head_id;
    float mix0, mix1;
    size_t tc_heads = 0, head_b_folded = 0;  // tensor-core path: W6 of the stage's heads; bias + W . id_embedding
  };
  // tensor-core path (exact six-product split): W6 images of every contraction, bf16
  uint16_t* tcw = nullptr;
  BlockTc tblk[SOPRO_MAX_SSM_LAYERS]{};
  size_t tc_pre = 0;
  bool tc_ok = false;
  std::vector<Stage> stages;
  // workspace
  float* ws = nullptr;
  size_t ws_bytes = 0;
  const int32_t* forced = nullptr;  // test hook: the previous codebooks every stage conditions on
  int tc_mode = -1;                 // -1 automatic (tensor cores above the skinny kernel's row count), 0 fp32 FMA kernels only
  // launch-bound streaming windows (one utterance, <= kNarGraphRows frames: 113..217 launches each) are replayed from
  // CUDA graphs captured over static buffers; every graph dies when the workspace is reallocated
  struct Replay {
    int T, tc;
    cudaGraphExec_t exec;
  };
  std::vector<Replay> replays;
  float* g_cond = nullptr;
  int32_t* g_rvq1 = nullptr;
  int32_t* g_codes = nullptr;
  bool graphs = true;
  cudaStream_t cap_stream = nullptr;
  cudaEvent_t g_done = nullptr;     // last replay's completion: the static buffers are reused across caller streams
  size_t reserve_bytes = 0;         // workspace floor (so that no graph-sized call reallocates)
};

constexpr int kNarGraphRows = 256;

static void nar_drop_replays(sopro_nar* n) {
  for (auto& r : n->replays) cudaGraphExecDestroy(r.exec);
  n->replays.clear();
}

extern "C" {

int sopro_nar_create(const sopro_nar_config_t* cfg, const sopro_nar_weights_t* w, int device, sopro_nar_t** out) {
  if (!cfg || !w || !out) return fail(SOPRO_ERR_INVALID, "null argument");
  *out = nullptr;
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev <= 0) return fail(SOPRO_ERR_UNSUPPORTED, "no CUDA device; the NAR refiner has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(SOPRO_ERR_INVALID, "device %d out of range", device);
  cudaDeviceProp prop;
  PCK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(SOPRO_ERR_UNSUPPORTED, "device is sm_%d%d; this build targets sm_100a only", prop.major, prop.minor);
  const int D = cfg->d_model, NL = cfg->n_layers, k = cfg->kernel, Q = cfg->n_codebooks, V = cfg->codebook_size, Hn = cfg->head_dim,
            AH = cfg->adapter_hidden, NS = cfg->n_stages;
  if (D < 32 || D > 512 || D % 16 || Hn % 16 || NL < 1 || NL > SOPRO_MAX_SSM_LAYERS || k < 1 || k > 64 || Q < 2 || Q > SOPRO_NAR_MAX_CODEBOOKS ||
      NS < 1 || NS > SOPRO_NAR_MAX_STAGES || V < 2 || AH < 1)
    return fail(SOPRO_ERR_INVALID, "unsupported NAR geometry (d_model=%d head_dim=%d layers=%d codebooks=%d stages=%d)", D, Hn, NL, Q, NS);
  for (int i = 0; i < NL; ++i)
    if (!block_ok(w->block[i]) || cfg->dilation[i] < 1) return fail(SOPRO_ERR_INVALID, "NAR block %d: null weight or bad dilation", i);
  if (!w->norm_w || !w->pre_w || !w->pre_b || !w->stage_emb || !w->adapter_norm_w || !w->adapter_w0 || !w->adapter_b0 || !w->adapter_w2 ||
      !w->adapter_b2 || !w->prev_cb_weights || !w->cb_embed)
    return fail(SOPRO_ERR_INVALID, "NAR: null weight pointer");
  int covered = 1;
  for (int s = 0; s < NS; ++s) {
    if (cfg->stage_first[s] != covered || cfg->stage_count[s] < 1 || !w->head_id_emb[s] || !w->mix[s])
      return fail(SOPRO_ERR_INVALID, "NAR stage %d: codebooks must be consecutive from 1 (first=%d count=%d)", s, cfg->stage_first[s],
                  cfg->stage_count[s]);
    for (int j = 0; j < cfg->stage_count[s]; ++j)
      if (covered + j >= Q || !w->head_w[covered + j] || !w->head_b[covered + j])
        return fail(SOPRO_ERR_INVALID, "NAR stage %d head %d: null weight or codebook out of range", s, j);
    covered += cfg->stage_count[s];
  }
  PCK(cudaSetDevice(device));
  sopro_nar* n = new sopro_nar();
  n->device = device;
  n->cfg = *cfg;
  FArena A;
  for (int i = 0; i < NL; ++i) add_block(A, w->block[i], D, k, &n->blk[i]);
  n->norm_w = A.add(w->norm_w, D);
  n->pre_w = A.add(w->pre_w, (size_t)Hn * D);
  n->pre_b = A.add(w->pre_b, Hn);
  n->adapter_norm_w = A.add(w->adapter_norm_w, D);
  n->emb = A.add(w->cb_embed, ((size_t)Q * V + 1) * D);
  for (int s = 0; s < NS; ++s) {
    sopro_nar::Stage S{};
    S.first = cfg->stage_first[s];
    S.count = cfg->stage_count[s];
    S.n_prev = S.first;  // codebooks 0 .. first-1 are decided when the stage runs
    // softmax over the previous codebooks' weights (model.py:332, nn/embeddings.py:94-108), in double
    {
      std::vector<double> e(S.n_prev);
      double mx = -1e300, sum = 0;
      for (int j = 0; j < S.n_prev; ++j) mx = std::max(mx, (double)w->prev_cb_weights[j]);
      for (int j = 0; j < S.n_prev; ++j) sum += (e[j] = exp((double)w->prev_cb_weights[j] - mx));
      std::vector<float> wp(S.n_prev);
      for (int j = 0; j < S.n_prev; ++j) wp[j] = (float)(e[j] / sum);
      S.w_prev = A.add(wp.data(), wp.size());
    }
    {
      const double a = w->mix[s][0], b = w->mix[s][1], mx = std::max(a, b);
      const double ea = exp(a - mx), eb = exp(b - mx);
      S.mix0 = (float)(ea / (ea + eb));
      S.mix1 = (float)(eb / (ea + eb));
    }
    // stage adapter MLP on the stage embedding (nn/nar.py:20-31): g, b = Linear(GELU(Linear(e))).chunk(2); constants
    {
      std::vector<double> hmid(AH);
      const float* e = w->stage_emb + (size_t)s * D;
      for (int i = 0; i < AH; ++i) {
        double acc = w->adapter_b0[i];
        for (int c = 0; c < D; ++c) acc += (double)w->adapter_w0[(size_t)i * D + c] * e[c];
        const double x = acc;
        hmid[i] = 0.5 * x * (1.0 + erf(x * 0.70710678118654752440));
      }
      std::vector<float> mul(D), add(D);
      for (int c = 0; c < 2 * D; ++c) {
        double acc = w->adapter_b2[c];
        for (int i = 0; i < AH; ++i) acc += (double)w->adapter_w2[(size_t)c * AH + i] * hmid[i];
        if (c < D) mul[c] = (float)(1.0 + tanh(acc));
        else add[c - D] = (float)tanh(acc);
      }
      S.mul = A.add(mul.data(), D);
      S.add = A.add(add.data(), D);
    }
    // the stage's heads, contiguous: W [count][V][Hn], bias [count][V], id embedding [count][Hn]
    S.head_w = A.add(nullptr, (size_t)S.count * V * Hn);
    S.head_b = A.add(nullptr, (size_t)S.count * V);
    for (int j = 0; j < S.count; ++j) {
      memcpy(A.host.data() + S.head_w + (size_t)j * V * Hn, w->head_w[S.first + j], (size_t)V * Hn * 4);
      memcpy(A.host.data() + S.head_b + (size_t)j * V, w->head_b[S.first + j], (size_t)V * 4);
    }
    S.head_id = A.add(w->head_id_emb[s], (size_t)S.count * Hn);
    {  // (z + e_h) . W_h^T + b_h = z . W_h^T + (b_h + W_h e_h): the head's id embedding folded into its bias
      std::vector<float> fb((size_t)S.count * V);
      for (int j = 0; j < S.count; ++j) {
        const float* Wh = w->head_w[S.first + j];
        const float* e = w->head_id_emb[s] + (size_t)j * Hn;
        for (int v = 0; v < V; ++v) {
          double acc = w->head_b[S.first + j][v];
          for (int c = 0; c < Hn; ++c) acc += (double)Wh[(size_t)v * Hn + c] * (double)e[c];
          fb[(size_t)j * V + v] = (float)acc;
        }
      }
      S.head_b_folded = A.add(fb.data(), fb.size());
    }
    n->stages.push_back(S);
  }
  // tensor-core images (W6) of every contraction; geometry the implicit-GEMM kernel takes: K blocks of 64, N tiles of 32+
  std::vector<uint16_t> T;
  const bool tc_ok = D % 64 == 0 && Hn % 64 == 0 && V % 32 == 0 && (2 * D) % 32 == 0;
  if (tc_ok) {
    for (int i = 0; i < NL; ++i) {
      n->tblk[i].glu = pack_w6(T, w->block[i].glu_w, (size_t)2 * D, D);
      n->tblk[i].w1 = pack_w6(T, w->block[i].ffn_w1, (size_t)4 * D, D);
      n->tblk[i].w2 = pack_w6(T, w->block[i].ffn_w2, D, (size_t)4 * D);
    }
    n->tc_pre = pack_w6(T, w->pre_w, Hn, D);
    for (auto& S : n->stages) {
      std::vector<float> hw((size_t)S.count * V * Hn);
      for (int j = 0; j < S.count; ++j) memcpy(hw.data() + (size_t)j * V * Hn, w->head_w[S.first + j], (size_t)V * Hn * 4);
      S.tc_heads = pack_w6(T, hw.data(), (size_t)S.count * V, Hn);
    }
  }
  n->n_floats = A.host.size();
  cudaError_t err = cudaMalloc(&n->dev, n->n_floats * 4);
  if (err == cudaSuccess) err = cudaMemcpy(n->dev, A.host.data(), n->n_floats * 4, cudaMemcpyHostToDevice);
  if (err == cudaSuccess && tc_ok) {
    err = cudaMalloc(&n->tcw, T.size() * 2);
    if (err == cudaSuccess) err = cudaMemcpy(n->tcw, T.data(), T.size() * 2, cudaMemcpyHostToDevice);
    n->tc_ok = err == cudaSuccess;
  }
  if (err != cudaSuccess) {
    if (n->dev) cudaFree(n->dev);
    if (n->tcw) cudaFree(n->tcw);
    delete n;
    return fail(SOPRO_ERR_CUDA, "NAR weight upload (%zu MB) failed: %s", (A.host.size() * 4 + T.size() * 2) >> 20, cudaGetErrorString(err));
  }
  *out = n;
  return SOPRO_OK;
}

int sopro_nar_destroy(sopro_nar_t* n) {
  if (!n) return SOPRO_OK;
  cudaSetDevice(n->device);
  nar_drop_replays(n);
  if (n->cap_stream) cudaStreamDestroy(n->cap_stream);
  if (n->g_done) cudaEventDestroy(n->g_done);
  cudaFree(n->g_cond);
  cudaFree(n->g_rvq1);
  cudaFree(n->g_codes);
  cudaFree(n->dev);
  cudaFree(n->tcw);
  cudaFree(n->ws);
  delete n;
  return SOPRO_OK;
}

// test hook (host only): the W6 image pack_w6 builds for W [N][K] -> out [N][6K] bf16 bit patterns
int sopro_debug_pack_w6(const float* W, int N, int K, uint16_t* out) {
  if (!W || !out || N < 1 || K < 1) return fail(SOPRO_ERR_INVALID, "bad argument");
  std::vector<uint16_t> T;
  const size_t off = pack_w6(T, W, (size_t)N, (size_t)K);
  memcpy(out, T.data() + off, (size_t)N * kPairs * K * 2);
  return SOPRO_OK;
}

int sopro_nar_set_contraction(sopro_nar_t* n, int mode) {
  if (!n || mode < -1 || mode > 1) return fail(SOPRO_ERR_INVALID, "bad argument");
  if (mode == 1 && !n->tc_ok) return fail(SOPRO_ERR_INVALID, "this NAR geometry has no tensor-core images");
  n->tc_mode = mode;
  return SOPRO_OK;
}

int sopro_nar_set_forced(sopro_nar_t* n, const int32_t* forced_codes) {
  if (!n) return fail(SOPRO_ERR_INVALID, "null argument");
  n->forced = forced_codes;
  return SOPRO_OK;
}

}  // extern "C"

// the refiner's launches on `st`; reserve_only: size (and grow) the workspace for this shape, launch nothing
static int nar_refine_impl(sopro_nar_t* n, const float* cond, int64_t cond_batch_stride, const int32_t* rvq1, const int32_t* lens, int B,
                           int Tmax, int32_t* codes, void* stream, bool reserve_only = false) {
  if (!n || (!reserve_only && (!cond || !rvq1 || !codes))) return fail(SOPRO_ERR_INVALID, "null argument");
  if (B < 1 || Tmax < 1 || (long long)B * Tmax > 0x3fffffffLL) return fail(SOPRO_ERR_INVALID, "bad B=%d Tmax=%d", B, Tmax);
  const sopro_nar_config_t& c = n->cfg;
  const int D = c.d_model, Q = c.n_codebooks, V = c.codebook_size, Hn = c.head_dim;
  if (cond_batch_stride < (int64_t)Tmax * D) return fail(SOPRO_ERR_INVALID, "cond_batch_stride smaller than Tmax*d_model");
  PCK(cudaSetDevice(n->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const long long M = (long long)B * Tmax;
  int max_heads = 1;
  for (const auto& S : n->stages) max_heads = std::max(max_heads, S.count);
  const size_t parts_max = (size_t)std::max(argmax_parts((int)M, V, 1), argmax_parts((int)M, V, max_heads));
  // Tensor cores (exact six-product split) for every row count the skinny fp32 kernel does not take; SOPRO_NAR_TC=0 keeps
  // the fp32 FMA tile kernels (the reference for tests/test_nar_gpu.py::test_tensor_core_path_equals_the_fp32_path)
  static const bool tc_env_off = getenv("SOPRO_NAR_TC") && atoi(getenv("SOPRO_NAR_TC")) == 0;
  const bool use_tc = n->tc_ok && !tc_env_off && n->tc_mode != 0 && M > dense::kSkinnyRows;
  // rows per head-logits chunk of the tensor-core path (logits [chunk][heads * V] fp32 reach memory there, <= 256 MB)
  long long mc = ((256ll << 20) / ((long long)max_heads * V * 4)) / 128 * 128;
  mc = std::max<long long>(128, std::min<long long>(mc, (M + 127) / 128 * 128));
  const size_t fx = (size_t)M * D, fh = (size_t)M * D, fhid = (size_t)M * 4 * D, fz = (size_t)M * Hn,
               famax = use_tc ? 0 : (size_t)max_heads * M * parts_max;
  auto al = [](size_t x) { return (x + 63) / 64 * 64; };
  const size_t fa3 = use_tc ? ((size_t)M * 3 * 4 * D + 1) / 2 : 0;          // bf16 [M][3 * 4D], in floats
  const size_t flog = use_tc ? (size_t)mc * max_heads * V : 0;
  const size_t need = std::max(n->reserve_bytes, (al(fx) + al(fh) + al(fhid) + al(fz) + 2 * al(famax) + al(fa3) + al(flog)) * 4);
  if (n->ws_bytes < need) {
    PCK(cudaStreamSynchronize(st));
    nar_drop_replays(n);  // the graphs hold pointers into the old workspace
    cudaFree(n->ws);
    n->ws = nullptr;
    n->ws_bytes = 0;
    cudaError_t e = cudaMalloc(&n->ws, need);
    if (e != cudaSuccess) return fail(SOPRO_ERR_CUDA, "NAR workspace %zu MB: %s", need >> 20, cudaGetErrorString(e));
    n->ws_bytes = need;
  }
  if (reserve_only) {
    n->reserve_bytes = std::max(n->reserve_bytes, need);
    return SOPRO_OK;
  }
  float* x = n->ws;
  float* h = x + al(fx);
  float* hid = h + al(fh);
  float* z = hid + al(fhid);
  float* amax_v = z + al(fz);
  int* amax_i = reinterpret_cast<int*>(amax_v + al(famax));
  __nv_bfloat16* a3 = reinterpret_cast<__nv_bfloat16*>(amax_v + 2 * al(famax));
  float* logits = amax_v + 2 * al(famax) + al(fa3);
  const float* W = n->dev;
  set_first_codebook_kernel<<<(unsigned)((M + 255) / 256), 256, 0, st>>>(rvq1, codes, M, Q);
  PCK(cudaGetLastError());
  for (const auto& S : n->stages) {
    EmbedMix em{};
    em.cond = cond; em.cond_bs = cond_batch_stride; em.codes = n->forced ? n->forced : codes; em.emb = W + n->emb; em.w_prev = W + S.w_prev;
    em.norm_w = W + n->adapter_norm_w; em.mul = W + S.mul; em.add = W + S.add; em.out = x; em.mix0 = S.mix0; em.mix1 = S.mix1;
    em.Tmax = Tmax; em.D = D; em.Q = Q; em.V = V; em.n_prev = S.n_prev;
    nar_embed_mix_kernel<<<(unsigned)((M + 7) / 8), 256, 0, st>>>(em, M);
    PCK(cudaGetLastError());
    int rc;
    if (use_tc) {
      for (int i = 0; i < c.n_layers; ++i)
        if ((rc = ssm_block_tc(W, n->blk[i], n->tcw, n->tblk[i], x, h, hid, a3, lens, B, Tmax, D, c.kernel, c.dilation[i], st))) return rc;
      const unsigned rb = (unsigned)((M + 7) / 8);
      split3_rows_kernel<<<rb, 256, 0, st>>>(x, W + n->norm_w, a3, M, D);
      if ((rc = launch_tc6(a3, n->tcw + n->tc_pre, W + n->pre_b, nullptr, z, M, Hn, D, tc::EPI_NONE, st))) return rc;
      split3_rows_kernel<<<rb, 256, 0, st>>>(z, nullptr, a3, M, Hn);
      for (long long m0 = 0; m0 < M; m0 += mc) {
        const long long rows = std::min<long long>(mc, M - m0);
        if ((rc = launch_tc6(a3 + m0 * 3 * Hn, n->tcw + S.tc_heads, W + S.head_b_folded, nullptr, logits, rows, S.count * V, Hn, tc::EPI_NONE, st)))
          return rc;
        argmax_heads_kernel<<<(unsigned)((rows * S.count + 7) / 8), 256, 0, st>>>(logits, rows, S.count, V, codes + m0 * Q + S.first, Q);
      }
      PCK(cudaGetLastError());
      continue;
    }
    for (int i = 0; i < c.n_layers; ++i)
      if ((rc = ssm_block(W, n->blk[i], x, h, hid, lens, B, Tmax, D, c.kernel, c.dilation[i], false, st))) return rc;
    dense::DenseOp g{};
    g.A = x; g.W = W + n->pre_w; g.bias = W + n->pre_b; g.norm_w = W + n->norm_w; g.C = z; g.M = (int)M; g.N = Hn; g.K = D; g.ldc = Hn;
    g.epi = dense::EPI_BIAS;
    if ((rc = launch_dense(g, 1, st))) return rc;
    g = dense::DenseOp{};
    g.A = z; g.W = W + S.head_w; g.bias = W + S.head_b; g.a_add = W + S.head_id; g.M = (int)M; g.N = V; g.K = Hn; g.epi = dense::EPI_ARGMAX;
    g.amax_val = amax_v; g.amax_idx = amax_i; g.zW = (size_t)V * Hn; g.zBias = V; g.zAdd = Hn;
    const int parts = argmax_parts((int)M, V, S.count);
    if ((rc = launch_dense(g, S.count, st))) return rc;
    dense::argmax_finish_kernel<<<dim3((unsigned)((M + 127) / 128), S.count), 128, 0, st>>>(amax_v, amax_i, (int)M, parts, codes + S.first, Q);
    PCK(cudaGetLastError());
  }
  return SOPRO_OK;
}

extern "C" {

int sopro_nar_set_graphs(sopro_nar_t* n, int enabled) {
  if (!n) return fail(SOPRO_ERR_INVALID, "null argument");
  n->graphs = enabled != 0;
  return SOPRO_OK;
}

int sopro_nar_refine(sopro_nar_t* n, const float* cond, int64_t cond_batch_stride, const int32_t* rvq1, const int32_t* lens, int B,
                     int Tmax, int32_t* codes, void* stream) {
  if (!n || !cond || !rvq1 || !codes) return fail(SOPRO_ERR_INVALID, "null argument");
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  cudaStreamCaptureStatus cap = cudaStreamCaptureStatusNone;
  PCK(cudaSetDevice(n->device));
  PCK(cudaStreamIsCapturing(st, &cap));
  // one utterance's streaming window: replay the whole pass (113..217 launches) from a graph over static buffers
  if (!n->graphs || B != 1 || Tmax < 1 || Tmax > kNarGraphRows || lens || n->forced || cap != cudaStreamCaptureStatusNone)
    return nar_refine_impl(n, cond, cond_batch_stride, rvq1, lens, B, Tmax, codes, stream);
  const sopro_nar_config_t& c = n->cfg;
  const int D = c.d_model, Q = c.n_codebooks;
  if (!n->g_cond) {
    PCK(cudaMalloc(&n->g_cond, (size_t)kNarGraphRows * D * 4));
    PCK(cudaMalloc(&n->g_rvq1, (size_t)kNarGraphRows * 4));
    PCK(cudaMalloc(&n->g_codes, (size_t)kNarGraphRows * Q * 4));
  }
  // no graph-sized call may reallocate the workspace: reserve the largest graph shape of either arithmetic path once
  if (n->reserve_bytes == 0) {
    int rc = nar_refine_impl(n, nullptr, (int64_t)kNarGraphRows * D, nullptr, nullptr, 1, kNarGraphRows, nullptr, stream, true);
    if (!rc) rc = nar_refine_impl(n, nullptr, (int64_t)dense::kSkinnyRows * D, nullptr, nullptr, 1, dense::kSkinnyRows, nullptr, stream, true);
    if (rc) return rc;
  }
  const int tc = n->tc_mode;
  cudaGraphExec_t exec = nullptr;
  for (auto& r : n->replays)
    if (r.T == Tmax && r.tc == tc) exec = r.exec;
  if (!exec) {
    if (n->replays.size() >= 96) nar_drop_replays(n);
    // warm-up outside the capture (first use of a kernel sets function attributes), then capture on a private stream
    int rc = nar_refine_impl(n, cond, cond_batch_stride, rvq1, nullptr, 1, Tmax, codes, stream);
    if (rc) return rc;
    if (!n->cap_stream) PCK(cudaStreamCreateWithFlags(&n->cap_stream, cudaStreamNonBlocking));
    PCK(cudaStreamBeginCapture(n->cap_stream, cudaStreamCaptureModeThreadLocal));
    rc = nar_refine_impl(n, n->g_cond, (int64_t)Tmax * D, n->g_rvq1, nullptr, 1, Tmax, n->g_codes, n->cap_stream);
    cudaGraph_t graph = nullptr;
    cudaError_t ce = cudaStreamEndCapture(n->cap_stream, &graph);
    if (rc || ce != cudaSuccess) {  // this call already ran eagerly; just do not cache
      if (graph) cudaGraphDestroy(graph);
      cudaGetLastError();
      return SOPRO_OK;
    }
    ce = cudaGraphInstantiate(&exec, graph, 0);
    cudaGraphDestroy(graph);
    if (ce == cudaSuccess) n->replays.push_back({Tmax, tc, exec});
    else cudaGetLastError();
    return SOPRO_OK;  // the eager warm-up produced this call's result
  }
  // replays from different caller streams share the static buffers: each waits for the previous one to finish
  if (!n->g_done) PCK(cudaEventCreateWithFlags(&n->g_done, cudaEventDisableTiming));
  else PCK(cudaStreamWaitEvent(st, n->g_done, 0));
  PCK(cudaMemcpyAsync(n->g_cond, cond, (size_t)Tmax * D * 4, cudaMemcpyDeviceToDevice, st));
  PCK(cudaMemcpyAsync(n->g_rvq1, rvq1, (size_t)Tmax * 4, cudaMemcpyDeviceToDevice, st));
  PCK(cudaGraphLaunch(exec, st));
  PCK(cudaMemcpyAsync(codes, n->g_codes, (size_t)Tmax * Q * 4, cudaMemcpyDeviceToDevice, st));
  PCK(cudaEventRecord(n->g_done, st));
  return SOPRO_OK;
}

}  // extern "C"

// =================================================================================================
// Prefill: SoproTTSModel.prepare_conditioning (reference model.py:172-216) batched over utterances that share one
// prepared reference voice:
//   TextEncoder (nn/text.py:29-44): embedding + sinusoid -> mask -> n SSMLiteBlocks (non-causal) -> RMSNorm -> masked mean
//   base[t] = txt_pool + frame_pos[t]                                 (model.py:200-202)
//   SpeakerFiLM (nn/speaker.py:76-85): LayerNorm(base) * (1 + s*tanh(gamma)) + s*tanh(beta)
//   3 x RefXAttnBlock with cached K/V (nn/ref.py:57-108): q = Wq RMSNorm(x); softmax(q K^T / sqrt(dh)) V; nan_to_num;
//       a *= clamp(rms(x) / rms(a), 0, 10); x += gmax*tanh(gate) * Wo a
//   cond_ar = RMSNorm(x)                                              (model.py:208)
// cond_ar and txt_seq are INPUTS of the id-exact AR kernel, hence fp32 everywhere.
// =================================================================================================
namespace pstage {

// x[b][l] = (emb[id] + pos[l]) * (l < len[b])      (nn/text.py:31-35)
__global__ void __launch_bounds__(128) text_embed_kernel(const int* __restrict__ ids, const int* __restrict__ len,
                                                         const float* __restrict__ emb, const float* __restrict__ pos,
                                                         float* __restrict__ x, int Lmax, int D, int vocab) {
  const int l = blockIdx.x, b = blockIdx.y;
  const bool live = l < len[b];
  const int id = min(max(ids[(size_t)b * Lmax + l], 0), vocab - 1);
  for (int c = threadIdx.x; c < D; c += blockDim.x)
    x[((size_t)b * Lmax + l) * D + c] = live ? __ldg(emb + (size_t)id * D + c) + __ldg(pos + (size_t)l * D + c) : 0.f;
}

// pool[b][c] = sum_{l < len} x[b][l][c] / (len + 1e-6)      (nn/text.py:41-43)
__global__ void __launch_bounds__(128) mean_pool_kernel(const float* __restrict__ x, const int* __restrict__ len,
                                                        float* __restrict__ pool, int Lmax, int D) {
  const int b = blockIdx.x;
  const int L = len[b];
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    float s = 0.f;
    for (int l = 0; l < L; ++l) s += x[((size_t)b * Lmax + l) * D + c];
    pool[(size_t)b * D + c] = s / ((float)L + 1e-6f);
  }
}

// one warp per (b, t) row: base = pool[b] + frame_pos[t]; LayerNorm (eps 1e-5, biased variance) * w + bias;
// y = ln * (1 + s*tanh(gamma[b])) + s*tanh(beta[b])         (film rows [Bf][2D], Bf = B or 1)
// film_index (per-utterance voices): utterance b reads film row film_index[b] instead
__global__ void __launch_bounds__(256) film_rows_kernel(const float* __restrict__ pool, const float* __restrict__ fpos,
                                                        const float* __restrict__ ln_w, const float* __restrict__ ln_b,
                                                        const float* __restrict__ film, int film_shared,
                                                        const int* __restrict__ film_index, float strength,
                                                        float* __restrict__ y, long long rows, int T, int D) {
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const long long b = row / T, t = row - b * T;
  constexpr int kMaxPer = 16;
  float v[kMaxPer];
  float s = 0.f;
  int n = 0;
  for (int k = lane; k < D; k += 32, ++n) {
    v[n] = pool[b * D + k] + __ldg(fpos + t * D + k);
    s += v[n];
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / (float)D;
  float var = 0.f;
  n = 0;
  for (int k = lane; k < D; k += 32, ++n) {
    const float d = v[n] - mean;
    var += d * d;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) var += __shfl_xor_sync(0xffffffffu, var, o);
  const float inv = 1.0f / sqrtf(var / (float)D + 1e-5f);
  const float* f = film + (film_index ? (long long)film_index[b] * 2 * D : film_shared ? 0 : b * 2 * D);
  n = 0;
  for (int k = lane; k < D; k += 32, ++n) {
    const float ln = (v[n] - mean) * inv * __ldg(ln_w + k) + __ldg(ln_b + k);
    y[row * D + k] = ln * (1.0f + strength * tanhf(f[k])) + strength * tanhf(f[D + k]);
  }
}

// Cached reference cross-attention core + RMS matching of ONE query row, by one warp (nn/ref.py:84-101):
//   per head: s_j = q.K_j / sqrt(dh); p = softmax(s); a = sum_j p_j V_j; nan_to_num
//   a *= clamp(rms(x) / rms(a), 0, 10) over the full row (both heads)
// K, V: [H][Tr][dh] (the row's reference voice).  Shared memory per warp: q [D] | p [Tr] | a [D], in regions sized for
// Tr_region >= Tr rows of p.  Both attention kernels below run this one instruction sequence, so a row's result depends
// only on its own voice.
__device__ __forceinline__ void ref_attn_row(const float* __restrict__ q, const float* __restrict__ x,
                                             const float* __restrict__ Kc, const float* __restrict__ Vc,
                                             float* __restrict__ out, long long row, int D, int H, int Tr, int Tr_region,
                                             float* rsm, int warp, int lane) {
  const int dh = D / H, Trp = (Tr + 3) & ~3;  // padded: the per-warp regions stay 16-byte aligned
  float* qs = rsm + (size_t)warp * (2 * D + ((Tr_region + 3) & ~3));
  float* ps = qs + D;
  float* as = ps + Trp;
  for (int k = lane; k < D; k += 32) qs[k] = q[row * D + k];
  __syncwarp();
  const float scale = 1.0f / sqrtf((float)dh);
  float ssa = 0.f;
  for (int h = 0; h < H; ++h) {
    const float* Kh = Kc + (size_t)h * Tr * dh;
    const float* Vh = Vc + (size_t)h * Tr * dh;
    float mx = -INFINITY;
    for (int j = lane; j < Tr; j += 32) {
      const float* kr = Kh + (size_t)j * dh;
      float s = 0.f;
      for (int d = 0; d < dh; d += 4) {
        const float4 kk = __ldg(reinterpret_cast<const float4*>(kr + d));
        const float4 qq = *reinterpret_cast<const float4*>(qs + h * dh + d);
        s += kk.x * qq.x + kk.y * qq.y + kk.z * qq.z + kk.w * qq.w;
      }
      s *= scale;
      ps[j] = s;
      mx = fmaxf(mx, s);
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
    float sum = 0.f;
    for (int j = lane; j < Tr; j += 32) {
      const float e = expf(ps[j] - mx);
      ps[j] = e;
      sum += e;
    }
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
    __syncwarp();
    const float inv = 1.0f / sum;
    for (int d = lane; d < dh; d += 32) {
      float o = 0.f;
      for (int j = 0; j < Tr; ++j) o += (ps[j] * inv) * __ldg(Vh + (size_t)j * dh + d);
      if (!isfinite(o)) o = 0.f;
      as[h * dh + d] = o;
      ssa += o * o;
    }
    __syncwarp();
  }
  float ssx = 0.f;
  for (int k = lane; k < D; k += 32) {
    const float xv = x[row * D + k];
    ssx += xv * xv;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    ssa += __shfl_xor_sync(0xffffffffu, ssa, o);
    ssx += __shfl_xor_sync(0xffffffffu, ssx, o);
  }
  const float rx = sqrtf(ssx / (float)D + 1e-6f), ra = sqrtf(ssa / (float)D + 1e-6f);
  const float sc = fminf(fmaxf(rx / ra, 0.0f), 10.0f);
  for (int k = lane; k < D; k += 32) out[row * D + k] = as[k] * sc;
}

// one shared reference voice: K, V [H][Tr][dh]
__global__ void __launch_bounds__(256) ref_attn_kernel(const float* __restrict__ q, const float* __restrict__ x,
                                                       const float* __restrict__ Kc, const float* __restrict__ Vc,
                                                       float* __restrict__ out, long long rows, int D, int H, int Tr) {
  extern __shared__ float rsm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + warp;
  if (row >= rows) return;
  ref_attn_row(q, x, Kc, Vc, out, row, D, H, Tr, Tr, rsm, warp, lane);
}

// a voice per utterance: row r belongs to utterance b = r / T and reads voice v = voice[b]: K, V = Kv[v], Vv[v]
// ([H][tr[v]][dh], this layer's).  The per-warp shared-memory regions are sized by Trmax, the largest tr[v].
__global__ void __launch_bounds__(256) ref_attn_voices_kernel(const float* __restrict__ q, const float* __restrict__ x,
                                                              const float* const* __restrict__ Kv, const float* const* __restrict__ Vv,
                                                              const int* __restrict__ voice, const int* __restrict__ tr,
                                                              float* __restrict__ out, long long rows, int T, int D, int H, int Trmax) {
  extern __shared__ float rsm[];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long row = (long long)blockIdx.x * 8 + warp;
  if (row >= rows) return;
  const int v = voice[(int)row / T];  // rows < 2^30 (sopro_prefill_run_voices checks B * n_frames)
  ref_attn_row(q, x, Kv[v], Vv[v], out, row, D, H, tr[v], Trmax, rsm, warp, lane);
}

}  // namespace pstage

struct sopro_prefill {
  int device = 0;
  sopro_prefill_config_t cfg{};
  float* dev = nullptr;
  size_t n_floats = 0;
  size_t text_emb = 0, text_pos = 0, frame_pos = 0, text_norm_w = 0, film_w0 = 0, film_b0 = 0, film_w2 = 0, film_b2 = 0, film_ln_w = 0,
         film_ln_b = 0, cond_norm_w = 0;
  BlockOff blk[SOPRO_MAX_SSM_LAYERS]{};
  struct Ref {
    size_t nq_w, q_w, o_w;
    float gate_eff;
  } ref[SOPRO_PREFILL_MAX_REF_LAYERS]{};
  float* ws = nullptr;
  size_t ws_bytes = 0;
  // pinned staging of sopro_prefill_run_voices' voice tables: the upload is asynchronous, pin_done marks when it has
  // read the buffer
  char* pin = nullptr;
  size_t pin_bytes = 0;
  cudaEvent_t pin_done = nullptr;
};

namespace pstage {

// The voices of sopro_prefill_run_voices, as the caller passed them (host arrays).
struct Voices {
  int n;                  // voices
  const int32_t* voice;   // [B] voice of each text
  const int32_t* tr;      // [n] Tr of each voice
  const float* const* k;  // [ref_layers * n] device pointers, entry l * n + v
  const float* const* v;
};

// Both prefill entry points after validation.  mv == nullptr: sopro_prefill_run (sv [B or 1], ref_k / ref_v / Tr of
// the shared voice).  Otherwise a voice per text: sv [mv->n][sv_dim], K / V and Tr from mv; the voice tables are staged
// in the workspace, and each voice's FiLM row is computed by the skinny kernel like a shared voice's (see below).
int prefill_run(sopro_prefill* p, const int32_t* text_ids, const int32_t* text_len, int B, int Lmax, const float* sv, int sv_shared,
                const float* const* ref_k, const float* const* ref_v, int Tr, const Voices* mv, float style_strength, int n_frames,
                float* txt_seq, float* txt_pool, float* cond_ar, void* stream) {
  const sopro_prefill_config_t& c = p->cfg;
  const int D = c.d_model, SV = c.sv_dim, H = c.ref_heads;
  PCK(cudaSetDevice(p->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const long long Mt = (long long)B * Lmax, Mc = (long long)B * n_frames;
  auto al = [](size_t x) { return (x + 63) / 64 * 64; };
  const size_t rows = (size_t)std::max(Mt, Mc);
  const int Bf = mv ? mv->n : sv_shared ? 1 : B;  // FiLM rows
  const int Bw = mv ? mv->n : B;
  // voice tables (mv): K / V pointers [ref_layers][2][n] | voice [B] | tr [n]
  const size_t n_ptr = mv ? (size_t)c.ref_layers * 2 * mv->n : 0, tab_bytes = mv ? n_ptr * 8 + ((size_t)B + mv->n) * 4 : 0;
  const size_t need = (al(rows * D) * 3 + al(rows * 4 * D) + al((size_t)Bw * D) + al((size_t)Bw * 2 * D) + al((tab_bytes + 3) / 4)) * 4;
  if (p->ws_bytes < need) {
    PCK(cudaStreamSynchronize(st));
    cudaFree(p->ws);
    p->ws = nullptr;
    p->ws_bytes = 0;
    cudaError_t e = cudaMalloc(&p->ws, need);
    if (e != cudaSuccess) return fail(SOPRO_ERR_CUDA, "prefill workspace %zu MB: %s", need >> 20, cudaGetErrorString(e));
    p->ws_bytes = need;
  }
  float* x = p->ws;
  float* h = x + al(rows * D);
  float* q = h + al(rows * D);
  float* hid = q + al(rows * D);
  float* fmid = hid + al(rows * 4 * D);      // [Bf][D] FiLM hidden
  float* film = fmid + al((size_t)Bw * D);   // [Bf][2D]
  float* tab = film + al((size_t)Bw * 2 * D);
  const float* const* tab_kv = reinterpret_cast<const float* const*>(tab);
  const int* tab_voice = reinterpret_cast<const int*>(reinterpret_cast<const char*>(tab) + n_ptr * 8);
  const int* tab_tr = mv ? tab_voice + B : nullptr;
  int Tra = Tr;  // the largest Tr of the call
  if (mv) {
    if (!p->pin_done) PCK(cudaEventCreateWithFlags(&p->pin_done, cudaEventDisableTiming));
    else PCK(cudaEventSynchronize(p->pin_done));  // the previous call's upload has read the staging buffer (normally long ago)
    if (p->pin_bytes < tab_bytes) {
      cudaFreeHost(p->pin);
      p->pin = nullptr;
      p->pin_bytes = 0;
      PCK(cudaMallocHost(reinterpret_cast<void**>(&p->pin), tab_bytes));
      p->pin_bytes = tab_bytes;
    }
    const float** kv = reinterpret_cast<const float**>(p->pin);
    for (int l = 0; l < c.ref_layers; ++l)
      for (int v = 0; v < mv->n; ++v) {
        kv[(size_t)(2 * l) * mv->n + v] = mv->k[(size_t)l * mv->n + v];
        kv[(size_t)(2 * l + 1) * mv->n + v] = mv->v[(size_t)l * mv->n + v];
      }
    memcpy(p->pin + n_ptr * 8, mv->voice, (size_t)B * 4);
    memcpy(p->pin + n_ptr * 8 + (size_t)B * 4, mv->tr, (size_t)mv->n * 4);
    PCK(cudaMemcpyAsync(tab, p->pin, tab_bytes, cudaMemcpyHostToDevice, st));
    PCK(cudaEventRecord(p->pin_done, st));
    Tra = *std::max_element(mv->tr, mv->tr + mv->n);
  }
  const float* W = p->dev;
  int rc;
  // ---- text encoder
  text_embed_kernel<<<dim3(Lmax, B), 128, 0, st>>>(text_ids, text_len, W + p->text_emb, W + p->text_pos, x, Lmax, D, c.text_vocab);
  PCK(cudaGetLastError());
  for (int i = 0; i < c.n_layers_text; ++i)
    if ((rc = ssm_block(W, p->blk[i], x, h, hid, text_len, B, Lmax, D, c.text_kernel, 1, false, st))) return rc;
  dense::rmsnorm_rows_kernel<<<(unsigned)((Mt + 7) / 8), 256, 0, st>>>(x, W + p->text_norm_w, nullptr, nullptr, txt_seq, Mt, D);
  PCK(cudaGetLastError());
  mean_pool_kernel<<<B, 128, 0, st>>>(txt_seq, text_len, txt_pool, Lmax, D);
  PCK(cudaGetLastError());
  // ---- FiLM parameters from the speaker vector(s).  Per voice in launches of at most 16 rows: the skinny kernel stages
  // 16 rows whatever M is and reduces every row through the same butterfly, so a voice's row is bit-equal to the M = 1
  // launch of a shared voice.  One launch of more than 16 rows would take the tile kernel, which sums in another order.
  const int chunk = mv ? dense::kSkinnyRows : Bf;
  for (int r0 = 0; r0 < Bf; r0 += chunk) {
    const int m = std::min(chunk, Bf - r0);
    dense::DenseOp g{};
    g.A = sv + (size_t)r0 * SV; g.W = W + p->film_w0; g.bias = W + p->film_b0; g.C = fmid + (size_t)r0 * D; g.M = m; g.N = D; g.K = SV;
    g.ldc = D; g.epi = dense::EPI_GELU;
    if ((rc = launch_dense(g, 1, st))) return rc;
    g = dense::DenseOp{};
    g.A = fmid + (size_t)r0 * D; g.W = W + p->film_w2; g.bias = W + p->film_b2; g.C = film + (size_t)r0 * 2 * D; g.M = m; g.N = 2 * D;
    g.K = D; g.ldc = 2 * D; g.epi = dense::EPI_BIAS;
    if ((rc = launch_dense(g, 1, st))) return rc;
  }
  film_rows_kernel<<<(unsigned)((Mc + 7) / 8), 256, 0, st>>>(txt_pool, W + p->frame_pos, W + p->film_ln_w, W + p->film_ln_b, film, sv_shared ? 1 : 0,
                                                            mv ? tab_voice : nullptr, style_strength, x, Mc, n_frames, D);
  PCK(cudaGetLastError());
  // ---- reference cross-attention stack
  const size_t rsmem = (size_t)8 * (2 * D + ((Tra + 3) & ~3)) * 4;
  if (c.ref_layers > 0 && rsmem > 48 * 1024) {
    static bool attr = false, attr_voices = false;
    bool& done = mv ? attr_voices : attr;
    if (!done) {
      if (mv) PCK(cudaFuncSetAttribute(ref_attn_voices_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      else PCK(cudaFuncSetAttribute(ref_attn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024));
      done = true;
    }
  }
  for (int i = 0; i < c.ref_layers; ++i) {
    dense::DenseOp g{};
    g.A = x; g.W = W + p->ref[i].q_w; g.norm_w = W + p->ref[i].nq_w; g.C = q; g.M = (int)Mc; g.N = D; g.K = D; g.ldc = D; g.epi = dense::EPI_BIAS;
    if ((rc = launch_dense(g, 1, st))) return rc;
    if (mv)
      ref_attn_voices_kernel<<<(unsigned)((Mc + 7) / 8), 256, rsmem, st>>>(q, x, tab_kv + (size_t)(2 * i) * mv->n, tab_kv + (size_t)(2 * i + 1) * mv->n,
                                                                           tab_voice, tab_tr, h, Mc, n_frames, D, H, Tra);
    else
      ref_attn_kernel<<<(unsigned)((Mc + 7) / 8), 256, rsmem, st>>>(q, x, ref_k[i], ref_v[i], h, Mc, D, H, Tr);
    PCK(cudaGetLastError());
    g = dense::DenseOp{};
    g.A = h; g.W = W + p->ref[i].o_w; g.R = x; g.C = x; g.M = (int)Mc; g.N = D; g.K = D; g.ldc = D; g.epi = dense::EPI_RES_GATE;
    g.gate = p->ref[i].gate_eff;
    if ((rc = launch_dense(g, 1, st))) return rc;
  }
  dense::rmsnorm_rows_kernel<<<(unsigned)((Mc + 7) / 8), 256, 0, st>>>(x, W + p->cond_norm_w, nullptr, nullptr, cond_ar, Mc, D);
  PCK(cudaGetLastError());
  return SOPRO_OK;
}

int check_batch(const sopro_prefill* p, int B, int Lmax, int n_frames) {
  const sopro_prefill_config_t& c = p->cfg;
  if (B < 1 || Lmax < 1 || Lmax > c.max_text_len || n_frames < 1 || n_frames > c.max_frames_pos || (long long)B * n_frames > 0x3fffffffLL)
    return fail(SOPRO_ERR_INVALID, "bad B=%d Lmax=%d (max %d) n_frames=%d (max %d)", B, Lmax, c.max_text_len, n_frames, c.max_frames_pos);
  return SOPRO_OK;
}

}  // namespace pstage

extern "C" {

int sopro_prefill_create(const sopro_prefill_config_t* cfg, const sopro_prefill_weights_t* w, int device, sopro_prefill_t** out) {
  if (!cfg || !w || !out) return fail(SOPRO_ERR_INVALID, "null argument");
  *out = nullptr;
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev <= 0) return fail(SOPRO_ERR_UNSUPPORTED, "no CUDA device; the prefill has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(SOPRO_ERR_INVALID, "device %d out of range", device);
  cudaDeviceProp prop;
  PCK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(SOPRO_ERR_UNSUPPORTED, "device is sm_%d%d; this build targets sm_100a only", prop.major, prop.minor);
  const int D = cfg->d_model, NL = cfg->n_layers_text, k = cfg->text_kernel, SV = cfg->sv_dim, RL = cfg->ref_layers, H = cfg->ref_heads;
  if (D < 32 || D > 512 || D % 16 || NL < 0 || NL > SOPRO_MAX_SSM_LAYERS || k < 1 || k > 64 || SV < 16 || SV % 16 || RL < 0 ||
      RL > SOPRO_PREFILL_MAX_REF_LAYERS || H < 1 || D % H || (D / H) % 4 || cfg->text_vocab < 1 || cfg->max_text_len < 1 || cfg->max_frames_pos < 1)
    return fail(SOPRO_ERR_INVALID, "unsupported prefill geometry");
  for (int i = 0; i < NL; ++i)
    if (!block_ok(w->text_block[i])) return fail(SOPRO_ERR_INVALID, "text block %d: null weight", i);
  if (!w->text_emb || !w->text_pos || !w->frame_pos || !w->text_norm_w || !w->film_w0 || !w->film_b0 || !w->film_w2 || !w->film_b2 ||
      !w->film_norm_w || !w->film_norm_b || !w->cond_norm_w)
    return fail(SOPRO_ERR_INVALID, "prefill: null weight pointer");
  for (int i = 0; i < RL; ++i)
    if (!w->ref_layer[i].nq_w || !w->ref_layer[i].q_w || !w->ref_layer[i].o_w) return fail(SOPRO_ERR_INVALID, "ref layer %d: null weight", i);
  PCK(cudaSetDevice(device));
  sopro_prefill* p = new sopro_prefill();
  p->device = device;
  p->cfg = *cfg;
  FArena A;
  p->text_emb = A.add(w->text_emb, (size_t)cfg->text_vocab * D);
  p->text_pos = A.add(w->text_pos, (size_t)cfg->max_text_len * D);
  p->frame_pos = A.add(w->frame_pos, (size_t)cfg->max_frames_pos * D);
  for (int i = 0; i < NL; ++i) add_block(A, w->text_block[i], D, k, &p->blk[i]);
  p->text_norm_w = A.add(w->text_norm_w, D);
  p->film_w0 = A.add(w->film_w0, (size_t)D * SV);
  p->film_b0 = A.add(w->film_b0, D);
  p->film_w2 = A.add(w->film_w2, (size_t)2 * D * D);
  p->film_b2 = A.add(w->film_b2, 2 * D);
  p->film_ln_w = A.add(w->film_norm_w, D);
  p->film_ln_b = A.add(w->film_norm_b, D);
  for (int i = 0; i < RL; ++i) {
    p->ref[i].nq_w = A.add(w->ref_layer[i].nq_w, D);
    p->ref[i].q_w = A.add(w->ref_layer[i].q_w, (size_t)D * D);
    p->ref[i].o_w = A.add(w->ref_layer[i].o_w, (size_t)D * D);
    p->ref[i].gate_eff = cfg->ref_gmax * tanhf(w->ref_layer[i].gate);
  }
  p->cond_norm_w = A.add(w->cond_norm_w, D);
  p->n_floats = A.host.size();
  cudaError_t err = cudaMalloc(&p->dev, p->n_floats * 4);
  if (err == cudaSuccess) err = cudaMemcpy(p->dev, A.host.data(), p->n_floats * 4, cudaMemcpyHostToDevice);
  if (err != cudaSuccess) {
    if (p->dev) cudaFree(p->dev);
    delete p;
    return fail(SOPRO_ERR_CUDA, "prefill weight upload failed: %s", cudaGetErrorString(err));
  }
  *out = p;
  return SOPRO_OK;
}

int sopro_prefill_destroy(sopro_prefill_t* p) {
  if (!p) return SOPRO_OK;
  cudaSetDevice(p->device);
  if (p->pin_done) {
    cudaEventSynchronize(p->pin_done);
    cudaEventDestroy(p->pin_done);
  }
  cudaFreeHost(p->pin);
  cudaFree(p->dev);
  cudaFree(p->ws);
  delete p;
  return SOPRO_OK;
}

int sopro_prefill_run(sopro_prefill_t* p, const int32_t* text_ids, const int32_t* text_len, int B, int Lmax, const float* sv,
                      int sv_shared, const float* const* ref_k, const float* const* ref_v, int Tr, float style_strength, int n_frames,
                      float* txt_seq, float* txt_pool, float* cond_ar, void* stream) {
  if (!p || !text_ids || !text_len || !sv || !txt_seq || !txt_pool || !cond_ar) return fail(SOPRO_ERR_INVALID, "null argument");
  int rc;
  if ((rc = check_batch(p, B, Lmax, n_frames))) return rc;
  if (p->cfg.ref_layers > 0 && (!ref_k || !ref_v || Tr < 1 || Tr > 4096)) return fail(SOPRO_ERR_INVALID, "reference K/V missing or Tr=%d out of range", Tr);
  return prefill_run(p, text_ids, text_len, B, Lmax, sv, sv_shared, ref_k, ref_v, Tr, nullptr, style_strength, n_frames, txt_seq, txt_pool,
                     cond_ar, stream);
}

int sopro_prefill_run_voices(sopro_prefill_t* p, const int32_t* text_ids, const int32_t* text_len, int B, int Lmax, const int32_t* voice,
                             int n_voices, const float* sv, const int32_t* ref_len, const float* const* ref_k, const float* const* ref_v,
                             float style_strength, int n_frames, float* txt_seq, float* txt_pool, float* cond_ar, void* stream) {
  if (!p || !text_ids || !text_len || !voice || !sv || !ref_len || !txt_seq || !txt_pool || !cond_ar)
    return fail(SOPRO_ERR_INVALID, "null argument");
  int rc;
  if ((rc = check_batch(p, B, Lmax, n_frames))) return rc;
  if (n_voices < 1) return fail(SOPRO_ERR_INVALID, "n_voices=%d: at least one voice is needed", n_voices);
  for (int b = 0; b < B; ++b)
    if (voice[b] < 0 || voice[b] >= n_voices) return fail(SOPRO_ERR_INVALID, "voice[%d]=%d out of range [0, %d)", b, voice[b], n_voices);
  for (int v = 0; v < n_voices; ++v)
    if (ref_len[v] < 1 || ref_len[v] > 4096) return fail(SOPRO_ERR_INVALID, "ref_len[%d]=%d out of range [1, 4096]", v, ref_len[v]);
  const int RL = p->cfg.ref_layers;
  if (RL > 0 && (!ref_k || !ref_v)) return fail(SOPRO_ERR_INVALID, "reference K/V tables missing");
  for (long long i = 0; i < (long long)RL * n_voices; ++i)
    if (!ref_k[i] || !ref_v[i])
      return fail(SOPRO_ERR_INVALID, "reference K/V of layer %lld, voice %lld is null", i / n_voices, i % n_voices);
  const Voices mv{n_voices, voice, ref_len, ref_k, ref_v};
  return prefill_run(p, text_ids, text_len, B, Lmax, sv, 0, nullptr, nullptr, 0, &mv, style_strength, n_frames, txt_seq, txt_pool, cond_ar,
                     stream);
}

}  // extern "C"

// =================================================================================================
// Reference preparation: SoproTTSModel.prepare_reference (reference model.py:152-170), once per voice, from the voice's
// codes [Tr][Q]:
//   Token2SV (nn/speaker.py:12-61): softmax(cb_weights)-weighted sum of per-codebook embeddings -> 2 x (depthwise conv k7,
//       non-causal, GELU) -> AttentiveStatsPool (nn/blocks.py:165-188: softmax_t(w2 . tanh(W0 h + b0) + b2), weighted mean
//       and std) -> Linear -> L2 normalise                                               -> sv_ref [sv_dim]
//   _encode_reference_seq (model.py:136-150): softmax(ref_cb_weights)-weighted sum of cb_embed rows -> SSMLiteBlocks
//       (non-causal) -> RMSNorm                                                           -> ref_seq [Tr][D]
//   RefXAttnStack.build_kv_caches (nn/ref.py): per layer K = Wk RMSNorm_kv(ref_seq), V = Wv RMSNorm_kv(ref_seq), stored
//       [H][Tr][D/H]                                                                      -> the prefill engine's ref_k / ref_v
// fp32 (everything here feeds cond_ar, an input of the id-exact AR kernel).
// =================================================================================================
namespace pstage {

// out[t][c] = sum_q w[q] * emb[(q*V + tok[t][q]) * dim + c], q ascending (the reference's loop order); a code outside
// [0, V) is clamped and flagged
__global__ void __launch_bounds__(128) codes_mix_kernel(const int* __restrict__ tok, const float* __restrict__ emb,
                                                        const float* __restrict__ w, float* __restrict__ out, int Q, int V, int dim,
                                                        int* __restrict__ bad) {
  const int t = blockIdx.x;
  extern __shared__ int ids[];
  for (int q = threadIdx.x; q < Q; q += blockDim.x) {
    int id = tok[(size_t)t * Q + q];
    if (id < 0 || id >= V) {
      atomicExch(bad, 1);
      id = min(max(id, 0), V - 1);
    }
    ids[q] = id;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < dim; c += blockDim.x) {
    float acc = 0.f;
    for (int q = 0; q < Q; ++q) acc = __fadd_rn(acc, __fmul_rn(__ldg(w + q), __ldg(emb + ((size_t)q * V + ids[q]) * dim + c)));
    out[(size_t)t * dim + c] = acc;
  }
}

// y[t][c] = gelu(bias[c] + sum_j x[t + j - left][c] * w[c][j])   (DepthwiseConv1d non-causal + GELU, zero padding)
__global__ void __launch_bounds__(128) dwconv_gelu_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                          const float* __restrict__ bias, float* __restrict__ y, int T, int D, int k,
                                                          int left) {
  const int t = blockIdx.x;
  for (int c = threadIdx.x; c < D; c += blockDim.x) {
    float acc = 0.f;
    for (int j = 0; j < k; ++j) {
      const int r = t + j - left;
      if (r >= 0 && r < T) acc = fmaf(x[(size_t)r * D + c], __ldg(w + c * k + j), acc);
    }
    y[(size_t)t * D + c] = dense::gelu_erf(acc + __ldg(bias + c));
  }
}

// AttentiveStatsPool tail: u [T][D] = W0 h + b0 (from the dense kernel); logits[t] = w2 . tanh(u[t]) + b2; a = softmax_t;
// mu = sum_t a h; std = sqrt(max(sum_t a (h - mu)^2, 1e-6)); out = [mu | std]  (one CTA; T floats of shared memory)
__global__ void __launch_bounds__(256) attn_stats_pool_kernel(const float* __restrict__ u, const float* __restrict__ h,
                                                              const float* __restrict__ w2, float b2, float* __restrict__ out, int T,
                                                              int D) {
  extern __shared__ float a[];
  __shared__ float red[8];
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  for (int t = warp; t < T; t += 8) {
    float s = 0.f;
    for (int c = lane; c < D; c += 32) s = fmaf(__ldg(w2 + c), tanhf(u[(size_t)t * D + c]), s);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
    if (lane == 0) a[t] = s + b2;
  }
  __syncthreads();
  float mx = -INFINITY;
  for (int t = threadIdx.x; t < T; t += 256) mx = fmaxf(mx, a[t]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if (lane == 0) red[warp] = mx;
  __syncthreads();
  mx = red[0];
  for (int i = 1; i < 8; ++i) mx = fmaxf(mx, red[i]);
  __syncthreads();
  float sum = 0.f;
  for (int t = threadIdx.x; t < T; t += 256) {
    const float e = expf(a[t] - mx);
    a[t] = e;
    sum += e;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  if (lane == 0) red[warp] = sum;
  __syncthreads();
  sum = 0.f;
  for (int i = 0; i < 8; ++i) sum += red[i];
  const float inv = 1.0f / sum;
  for (int c = threadIdx.x; c < D; c += 256) {
    float mu = 0.f;
    for (int t = 0; t < T; ++t) mu = fmaf(h[(size_t)t * D + c], a[t] * inv, mu);
    float var = 0.f;
    for (int t = 0; t < T; ++t) {
      const float d = h[(size_t)t * D + c] - mu;
      var = fmaf(a[t] * inv, d * d, var);
    }
    out[c] = mu;
    out[D + c] = sqrtf(fmaxf(var, 1e-6f));
  }
}

// F.normalize(e, eps): e / max(||e||, eps), one warp
__global__ void l2_normalize_kernel(const float* __restrict__ e, float* __restrict__ out, int n, float eps) {
  const int lane = threadIdx.x;
  float s = 0.f;
  for (int i = lane; i < n; i += 32) s = fmaf(e[i], e[i], s);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float d = fmaxf(sqrtf(s), eps);
  for (int i = lane; i < n; i += 32) out[i] = e[i] / d;
}

// [T][H*Dh] -> [H][T][Dh]
__global__ void heads_major_kernel(const float* __restrict__ x, float* __restrict__ y, int T, int H, int Dh) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)T * H * Dh) return;
  const int d = (int)(i % Dh), t = (int)((i / Dh) % T), h = (int)(i / ((long long)Dh * T));
  y[i] = x[(size_t)t * H * Dh + h * Dh + d];
}

}  // namespace pstage

struct sopro_refprep {
  int device = 0;
  sopro_refprep_config_t cfg{};
  float* dev = nullptr;
  size_t sv_emb = 0, sv_w = 0, dw0_w = 0, dw0_b = 0, dw1_w = 0, dw1_b = 0, pool_w0 = 0, pool_b0 = 0, pool_w2 = 0, proj_w = 0, proj_b = 0,
         cb_embed = 0, ref_w = 0, ref_norm_w = 0;
  float pool_b2 = 0.f;
  BlockOff blk[SOPRO_MAX_SSM_LAYERS]{};
  struct Layer {
    size_t nkv_w, k_w, v_w;
  } layer[SOPRO_PREFILL_MAX_REF_LAYERS]{};
  float* ws = nullptr;
  size_t ws_bytes = 0;
  int* bad = nullptr;
};

extern "C" {

int sopro_refprep_create(const sopro_refprep_config_t* cfg, const sopro_refprep_weights_t* w, int device, sopro_refprep_t** out) {
  if (!cfg || !w || !out) return fail(SOPRO_ERR_INVALID, "null argument");
  *out = nullptr;
  int ndev = 0;
  cudaError_t ce = cudaGetDeviceCount(&ndev);
  if (ce != cudaSuccess || ndev <= 0) return fail(SOPRO_ERR_UNSUPPORTED, "no CUDA device; the reference preparation has no CPU fallback");
  if (device < 0 || device >= ndev) return fail(SOPRO_ERR_INVALID, "device %d out of range", device);
  cudaDeviceProp prop;
  PCK(cudaGetDeviceProperties(&prop, device));
  if (prop.major != 10) return fail(SOPRO_ERR_UNSUPPORTED, "device is sm_%d%d; this build targets sm_100a only", prop.major, prop.minor);
  const int D = cfg->d_model, d = cfg->sv_embed_dim, SV = cfg->sv_dim, Q = cfg->n_codebooks, V = cfg->codebook_size, NL = cfg->ref_enc_layers,
            RL = cfg->ref_layers, H = cfg->ref_heads;
  if (D < 32 || D > 512 || D % 16 || d < 16 || d % 16 || SV < 16 || SV % 16 || Q < 1 || Q > 64 || V < 1 || NL < 0 || NL > SOPRO_MAX_SSM_LAYERS ||
      RL < 0 || RL > SOPRO_PREFILL_MAX_REF_LAYERS || H < 1 || D % H || cfg->sv_kernel < 1 || cfg->sv_kernel > 64 || cfg->ref_enc_kernel < 1 ||
      cfg->ref_enc_kernel > 64)
    return fail(SOPRO_ERR_INVALID, "unsupported reference-preparation geometry");
  if (!w->sv_emb || !w->sv_cb_weights || !w->sv_dw0_w || !w->sv_dw0_b || !w->sv_dw1_w || !w->sv_dw1_b || !w->pool_w0 || !w->pool_b0 || !w->pool_w2 ||
      !w->proj_w || !w->proj_b || !w->cb_embed || !w->ref_cb_weights || !w->ref_norm_w)
    return fail(SOPRO_ERR_INVALID, "reference preparation: null weight pointer");
  for (int i = 0; i < NL; ++i)
    if (!block_ok(w->ref_block[i])) return fail(SOPRO_ERR_INVALID, "reference encoder block %d: null weight", i);
  for (int i = 0; i < RL; ++i)
    if (!w->layer[i].nkv_w || !w->layer[i].k_w || !w->layer[i].v_w) return fail(SOPRO_ERR_INVALID, "ref layer %d: null weight", i);
  PCK(cudaSetDevice(device));
  sopro_refprep* p = new sopro_refprep();
  p->device = device;
  p->cfg = *cfg;
  FArena A;
  auto softmax = [&](const float* x) {  // F.softmax(cb_weights, dim=0), fp32
    std::vector<float> s(Q);
    float mx = x[0];
    for (int q = 1; q < Q; ++q) mx = std::max(mx, x[q]);
    float sum = 0.f;
    for (int q = 0; q < Q; ++q) sum += (s[q] = expf(x[q] - mx));
    for (int q = 0; q < Q; ++q) s[q] /= sum;
    return A.add(s.data(), Q);
  };
  p->sv_emb = A.add(w->sv_emb, (size_t)Q * V * d);
  p->sv_w = softmax(w->sv_cb_weights);
  p->dw0_w = A.add(w->sv_dw0_w, (size_t)d * cfg->sv_kernel);
  p->dw0_b = A.add(w->sv_dw0_b, d);
  p->dw1_w = A.add(w->sv_dw1_w, (size_t)d * cfg->sv_kernel);
  p->dw1_b = A.add(w->sv_dw1_b, d);
  p->pool_w0 = A.add(w->pool_w0, (size_t)d * d);
  p->pool_b0 = A.add(w->pool_b0, d);
  p->pool_w2 = A.add(w->pool_w2, d);
  p->pool_b2 = w->pool_b2;
  p->proj_w = A.add(w->proj_w, (size_t)SV * 2 * d);
  p->proj_b = A.add(w->proj_b, SV);
  p->cb_embed = A.add(w->cb_embed, (size_t)Q * V * D);
  p->ref_w = softmax(w->ref_cb_weights);
  for (int i = 0; i < NL; ++i) add_block(A, w->ref_block[i], D, cfg->ref_enc_kernel, &p->blk[i]);
  p->ref_norm_w = A.add(w->ref_norm_w, D);
  for (int i = 0; i < RL; ++i) {
    p->layer[i].nkv_w = A.add(w->layer[i].nkv_w, D);
    p->layer[i].k_w = A.add(w->layer[i].k_w, (size_t)D * D);
    p->layer[i].v_w = A.add(w->layer[i].v_w, (size_t)D * D);
  }
  cudaError_t err = cudaMalloc(&p->dev, A.host.size() * 4);
  if (err == cudaSuccess) err = cudaMemcpy(p->dev, A.host.data(), A.host.size() * 4, cudaMemcpyHostToDevice);
  if (err == cudaSuccess) err = cudaMalloc(&p->bad, 256);
  if (err == cudaSuccess) err = cudaMemset(p->bad, 0, 256);
  if (err != cudaSuccess) {
    if (p->dev) cudaFree(p->dev);
    if (p->bad) cudaFree(p->bad);
    delete p;
    return fail(SOPRO_ERR_CUDA, "reference-preparation weight upload failed: %s", cudaGetErrorString(err));
  }
  *out = p;
  return SOPRO_OK;
}

int sopro_refprep_destroy(sopro_refprep_t* p) {
  if (!p) return SOPRO_OK;
  cudaSetDevice(p->device);
  cudaFree(p->dev);
  cudaFree(p->ws);
  cudaFree(p->bad);
  delete p;
  return SOPRO_OK;
}

int sopro_refprep_run(sopro_refprep_t* p, const int32_t* tokens, int Tr, float* sv, float* ref_seq, float* const* ref_k, float* const* ref_v,
                      void* stream) {
  if (!p || !tokens || !sv || !ref_seq) return fail(SOPRO_ERR_INVALID, "null argument");
  const sopro_refprep_config_t& c = p->cfg;
  if (Tr < 1 || Tr > 4096) return fail(SOPRO_ERR_INVALID, "Tr=%d outside [1, 4096]", Tr);
  if (c.ref_layers > 0 && (!ref_k || !ref_v)) return fail(SOPRO_ERR_INVALID, "ref_k / ref_v missing");
  for (int i = 0; i < c.ref_layers; ++i)
    if (!ref_k[i] || !ref_v[i]) return fail(SOPRO_ERR_INVALID, "ref_k[%d] / ref_v[%d] is null", i, i);
  PCK(cudaSetDevice(p->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  const int D = c.d_model, d = c.sv_embed_dim, SV = c.sv_dim, Q = c.n_codebooks, V = c.codebook_size, H = c.ref_heads;
  auto al = [](size_t x) { return (x + 63) / 64 * 64; };
  const size_t rows = (size_t)Tr;
  const size_t need = (al(rows * D) * 3 + al(rows * 4 * D) + al(2 * (size_t)d) + al((size_t)SV)) * 4;
  if (p->ws_bytes < need) {
    PCK(cudaStreamSynchronize(st));
    cudaFree(p->ws);
    p->ws = nullptr;
    p->ws_bytes = 0;
    cudaError_t e = cudaMalloc(&p->ws, need);
    if (e != cudaSuccess) return fail(SOPRO_ERR_CUDA, "reference-preparation workspace: %s", cudaGetErrorString(e));
    p->ws_bytes = need;
  }
  float* x = p->ws;
  float* h = x + al(rows * D);
  float* q = h + al(rows * D);
  float* hid = q + al(rows * D);
  float* stats = hid + al(rows * 4 * D);  // [2d]
  float* e = stats + al(2 * (size_t)d);   // [SV]
  const float* W = p->dev;
  int rc;
  dense::DenseOp g{};
  // ---- Token2SV (d <= D: the [Tr][d] buffers live in x / h / q)
  codes_mix_kernel<<<Tr, 128, Q * sizeof(int), st>>>(tokens, W + p->sv_emb, W + p->sv_w, x, Q, V, d, p->bad);
  PCK(cudaGetLastError());
  const int left = (c.sv_kernel - 1) / 2;
  dwconv_gelu_kernel<<<Tr, 128, 0, st>>>(x, W + p->dw0_w, W + p->dw0_b, h, Tr, d, c.sv_kernel, left);
  dwconv_gelu_kernel<<<Tr, 128, 0, st>>>(h, W + p->dw1_w, W + p->dw1_b, x, Tr, d, c.sv_kernel, left);
  PCK(cudaGetLastError());
  g.A = x; g.W = W + p->pool_w0; g.bias = W + p->pool_b0; g.C = q; g.M = Tr; g.N = d; g.K = d; g.ldc = d; g.epi = dense::EPI_BIAS;
  if ((rc = launch_dense(g, 1, st))) return rc;
  attn_stats_pool_kernel<<<1, 256, (size_t)Tr * 4, st>>>(q, x, W + p->pool_w2, p->pool_b2, stats, Tr, d);
  PCK(cudaGetLastError());
  g = dense::DenseOp{};
  g.A = stats; g.W = W + p->proj_w; g.bias = W + p->proj_b; g.C = e; g.M = 1; g.N = SV; g.K = 2 * d; g.ldc = SV; g.epi = dense::EPI_BIAS;
  if ((rc = launch_dense(g, 1, st))) return rc;
  l2_normalize_kernel<<<1, 32, 0, st>>>(e, sv, SV, 1e-6f);
  PCK(cudaGetLastError());
  // ---- reference encoder
  codes_mix_kernel<<<Tr, 128, Q * sizeof(int), st>>>(tokens, W + p->cb_embed, W + p->ref_w, x, Q, V, D, p->bad);
  PCK(cudaGetLastError());
  for (int i = 0; i < c.ref_enc_layers; ++i)
    if ((rc = ssm_block(W, p->blk[i], x, h, hid, nullptr, 1, Tr, D, c.ref_enc_kernel, 1, false, st))) return rc;
  dense::rmsnorm_rows_kernel<<<(unsigned)((Tr + 7) / 8), 256, 0, st>>>(x, W + p->ref_norm_w, nullptr, nullptr, ref_seq, (long long)Tr, D);
  PCK(cudaGetLastError());
  // ---- cached K / V of every reference cross-attention layer, heads-major
  const long long tot = (long long)Tr * D;
  for (int i = 0; i < c.ref_layers; ++i) {
    for (int kv = 0; kv < 2; ++kv) {
      g = dense::DenseOp{};
      g.A = ref_seq; g.W = W + (kv ? p->layer[i].v_w : p->layer[i].k_w); g.norm_w = W + p->layer[i].nkv_w; g.C = h; g.M = Tr; g.N = D; g.K = D;
      g.ldc = D; g.epi = dense::EPI_BIAS;
      if ((rc = launch_dense(g, 1, st))) return rc;
      heads_major_kernel<<<(unsigned)((tot + 255) / 256), 256, 0, st>>>(h, kv ? ref_v[i] : ref_k[i], Tr, H, D / H);
      PCK(cudaGetLastError());
    }
  }
  return SOPRO_OK;
}

/* Synchronises `stream`; SOPRO_ERR_INVALID if a run since the last check met a code outside [0, codebook_size). */
int sopro_refprep_check(sopro_refprep_t* p, void* stream) {
  if (!p) return fail(SOPRO_ERR_INVALID, "null argument");
  PCK(cudaSetDevice(p->device));
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  int bad = 0;
  PCK(cudaMemcpyAsync(&bad, p->bad, 4, cudaMemcpyDeviceToHost, st));
  PCK(cudaStreamSynchronize(st));
  if (bad) {
    PCK(cudaMemsetAsync(p->bad, 0, 4, st));
    return fail(SOPRO_ERR_INVALID, "reference codes outside [0, %d)", p->cfg.codebook_size);
  }
  return SOPRO_OK;
}

}  // extern "C"
