// CUDA-core (fp32) kernels of the dsx sampler: weight packing, the step-embedding table, layout
// packing of the conditioner, the DiffNet input/output projections, an exact-fp32 residual-layer
// path (DSX_PREC_FP32_SIMT: any channel count; also the on-device cross-check for the tcgen05
// path), and the DDPM / PLMS state updates with their Philox noise generator.
//
// Reference semantics followed (paths relative to the reference tree):
//   usr/diff/net.py:32-44,94-98,119-120  step embedding + MLP (Mish: usr/diff/diffusion.py:68-70)
//   usr/diff/net.py:66-78                ResidualBlock
//   usr/diff/net.py:115-130              DiffNet.forward head / tail
//   usr/diff/shallow_diffusion_tts.py:134-166   p_sample
//   usr/diff/shallow_diffusion_tts.py:174-199   get_x_pred + linear multistep combination
#include <math.h>

#include "dsx_internal.h"
#include "dsx_rng.cuh"
#include "dsx_update.cuh"

namespace dsx {

// ------------------------------------------------------------------------------------------
// weight packing (fp32 layouts used by the SIMT kernels and as the source of the fp16 packs)
// ------------------------------------------------------------------------------------------
__global__ void k_pack_w1f(const float* __restrict__ dil_w, const float* __restrict__ cond_w,
                           const float* __restrict__ dil_b, const float* __restrict__ cond_b,
                           float* __restrict__ w1f, float* __restrict__ b1f, int C, int H) {
  // dil_w [2C][C][3], cond_w [2C][H] -> w1f [2C][3C+H] with k = tap*C + c | 3C + h
  const int K = 3 * C + H;
  const int j = blockIdx.x;
  for (int k = threadIdx.x; k < K; k += blockDim.x) {
    float v;
    if (k < 3 * C) {
      int tap = k / C, c = k % C;
      v = dil_w[(static_cast<size_t>(j) * C + c) * 3 + tap];
    } else {
      v = cond_w[static_cast<size_t>(j) * H + (k - 3 * C)];
    }
    w1f[static_cast<size_t>(j) * K + k] = v;
  }
  if (threadIdx.x == 0) b1f[j] = dil_b[j] + cond_b[j];
}

int simt_pack_model(dsx_handle* h, const dsx_diffnet_params* p, cudaStream_t s) {
  ModelDev& m = h->m;
  const int C = m.C, H = m.H, M = m.M, L = m.L;
  const size_t K1 = 3 * static_cast<size_t>(C) + H;
  float *in_w, *in_b, *mlp0_w, *mlp0_b, *mlp2_w, *mlp2_b, *dif_w, *dif_b, *w1f, *b1f, *w2f, *b2f, *skip_w, *skip_b,
      *fin_w, *fin_b;
#define ALLOC(ptr, n) DSX_TRY(dev_alloc(h, reinterpret_cast<void**>(&ptr), (n) * sizeof(float), true))
#define COPY(dst, src, n) DSX_CUDA(cudaMemcpyAsync(dst, src, (n) * sizeof(float), cudaMemcpyDeviceToDevice, s))
  ALLOC(in_w, static_cast<size_t>(C) * M);
  ALLOC(in_b, C);
  ALLOC(mlp0_w, static_cast<size_t>(4) * C * C);
  ALLOC(mlp0_b, 4 * C);
  ALLOC(mlp2_w, static_cast<size_t>(4) * C * C);
  ALLOC(mlp2_b, C);
  ALLOC(dif_w, static_cast<size_t>(L) * C * C);
  ALLOC(dif_b, static_cast<size_t>(L) * C);
  ALLOC(w1f, static_cast<size_t>(L) * 2 * C * K1);
  ALLOC(b1f, static_cast<size_t>(L) * 2 * C);
  ALLOC(w2f, static_cast<size_t>(L) * 2 * C * C);
  ALLOC(b2f, static_cast<size_t>(L) * 2 * C);
  ALLOC(skip_w, static_cast<size_t>(C) * C);
  ALLOC(skip_b, C);
  ALLOC(fin_w, static_cast<size_t>(M) * C);
  ALLOC(fin_b, M);
  COPY(in_w, p->in_w, static_cast<size_t>(C) * M);
  COPY(in_b, p->in_b, C);
  COPY(mlp0_w, p->mlp0_w, static_cast<size_t>(4) * C * C);
  COPY(mlp0_b, p->mlp0_b, 4 * C);
  COPY(mlp2_w, p->mlp2_w, static_cast<size_t>(4) * C * C);
  COPY(mlp2_b, p->mlp2_b, C);
  COPY(skip_w, p->skip_w, static_cast<size_t>(C) * C);
  COPY(skip_b, p->skip_b, C);
  COPY(fin_w, p->fin_w, static_cast<size_t>(M) * C);
  COPY(fin_b, p->fin_b, M);
  for (int l = 0; l < L; ++l) {
    COPY(dif_w + static_cast<size_t>(l) * C * C, p->dif_w[l], static_cast<size_t>(C) * C);
    COPY(dif_b + static_cast<size_t>(l) * C, p->dif_b[l], C);
    COPY(w2f + static_cast<size_t>(l) * 2 * C * C, p->out_w[l], static_cast<size_t>(2) * C * C);
    COPY(b2f + static_cast<size_t>(l) * 2 * C, p->out_b[l], 2 * C);
    k_pack_w1f<<<2 * C, 256, 0, s>>>(p->dil_w[l], p->cond_w[l], p->dil_b[l], p->cond_b[l],
                                     w1f + static_cast<size_t>(l) * 2 * C * K1, b1f + static_cast<size_t>(l) * 2 * C,
                                     C, H);
    h->launches++;
  }
  DSX_CUDA(cudaGetLastError());
#undef ALLOC
#undef COPY
  m.in_w = in_w; m.in_b = in_b; m.mlp0_w = mlp0_w; m.mlp0_b = mlp0_b; m.mlp2_w = mlp2_w; m.mlp2_b = mlp2_b;
  m.dif_w = dif_w; m.dif_b = dif_b; m.w1f = w1f; m.b1f = b1f; m.w2f = w2f; m.b2f = b2f;
  m.skip_w = skip_w; m.skip_b = skip_b; m.fin_w = fin_w; m.fin_b = fin_b;
  return DSX_OK;
}

// ------------------------------------------------------------------------------------------
// step-embedding table: DTAB[row][l][c] = W_d,l . mlp(sinusoid(t_row)) + b_d,l
// One block per row.  net.py:37-44 computes the frequencies and angles in fp32 (exp, mul, sin,
// cos as separate fp32 ops); here each transcendental is evaluated in double and rounded once,
// which is within 1 ulp of any conforming fp32 libm.
// ------------------------------------------------------------------------------------------
__global__ void k_embed_table(ModelDev m, const int64_t* __restrict__ tvals, float* __restrict__ emb_out) {
  extern __shared__ float sm[];
  const int C = m.C;
  float* e0 = sm;           // [C]  sinusoid
  float* h1 = sm + C;       // [4C] hidden
  const int row = blockIdx.x;
  const float t = static_cast<float>(tvals[row]);
  const int half = C / 2;
  const double step = log(10000.0) / (half - 1);
  const float stepf = static_cast<float>(step);   // python float -> fp32 scalar multiply
  for (int i = threadIdx.x; i < half; i += blockDim.x) {
    float arg = static_cast<float>(i) * -stepf;                    // arange(half) * -emb   (fp32)
    float f = static_cast<float>(exp(static_cast<double>(arg)));   // torch.exp            (fp32)
    float ang = t * f;                                             // x[:,None]*emb[None,:] (fp32)
    e0[i] = static_cast<float>(sin(static_cast<double>(ang)));
    e0[half + i] = static_cast<float>(cos(static_cast<double>(ang)));
  }
  __syncthreads();
  // matvecs: one warp per output, lanes stride over k (coalesced weight rows), shuffle reduction
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, nwarps = blockDim.x >> 5;
  auto dot = [&](const float* __restrict__ w, const float* __restrict__ v, int n) {
    float acc = 0.f;
    for (int k = lane; k < n; k += 32) acc = fmaf(w[k], v[k], acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    return acc;
  };
  for (int j = warp; j < 4 * C; j += nwarps) {
    float acc = dot(m.mlp0_w + static_cast<size_t>(j) * C, e0, C) + m.mlp0_b[j];
    // Mish: x * tanh(softplus(x)); softplus with torch's threshold (20) semantics
    float sp = acc > 20.f ? acc : log1pf(expf(acc));
    if (lane == 0) h1[j] = acc * tanhf(sp);
  }
  __syncthreads();
  for (int j = warp; j < C; j += nwarps) {
    float acc = dot(m.mlp2_w + static_cast<size_t>(j) * 4 * C, h1, 4 * C) + m.mlp2_b[j];
    if (lane == 0) emb_out[static_cast<size_t>(row) * C + j] = acc;
  }
}

// per-layer FiLM vectors d_l(t) = diffusion_projection_l(emb(t)) (net.py:62,67) for every row of the table: one warp
// per output channel keeps its weight row in registers and walks over the rows
__global__ void k_embed_proj(ModelDev m, const float* __restrict__ emb, float* __restrict__ dtab, int rows) {
  const int C = m.C, L = m.L;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int idx = blockIdx.x * (blockDim.x >> 5) + warp;
  if (idx >= L * C) return;
  const float* w = m.dif_w + static_cast<size_t>(idx) * C;
  const float bias = m.dif_b[idx];
  for (int row = 0; row < rows; ++row) {
    const float* v = emb + static_cast<size_t>(row) * C;
    float acc = 0.f;
    for (int k = lane; k < C; k += 32) acc = fmaf(w[k], v[k], acc);
#pragma unroll
    for (int o = 16; o > 0; o >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, o);
    if (lane == 0) dtab[static_cast<size_t>(row) * L * C + idx] = acc + bias;
  }
}

int launch_embed_table(dsx_handle* h, const int64_t* t_dev, int rows, cudaStream_t s) {
  const size_t smem = static_cast<size_t>(5) * h->m.C * sizeof(float);
  k_embed_table<<<rows, 512, smem, s>>>(h->m, t_dev, h->ws.EMB);
  h->launches++;
  DSX_CUDA(cudaGetLastError());
  k_embed_proj<<<(h->m.L * h->m.C + 15) / 16, 512, 0, s>>>(h->m, h->ws.EMB, h->ws.DTAB, rows);
  h->launches++;
  DSX_CUDA(cudaGetLastError());
  return DSX_OK;
}

// ------------------------------------------------------------------------------------------
// conditioner packing: cond[b][h][t] (arbitrary strides) -> frames-major fp32 and fp16 hi/lo
// ------------------------------------------------------------------------------------------
__global__ void k_pack_cond(const float* __restrict__ cond, dsx_strides cs, int B, int T, int Tp, int H,
                            float* __restrict__ condf, __half* __restrict__ condh, size_t plane_elems) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const int t0 = blockIdx.x * 32, h0 = blockIdx.y * 32;
  // read: pick the thread->element mapping along the input's unit-stride axis
  const bool h_fast = (cs.c == 1);
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int t = h_fast ? t0 + i : t0 + threadIdx.x;
    int hh = h_fast ? h0 + threadIdx.x : h0 + i;
    float v = 0.f;
    if (t < T && hh < H) v = cond[b * cs.b + hh * cs.c + t * cs.t];
    if (h_fast) tile[i][threadIdx.x] = v; else tile[threadIdx.x][i] = v;   // tile[t][h]
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int t = t0 + i, hh = h0 + threadIdx.x;
    if (t < Tp && hh < H) {
      float v = (t < T) ? tile[i][threadIdx.x] : 0.f;
      size_t o = (static_cast<size_t>(b) * Tp + t) * H + hh;
      if (condf) condf[o] = v;
      if (condh) {
        __half hi = __float2half_rn(v);
        condh[o] = hi;
        condh[plane_elems + o] = __float2half_rn(v - __half2float(hi));
      }
    }
  }
}

int launch_pack_cond(dsx_handle* h, const float* cond, dsx_strides cs, const Geom& g, cudaStream_t s) {
  dim3 grid((g.Tp + 31) / 32, (h->m.H + 31) / 32, g.B), block(32, 8);
  const bool tc = h->precision != DSX_PREC_FP32_SIMT;
  k_pack_cond<<<grid, block, 0, s>>>(cond, cs, g.B, g.T, g.Tp, h->m.H, tc ? nullptr : h->ws.CONDF,
                                     tc ? h->ws.CONDH : nullptr, g.frames_padded() * h->m.H);
  h->launches++;
  DSX_CUDA(cudaGetLastError());
  return DSX_OK;
}

// ------------------------------------------------------------------------------------------
// input projection of the fp32 path (net.py:116-118): X[n][c] = relu(W_in[c][:] . x[b][:][t] + b_in[c]).  The tensor-core
// paths project in k_tc_head / k_tc_stack.
// ------------------------------------------------------------------------------------------
constexpr int kInFrames = 16;
__global__ void k_inproj(ModelDev m, const float* __restrict__ x, dsx_strides xs, int T, int Tp, float* __restrict__ X) {
  extern __shared__ float xt[];   // [kInFrames][M]
  const int b = blockIdx.y, t0 = blockIdx.x * kInFrames, M = m.M, C = m.C;
  for (int i = threadIdx.x; i < kInFrames * M; i += blockDim.x) {
    int f = i % kInFrames, mm = i / kInFrames;
    int t = t0 + f;
    xt[f * M + mm] = (t < T) ? x[b * xs.b + mm * xs.c + t * xs.t] : 0.f;
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const float* w = m.in_w + static_cast<size_t>(c) * M;
    float acc[kInFrames];
#pragma unroll
    for (int f = 0; f < kInFrames; ++f) acc[f] = 0.f;
    for (int mm = 0; mm < M; ++mm) {
      float wv = w[mm];
#pragma unroll
      for (int f = 0; f < kInFrames; ++f) acc[f] = fmaf(wv, xt[f * M + mm], acc[f]);
    }
    const float bias = m.in_b[c];
#pragma unroll
    for (int f = 0; f < kInFrames; ++f) {
      int t = t0 + f;
      if (t >= T) continue;
      X[(static_cast<size_t>(b) * Tp + t) * C + c] = fmaxf(acc[f] + bias, 0.f);
    }
  }
}

int launch_inproj(dsx_handle* h, const float* x, dsx_strides xs, const Geom& g, cudaStream_t s) {
  dim3 grid((g.T + kInFrames - 1) / kInFrames, g.B);
  k_inproj<<<grid, 256, kInFrames * h->m.M * sizeof(float), s>>>(h->m, x, xs, g.T, g.Tp, h->ws.X);
  h->launches++;
  DSX_CUDA(cudaGetLastError());
  return DSX_OK;
}

// ------------------------------------------------------------------------------------------
// generic fp32 GEMM: out[n][j] = sum_k A(n,k) * W[j][k]   (64x64 tile, 4x4 per thread)
// A is virtual: PLAIN rows of a frames-major matrix (optionally scaled), or CONV = the dilated
// 3-tap gather of (X + d_l) with zero padding applied AFTER the FiLM add (net.py:69-71) followed by
// the conditioner columns.
// ------------------------------------------------------------------------------------------
struct GemmA {
  const float* X;      // [B][Tp][lda]
  const float* dl;     // [B?][C] FiLM row base (CONV), indexed by d_row_stride * b
  const float* cond;   // [B][Tp][H]          (CONV)
  int lda, C, H, T, Tp, dil, d_row_stride;
  float scale;
};

template <int CONV>
__global__ void __launch_bounds__(256) k_simt_gemm(GemmA a, const float* __restrict__ W, int K, int J,
                                                   float* __restrict__ out, int ldo) {
  __shared__ float As[16][68];
  __shared__ float Ws[16][68];
  const int n0 = blockIdx.x * 64, j0 = blockIdx.y * 64;
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += 16) {
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      int e = threadIdx.x + i * 256;
      int kk = e % 16, nn = e / 16;
      int n = n0 + nn, k = k0 + kk;
      int b = n / a.Tp, t = n % a.Tp;
      float v = 0.f;
      if (CONV) {
        if (t < a.T) {
          if (k < 3 * a.C) {
            int tap = k / a.C, c = k % a.C;
            int tt = t + (tap - 1) * a.dil;
            if (tt >= 0 && tt < a.T)
              v = a.X[(static_cast<size_t>(b) * a.Tp + tt) * a.lda + c] + a.dl[static_cast<size_t>(b) * a.d_row_stride + c];
          } else {
            v = a.cond[(static_cast<size_t>(b) * a.Tp + t) * a.H + (k - 3 * a.C)];
          }
        }
      } else {
        v = a.X[static_cast<size_t>(n) * a.lda + k] * a.scale;
      }
      As[kk][nn] = v;
      int j = j0 + nn;
      Ws[kk][nn] = (j < J) ? W[static_cast<size_t>(j) * K + k] : 0.f;
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < 16; ++kk) {
      float av[4], wv[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) { av[i] = As[kk][ty * 4 + i]; wv[i] = Ws[kk][tx * 4 + i]; }
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int jj = 0; jj < 4; ++jj) acc[i][jj] = fmaf(av[i], wv[jj], acc[i][jj]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    int n = n0 + ty * 4 + i;
#pragma unroll
    for (int jj = 0; jj < 4; ++jj) {
      int j = j0 + tx * 4 + jj;
      if (j < J) out[static_cast<size_t>(n) * ldo + j] = acc[i][jj];
    }
  }
}

__global__ void k_gate(const float* __restrict__ g1, const float* __restrict__ b1, float* __restrict__ z, int C,
                       size_t n_elems) {
  size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i >= n_elems) return;
  size_t n = i / C;
  int c = static_cast<int>(i % C);
  float g = g1[n * 2 * C + c] + b1[c];
  float f = g1[n * 2 * C + C + c] + b1[C + c];
  z[i] = (1.f / (1.f + expf(-g))) * tanhf(f);
}

__global__ void k_resid(const float* __restrict__ g1, const float* __restrict__ b2, float* __restrict__ X,
                        float* __restrict__ SKIP, int C, size_t n_elems, int first) {
  size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i >= n_elems) return;
  size_t n = i / C;
  int c = static_cast<int>(i % C);
  float r = g1[n * 2 * C + c] + b2[c];
  float sk = g1[n * 2 * C + C + c] + b2[C + c];
  X[i] = (X[i] + r) * 0.70710678118654752440f;
  SKIP[i] = first ? sk : SKIP[i] + sk;
}

int launch_simt_layer(dsx_handle* h, int layer, const Geom& g, int row0, int row_per_b, cudaStream_t s) {
  const ModelDev& m = h->m;
  const int C = m.C, H = m.H;
  const int K1 = 3 * C + H;
  const size_t nf = g.frames_padded();
  GemmA a{};
  a.X = h->ws.X; a.lda = C; a.C = C; a.H = H; a.T = g.T; a.Tp = g.Tp; a.dil = 1 << (layer % m.cycle);
  a.dl = h->ws.DTAB + (static_cast<size_t>(row0) * m.L + layer) * C;
  a.d_row_stride = row_per_b * m.L * C;
  a.cond = h->ws.CONDF; a.scale = 1.f;
  dim3 grid1(static_cast<unsigned>(nf / 64), (2 * C + 63) / 64);
  k_simt_gemm<1><<<grid1, 256, 0, s>>>(a, m.w1f + static_cast<size_t>(layer) * 2 * C * K1, K1, 2 * C, h->ws.G1, 2 * C);
  const size_t ne = nf * C;
  const unsigned eb = static_cast<unsigned>((ne + 255) / 256);
  k_gate<<<eb, 256, 0, s>>>(h->ws.G1, m.b1f + static_cast<size_t>(layer) * 2 * C, h->ws.Zf, C, ne);
  GemmA a2{};
  a2.X = h->ws.Zf; a2.lda = C; a2.Tp = g.Tp; a2.scale = 1.f;
  k_simt_gemm<0><<<grid1, 256, 0, s>>>(a2, m.w2f + static_cast<size_t>(layer) * 2 * C * C, C, 2 * C, h->ws.G1, 2 * C);
  k_resid<<<eb, 256, 0, s>>>(h->ws.G1, m.b2f + static_cast<size_t>(layer) * 2 * C, h->ws.X, h->ws.SKIP, C, ne,
                             layer == 0);
  h->launches += 4;
  DSX_CUDA(cudaGetLastError());
  return DSX_OK;
}

// ------------------------------------------------------------------------------------------
// head (net.py:126-130): eps = W_out . relu(W_s . (skip/sqrt(L)) + b_s) + b_out, written in the
// reference's [B,1,M,T] layout.
// ------------------------------------------------------------------------------------------
__global__ void k_bias_relu(float* __restrict__ v, const float* __restrict__ b, int C, size_t n_elems) {
  size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i >= n_elems) return;
  v[i] = fmaxf(v[i] + b[i % C], 0.f);
}

__global__ void k_eps_out(const float* __restrict__ g, const float* __restrict__ b, float* __restrict__ eps, int M,
                          int T, int Tp, int ldg) {
  __shared__ float tile[32][33];
  const int bb = blockIdx.z, t0 = blockIdx.x * 32, m0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int t = t0 + i, mm = m0 + threadIdx.x;
    tile[i][threadIdx.x] = (t < T && mm < M) ? g[(static_cast<size_t>(bb) * Tp + t) * ldg + mm] + b[mm] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int mm = m0 + i, t = t0 + threadIdx.x;
    if (mm < M && t < T) eps[(static_cast<size_t>(bb) * M + mm) * T + t] = tile[threadIdx.x][i];
  }
}

int launch_head(dsx_handle* h, const Geom& g, float* eps, cudaStream_t s) {
  const ModelDev& m = h->m;
  const int C = m.C, M = m.M;
  const size_t nf = g.frames_padded();
  GemmA a{};
  a.X = h->ws.SKIP; a.lda = C; a.Tp = g.Tp; a.scale = 1.f / sqrtf(static_cast<float>(m.L));
  dim3 grid1(static_cast<unsigned>(nf / 64), (C + 63) / 64);
  k_simt_gemm<0><<<grid1, 256, 0, s>>>(a, m.skip_w, C, C, h->ws.Zf, C);
  const size_t ne = nf * C;
  k_bias_relu<<<static_cast<unsigned>((ne + 255) / 256), 256, 0, s>>>(h->ws.Zf, m.skip_b, C, ne);
  GemmA a2{};
  a2.X = h->ws.Zf; a2.lda = C; a2.Tp = g.Tp; a2.scale = 1.f;
  dim3 grid2(static_cast<unsigned>(nf / 64), (M + 63) / 64);
  k_simt_gemm<0><<<grid2, 256, 0, s>>>(a2, m.fin_w, C, M, h->ws.G1, 2 * C);
  dim3 grid3((g.T + 31) / 32, (M + 31) / 32, g.B), block3(32, 8);
  k_eps_out<<<grid3, block3, 0, s>>>(h->ws.G1, m.fin_b, eps, M, g.T, g.Tp, 2 * C);
  h->launches += 4;
  DSX_CUDA(cudaGetLastError());
  return DSX_OK;
}

// p_sample after the network (shallow_diffusion_tts.py:134-166, ddpm_step) with injected or Philox noise
__global__ void k_ddpm_update(float* __restrict__ x, const float* __restrict__ eps, const float* __restrict__ noise,
                              uint64_t seed, uint64_t offset, DdpmCoef c, size_t n, int M, int T, int b_off) {
  size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  const float xv = x[i], ev = eps[i];
  float z = 0.f;
  if (c.sigma != 0.f) {
    if (noise) {
      z = noise[i];
    } else {
      const int t = static_cast<int>(i % T), m = static_cast<int>((i / T) % M), b = static_cast<int>(i / (static_cast<size_t>(T) * M));
      const float4 z4 = philox_normal4(seed, offset, mel_noise_block(b + b_off, m, t, M, T));
      z = (m & 3) == 0 ? z4.x : (m & 3) == 1 ? z4.y : (m & 3) == 2 ? z4.z : z4.w;
    }
  }
  x[i] = ddpm_step(c, xv, ev, z);
}

int launch_ddpm_update(dsx_handle* h, float* x, const float* eps, const float* noise, uint64_t seed, uint64_t offset,
                       DdpmCoef c, size_t n, int T, cudaStream_t s) {
  k_ddpm_update<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(x, eps, noise, seed, offset, c, n, h->m.M, T, h->batch_offset);
  h->launches++;
  DSX_CUDA(cudaGetLastError());
  return DSX_OK;
}

// PLMS (shallow_diffusion_tts.py:174-199, plms_step) over e0 and the history e1..e3 that is given
__global__ void k_plms_update(float* __restrict__ xo, const float* __restrict__ xi, const float* __restrict__ e0,
                              const float* __restrict__ e1, const float* __restrict__ e2,
                              const float* __restrict__ e3, PlmsCoef c, size_t n) {
  size_t i = blockIdx.x * static_cast<size_t>(blockDim.x) + threadIdx.x;
  if (i >= n) return;
  xo[i] = plms_step(c, xi[i], e0[i], e1 ? e1[i] : 0.f, e2 ? e2[i] : 0.f, e3 ? e3[i] : 0.f, e1, e2, e3);
}

int launch_plms_update(dsx_handle* h, float* x_out, const float* x_in, const float* e0, const float* e1,
                       const float* e2, const float* e3, PlmsCoef c, size_t n, cudaStream_t s) {
  k_plms_update<<<static_cast<unsigned>((n + 255) / 256), 256, 0, s>>>(x_out, x_in, e0, e1, e2, e3, c, n);
  h->launches++;
  DSX_CUDA(cudaGetLastError());
  return DSX_OK;
}

// prologue of the infer branch (shallow_diffusion_tts.py:249-255): norm_spec (:278-279), transpose to
// [B,1,M,T], q_sample at K_step-1 (:206-211).
__global__ void k_prologue(float* __restrict__ x, const float* __restrict__ fs2_mel, const float* __restrict__ noise,
                           uint64_t seed, const float* __restrict__ smin, const float* __restrict__ smax, float sa,
                           float s1a, int T, int M, int b_off) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, t0 = blockIdx.x * 32, m0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int t = t0 + i, mm = m0 + threadIdx.x;
    float v = 0.f;
    if (t < T && mm < M) {
      float lo = smin[mm], hi = smax[mm];
      v = __fsub_rn(__fmul_rn(__fdiv_rn(__fsub_rn(fs2_mel[(static_cast<size_t>(b) * T + t) * M + mm], lo),
                                        __fsub_rn(hi, lo)), 2.f), 1.f);
    }
    tile[i][threadIdx.x] = v;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int mm = m0 + i, t = t0 + threadIdx.x;
    if (mm < M && t < T) {
      size_t o = (static_cast<size_t>(b) * M + mm) * T + t;
      float z = noise ? noise[o] : philox_normal(seed, 0xFFFFFFFFull, o + static_cast<size_t>(b_off) * M * T);
      x[o] = __fadd_rn(__fmul_rn(sa, tile[threadIdx.x][i]), __fmul_rn(s1a, z));
    }
  }
}

int launch_prologue(dsx_handle* h, float* x, const float* fs2_mel, const float* start_noise, uint64_t seed,
                    const float* spec_min, const float* spec_max, float sa, float s1a, int B, int T, int M,
                    cudaStream_t s) {
  dim3 grid((T + 31) / 32, (M + 31) / 32, B), block(32, 8);
  k_prologue<<<grid, block, 0, s>>>(x, fs2_mel, start_noise, seed, spec_min, spec_max, sa, s1a, T, M, h->batch_offset);
  h->launches++;
  DSX_CUDA(cudaGetLastError());
  return DSX_OK;
}

// epilogue (:271-275): x[:,0].transpose(1,2) -> denorm_spec (:281-282) -> * (mel2ph > 0)
__global__ void k_epilogue(const float* __restrict__ x, const int64_t* __restrict__ mel2ph,
                           const float* __restrict__ smin, const float* __restrict__ smax, float* __restrict__ out,
                           int T, int M) {
  __shared__ float tile[32][33];
  const int b = blockIdx.z, t0 = blockIdx.x * 32, m0 = blockIdx.y * 32;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int mm = m0 + i, t = t0 + threadIdx.x;
    tile[i][threadIdx.x] = (mm < M && t < T) ? x[(static_cast<size_t>(b) * M + mm) * T + t] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    int t = t0 + i, mm = m0 + threadIdx.x;
    if (t < T && mm < M) {
      float lo = smin[mm], hi = smax[mm];
      float v = __fadd_rn(__fmul_rn(__fdiv_rn(__fadd_rn(tile[threadIdx.x][i], 1.f), 2.f), __fsub_rn(hi, lo)), lo);
      if (mel2ph) v = __fmul_rn(v, mel2ph[static_cast<size_t>(b) * T + t] > 0 ? 1.f : 0.f);
      out[(static_cast<size_t>(b) * T + t) * M + mm] = v;
    }
  }
}

int launch_epilogue(dsx_handle* h, const float* x, const int64_t* mel2ph, const float* spec_min,
                    const float* spec_max, float* mel_out, int B, int T, int M, cudaStream_t s) {
  dim3 grid((T + 31) / 32, (M + 31) / 32, B), block(32, 8);
  k_epilogue<<<grid, block, 0, s>>>(x, mel2ph, spec_min, spec_max, mel_out, T, M);
  h->launches++;
  DSX_CUDA(cudaGetLastError());
  return DSX_OK;
}

}  // namespace dsx
