// FourCastNet v1 (AFNO backbone) 6-h step operator on sm_100a (SURVEY.md Appendix D, DESIGN.md section 4d).
//
// Token stream: x fp32 (B*h*w, E), (member, h, w)-major, the residual stream.  Per block
//   LN1                      x -> u (fp32: the filter adds its own input back)
//   AFNO2D filter            u -> W-DFT (kw kept modes) -> H-DFT (kept H rows) -> complex block MLP + softshrink
//                            -> inverse H-DFT -> inverse W-DFT (c2r) whose epilogue adds u and the residual to x
//   LN2                      x -> v (fp16 operand rows)
//   fc1 + GELU, fc2          tcgen05 GEMMs (gemm_tc.cuh); fc2's epilogue adds into x
// The patch embedding (normalise + im2col in the producer, bias + pos_embed in the epilogue) and the head (de-normalise,
// scatter of the (p1, p2, c) columns to the output planes in the epilogue) are tcgen05 GEMMs as well.  The spectral
// filter (8 % of the step's FLOPs) runs on the CUDA cores in fp32.  No atomics: every reduction has one owner.
#include <cstring>
#include <vector>

#include "engine.h"
#include "gemm_tc.cuh"

namespace sky {
namespace {

constexpr int FCN_BS = 96;      // spectral block width the block-MLP kernel is written for
constexpr int FCN_MAXH = 128;   // token-grid height limit of the H-DFT tiles

// fp32 W [N, K] -> tile image [N/BN][Kp/64][BN rows x 128 B, SWIZZLE_128B] (the B operand of k_gemm_tc)
__global__ void k_fcn_pack(const float* __restrict__ W, int N, int K, int Kp, int BN, uint8_t* __restrict__ img) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;  // one 8-half chunk each
  const int cpr = Kp / 8;
  if (idx >= (long long)N * cpr) return;
  const int n = (int)(idx / cpr), kc = (int)(idx % cpr);
  __half h[8];
#pragma unroll
  for (int e = 0; e < 8; ++e) {
    const int k = kc * 8 + e;
    h[e] = __float2half_rn(k < K ? W[(long long)n * K + k] : 0.f);
  }
  const int nt = n / BN, nr = n % BN, kb = kc / 8, ch = kc % 8;
  *reinterpret_cast<uint4*>(img + ((size_t)nt * (Kp / 64) + kb) * (size_t)BN * 128 + sw128_offset(nr, ch)) =
      *reinterpret_cast<uint4*>(h);
}

// complex block weight w (2, nb, bs, bs) [re/im part, block, in, out] -> per block the real (2 bs x 2 bs) matrix
// [in][out] that maps the rows [re | im] of a mode to [re | im] of the complex product
__global__ void k_fcn_cplx_weight(const float* __restrict__ w, int nb, int bs, float* __restrict__ out) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const int n2 = 2 * bs;
  if (idx >= (long long)nb * n2 * n2) return;
  const int o = (int)(idx % n2), i = (int)(idx / n2 % n2), g = (int)(idx / ((long long)n2 * n2));
  const int ii = i % bs, oo = o % bs;
  const bool ire = i < bs, ore = o < bs;
  const float w0 = w[(((long long)0 * nb + g) * bs + ii) * bs + oo], w1 = w[(((long long)1 * nb + g) * bs + ii) * bs + oo];
  out[idx] = ire == ore ? w0 : (ore ? -w1 : w1);
}

// ---------------------------------------------------------------------------------------------------------------
// GEMM producers / epilogues (k_gemm_tc: one lane owns one accumulator row)
// ---------------------------------------------------------------------------------------------------------------
// patch embedding: row = (member, hh, ww), k = (c, p1, p2) of the 8x8 patch; normalised on the fly
struct ProdFcnEmbed {
  const float* state; const float* mean; const float* stdv;
  int C, nlat, nlon, w; long long T, M;
  __device__ RowInfo prep(long long row) const {
    if (row >= M) return {-1, 0};
    const long long b = row / T, t = row % T;
    const int hh = (int)(t / w), ww = (int)(t % w);
    return {b * C * (long long)nlat * nlon + (long long)(8 * hh) * nlon + 8 * ww, 0};
  }
  __device__ uint4 load8(const RowInfo& ri, int k) const {
    if (ri.base < 0) return make_uint4(0, 0, 0, 0);
    const int c = k >> 6, p1 = (k >> 3) & 7;
    const float mu = __ldg(mean + c), rs = 1.0f / __ldg(stdv + c);
    const float4* p = reinterpret_cast<const float4*>(state + ri.base + ((long long)c * nlat + p1) * nlon);
    float4 a = __ldg(p), b = __ldg(p + 1);
    a.x = (a.x - mu) * rs; a.y = (a.y - mu) * rs; a.z = (a.z - mu) * rs; a.w = (a.w - mu) * rs;
    b.x = (b.x - mu) * rs; b.y = (b.y - mu) * rs; b.z = (b.z - mu) * rs; b.w = (b.w - mu) * rs;
    return f32x8_to_h8(a, b);
  }
};

// x[row, n] = acc + bias[n] + pos[row % T, n]
struct EpiFcnEmbed {
  float* x; const float* bias; const float* pos; int E; long long T, M;
  template <class Acc>
  __device__ void run(Acc& acc, long long row, int n0, int BN) const {
    for (int c = 0; c < BN; c += 32) {
      float v[32];
      acc.load32(c, v);
      if (row < M) {
        const float* pr = pos + (row % T) * E + n0 + c;
#pragma unroll
        for (int j = 0; j < 32; ++j) v[j] += __ldg(bias + n0 + c + j) + __ldg(pr + j);
        float* o = x + row * E + n0 + c;
#pragma unroll
        for (int j = 0; j < 4; ++j) stg_f32x8(o + 8 * j, v + 8 * j);
      }
    }
  }
};

// x[row, n] += acc + bias[n]     (fc2: the MLP branch joins the residual stream)
struct EpiFcnResidual {
  float* x; const float* bias; int E; long long M;
  template <class Acc>
  __device__ void run(Acc& acc, long long row, int n0, int BN) const {
    for (int c = 0; c < BN; c += 32) {
      float v[32];
      acc.load32(c, v);
      if (row < M) {
        float* o = x + row * E + n0 + c;
        float r[8];
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          ldg_f32x8(o + 8 * j, r);
#pragma unroll
          for (int e = 0; e < 8; ++e) r[e] += v[8 * j + e] + __ldg(bias + n0 + c + 8 * j + e);
          stg_f32x8(o + 8 * j, r);
        }
      }
    }
  }
};

// head: column n = (p1 * 8 + p2) * C + c  ->  y[b, c, 8 hh + p1, 8 ww + p2] = acc * std[c] + mean[c]
struct EpiFcnHead {
  float* y; const float* mean; const float* stdv; int C, nlat, nlon, w; long long T, M;
  template <class Acc>
  __device__ void run(Acc& acc, long long row, int n0, int BN) const {
    const long long b = row / T, t = row % T;
    const int hh = (int)(t / w), ww = (int)(t % w);
    for (int c = 0; c < BN; c += 32) {
      float v[32];
      acc.load32(c, v);
      if (row < M) {
#pragma unroll 4
        for (int j = 0; j < 32; ++j) {
          const int n = n0 + c + j, ch = n % C, pp = n / C;
          y[((b * C + ch) * nlat + 8 * hh + (pp >> 3)) * (long long)nlon + 8 * ww + (pp & 7)] =
              v[j] * __ldg(stdv + ch) + __ldg(mean + ch);
        }
      }
    }
  }
};

// ---------------------------------------------------------------------------------------------------------------
// LayerNorm over E columns: one warp per row, lane owns 4 consecutive features per 128-feature slab
// ---------------------------------------------------------------------------------------------------------------
template <bool kHalf>
__global__ void __launch_bounds__(256) k_fcn_ln(const float* __restrict__ x, void* __restrict__ out,
                                                const float* __restrict__ gamma, const float* __restrict__ beta,
                                                float eps, long long rows, int E) {
  constexpr int MAXS = 8;   // E <= 1024
  const long long row = (long long)blockIdx.x * 8 + threadIdx.x / 32;
  const int lane = threadIdx.x % 32, ns = E / 128;
  if (row >= rows) return;
  float4 v[MAXS];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < MAXS; ++i)
    if (i < ns) {
      v[i] = __ldg(reinterpret_cast<const float4*>(x + row * E + 128 * i + 4 * lane));
      s += (v[i].x + v[i].y) + (v[i].z + v[i].w);
    }
  const float mean = warp_sum(s) / E;
  float ss = 0.f;
#pragma unroll
  for (int i = 0; i < MAXS; ++i)
    if (i < ns) {
      const float a = v[i].x - mean, b = v[i].y - mean, c = v[i].z - mean, d = v[i].w - mean;
      ss += (a * a + b * b) + (c * c + d * d);
    }
  const float rstd = rsqrtf(warp_sum(ss) / E + eps);
#pragma unroll
  for (int i = 0; i < MAXS; ++i)
    if (i < ns) {
      const int e = 128 * i + 4 * lane;
      const float4 g = __ldg(reinterpret_cast<const float4*>(gamma + e)), b = __ldg(reinterpret_cast<const float4*>(beta + e));
      const float4 r = make_float4((v[i].x - mean) * rstd * g.x + b.x, (v[i].y - mean) * rstd * g.y + b.y,
                                   (v[i].z - mean) * rstd * g.z + b.z, (v[i].w - mean) * rstd * g.w + b.w);
      if (kHalf) {
        uint2 pk;
        pk.x = pack_half2(r.x, r.y); pk.y = pack_half2(r.z, r.w);
        *reinterpret_cast<uint2*>(static_cast<__half*>(out) + row * E + e) = pk;
      } else {
        *reinterpret_cast<float4*>(static_cast<float*>(out) + row * E + e) = r;
      }
    }
}

// ---------------------------------------------------------------------------------------------------------------
// spectral filter (fp32)
// ---------------------------------------------------------------------------------------------------------------
// W-DFT twiddles (cos, sin)(2 pi m x / w) as a [x][KW] table with zero columns for m >= kw: the W-DFT kernels read one
// float4 (two modes) per load, the same address across the warp (an L1 broadcast)
__global__ void k_fcn_twiddle(float2* __restrict__ t, int w, int kw, int KW) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= w * KW) return;
  const int x = idx / KW, m = idx % KW;
  float2 r = make_float2(0.f, 0.f);
  if (m < kw) {
    double s, c;
    sincospi(2.0 * ((m * x) % w) / w, &s, &c);
    r = make_float2((float)c, (float)s);
  }
  t[idx] = r;
}

// forward W-DFT of one latitude row of tokens: F[b, hh, m, e] = scale * sum_x u[b, hh, x, e] e^{-2 pi i m x / w}, m < kw
template <int KW>
__global__ void __launch_bounds__(128) k_fcn_dft_w(const float* __restrict__ u, const float4* __restrict__ tw,
                                                   float2* __restrict__ F, int w, int kw, int E, float scale) {
  const long long bh = blockIdx.x;
  const int e = blockIdx.y * 128 + threadIdx.x;
  float ar[KW], ai[KW];
#pragma unroll
  for (int m = 0; m < KW; ++m) { ar[m] = 0.f; ai[m] = 0.f; }
  const float* src = u + bh * w * E + e;
  for (int x = 0; x < w; ++x) {
    const float v = __ldg(src + (long long)x * E);
    const float4* t = tw + (size_t)x * (KW / 2);
#pragma unroll
    for (int q = 0; q < KW / 2; ++q) {
      const float4 c = __ldg(t + q);
      ar[2 * q] = fmaf(v, c.x, ar[2 * q]); ai[2 * q] = fmaf(-v, c.y, ai[2 * q]);
      ar[2 * q + 1] = fmaf(v, c.z, ar[2 * q + 1]); ai[2 * q + 1] = fmaf(-v, c.w, ai[2 * q + 1]);
    }
  }
#pragma unroll
  for (int m = 0; m < KW; ++m)
    if (m < kw) F[(bh * kw + m) * E + e] = make_float2(ar[m] * scale, ai[m] * scale);
}

// complex DFT along H of the (B, n_in, kw, E) spectra -> (B, n_out, kw, E):
//   forward (n_in = h rows, n_out = kept frequencies f = h_lo + o):  out[o] = scale * sum_i in[i] e^{-2 pi i f i / h}
//   inverse (n_in = kept frequencies f = h_lo + i, n_out = h rows):  out[o] = scale * sum_i in[i] e^{+2 pi i f o / h}
// Block = (member, mode m) x 32 channels; the input column sits in shared memory, warp q owns outputs q, q + 8, ...
__global__ void __launch_bounds__(256) k_fcn_dft_h(const float2* __restrict__ in, float2* __restrict__ out, int h,
                                                   int h_lo, int n_in, int n_out, int kw, int E, int forward,
                                                   float scale) {
  __shared__ float2 tile[FCN_MAXH][32];
  __shared__ float cs[FCN_MAXH], sn[FCN_MAXH];
  const int b = blockIdx.x / kw, m = blockIdx.x % kw, e0 = blockIdx.y * 32;
  const int lane = threadIdx.x % 32, q = threadIdx.x / 32;
  for (int j = threadIdx.x; j < h; j += blockDim.x) {
    double s, c;
    sincospi(2.0 * j / h, &s, &c);
    cs[j] = (float)c; sn[j] = (float)(forward ? -s : s);
  }
  for (int idx = threadIdx.x; idx < n_in * 32; idx += blockDim.x) {
    const int i = idx / 32, l = idx % 32;
    tile[i][l] = in[(((long long)b * n_in + i) * kw + m) * E + e0 + l];
  }
  __syncthreads();
  for (int o = q; o < n_out; o += 8) {
    const int d = forward ? (h_lo + o) % h : o % h;   // phase index step per input row
    int j = forward ? 0 : (int)((long long)h_lo * o % h);
    float re = 0.f, im = 0.f;
    for (int i = 0; i < n_in; ++i) {
      const float2 z = tile[i][lane];
      const float c = cs[j], s = sn[j];
      re = fmaf(z.x, c, fmaf(-z.y, s, re));
      im = fmaf(z.x, s, fmaf(z.y, c, im));
      j += d; if (j >= h) j -= h;
    }
    out[(((long long)b * n_out + o) * kw + m) * E + e0 + lane] = make_float2(re * scale, im * scale);
  }
}

// complex block MLP on the kept modes: per mode pixel p and block g the rows [re | im] (2 BS values) go through
//   o1 = relu(x Wc1 + b1), o2 = o1 Wc2 + b2, softshrink(lambda)
// Block = 32 mode pixels x one spectral block; thread o owns output column o of all 32 pixels.
template <int BS>
__global__ void __launch_bounds__(2 * BS) k_fcn_block_mlp(const float2* __restrict__ Y, float2* __restrict__ Z,
                                                          const float* __restrict__ W1, const float* __restrict__ b1,
                                                          const float* __restrict__ W2, const float* __restrict__ b2,
                                                          long long P, int E, int nb, float lambda) {
  constexpr int N2 = 2 * BS, PT = 32;
  __shared__ __align__(16) float xs[PT][N2];
  const int g = blockIdx.y, o = threadIdx.x;
  const long long p0 = (long long)blockIdx.x * PT;
  for (int idx = threadIdx.x; idx < PT * BS; idx += N2) {
    const int p = idx / BS, j = idx % BS;
    const float2 z = p0 + p < P ? Y[(p0 + p) * E + g * BS + j] : make_float2(0.f, 0.f);
    xs[p][j] = z.x; xs[p][BS + j] = z.y;
  }
  __syncthreads();
  const int bo = (o < BS ? 0 : nb) * BS + g * BS + o % BS;
  float acc[PT];
  for (int layer = 0; layer < 2; ++layer) {
    const float* Wg = (layer ? W2 : W1) + (size_t)g * N2 * N2;
#pragma unroll
    for (int p = 0; p < PT; ++p) acc[p] = 0.f;
    for (int i = 0; i < N2; i += 4) {
      const float w0 = __ldg(Wg + (i + 0) * N2 + o), w1 = __ldg(Wg + (i + 1) * N2 + o);
      const float w2 = __ldg(Wg + (i + 2) * N2 + o), w3 = __ldg(Wg + (i + 3) * N2 + o);
#pragma unroll
      for (int p = 0; p < PT; ++p) {
        const float4 xv = *reinterpret_cast<const float4*>(&xs[p][i]);
        acc[p] = fmaf(xv.x, w0, fmaf(xv.y, w1, fmaf(xv.z, w2, fmaf(xv.w, w3, acc[p]))));
      }
    }
    const float bias = __ldg((layer ? b2 : b1) + bo);
    __syncthreads();   // every thread has finished reading xs
    if (layer == 0) {
#pragma unroll
      for (int p = 0; p < PT; ++p) xs[p][o] = fmaxf(acc[p] + bias, 0.f);
      __syncthreads();
    } else {
      float* Zf = reinterpret_cast<float*>(Z);
#pragma unroll
      for (int p = 0; p < PT; ++p) {
        const float v = acc[p] + bias;
        const float r = v > lambda ? v - lambda : (v < -lambda ? v + lambda : 0.f);
        if (p0 + p < P) Zf[((p0 + p) * E + g * BS + o % BS) * 2 + (o < BS ? 0 : 1)] = r;
      }
    }
  }
}

// inverse W-DFT (c2r: the imaginary parts of mode 0 and of the Nyquist mode do not contribute) of one latitude row,
// plus the filter's own skip and the block's residual:  x[b, hh, xw, e] += scale * irfft(G)[xw] + u[b, hh, xw, e]
template <int KW>
__global__ void __launch_bounds__(128) k_fcn_idft_w(const float2* __restrict__ G, const float4* __restrict__ tw,
                                                    const float* __restrict__ u, float* __restrict__ x, int w, int kw,
                                                    int E, float scale) {
  const long long bh = blockIdx.x;
  const int e = blockIdx.y * 128 + threadIdx.x;
  float gr[KW], gi[KW];
#pragma unroll
  for (int m = 0; m < KW; ++m) {
    gr[m] = 0.f; gi[m] = 0.f;
    if (m < kw) {
      const float2 z = G[(bh * kw + m) * E + e];
      const float c = (m == 0 || 2 * m == w) ? scale : 2.f * scale;
      gr[m] = z.x * c; gi[m] = z.y * c;
    }
  }
  for (int xw = 0; xw < w; ++xw) {
    const float4* t = tw + (size_t)xw * (KW / 2);
    float acc = 0.f;
#pragma unroll
    for (int q = 0; q < KW / 2; ++q) {
      const float4 c = __ldg(t + q);
      acc = fmaf(gr[2 * q], c.x, fmaf(-gi[2 * q], c.y, acc));
      acc = fmaf(gr[2 * q + 1], c.z, fmaf(-gi[2 * q + 1], c.w, acc));
    }
    const long long off = (bh * w + xw) * E + e;
    x[off] += acc + __ldg(u + off);
  }
}

__global__ void k_fcn_copy(const float* __restrict__ src, float* __restrict__ dst, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) dst[i] = src[i];
}

// ---------------------------------------------------------------------------------------------------------------
// engine
// ---------------------------------------------------------------------------------------------------------------
struct FcnBlock {
  uint8_t *fc1, *fc2;
  const float *ln1_g, *ln1_b, *ln2_g, *ln2_b, *fc1_b, *fc2_b, *b1, *b2;
  float *w1c, *w2c;
};

struct FcnEngine : Engine {
  sky_afno_config_t cfg;
  int h, w, T, E, C, hid, kw, h_lo, h_hi, nk;
  std::vector<void*> owned;
  std::vector<FcnBlock> blocks;
  uint8_t *embed_img = nullptr, *head_img = nullptr;
  int kwt = 0;                 // W-DFT kernel instantiation (kept-mode capacity: 8, 24 or 48)
  float2* twiddle = nullptr;   // [w][kwt] (cos, sin) table of the W-DFT kernels
  const float *mean = nullptr, *stdv = nullptr, *embed_b = nullptr, *pos = nullptr;

  FcnEngine(const sky_afno_config_t& c, int dev) : cfg(c) {
    device = dev;
    h = c.nlat / c.patch; w = c.nlon / c.patch; T = h * w;
    E = c.embed; C = c.n_channels; hid = c.mlp_ratio * c.embed;
    const int total = h / 2 + 1;
    const int kept = (int)(total * (double)c.hard_thresholding_fraction);
    h_lo = total - kept; h_hi = total + kept < h ? total + kept : h; nk = h_hi - h_lo;
    kw = kept < w / 2 + 1 ? kept : w / 2 + 1;
    kwt = kw <= 8 ? 8 : kw <= 24 ? 24 : 48;
  }
  ~FcnEngine() override {
    for (void* p : owned) cudaFree(p);
  }

  template <class T_>
  T_* dalloc(size_t n) {
    void* p = nullptr;
    if (cudaMalloc(&p, n * sizeof(T_)) != cudaSuccess) { set_error("cudaMalloc(%zu) failed", n * sizeof(T_)); return nullptr; }
    owned.push_back(p);
    return reinterpret_cast<T_*>(p);
  }
  uint8_t* pack(const char* name, int N, int K, int BN, cudaStream_t st) {
    const float* src = param(name, (uint64_t)N * K);
    if (!src) return nullptr;
    const int Kp = (K + 63) / 64 * 64;
    uint8_t* img = dalloc<uint8_t>((size_t)N * Kp * 2);
    if (!img) return nullptr;
    const long long chunks = (long long)N * Kp / 8;
    k_fcn_pack<<<(unsigned)((chunks + 255) / 256), 256, 0, st>>>(src, N, K, Kp, BN, img);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? img : nullptr;
  }
  float* cplx(const char* name, cudaStream_t st) {
    const int nb = cfg.num_blocks, bs = E / nb;
    const float* src = param(name, 2ull * nb * bs * bs);
    if (!src) return nullptr;
    const long long n = (long long)nb * 4 * bs * bs;
    float* out = dalloc<float>((size_t)n);
    if (!out) return nullptr;
    k_fcn_cplx_weight<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(src, nb, bs, out);
    count_launch();
    return cudaGetLastError() == cudaSuccess ? out : nullptr;
  }

  int prepare(cudaStream_t st) override {
    for (void* p : owned) cudaFree(p);
    owned.clear();
    blocks.assign(cfg.depth, FcnBlock{});
    const int nb = cfg.num_blocks, bs = E / nb;
    char nm[96];
#define FCN_KEEP(dst, name, cnt) if (!((dst) = keep(name, (uint64_t)(cnt), st))) return SKY_ERR_ARG;
#define FCN_NZ(expr) if (!(expr)) return SKY_ERR_ARG;
    FCN_KEEP(mean, "norm.mean", C); FCN_KEEP(stdv, "norm.std", C);
    FCN_KEEP(embed_b, "patch_embed.proj.bias", E);
    FCN_KEEP(pos, "pos_embed", (uint64_t)T * E);
    FCN_NZ(embed_img = pack("patch_embed.proj.weight", E, C * 64, 128, st));
    FCN_NZ(head_img = pack("head.weight", C * 64, E, 128, st));
    FCN_NZ(twiddle = dalloc<float2>((size_t)w * kwt));
    k_fcn_twiddle<<<(unsigned)((w * kwt + 255) / 256), 256, 0, st>>>(twiddle, w, kw, kwt);
    count_launch();
    for (int i = 0; i < cfg.depth; ++i) {
      FcnBlock& b = blocks[i];
#define FCN_NAME(s) (snprintf(nm, sizeof nm, "blocks.%d.%s", i, s), nm)
      FCN_KEEP(b.ln1_g, FCN_NAME("norm1.weight"), E); FCN_KEEP(b.ln1_b, FCN_NAME("norm1.bias"), E);
      FCN_KEEP(b.ln2_g, FCN_NAME("norm2.weight"), E); FCN_KEEP(b.ln2_b, FCN_NAME("norm2.bias"), E);
      FCN_KEEP(b.fc1_b, FCN_NAME("mlp.fc1.bias"), hid); FCN_KEEP(b.fc2_b, FCN_NAME("mlp.fc2.bias"), E);
      FCN_KEEP(b.b1, FCN_NAME("filter.b1"), 2 * nb * bs); FCN_KEEP(b.b2, FCN_NAME("filter.b2"), 2 * nb * bs);
      FCN_NZ(b.w1c = cplx(FCN_NAME("filter.w1"), st)); FCN_NZ(b.w2c = cplx(FCN_NAME("filter.w2"), st));
      FCN_NZ(b.fc1 = pack(FCN_NAME("mlp.fc1.weight"), hid, E, 256, st));
      FCN_NZ(b.fc2 = pack(FCN_NAME("mlp.fc2.weight"), E, hid, 128, st));
#undef FCN_NAME
    }
#undef FCN_KEEP
#undef FCN_NZ
    SKY_CUDA_OK(cudaGetLastError());
    return 0;
  }

  // workspace: x, u (fp32 tokens), v (fp16 LN2 rows), hidden (fp16), two spectral buffers
  struct Ws { float* x; float* u; __half* v; __half* hid; float2* s0; float2* s1; };
  static size_t al(size_t b) { return (b + 255) / 256 * 256; }
  size_t spec_elems(int batch) const { return (size_t)batch * (h > nk ? h : nk) * kw * E; }
  Ws carve(void* ws, int batch) const {
    const size_t M = (size_t)batch * T;
    uint8_t* p = static_cast<uint8_t*>(ws);
    Ws r;
    r.x = reinterpret_cast<float*>(p); p += al(M * E * 4);
    r.u = reinterpret_cast<float*>(p); p += al(M * E * 4);
    r.v = reinterpret_cast<__half*>(p); p += al(M * E * 2);
    r.hid = reinterpret_cast<__half*>(p); p += al(M * hid * 2);
    r.s0 = reinterpret_cast<float2*>(p); p += al(spec_elems(batch) * 8);
    r.s1 = reinterpret_cast<float2*>(p);
    return r;
  }
  size_t workspace_bytes(int batch) const override {
    const size_t M = (size_t)batch * T;
    return al(M * E * 4) * 2 + al(M * E * 2) + al(M * hid * 2) + 2 * al(spec_elems(batch) * 8);
  }

  template <int KW>
  int filter_w(const float* u, float2* F, float2* G, float* x, int batch, bool inverse, cudaStream_t st) {
    const dim3 grid((unsigned)(batch * h), (unsigned)(E / 128));
    const float scale = (float)(1.0 / sqrt((double)w));
    const float4* tw = reinterpret_cast<const float4*>(twiddle);
    if (!inverse) k_fcn_dft_w<KW><<<grid, 128, 0, st>>>(u, tw, F, w, kw, E, scale);
    else k_fcn_idft_w<KW><<<grid, 128, 0, st>>>(G, tw, u, x, w, kw, E, scale);
    SKY_CUDA_OK(cudaGetLastError());
    return 0;
  }
  int filter_w_any(const float* u, float2* F, float2* G, float* x, int batch, bool inverse, cudaStream_t st) {
    if (kwt == 8) return filter_w<8>(u, F, G, x, batch, inverse, st);
    if (kwt == 24) return filter_w<24>(u, F, G, x, batch, inverse, st);
    return filter_w<48>(u, F, G, x, batch, inverse, st);
  }

  int step(const float* x_in, float* x_out, int batch, void* ws, size_t ws_bytes, cudaStream_t st) override {
    if (!loaded) { set_error("weights not loaded"); return SKY_ERR_STATE; }
    if (ws_bytes < workspace_bytes(batch)) { set_error("workspace too small"); return SKY_ERR_ARG; }
    const Ws b = carve(ws, batch);
    const long long M = (long long)batch * T;
    const int nbk = cfg.num_blocks;
    const float hs = (float)(1.0 / sqrt((double)h));
    const long long P = (long long)batch * nk * kw;
    int rc = 0;
#define FCN_L(tag, n, ...) do { prof_begin(tag, st); if ((rc = (__VA_ARGS__))) return rc; prof_end(tag, st); count_launch(n); } while (0)
#define FCN_K(tag, ...) do { prof_begin(tag, st); __VA_ARGS__; SKY_CUDA_OK(cudaGetLastError()); prof_end(tag, st); count_launch(); } while (0)
    FCN_L(KT_FCN_EMBED, 1, launch_gemm_tc<ProdFcnEmbed, EpiFcnEmbed, 128>(
        ProdFcnEmbed{x_in, mean, stdv, C, cfg.nlat, cfg.nlon, w, T, M}, EpiFcnEmbed{b.x, embed_b, pos, E, T, M},
        embed_img, M, E, C * 64, num_sms, st));
    if (stop_after == 0) return 0;
    const unsigned ln_grid = (unsigned)((M + 7) / 8);
    for (int i = 0; i < cfg.depth; ++i) {
      const FcnBlock& k = blocks[i];
      FCN_K(KT_FCN_LN, k_fcn_ln<false><<<ln_grid, 256, 0, st>>>(b.x, b.u, k.ln1_g, k.ln1_b, cfg.ln_eps, M, E));
      FCN_L(KT_FCN_SPEC, 1, filter_w_any(b.u, b.s0, nullptr, nullptr, batch, false, st));
      FCN_K(KT_FCN_SPEC, k_fcn_dft_h<<<dim3((unsigned)(batch * kw), (unsigned)(E / 32)), 256, 0, st>>>(
                             b.s0, b.s1, h, h_lo, h, nk, kw, E, 1, hs));
      FCN_K(KT_FCN_SPEC, k_fcn_block_mlp<FCN_BS><<<dim3((unsigned)((P + 31) / 32), (unsigned)nbk), 2 * FCN_BS, 0, st>>>(
                             b.s1, b.s0, k.w1c, k.b1, k.w2c, k.b2, P, E, nbk, cfg.sparsity));
      FCN_K(KT_FCN_SPEC, k_fcn_dft_h<<<dim3((unsigned)(batch * kw), (unsigned)(E / 32)), 256, 0, st>>>(
                             b.s0, b.s1, h, h_lo, nk, h, kw, E, 0, hs));
      FCN_L(KT_FCN_SPEC, 1, filter_w_any(b.u, nullptr, b.s1, b.x, batch, true, st));
      if (stop_after == 2 * i + 1) return 0;
      FCN_K(KT_FCN_LN, k_fcn_ln<true><<<ln_grid, 256, 0, st>>>(b.x, b.v, k.ln2_g, k.ln2_b, cfg.ln_eps, M, E));
      if ((rc = range_scan(0, b.v, (size_t)M * E * 2, st))) return rc;
      FCN_L(KT_FCN_MLP, 1, launch_gemm_tc<ProdPlainF16, EpiStoreF16<true>, 256>(
          ProdPlainF16{b.v, E, M, E}, EpiStoreF16<true>{b.hid, hid, k.fc1_b, M}, k.fc1, M, hid, E, num_sms, st));
      if ((rc = range_scan(5, b.hid, (size_t)M * hid * 2, st))) return rc;
      FCN_L(KT_FCN_MLP, 1, launch_gemm_tc<ProdPlainF16, EpiFcnResidual, 128>(
          ProdPlainF16{b.hid, hid, M, hid}, EpiFcnResidual{b.x, k.fc2_b, E, M}, k.fc2, M, E, hid, num_sms, st));
      if (stop_after == 2 * i + 2) return 0;
    }
    FCN_L(KT_FCN_HEAD, 1, launch_gemm_tc<ProdPlainF32, EpiFcnHead, 128>(
        ProdPlainF32{b.x, E, M, E}, EpiFcnHead{x_out, mean, stdv, C, cfg.nlat, cfg.nlon, w, T, M}, head_img, M, C * 64, E,
        num_sms, st));
#undef FCN_L
#undef FCN_K
    return 0;
  }

  int debug_copy(const char* what, float* dst, uint64_t max_floats, void* ws, int batch, cudaStream_t st) override {
    if (!strcmp(what, "range")) {
      if (!range_dev) { set_error("range guard is off"); return SKY_ERR_STATE; }
      SKY_CUDA_OK(cudaMemcpyAsync(dst, range_dev, 8 * sizeof(float), cudaMemcpyDeviceToDevice, st));
      return 0;
    }
    if (strcmp(what, "tokens")) { set_error("unknown tap '%s' (FourCastNet has 'tokens' and 'range')", what); return SKY_ERR_ARG; }
    const long long n = (long long)batch * T * E;
    if ((uint64_t)n > max_floats) { set_error("tap needs %lld floats", n); return SKY_ERR_ARG; }
    k_fcn_copy<<<(unsigned)((n + 255) / 256), 256, 0, st>>>(carve(ws, batch).x, dst, n);
    SKY_CUDA_OK(cudaGetLastError());
    return 0;
  }
};

}  // namespace

Engine* make_fcn_engine(const sky_afno_config_t& c, int device) {
  if (c.patch != 8 || c.nlat % 8 || c.nlon % 8 || c.nlat <= 0 || c.nlon <= 0) { set_error("FourCastNet: patch 8 and a grid that tiles by it"); return nullptr; }
  if (c.embed % 128 || c.embed > 1024 || c.num_blocks <= 0 || c.embed != c.num_blocks * FCN_BS) {
    set_error("FourCastNet: embed must be num_blocks x %d, a multiple of 128 and <= 1024 (got %d / %d)", FCN_BS, c.embed, c.num_blocks);
    return nullptr;
  }
  if ((c.n_channels * 64) % 128 || c.n_channels <= 0) { set_error("FourCastNet: an even channel count"); return nullptr; }
  if ((c.mlp_ratio * c.embed) % 256 || c.depth <= 0) { set_error("FourCastNet: mlp width must tile by 256"); return nullptr; }
  if (c.nlat / 8 > FCN_MAXH) { set_error("FourCastNet: more than %d token rows", FCN_MAXH); return nullptr; }
  FcnEngine* e = new FcnEngine(c, device);
  if (e->kw > 48 || e->kw <= 0 || e->nk <= 0) { set_error("FourCastNet: %d kept W-modes (1 ... 48 supported)", e->kw); delete e; return nullptr; }
  return e;
}

}  // namespace sky
