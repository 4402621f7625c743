// HBM-bound kernels of the denoise + decode path: normalisations, modulation, RoPE, layout shuffles, sampler update.
// All of them move 128-bit vectors per thread, reduce with warp shuffles, and do their arithmetic in fp32.
#include "common.cuh"
#include "host.h"

namespace dk {

template <typename T>
__device__ __forceinline__ void load8(const T* p, float (&v)[8]) {
  const uint4 u = *reinterpret_cast<const uint4*>(p);
  const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const float2 f = Half16<T>::unpack(w[i]);
    v[2 * i] = f.x;
    v[2 * i + 1] = f.y;
  }
}
template <typename T>
__device__ __forceinline__ void store8(T* p, const float (&v)[8]) {
  uint4 o;
  o.x = Half16<T>::pack(v[0], v[1]);
  o.y = Half16<T>::pack(v[2], v[3]);
  o.z = Half16<T>::pack(v[4], v[5]);
  o.w = Half16<T>::pack(v[6], v[7]);
  *reinterpret_cast<uint4*>(p) = o;
}
template <typename T>
__device__ __forceinline__ float round16(float v) {
  return Half16<T>::to_f(Half16<T>::from_f(v));
}

// block-wide sum for blockDim.x = NT (multiple of 32); every thread gets the result
template <int NT>
__device__ __forceinline__ float block_sum(float v, float* red) {
  v = warp_sum(v);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = (lane < NT / 32) ? red[lane] : 0.f;
  t = warp_sum(t);
  return t;
}
template <int NT>
__device__ __forceinline__ float block_max(float v, float* red) {
  v = warp_max(v);
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  __syncthreads();
  if (lane == 0) red[warp] = v;
  __syncthreads();
  float t = (lane < NT / 32) ? red[lane] : -INFINITY;
  t = warp_max(t);
  return t;
}

// ------------------------------------------------------------------------------------------------
// K2: LayerNorm (no affine) + adaLN modulate.  One 128-thread block per row, row kept in registers.
//     mlx.fast.layer_norm semantics: biased variance, fp32 accumulation, (x-mu)*rsqrt(var+eps)*w + b with
//     w = 1 + scale, b = shift (reference mlx/mmdit.py:958-972).
// ------------------------------------------------------------------------------------------------
constexpr int LN_WARPS = 4;     // rows per block
constexpr int LN_MAXV = 16;     // h <= 32 lanes * 8 * 16 = 4096

// One warp per row: the row lives in registers (<= 16 x 128-bit loads in flight per lane), statistics via warp
// shuffles only — no shared memory, no block barriers.
template <typename T, int NV>
__global__ void __launch_bounds__(LN_WARPS * 32)
ln_modulate_kernel(const T* __restrict__ x, T* __restrict__ y, const T* __restrict__ shift, const T* __restrict__ scale,
                   long long mod_ld, int rows, int rows_per_batch, int h, float eps) {
  const int row = blockIdx.x * LN_WARPS + (threadIdx.x >> 5);
  if (row >= rows) return;
  const int lane = threadIdx.x & 31;
  const int b = row / rows_per_batch;
  const T* xr = x + static_cast<long long>(row) * h;
  T* yr = y + static_cast<long long>(row) * h;
  const int nvec = h / 8;
  float v[NV][8];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int vec = lane + i * 32;
    if (vec < nvec) {
      load8(xr + vec * 8, v[i]);
#pragma unroll
      for (int j = 0; j < 8; ++j) s += v[i][j];
    }
  }
  const float mean = warp_sum(s) / h;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int vec = lane + i * 32;
    if (vec < nvec) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float d = v[i][j] - mean;
        q += d * d;
      }
    }
  }
  const float rstd = rsqrtf(warp_sum(q) / h + eps);
  const T* sh = shift + static_cast<long long>(b) * mod_ld;
  const T* sc = scale + static_cast<long long>(b) * mod_ld;
#pragma unroll
  for (int i = 0; i < NV; ++i) {
    const int vec = lane + i * 32;
    if (vec < nvec) {
      float a[8], c[8], o[8];
      load8(sc + vec * 8, a);
      load8(sh + vec * 8, c);
#pragma unroll
      for (int j = 0; j < 8; ++j) o[j] = (v[i][j] - mean) * rstd * (1.0f + a[j]) + c[j];
      store8(yr + vec * 8, o);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// QK-RMSNorm + RoPE, in place on the q and k thirds of the packed QKV buffer.  One warp per (row, head, q|k).
// ------------------------------------------------------------------------------------------------
template <typename T, int D>
__global__ void __launch_bounds__(256)
qk_norm_rope_kernel(T* __restrict__ qkv, int rows, int S, int heads, int split, const T* __restrict__ q_w,
                    const T* __restrict__ k_w, const T* __restrict__ q_w2, const T* __restrict__ k_w2,
                    const float* __restrict__ rope, float eps) {
  constexpr int EPL = D / 32;  // elements per lane: 2 (d=64) or 4 (d=128)
  const long long gw = (static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  const long long total = static_cast<long long>(rows) * heads * 2;
  if (gw >= total) return;
  const int which = static_cast<int>(gw % 2);  // 0 = q, 1 = k
  const int head = static_cast<int>((gw / 2) % heads);
  const long long row = gw / (2LL * heads);
  const int pos = static_cast<int>(row % S);
  const int h = heads * D;
  T* p = qkv + row * (3LL * h) + static_cast<long long>(which) * h + head * D + lane * EPL;

  float v[EPL];
  if (EPL == 4) {
    const uint2 u = *reinterpret_cast<const uint2*>(p);
    const float2 a = Half16<T>::unpack(u.x), b = Half16<T>::unpack(u.y);
    v[0] = a.x;
    v[1] = a.y;
    v[EPL - 2] = b.x;
    v[EPL - 1] = b.y;
  } else {
    const uint32_t u = *reinterpret_cast<const uint32_t*>(p);
    const float2 a = Half16<T>::unpack(u);
    v[0] = a.x;
    v[1] = a.y;
  }
  const T* w = (pos < split) ? (which == 0 ? q_w : k_w) : (which == 0 ? q_w2 : k_w2);
  if (w != nullptr) {
    float ss = 0.f;
#pragma unroll
    for (int i = 0; i < EPL; ++i) ss += v[i] * v[i];
    ss = warp_sum(ss);
    const float rstd = rsqrtf(ss / D + eps);
#pragma unroll
    for (int i = 0; i < EPL; ++i)
      v[i] = round16<T>(v[i] * rstd * Half16<T>::to_f(w[lane * EPL + i]));  // nn.RMSNorm output in the activation dtype
  }
  if (rope != nullptr) {
    // rope[pos][pair] = (cos, sin); out = (x0 cos - x1 sin, x0 sin + x1 cos)  — mlx/mmdit.py:934-942
    const float* rp = rope + (static_cast<long long>(pos) * (D / 2) + lane * (EPL / 2)) * 2;
#pragma unroll
    for (int i = 0; i < EPL / 2; ++i) {
      const float c = rp[2 * i], sn = rp[2 * i + 1];
      const float x0 = v[2 * i], x1 = v[2 * i + 1];
      v[2 * i] = x0 * c - x1 * sn;
      v[2 * i + 1] = x0 * sn + x1 * c;
    }
  }
  if (EPL == 4) {
    uint2 o;
    o.x = Half16<T>::pack(v[0], v[1]);
    o.y = Half16<T>::pack(v[EPL - 2], v[EPL - 1]);
    *reinterpret_cast<uint2*>(p) = o;
  } else {
    *reinterpret_cast<uint32_t*>(p) = Half16<T>::pack(v[0], v[1]);
  }
}

// ------------------------------------------------------------------------------------------------
// small elementwise kernels (grid-stride over 8-element vectors)
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void silu_add_kernel(const T* __restrict__ y, const T* __restrict__ temb, T* __restrict__ c, int n_t, int B,
                                int h) {
  const long long nvec = static_cast<long long>(n_t) * B * h / 8;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < nvec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long e = i * 8;
    const int col = static_cast<int>(e % h);
    const long long row = e / h;
    const int b = static_cast<int>(row % B);
    const int t = static_cast<int>(row / B);
    float a[8], d[8], o[8];
    load8(y + static_cast<long long>(b) * h + col, a);
    load8(temb + static_cast<long long>(t) * h + col, d);
#pragma unroll
    for (int j = 0; j < 8; ++j) o[j] = silu_f(round16<T>(a[j] + d[j]));
    store8(c + e, o);
  }
}

template <typename T>
__global__ void act_kernel(const T* __restrict__ x, T* __restrict__ y, long long n, int act) {
  const long long nvec = n / 8;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < nvec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    float a[8];
    load8(x + i * 8, a);
#pragma unroll
    for (int j = 0; j < 8; ++j) a[j] = act == DK_ACT_SILU ? silu_f(a[j]) : (act == DK_ACT_GELU_ERF ? gelu_erf(a[j]) : (act == DK_ACT_QUICK_GELU ? quick_gelu_f(a[j]) : a[j]));
    store8(y + i * 8, a);
  }
}

// patchify / unpatchify: one thread per (token, output feature)
template <typename T>
__global__ void patchify_kernel(const T* __restrict__ latent, T* __restrict__ rows, int B, int H, int W, int C,
                                int order) {
  const int F = 4 * C;
  const long long total = static_cast<long long>(B) * (H / 2) * (W / 2) * F;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int f = static_cast<int>(i % F);
    const long long tok = i / F;
    const int wp = static_cast<int>(tok % (W / 2));
    const int hp = static_cast<int>((tok / (W / 2)) % (H / 2));
    const int b = static_cast<int>(tok / (static_cast<long long>(W / 2) * (H / 2)));
    int c, ph, pw;
    if (order == 0) {  // (c, ph, pw)
      c = f / 4;
      ph = (f / 2) % 2;
      pw = f % 2;
    } else {  // (ph, pw, c)
      ph = f / (2 * C);
      pw = (f / C) % 2;
      c = f % C;
    }
    rows[i] = latent[((static_cast<long long>(b) * H + 2 * hp + ph) * W + 2 * wp + pw) * C + c];
  }
}
template <typename T>
__global__ void unpatchify_kernel(const T* __restrict__ rows, T* __restrict__ latent, int B, int H, int W, int C,
                                  int order) {
  const int F = 4 * C;
  const long long total = static_cast<long long>(B) * H * W * C;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < total;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const int c = static_cast<int>(i % C);
    const int x = static_cast<int>((i / C) % W);
    const int y = static_cast<int>((i / (static_cast<long long>(C) * W)) % H);
    const int b = static_cast<int>(i / (static_cast<long long>(C) * W * H));
    const int ph = y & 1, pw = x & 1;
    const long long tok = (static_cast<long long>(b) * (H / 2) + y / 2) * (W / 2) + x / 2;
    const int f = order == 0 ? (c * 4 + ph * 2 + pw) : ((ph * 2 + pw) * C + c);
    latent[i] = rows[tok * F + f];
  }
}

template <typename T>
__global__ void pos_embed_crop_kernel(const T* __restrict__ table, T* __restrict__ out, int max_hw, int hp, int wp,
                                      int h) {
  const int y0 = (max_hw - hp) / 2, x0 = (max_hw - wp) / 2;
  const long long nvec = static_cast<long long>(hp) * wp * h / 8;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < nvec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long e = i * 8;
    const int col = static_cast<int>(e % h);
    const long long tok = e / h;
    const int xx = static_cast<int>(tok % wp), yy = static_cast<int>(tok / wp);
    *reinterpret_cast<uint4*>(out + e) =
        *reinterpret_cast<const uint4*>(table + (static_cast<long long>(y0 + yy) * max_hw + x0 + xx) * h + col);
  }
}

template <typename T>
__global__ void copy_rows_kernel(const T* __restrict__ src, T* __restrict__ dst, int B, int rows, int h, int dst_rows,
                                 int dst_off, int src_rows, int src_off) {
  const long long nvec = static_cast<long long>(B) * rows * h / 8;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < nvec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long e = i * 8;
    const int col = static_cast<int>(e % h);
    const long long rr = e / h;
    const int r = static_cast<int>(rr % rows);
    const int b = static_cast<int>(rr / rows);
    *reinterpret_cast<uint4*>(dst + (static_cast<long long>(b) * dst_rows + dst_off + r) * h + col) =
        *reinterpret_cast<const uint4*>(src + (static_cast<long long>(b) * src_rows + src_off + r) * h + col);
  }
}

// ------------------------------------------------------------------------------------------------
// sampler (fp32 state) — reference mlx/__init__.py:691-719, 775-782; mlx/sampler.py:37-39
// ------------------------------------------------------------------------------------------------
template <typename T>
__global__ void sampler_prepare_kernel(const float* __restrict__ x, T* __restrict__ xin, long long n, int reps) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const T v = Half16<T>::from_f(x[i]);
    for (int k = 0; k < reps; ++k) xin[k * n + i] = v;
  }
}
template <typename T>
__global__ void sampler_step_kernel(float* __restrict__ x, const T* __restrict__ xin, const T* __restrict__ out,
                                    long long n, float sigma, float sigma_next, float cfg) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    // calculate_denoised: model_input - model_output * sigma (fp32 sigma promotes to fp32)
    float den = Half16<T>::to_f(xin[i]) - Half16<T>::to_f(out[i]) * sigma;
    if (cfg > 0.f) {
      const float den_neg = Half16<T>::to_f(xin[n + i]) - Half16<T>::to_f(out[n + i]) * sigma;
      den = den_neg + cfg * (den - den_neg);
    }
    const float xv = x[i];
    const float d = (xv - den) / sigma;          // to_d
    x[i] = xv + d * (sigma_next - sigma);        // Euler
  }
}
__global__ void axpb_kernel(const float* __restrict__ x, float* __restrict__ y, long long n, float a, float b) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    y[i] = x[i] * a + b;
}
// MLX affine 4-bit weights (mx.quantize, group_size 64, bits 4; reference nn.quantize call sites mlx/model_io.py:728-734,
// 772-775) -> dense 16-bit: w[n, k] = scales[n, k / group] * q[n, k] + biases[n, k / group], q = nibble (k % 8) of
// word wq[n, k / 8] (element 0 in the low bits).  One thread = one word = 8 outputs = one 16-byte store.
template <typename T>
__global__ void dequant_q4_kernel(const uint32_t* __restrict__ wq, const T* __restrict__ scales,
                                  const T* __restrict__ biases, T* __restrict__ out, long long N, int K, int group) {
  const int wpr = K / 8;  // words per row
  const int gpr = K / group;
  const long long nwords = N * wpr;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < nwords;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long n = i / wpr;
    const int k0 = static_cast<int>(i - n * wpr) * 8;
    const uint32_t w = wq[i];
    const float sc = Half16<T>::to_f(scales[n * gpr + k0 / group]);
    const float bi = Half16<T>::to_f(biases[n * gpr + k0 / group]);
    uint32_t o[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float a = __fmaf_rn(sc, static_cast<float>((w >> (8 * j)) & 0xFu), bi);
      const float b = __fmaf_rn(sc, static_cast<float>((w >> (8 * j + 4)) & 0xFu), bi);
      o[j] = Half16<T>::pack(a, b);
    }
    *reinterpret_cast<uint4*>(out + n * K + k0) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

// read_image (reference mlx/__init__.py:536-551): uint8 [pixels, src_c >= 3] -> 16-bit [pixels, cpad], channels 0..2 =
// u8 / 255 * 2 - 1 (fp32 arithmetic, then rounded to T), channels 3.. = 0 (the tensor-core conv wants Cin % 64 == 0)
template <typename T>
__global__ void image_pre_kernel(const uint8_t* __restrict__ img, T* __restrict__ out, long long pixels, int src_c,
                                 int cpad) {
  const int vpp = cpad / 8;
  const long long nvec = pixels * vpp;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < nvec;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long p = i / vpp;
    const int v = static_cast<int>(i - p * vpp);
    uint4 w = make_uint4(0u, 0u, 0u, 0u);
    if (v == 0) {
      const uint8_t* px = img + p * src_c;
      // three separately rounded fp32 ops like the reference's (x / 255) * 2 - 1 (no FMA contraction)
      const float r = __fsub_rn(__fmul_rn(__fdiv_rn(static_cast<float>(px[0]), 255.f), 2.f), 1.f);
      const float g = __fsub_rn(__fmul_rn(__fdiv_rn(static_cast<float>(px[1]), 255.f), 2.f), 1.f);
      const float b = __fsub_rn(__fmul_rn(__fdiv_rn(static_cast<float>(px[2]), 255.f), 2.f), 1.f);
      w.x = Half16<T>::pack(r, g);
      w.y = Half16<T>::pack(b, 0.f);
    }
    *reinterpret_cast<uint4*>(out + p * cpad + v * 8) = w;
  }
}
__global__ void axpby_kernel(const float* __restrict__ x, const float* __restrict__ y, float* __restrict__ o,
                             long long n, float a, float b) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    o[i] = a * x[i] + b * y[i];
}
// VAE encoder posterior sample (reference mlx/__init__.py:586-594) + latent_format.process_in (:729-730):
//   hidden [pixels, 2C] = (mean | logvar); z = mean + exp(0.5 * clip(logvar, -30, 20)) * noise; out = (z - shift) * scale
template <typename T>
__global__ void vae_sample_latent_kernel(const T* __restrict__ hidden, const float* __restrict__ noise,
                                         float* __restrict__ out, long long pixels, int C, float shift, float scale) {
  const long long n = pixels * C;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long p = i / C;
    const int c = static_cast<int>(i - p * C);
    const float mean = Half16<T>::to_f(hidden[p * 2 * C + c]);
    const float logvar = fminf(fmaxf(Half16<T>::to_f(hidden[p * 2 * C + C + c]), -30.f), 20.f);
    const float z = mean + __expf(0.5f * logvar) * noise[i];
    out[i] = (z - shift) * scale;
  }
}
template <typename T>
__global__ void cast_f32_to_16_kernel(const float* __restrict__ x, T* __restrict__ y, long long n) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    y[i] = Half16<T>::from_f(x[i]);
}
template <typename T>
__global__ void cast_16_to_f32_kernel(const T* __restrict__ x, float* __restrict__ y, long long n) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x)
    y[i] = Half16<T>::to_f(x[i]);
}

// ------------------------------------------------------------------------------------------------
// GroupNorm (VAE).  stats: two-stage, deterministic (no atomics across blocks):
//   stage 1: grid (chunks, B); each block reduces its pixel slab to per-group (sum, sumsq) partials
//   stage 2: one thread per (b, g) folds the partials in double and writes (mean, rstd)
// apply: grid (blocks, B); a thread keeps its 8 channels' (scale, shift) in registers and streams pixels.
// ------------------------------------------------------------------------------------------------
constexpr int GN_MAX_CHUNKS = 1024;
constexpr int GN_THREADS = 256;

static inline int gn_chunks(int HW) {
  // >= 64 pixels per block, at most GN_MAX_CHUNKS blocks per image
  int c = (HW + 63) / 64;
  if (c > GN_MAX_CHUNKS) c = GN_MAX_CHUNKS;
  if (c < 1) c = 1;
  return c;
}

template <typename T>
__global__ void __launch_bounds__(GN_THREADS)
groupnorm_partial_kernel(const T* __restrict__ x, float* __restrict__ partial, int HW, int C, int G, int chunks) {
  extern __shared__ float sm[];  // [2*C] channel totals + 2 x [GN_THREADS*8] staging
  const int b = blockIdx.y, chunk = blockIdx.x;
  const int per = (HW + chunks - 1) / chunks;
  const int p0 = chunk * per;
  const int p1 = min(HW, p0 + per);
  const int vec_per_pix = C / 8;
  const int pix_per_iter = GN_THREADS / vec_per_pix;  // C <= 2048
  const int my_vec = threadIdx.x % vec_per_pix;
  const int my_pix = threadIdx.x / vec_per_pix;
  float s[8], q[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = q[j] = 0.f;
  if (my_pix < pix_per_iter) {
    const T* base = x + static_cast<long long>(b) * HW * C + my_vec * 8;
    int p = p0 + my_pix;
    // four independent 128-bit loads in flight per thread (HBM latency hiding)
    for (; p + 3 * pix_per_iter < p1; p += 4 * pix_per_iter) {
      uint4 u[4];
#pragma unroll
      for (int k = 0; k < 4; ++k)
        u[k] = *reinterpret_cast<const uint4*>(base + static_cast<long long>(p + k * pix_per_iter) * C);
#pragma unroll
      for (int k = 0; k < 4; ++k) {
        const uint32_t w[4] = {u[k].x, u[k].y, u[k].z, u[k].w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const float2 f = Half16<T>::unpack(w[i]);
          s[2 * i] += f.x;
          s[2 * i + 1] += f.y;
          q[2 * i] += f.x * f.x;
          q[2 * i + 1] += f.y * f.y;
        }
      }
    }
    for (; p < p1; p += pix_per_iter) {
      float v[8];
      load8(base + static_cast<long long>(p) * C, v);
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        s[j] += v[j];
        q[j] += v[j] * v[j];
      }
    }
  }
  // deterministic in-block reduction (fixed summation order, no atomics): stage every thread's 8 channel sums as
  // [pixel slot][channel], then one thread per channel folds the pixel slots in order
  float* st_s = sm + 2 * C;                    // [pix_per_iter][C]
  float* st_q = st_s + GN_THREADS * 8;         // [pix_per_iter][C]
  if (my_pix < pix_per_iter) {
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      st_s[my_pix * C + my_vec * 8 + j] = s[j];
      st_q[my_pix * C + my_vec * 8 + j] = q[j];
    }
  }
  __syncthreads();
  for (int c = threadIdx.x; c < C; c += GN_THREADS) {
    float ts = 0.f, tq = 0.f;
    for (int pp = 0; pp < pix_per_iter; ++pp) {
      ts += st_s[pp * C + c];
      tq += st_q[pp * C + c];
    }
    sm[c] = ts;
    sm[C + c] = tq;
  }
  __syncthreads();
  const int cpg = C / G;
  for (int g = threadIdx.x; g < G; g += GN_THREADS) {
    float ts = 0.f, tq = 0.f;
    for (int c = 0; c < cpg; ++c) {
      ts += sm[g * cpg + c];
      tq += sm[C + g * cpg + c];
    }
    float* dst = partial + ((static_cast<long long>(b) * chunks + chunk) * G + g) * 2;
    dst[0] = ts;
    dst[1] = tq;
  }
}
// one 256-thread block per (b, g): threads stride over the chunk partials four at a time (independent loads in
// flight: with one warp per (b, g) the 8192 partials of a 1024^2 image were a 256-deep chain of dependent-latency
// loads per lane, 45 us per launch x 30 launches = 11 % of a batch-1 decode), accumulation in double; fixed
// thread -> chunk assignment, fixed shuffle tree and fixed cross-warp order: deterministic
constexpr int GNF_THREADS = 256;
__global__ void __launch_bounds__(GNF_THREADS)
groupnorm_finalize_kernel(const float* __restrict__ partial, float* __restrict__ stats, int B, int G, int chunks,
                          double count, float eps) {
  const int idx = blockIdx.x;   // b * G + g
  const int b = idx / G, g = idx % G;
  const int t = threadIdx.x, lane = t & 31, warp = t >> 5;
  const float2* base = reinterpret_cast<const float2*>(partial) + static_cast<long long>(b) * chunks * G + g;
  double s = 0.0, q = 0.0;
  int c = t;
  for (; c + 3 * GNF_THREADS < chunks; c += 4 * GNF_THREADS) {
    const float2 p0 = base[static_cast<long long>(c) * G];
    const float2 p1 = base[static_cast<long long>(c + GNF_THREADS) * G];
    const float2 p2 = base[static_cast<long long>(c + 2 * GNF_THREADS) * G];
    const float2 p3 = base[static_cast<long long>(c + 3 * GNF_THREADS) * G];
    s += (static_cast<double>(p0.x) + p1.x) + (static_cast<double>(p2.x) + p3.x);
    q += (static_cast<double>(p0.y) + p1.y) + (static_cast<double>(p2.y) + p3.y);
  }
  for (; c < chunks; c += GNF_THREADS) {
    const float2 p = base[static_cast<long long>(c) * G];
    s += p.x;
    q += p.y;
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) {
    s += __shfl_xor_sync(0xffffffffu, s, o);
    q += __shfl_xor_sync(0xffffffffu, q, o);
  }
  __shared__ double red[2][GNF_THREADS / 32];
  if (lane == 0) {
    red[0][warp] = s;
    red[1][warp] = q;
  }
  __syncthreads();
  if (t == 0) {
    double ss = 0.0, qq = 0.0;
#pragma unroll
    for (int w = 0; w < GNF_THREADS / 32; ++w) {
      ss += red[0][w];
      qq += red[1][w];
    }
    const double mean = ss / count;
    double var = qq / count - mean * mean;
    if (var < 0.0) var = 0.0;
    stats[idx * 2] = static_cast<float>(mean);
    stats[idx * 2 + 1] = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
  }
}
template <typename T>
__global__ void __launch_bounds__(GN_THREADS)
groupnorm_apply_kernel(const T* __restrict__ x, T* __restrict__ y, const float* __restrict__ stats,
                       const T* __restrict__ gamma, const T* __restrict__ beta, int HW, int C, int G, int silu) {
  const int b = blockIdx.y;
  const int vec_per_pix = C / 8;
  const int pix_per_iter = GN_THREADS / vec_per_pix;
  const int my_vec = threadIdx.x % vec_per_pix;
  const int my_pix = threadIdx.x / vec_per_pix;
  if (my_pix >= pix_per_iter) return;
  const int cpg = C / G;
  float sc[8], sh[8];
  {
    float ga[8], be[8];
    load8(gamma + my_vec * 8, ga);
    load8(beta + my_vec * 8, be);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int g = (my_vec * 8 + j) / cpg;
      const float mean = stats[(b * G + g) * 2], rstd = stats[(b * G + g) * 2 + 1];
      sc[j] = rstd * ga[j];
      sh[j] = be[j] - mean * rstd * ga[j];
    }
  }
  const long long img = static_cast<long long>(b) * HW * C + my_vec * 8;
  const int step = gridDim.x * pix_per_iter;
  int p = blockIdx.x * pix_per_iter + my_pix;
  // four pixels per iteration: all loads issued before the first use
  for (; p + 3 * step < HW; p += 4 * step) {
    uint4 u[4];
#pragma unroll
    for (int k = 0; k < 4; ++k)
      u[k] = *reinterpret_cast<const uint4*>(x + img + static_cast<long long>(p + k * step) * C);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const uint32_t w[4] = {u[k].x, u[k].y, u[k].z, u[k].w};
      float v[8];
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float2 f = Half16<T>::unpack(w[i]);
        v[2 * i] = f.x;
        v[2 * i + 1] = f.y;
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        float o = fmaf(v[j], sc[j], sh[j]);
        if (silu) o = silu_f(round16<T>(o));
        v[j] = o;
      }
      store8(y + img + static_cast<long long>(p + k * step) * C, v);
    }
  }
  for (; p < HW; p += step) {
    float v[8];
    load8(x + img + static_cast<long long>(p) * C, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      float o = fmaf(v[j], sc[j], sh[j]);
      if (silu) o = silu_f(round16<T>(o));
      v[j] = o;
    }
    store8(y + img + static_cast<long long>(p) * C, v);
  }
}

// nearest 2x: grid (output rows / rows-per-block, B); a thread owns one 128-bit channel vector of one output column
// and walks output rows — no per-element divisions
template <typename T>
__global__ void __launch_bounds__(256)
upsample2x_kernel(const T* __restrict__ x, T* __restrict__ y, int H, int W, int C, int rows_per_block) {
  const int b = blockIdx.y;
  const int vpp = C / 8;                 // vectors per pixel
  const int row_vecs = 2 * W * vpp;      // vectors per output row
  const int oy0 = blockIdx.x * rows_per_block;
  const int oy1 = min(2 * H, oy0 + rows_per_block);
  const T* xin = x + static_cast<long long>(b) * H * W * C;
  T* yout = y + static_cast<long long>(b) * 4 * H * W * C;
  for (int v = threadIdx.x; v < row_vecs; v += blockDim.x) {
    const int ox = v / vpp;
    const int cv = v - ox * vpp;
    const long long in_col = static_cast<long long>(ox >> 1) * C + cv * 8;
    const long long out_col = static_cast<long long>(ox) * C + cv * 8;
    for (int oy = oy0; oy < oy1; oy += 2) {   // rows oy, oy+1 replicate input row oy/2 (oy0 is even)
      const uint4 u = *reinterpret_cast<const uint4*>(xin + static_cast<long long>(oy >> 1) * W * C + in_col);
      __stcs(reinterpret_cast<uint4*>(yout + static_cast<long long>(oy) * 2 * W * C + out_col), u);
      if (oy + 1 < oy1) __stcs(reinterpret_cast<uint4*>(yout + static_cast<long long>(oy + 1) * 2 * W * C + out_col), u);
    }
  }
}

// row softmax (VAE mid-block attention, reference mlx/vae.py:49-52): p = softmax(scale * s), fp32 math, 16-bit out
template <typename T>
__global__ void __launch_bounds__(256)
softmax_rows_kernel(T* __restrict__ x, int n, long long ld, float scale) {
  __shared__ float red[8];
  T* row = x + static_cast<long long>(blockIdx.x) * ld;
  const int nvec = n / 8;
  float mx = -INFINITY;
  for (int i = threadIdx.x; i < nvec; i += 256) {
    float v[8];
    load8(row + i * 8, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) mx = fmaxf(mx, v[j]);
  }
  mx = block_max<256>(mx, red);
  const float k = scale * 1.44269504088896341f;
  float sum = 0.f;
  for (int i = threadIdx.x; i < nvec; i += 256) {
    float v[8];
    load8(row + i * 8, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) sum += exp2f((v[j] - mx) * k);
  }
  sum = block_sum<256>(sum, red);
  const float inv = 1.0f / sum;
  for (int i = threadIdx.x; i < nvec; i += 256) {
    float v[8];
    load8(row + i * 8, v);
#pragma unroll
    for (int j = 0; j < 8; ++j) v[j] = exp2f((v[j] - mx) * k) * inv;
    store8(row + i * 8, v);
  }
}

// decode tail of one channel value: clip(x/2 + 0.5, 0, 1) in the activation dtype (mlx/__init__.py:583) and
// uint8 = trunc(v * 255) (:526).  image_post and image_post_masked both go through these two helpers, so the
// regenerated pixels of an inpainting composite are bit-identical to the plain decode's.
template <typename T>
__device__ __forceinline__ float image_post_unit(T x) {
  const float v = round16<T>(round16<T>(Half16<T>::to_f(x) * 0.5f) + 0.5f);
  return fminf(fmaxf(v, 0.f), 1.f);
}
template <typename T>
__device__ __forceinline__ uint8_t image_post_u8(float v) {
  return static_cast<uint8_t>(round16<T>(v * 255.f));
}
template <typename T>
__global__ void image_post_kernel(const T* __restrict__ x, int c_stride, float* __restrict__ img_f32,
                                  uint8_t* __restrict__ img_u8, long long pixels) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < pixels * 3;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long p = i / 3;
    const int c = static_cast<int>(i % 3);
    const float v = image_post_unit<T>(x[p * c_stride + c]);
    if (img_f32 != nullptr) img_f32[i] = v;
    if (img_u8 != nullptr) img_u8[i] = image_post_u8<T>(v);
  }
}
// inpainting composite: img_u8 = mask ? image_post's uint8 : orig  (orig [pixels, 3] uint8, mask one byte / pixel)
template <typename T>
__global__ void image_post_masked_kernel(const T* __restrict__ x, int c_stride, const uint8_t* __restrict__ orig,
                                         const uint8_t* __restrict__ mask, uint8_t* __restrict__ img_u8,
                                         long long pixels) {
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < pixels * 3;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    const long long p = i / 3;
    const int c = static_cast<int>(i % 3);
    img_u8[i] = mask[p] ? image_post_u8<T>(image_post_unit<T>(x[p * c_stride + c])) : orig[i];
  }
}

// inpainting re-noise of the kept latent cells after an Euler step (fp32, one float4 per thread, Q = C / 4 float4s per
// pixel; QC > 0 fixes Q at compile time so the pixel index is a shift):
//   x = mask ? x : sigma_next * noise + (1 - sigma_next) * x0
// Cells being regenerated (mask != 0) read nothing but their mask byte and are not written.
template <int QC>
__global__ void inpaint_blend_kernel(const float4* __restrict__ x0, const float4* __restrict__ noise,
                                     const uint8_t* __restrict__ mask, float4* __restrict__ x, long long pixels, int Q,
                                     float sigma_next) {
  const int q = QC > 0 ? QC : Q;
  const long long n = pixels * q;
  const float keep = 1.f - sigma_next;
  for (long long i = static_cast<long long>(blockIdx.x) * blockDim.x + threadIdx.x; i < n;
       i += static_cast<long long>(gridDim.x) * blockDim.x) {
    if (mask[i / q]) continue;
    const float4 a = x0[i], b = noise[i];
    float4 o;
    o.x = sigma_next * b.x + keep * a.x;
    o.y = sigma_next * b.y + keep * a.y;
    o.z = sigma_next * b.z + keep * a.z;
    o.w = sigma_next * b.w + keep * a.w;
    x[i] = o;
  }
}

static inline int grid_for(long long work_items, int threads, int sm_count) {
  long long blocks = (work_items + threads - 1) / threads;
  const long long cap = static_cast<long long>(sm_count) * 16;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  return static_cast<int>(blocks);
}

}  // namespace dk

using namespace dk;

#define DK_DTYPE_OK(dt) DK_REQUIRE((dt) == DK_BF16 || (dt) == DK_FP16, "%s: bad dtype %d", __func__, (dt))
#define DK_DISPATCH(dt, ...)                      \
  do {                                            \
    if ((dt) == DK_BF16) {                        \
      using T = __nv_bfloat16;                    \
      __VA_ARGS__;                                \
    } else {                                      \
      using T = __half;                           \
      __VA_ARGS__;                                \
    }                                             \
  } while (0)

extern "C" int dk_ln_modulate(dk_ctx* ctx, int dtype, const void* x, void* y, const void* shift, const void* scale,
                              long long mod_ld, int rows, int rows_per_batch, int h, float eps, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_ln_modulate: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(rows > 0 && rows_per_batch > 0, "dk_ln_modulate: empty input");
  DK_REQUIRE(h % 8 == 0 && h <= 32 * 8 * LN_MAXV, "dk_ln_modulate: h=%d unsupported (multiple of 8, <= %d)", h,
             32 * 8 * LN_MAXV);
  DK_REQUIRE(mod_ld % 8 == 0, "dk_ln_modulate: mod_ld must be a multiple of 8");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int blocks = (rows + LN_WARPS - 1) / LN_WARPS;
  const int nv = (h / 8 + 31) / 32;   // vectors per lane
  DK_DISPATCH(dtype, {
    const T* xp = static_cast<const T*>(x);
    T* yp = static_cast<T*>(y);
    const T* shp = static_cast<const T*>(shift);
    const T* scp = static_cast<const T*>(scale);
    if (nv <= 4)
      ln_modulate_kernel<T, 4><<<blocks, LN_WARPS * 32, 0, stream>>>(xp, yp, shp, scp, mod_ld, rows, rows_per_batch, h, eps);
    else if (nv <= 8)
      ln_modulate_kernel<T, 8><<<blocks, LN_WARPS * 32, 0, stream>>>(xp, yp, shp, scp, mod_ld, rows, rows_per_batch, h, eps);
    else if (nv <= 12)
      ln_modulate_kernel<T, 12><<<blocks, LN_WARPS * 32, 0, stream>>>(xp, yp, shp, scp, mod_ld, rows, rows_per_batch, h, eps);
    else
      ln_modulate_kernel<T, 16><<<blocks, LN_WARPS * 32, 0, stream>>>(xp, yp, shp, scp, mod_ld, rows, rows_per_batch, h, eps);
  });
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_qk_norm_rope(dk_ctx* ctx, int dtype, void* qkv, int rows, int S, int heads, int d, int split,
                               const void* q_w, const void* k_w, const void* q_w2, const void* k_w2, const float* rope,
                               float eps, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_qk_norm_rope: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(d == 64 || d == 128, "dk_qk_norm_rope: head dim %d unsupported (64 or 128)", d);
  DK_REQUIRE(rows > 0 && S > 0 && rows % S == 0, "dk_qk_norm_rope: rows %d must be a multiple of S %d", rows, S);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const long long warps = static_cast<long long>(rows) * heads * 2;
  const int blocks = static_cast<int>((warps * 32 + 255) / 256);
  if (q_w2 == nullptr) q_w2 = q_w;
  if (k_w2 == nullptr) k_w2 = k_w;
  DK_DISPATCH(dtype, {
    if (d == 128)
      qk_norm_rope_kernel<T, 128><<<blocks, 256, 0, stream>>>(
          static_cast<T*>(qkv), rows, S, heads, split, static_cast<const T*>(q_w), static_cast<const T*>(k_w),
          static_cast<const T*>(q_w2), static_cast<const T*>(k_w2), rope, eps);
    else
      qk_norm_rope_kernel<T, 64><<<blocks, 256, 0, stream>>>(
          static_cast<T*>(qkv), rows, S, heads, split, static_cast<const T*>(q_w), static_cast<const T*>(k_w),
          static_cast<const T*>(q_w2), static_cast<const T*>(k_w2), rope, eps);
  });
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_silu_add(dk_ctx* ctx, int dtype, const void* y, const void* temb, void* c, int n_t, int B, int h,
                           void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_silu_add: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(h % 8 == 0, "dk_silu_add: h must be a multiple of 8");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const long long nvec = static_cast<long long>(n_t) * B * h / 8;
  DK_DISPATCH(dtype, (silu_add_kernel<T><<<grid_for(nvec, 256, ctx->sm_count), 256, 0, stream>>>(
                         static_cast<const T*>(y), static_cast<const T*>(temb), static_cast<T*>(c), n_t, B, h)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_act(dk_ctx* ctx, int dtype, const void* x, void* y, long long n, int act, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_act: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(n % 8 == 0, "dk_act: n must be a multiple of 8");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DK_DISPATCH(dtype, (act_kernel<T><<<grid_for(n / 8, 256, ctx->sm_count), 256, 0, stream>>>(
                         static_cast<const T*>(x), static_cast<T*>(y), n, act)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_patchify(dk_ctx* ctx, int dtype, const void* latent, void* rows, int B, int H, int W, int C, int order,
                           void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_patchify: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(H % 2 == 0 && W % 2 == 0, "dk_patchify: latent size must be even (got %dx%d)", H, W);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const long long total = static_cast<long long>(B) * H * W * C;
  DK_DISPATCH(dtype, (patchify_kernel<T><<<grid_for(total, 256, ctx->sm_count), 256, 0, stream>>>(
                         static_cast<const T*>(latent), static_cast<T*>(rows), B, H, W, C, order)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_unpatchify(dk_ctx* ctx, int dtype, const void* rows, void* latent, int B, int H, int W, int C,
                             int order, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_unpatchify: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(H % 2 == 0 && W % 2 == 0, "dk_unpatchify: latent size must be even (got %dx%d)", H, W);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const long long total = static_cast<long long>(B) * H * W * C;
  DK_DISPATCH(dtype, (unpatchify_kernel<T><<<grid_for(total, 256, ctx->sm_count), 256, 0, stream>>>(
                         static_cast<const T*>(rows), static_cast<T*>(latent), B, H, W, C, order)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_pos_embed_crop(dk_ctx* ctx, int dtype, const void* table, void* out, int max_hw, int hp, int wp, int h,
                                 void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_pos_embed_crop: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(hp <= max_hw && wp <= max_hw, "dk_pos_embed_crop: %dx%d exceeds the %d table", hp, wp, max_hw);
  DK_REQUIRE(h % 8 == 0, "dk_pos_embed_crop: h must be a multiple of 8");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const long long nvec = static_cast<long long>(hp) * wp * h / 8;
  DK_DISPATCH(dtype, (pos_embed_crop_kernel<T><<<grid_for(nvec, 256, ctx->sm_count), 256, 0, stream>>>(
                         static_cast<const T*>(table), static_cast<T*>(out), max_hw, hp, wp, h)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_copy_rows(dk_ctx* ctx, int dtype, const void* src, void* dst, int B, int rows, int h, int dst_rows,
                            int dst_off, int src_rows, int src_off, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_copy_rows: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(h % 8 == 0, "dk_copy_rows: h must be a multiple of 8");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const long long nvec = static_cast<long long>(B) * rows * h / 8;
  DK_DISPATCH(dtype, (copy_rows_kernel<T><<<grid_for(nvec, 256, ctx->sm_count), 256, 0, stream>>>(
                         static_cast<const T*>(src), static_cast<T*>(dst), B, rows, h, dst_rows, dst_off, src_rows,
                         src_off)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_sampler_prepare(dk_ctx* ctx, int dtype, const float* x, void* xin, long long n_per_rep, int reps,
                                  void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_sampler_prepare: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DK_DISPATCH(dtype, (sampler_prepare_kernel<T><<<grid_for(n_per_rep, 256, ctx->sm_count), 256, 0, stream>>>(
                         x, static_cast<T*>(xin), n_per_rep, reps)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_sampler_step(dk_ctx* ctx, int dtype, float* x, const void* xin, const void* out, long long n,
                               float sigma, float sigma_next, float cfg_weight, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_sampler_step: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(sigma != 0.f, "dk_sampler_step: sigma must be non-zero");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DK_DISPATCH(dtype, (sampler_step_kernel<T><<<grid_for(n, 256, ctx->sm_count), 256, 0, stream>>>(
                         x, static_cast<const T*>(xin), static_cast<const T*>(out), n, sigma, sigma_next, cfg_weight)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_axpb_f32(dk_ctx* ctx, const float* x, float* y, long long n, float a, float b, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_axpb_f32: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  axpb_kernel<<<grid_for(n, 256, ctx->sm_count), 256, 0, stream>>>(x, y, n, a, b);
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_dequant_q4(dk_ctx* ctx, int dtype, const uint32_t* wq, const void* scales, const void* biases,
                             void* out, long long N, int K, int group_size, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_dequant_q4: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(N > 0 && K > 0, "dk_dequant_q4: empty weight");
  DK_REQUIRE(group_size >= 8 && group_size % 8 == 0 && K % group_size == 0,
             "dk_dequant_q4: K (%d) must be a multiple of group_size (%d), itself a multiple of 8", K, group_size);
  DK_REQUIRE((reinterpret_cast<uintptr_t>(out) & 15u) == 0, "dk_dequant_q4: out must be 16-byte aligned");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DK_DISPATCH(dtype, (dequant_q4_kernel<T><<<grid_for(N * (K / 8), 256, ctx->sm_count), 256, 0, stream>>>(
                         wq, static_cast<const T*>(scales), static_cast<const T*>(biases), static_cast<T*>(out), N, K,
                         group_size)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_image_pre(dk_ctx* ctx, int dtype, const uint8_t* img, void* out, long long pixels, int src_channels,
                            int cpad, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_image_pre: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(src_channels >= 3, "dk_image_pre: image needs at least 3 channels (got %d)", src_channels);
  DK_REQUIRE(cpad >= 8 && cpad % 8 == 0, "dk_image_pre: cpad (%d) must be a positive multiple of 8", cpad);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DK_DISPATCH(dtype, (image_pre_kernel<T><<<grid_for(pixels * (cpad / 8), 256, ctx->sm_count), 256, 0, stream>>>(
                         img, static_cast<T*>(out), pixels, src_channels, cpad)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_axpby_f32(dk_ctx* ctx, const float* x, const float* y, float* out, long long n, float a, float b,
                            void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_axpby_f32: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  axpby_kernel<<<grid_for(n, 256, ctx->sm_count), 256, 0, stream>>>(x, y, out, n, a, b);
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_vae_sample_latent(dk_ctx* ctx, int dtype, const void* hidden, const float* noise, float* out,
                                    long long pixels, int C, float shift, float scale, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_vae_sample_latent: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DK_DISPATCH(dtype, (vae_sample_latent_kernel<T><<<grid_for(pixels * C, 256, ctx->sm_count), 256, 0, stream>>>(
                         static_cast<const T*>(hidden), noise, out, pixels, C, shift, scale)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_cast_f32_to_16(dk_ctx* ctx, int dtype, const float* x, void* y, long long n, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_cast_f32_to_16: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DK_DISPATCH(dtype, (cast_f32_to_16_kernel<T><<<grid_for(n, 256, ctx->sm_count), 256, 0, stream>>>(
                         x, static_cast<T*>(y), n)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}
extern "C" int dk_cast_16_to_f32(dk_ctx* ctx, int dtype, const void* x, float* y, long long n, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_cast_16_to_f32: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DK_DISPATCH(dtype, (cast_16_to_f32_kernel<T><<<grid_for(n, 256, ctx->sm_count), 256, 0, stream>>>(
                         static_cast<const T*>(x), y, n)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_groupnorm_ws_floats(int B, int G) { return B * GN_MAX_CHUNKS * G * 2; }

extern "C" int dk_groupnorm_stats(dk_ctx* ctx, int dtype, const void* x, float* stats, float* ws, int B, int HW, int C,
                                  int G, float eps, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_groupnorm_stats: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(C % 8 == 0 && C % G == 0 && C <= 2048, "dk_groupnorm_stats: C=%d G=%d unsupported", C, G);
  DK_REQUIRE(ws != nullptr, "dk_groupnorm_stats: workspace of dk_groupnorm_ws_floats(B, G) floats required");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int chunks = gn_chunks(HW);
  dim3 grid(chunks, B);
  DK_DISPATCH(dtype, (groupnorm_partial_kernel<T><<<grid, GN_THREADS, (2 * C + 2 * GN_THREADS * 8) * sizeof(float), stream>>>(
                         static_cast<const T*>(x), ws, HW, C, G, chunks)));
  DK_LAUNCH_CHECK(ctx);
  groupnorm_finalize_kernel<<<B * G, GNF_THREADS, 0, stream>>>(ws, stats, B, G, chunks,
                                                                static_cast<double>(HW) * (C / G), eps);
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_groupnorm_finalize(dk_ctx* ctx, const float* partial, float* stats, int B, int G, int slots,
                                     double count, float eps, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_groupnorm_finalize: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_REQUIRE(partial != nullptr && stats != nullptr && B > 0 && G > 0 && slots > 0 && count > 0,
             "dk_groupnorm_finalize: bad arguments");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  groupnorm_finalize_kernel<<<B * G, GNF_THREADS, 0, stream>>>(partial, stats, B, G, slots, count, eps);
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_groupnorm_apply(dk_ctx* ctx, int dtype, const void* x, void* y, const float* stats, const void* gamma,
                                  const void* beta, int B, int HW, int C, int G, int silu, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_groupnorm_apply: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(C % 8 == 0 && C % G == 0 && C <= 2048, "dk_groupnorm_apply: C=%d G=%d unsupported", C, G);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int pix_per_iter = GN_THREADS / (C / 8);
  int blocks = (HW + pix_per_iter * 4 - 1) / (pix_per_iter * 4);   // >= 4 pixels per thread
  const int cap = (ctx->sm_count * 16 + B - 1) / B;
  if (blocks > cap) blocks = cap;
  if (blocks < 1) blocks = 1;
  dim3 grid(blocks, B);
  DK_DISPATCH(dtype, (groupnorm_apply_kernel<T><<<grid, GN_THREADS, 0, stream>>>(
                         static_cast<const T*>(x), static_cast<T*>(y), stats, static_cast<const T*>(gamma),
                         static_cast<const T*>(beta), HW, C, G, silu)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_upsample_nearest2x(dk_ctx* ctx, int dtype, const void* x, void* y, int B, int H, int W, int C,
                                     void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_upsample_nearest2x: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(C % 8 == 0, "dk_upsample_nearest2x: C must be a multiple of 8");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int rows_per_block = 2;   // even: both replicas of an input row are written by the same thread
  dim3 grid((2 * H + rows_per_block - 1) / rows_per_block, B);
  DK_DISPATCH(dtype, (upsample2x_kernel<T><<<grid, 256, 0, stream>>>(static_cast<const T*>(x), static_cast<T*>(y), H,
                                                                       W, C, rows_per_block)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_softmax_rows(dk_ctx* ctx, int dtype, void* x, long long rows, int n, long long ld, float scale,
                               void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_softmax_rows: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(n % 8 == 0 && ld % 8 == 0, "dk_softmax_rows: n and ld must be multiples of 8");
  DK_REQUIRE(rows > 0 && rows < (1LL << 31), "dk_softmax_rows: bad row count");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DK_DISPATCH(dtype, (softmax_rows_kernel<T><<<static_cast<unsigned>(rows), 256, 0, stream>>>(static_cast<T*>(x), n, ld,
                                                                                             scale)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_image_post(dk_ctx* ctx, int dtype, const void* x, int c_stride, float* img_f32, uint8_t* img_u8,
                             long long pixels, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_image_post: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DK_DISPATCH(dtype, (image_post_kernel<T><<<grid_for(pixels * 3, 256, ctx->sm_count), 256, 0, stream>>>(
                         static_cast<const T*>(x), c_stride, img_f32, img_u8, pixels)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_image_post_masked(dk_ctx* ctx, int dtype, const void* x, int c_stride, const uint8_t* orig,
                                    const uint8_t* mask, uint8_t* img_u8, long long pixels, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_image_post_masked: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_DTYPE_OK(dtype);
  DK_REQUIRE(x != nullptr && orig != nullptr && mask != nullptr && img_u8 != nullptr,
             "dk_image_post_masked: null tensor");
  DK_REQUIRE(c_stride >= 3, "dk_image_post_masked: c_stride (%d) must be >= 3", c_stride);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  DK_DISPATCH(dtype, (image_post_masked_kernel<T><<<grid_for(pixels * 3, 256, ctx->sm_count), 256, 0, stream>>>(
                         static_cast<const T*>(x), c_stride, orig, mask, img_u8, pixels)));
  DK_LAUNCH_CHECK(ctx);
  return 0;
}

extern "C" int dk_inpaint_blend(dk_ctx* ctx, const float* x0, const float* noise, const uint8_t* mask, float* x,
                                long long pixels, int C, float sigma_next, void* stream_) {
  DK_REQUIRE(ctx != nullptr, "dk_inpaint_blend: null ctx");
  DkDeviceGuard dk_guard_(ctx);
  DK_REQUIRE(x0 != nullptr && noise != nullptr && mask != nullptr && x != nullptr, "dk_inpaint_blend: null tensor");
  DK_REQUIRE(C > 0 && C % 4 == 0, "dk_inpaint_blend: C (%d) must be a positive multiple of 4", C);
  DK_REQUIRE(((reinterpret_cast<uintptr_t>(x0) | reinterpret_cast<uintptr_t>(noise) | reinterpret_cast<uintptr_t>(x)) &
              15u) == 0,
             "dk_inpaint_blend: x0, noise and x must be 16-byte aligned");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  const int grid = grid_for(pixels * (C / 4), 256, ctx->sm_count);
  const float4* a = reinterpret_cast<const float4*>(x0);
  const float4* b = reinterpret_cast<const float4*>(noise);
  float4* o = reinterpret_cast<float4*>(x);
  if (C == 16)
    inpaint_blend_kernel<4><<<grid, 256, 0, stream>>>(a, b, mask, o, pixels, 4, sigma_next);
  else
    inpaint_blend_kernel<0><<<grid, 256, 0, stream>>>(a, b, mask, o, pixels, C / 4, sigma_next);
  DK_LAUNCH_CHECK(ctx);
  return 0;
}
