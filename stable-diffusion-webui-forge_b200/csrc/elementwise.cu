// b200forge — HBM-bound kernels of the denoise path: GroupNorm (stats + apply/SiLU/concat), LayerNorm,
// layout conversion, nearest upsample, im2col for the few convolutions the TMA path does not cover,
// timestep embedding.  All activations are channels-last; every global access is a 16-byte vector.
#include "common.cuh"
#include "host_util.h"

namespace b200 {

template <bool BF16>
__device__ __forceinline__ void load8(const void* p, size_t elem_off, float (&x)[8]) {
  uint4 r = *reinterpret_cast<const uint4*>(reinterpret_cast<const char*>(p) + elem_off * 2);
  float2 f;
  f = unpack2<BF16>(r.x); x[0] = f.x; x[1] = f.y;
  f = unpack2<BF16>(r.y); x[2] = f.x; x[3] = f.y;
  f = unpack2<BF16>(r.z); x[4] = f.x; x[5] = f.y;
  f = unpack2<BF16>(r.w); x[6] = f.x; x[7] = f.y;
}
template <bool BF16>
__device__ __forceinline__ void store8(void* p, size_t elem_off, const float (&x)[8]) {
  uint4 o;
  o.x = pack2<BF16>(x[0], x[1]);
  o.y = pack2<BF16>(x[2], x[3]);
  o.z = pack2<BF16>(x[4], x[5]);
  o.w = pack2<BF16>(x[6], x[7]);
  *reinterpret_cast<uint4*>(reinterpret_cast<char*>(p) + elem_off * 2) = o;
}

// ------------------------------------------------------------------------------------------ GroupNorm
// Statistics are deterministic and cancellation-free:
//   * every block reduces its slab of pixels in a fixed order (per-thread sums -> smem table -> fixed-order tree), no atomics
//     on data;
//   * sums are taken of (x - pivot) with pivot = x[n, pixel 0, first channel of the group], the same for every block of a
//     sample, so block partials simply add and a large group mean does not cancel in sumsq/cnt - mean^2;
//   * the last block of a sample to finish (ticket counter, self-resetting) adds the slab partials in slab order and writes
//     (mean, rstd) per group — one launch, nothing to zero-fill per call.
// Workspace layout (b200_groupnorm_ws_bytes): int tickets[N] (padded to 256 B) | float final[N][G][2] | float part[N][slabs][G][2].
// grid (slabs, N), 256 threads arranged as (ry, tx): tx walks channel vectors, ry walks pixels.
__device__ __forceinline__ float gn_tree8(float v) {  // fixed-order sum over the 8 lanes of a group team
  v += __shfl_xor_sync(0xffffffffu, v, 1);
  v += __shfl_xor_sync(0xffffffffu, v, 2);
  v += __shfl_xor_sync(0xffffffffu, v, 4);
  return v;
}

template <bool BF16>
__global__ void __launch_bounds__(256) gn_stats_kernel(const void* __restrict__ x1, const void* __restrict__ x2,
                                                       int* __restrict__ tickets, float* __restrict__ final_stats,
                                                       float* __restrict__ part, int HW, int C1, int C2, int groups,
                                                       int pix_per_slab, float eps) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sh[];  // piv[C] | tab_s[RY][C] | tab_q[RY][C]
  __shared__ int is_last;
  const int C = C1 + C2;
  const int CV = C >> 3;
  const int cpg = C / groups;
  const int TX = CV < 256 ? CV : 256;
  const int RY = 256 / TX;
  const int tx = threadIdx.x % TX;
  const int ry = threadIdx.x / TX;
  const int n = blockIdx.y;
  const int slabs = gridDim.x;
  float* piv = sh;
  float* tab_s = sh + C;
  float* tab_q = tab_s + (size_t)RY * C;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const int c0 = (c / cpg) * cpg;
    piv[c] = c0 < C1 ? ld1<BF16>(x1, (size_t)n * HW * C1 + c0) : ld1<BF16>(x2, (size_t)n * HW * C2 + (c0 - C1));
  }
  __syncthreads();
  const int p0 = blockIdx.x * pix_per_slab;
  int p1 = p0 + pix_per_slab;
  if (p1 > HW) p1 = HW;
  if (ry < RY) {
    for (int cv = tx; cv < CV; cv += TX) {
      const int c = cv << 3;
      const bool first = c < C1;
      const void* src = first ? x1 : x2;
      const int Cs = first ? C1 : C2;
      const int cs = first ? c : c - C1;
      float s[8], q[8], pv[8];
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        s[i] = q[i] = 0.f;
        pv[i] = piv[c + i];
      }
      for (int px = p0 + ry; px < p1; px += RY) {
        float v[8];
        load8<BF16>(src, ((size_t)n * HW + px) * Cs + cs, v);
#pragma unroll
        for (int i = 0; i < 8; ++i) {
          const float dv = v[i] - pv[i];
          s[i] += dv;
          q[i] = fmaf(dv, dv, q[i]);
        }
      }
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        tab_s[(size_t)ry * C + c + i] = s[i];
        tab_q[(size_t)ry * C + c + i] = q[i];
      }
    }
  }
  __syncthreads();
  // teams of 8 lanes per group: lane j adds table entries j, j + 8, ... in index order, then a fixed shuffle tree
  const int team = threadIdx.x >> 3, tj = threadIdx.x & 7;
  const int per_group = RY * cpg;
  for (int g0 = 0; g0 < groups; g0 += 32) {  // warp-uniform trip count: the shuffles below use the full mask
    const int g = g0 + team;
    const bool g_ok = g < groups;
    float s = 0.f, q = 0.f;
    for (int e = tj; g_ok && e < per_group; e += 8) {
      const int r = e / cpg, c = g * cpg + (e - r * cpg);
      s += tab_s[(size_t)r * C + c];
      q += tab_q[(size_t)r * C + c];
    }
    s = gn_tree8(s);
    q = gn_tree8(q);
    if (tj == 0 && g_ok) {
      float* dst = part + (((size_t)n * slabs + blockIdx.x) * groups + g) * 2;
      dst[0] = s;
      dst[1] = q;
    }
  }
  __threadfence();
  __syncthreads();
  if (threadIdx.x == 0) {
    const int t = atomicAdd(&tickets[n], 1);
    is_last = (t == slabs - 1);
  }
  __syncthreads();
  if (!is_last) return;
  __threadfence();
  const float inv_cnt = 1.0f / ((float)HW * (float)cpg);
  for (int g0 = 0; g0 < groups; g0 += 32) {
    const int g = g0 + team;
    const bool g_ok = g < groups;
    float s = 0.f, q = 0.f;
    for (int sl = tj; g_ok && sl < slabs; sl += 8) {
      const float* src = part + (((size_t)n * slabs + sl) * groups + g) * 2;
      s += __ldcg(src);
      q += __ldcg(src + 1);
    }
    s = gn_tree8(s);
    q = gn_tree8(q);
    if (tj == 0 && g_ok) {
      const float dm = s * inv_cnt;
      const float var = fmaxf(fmaf(-dm, dm, q * inv_cnt), 0.f);
      final_stats[((size_t)n * groups + g) * 2 + 0] = piv[g * cpg] + dm;
      final_stats[((size_t)n * groups + g) * 2 + 1] = rsqrtf(var + eps);
    }
  }
  if (threadIdx.x == 0) tickets[n] = 0;  // ready for the next launch on this stream
}

template <bool BF16>
__global__ void __launch_bounds__(256) gn_apply_kernel(const void* __restrict__ x1, const void* __restrict__ x2,
                                                       const float* __restrict__ final_stats, const void* __restrict__ gamma,
                                                       const void* __restrict__ beta, void* __restrict__ y, int HW,
                                                       int C1, int C2, int groups, int silu, int pix_per_slab) {
  pdl_launch_dependents();
  pdl_wait();
  extern __shared__ float sh[];  // [C] scale, [C] shift
  const int C = C1 + C2;
  const int CV = C >> 3;
  const int n = blockIdx.y;
  const int cpg = C / groups;
  float* sc = sh;
  float* sf = sh + C;
  for (int c = threadIdx.x; c < C; c += blockDim.x) {
    const int g = c / cpg;
    const float mean = final_stats[((size_t)n * groups + g) * 2 + 0];
    const float rstd = final_stats[((size_t)n * groups + g) * 2 + 1];
    const float a = ld1<BF16>(gamma, c) * rstd;
    sc[c] = a;
    sf[c] = ld1<BF16>(beta, c) - mean * a;
  }
  __syncthreads();
  const int TX = CV < 256 ? CV : 256;
  const int RY = 256 / TX;
  const int tx = threadIdx.x % TX;
  const int ry = threadIdx.x / TX;
  const int p0 = blockIdx.x * pix_per_slab;
  int p1 = p0 + pix_per_slab;
  if (p1 > HW) p1 = HW;
  if (ry >= RY) return;
  for (int cv = tx; cv < CV; cv += TX) {
    const int c = cv << 3;
    const bool first = c < C1;
    const void* src = first ? x1 : x2;
    const int Cs = first ? C1 : C2;
    const int cs = first ? c : c - C1;
    float a[8], b[8];
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      a[i] = sc[c + i];
      b[i] = sf[c + i];
    }
    for (int px = p0 + ry; px < p1; px += RY) {
      float v[8];
      load8<BF16>(src, ((size_t)n * HW + px) * Cs + cs, v);
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        float t = fmaf(v[i], a[i], b[i]);
        v[i] = silu ? silu_fast_f(t) : t;
      }
      store8<BF16>(y, ((size_t)n * HW + px) * C + c, v);
    }
  }
}

// ------------------------------------------------------------------------------------------ LayerNorm
// one warp per row, row cached in registers (C <= 8*32*MAXV)
template <bool BF16, int MAXV>
__global__ void __launch_bounds__(256) layernorm_kernel(const void* __restrict__ x, const void* __restrict__ gamma,
                                                        const void* __restrict__ beta, void* __restrict__ y, int rows,
                                                        int C, float eps) {
  const int warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (warp >= rows) return;
  const int CV = C >> 3;
  float v[MAXV][8];
  float s = 0.f;
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int cv = lane + k * 32;
    if (cv < CV) {
      load8<BF16>(x, (size_t)warp * C + (cv << 3), v[k]);
#pragma unroll
      for (int i = 0; i < 8; ++i) s += v[k][i];
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  const float mean = s / (float)C;
  float q = 0.f;
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int cv = lane + k * 32;
    if (cv < CV) {
#pragma unroll
      for (int i = 0; i < 8; ++i) {
        const float d = v[k][i] - mean;
        q = fmaf(d, d, q);
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) q += __shfl_xor_sync(0xffffffffu, q, o);
  const float rstd = rsqrtf(q / (float)C + eps);
#pragma unroll
  for (int k = 0; k < MAXV; ++k) {
    const int cv = lane + k * 32;
    if (cv < CV) {
      float o8[8];
      if (gamma) {
        float g[8], bt[8];
        load8<BF16>(gamma, (size_t)(cv << 3), g);
        if (beta) load8<BF16>(beta, (size_t)(cv << 3), bt);
#pragma unroll
        for (int i = 0; i < 8; ++i) o8[i] = (v[k][i] - mean) * rstd * g[i] + (beta ? bt[i] : 0.f);
      } else {
#pragma unroll
        for (int i = 0; i < 8; ++i) o8[i] = (v[k][i] - mean) * rstd;
      }
      store8<BF16>(y, (size_t)warp * C + (cv << 3), o8);
    }
  }
}

// ------------------------------------------------------------------------------------------ layout helpers
__global__ void upsample2x_kernel(const uint4* __restrict__ x, uint4* __restrict__ y, int N, int H, int W, int CV) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t total = (size_t)N * (2 * H) * (2 * W) * CV;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int cv = (int)(i % CV);
    size_t t = i / CV;
    const int wo = (int)(t % (2 * W));
    t /= (2 * W);
    const int ho = (int)(t % (2 * H));
    const int n = (int)(t / (2 * H));
    y[i] = x[(((size_t)n * H + (ho >> 1)) * W + (wo >> 1)) * CV + cv];
  }
}

// vector path: C % 8 == 0.  out row = (n, ho, wo); column = tap*C + c; columns [9C, ldo) zero.
__global__ void im2col3x3_vec_kernel(const uint4* __restrict__ x, uint4* __restrict__ out, int N, int H, int W, int CV,
                                     int stride, int pad_lo, int Ho, int Wo, int ldoV) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t total = (size_t)N * Ho * Wo * ldoV;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int kv = (int)(i % ldoV);
    size_t t = i / ldoV;
    const int wo = (int)(t % Wo);
    t /= Wo;
    const int ho = (int)(t % Ho);
    const int n = (int)(t / Ho);
    uint4 v = make_uint4(0, 0, 0, 0);
    if (kv < 9 * CV) {
      const int tap = kv / CV, cv = kv - tap * CV;
      const int ky = tap / 3, kx = tap - ky * 3;
      const int hi = ho * stride + ky - pad_lo, wi = wo * stride + kx - pad_lo;
      if (hi >= 0 && hi < H && wi >= 0 && wi < W) v = x[(((size_t)n * H + hi) * W + wi) * CV + cv];
    }
    out[i] = v;
  }
}

// scalar path for odd channel counts (C = 3 or 4): 16-bit elements.
__global__ void im2col3x3_scalar_kernel(const uint16_t* __restrict__ x, uint16_t* __restrict__ out, int N, int H, int W,
                                        int C, int stride, int pad_lo, int Ho, int Wo, int ldo) {
  const size_t total = (size_t)N * Ho * Wo * ldo;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int k = (int)(i % ldo);
    size_t t = i / ldo;
    const int wo = (int)(t % Wo);
    t /= Wo;
    const int ho = (int)(t % Ho);
    const int n = (int)(t / Ho);
    uint16_t v = 0;
    if (k < 9 * C) {
      const int tap = k / C, c = k - tap * C;
      const int ky = tap / 3, kx = tap - ky * 3;
      const int hi = ho * stride + ky - pad_lo, wi = wo * stride + kx - pad_lo;
      if (hi >= 0 && hi < H && wi >= 0 && wi < W) v = x[(((size_t)n * H + hi) * W + wi) * C + c];
    }
    out[i] = v;
  }
}

template <bool BF16>
__global__ void nchw_to_nhwc_kernel(const void* __restrict__ x, void* __restrict__ y, int N, int C, int H, int W,
                                    int ldy, float scale, int in_is_f32) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t total = (size_t)N * H * W * ldy;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int c = (int)(i % ldy);
    size_t t = i / ldy;
    const int w = (int)(t % W);
    t /= W;
    const int h = (int)(t % H);
    const int n = (int)(t / H);
    float v = 0.f;
    if (c < C) {
      const size_t src = (((size_t)n * C + c) * H + h) * W + w;
      v = in_is_f32 ? reinterpret_cast<const float*>(x)[src] : ld1<BF16>(x, src);
      if (scale != 1.0f) v = v * scale;
    }
    st1<BF16>(y, i, v);
  }
}

template <bool BF16>
__global__ void nhwc_to_nchw_kernel(const void* __restrict__ x, void* __restrict__ y, int N, int C, int H, int W,
                                    int ldx, int out_is_f32) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t total = (size_t)N * C * H * W;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int w = (int)(i % W);
    size_t t = i / W;
    const int h = (int)(t % H);
    t /= H;
    const int c = (int)(t % C);
    const int n = (int)(t / C);
    const float v = ld1<BF16>(x, (((size_t)n * H + h) * W + w) * ldx + c);
    if (out_is_f32) reinterpret_cast<float*>(y)[i] = v;
    else st1<BF16>(y, i, v);
  }
}

template <bool BF16>
__global__ void silu_kernel(const void* __restrict__ x, void* __restrict__ y, size_t n) {
  pdl_launch_dependents();
  pdl_wait();
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (size_t)gridDim.x * blockDim.x)
    st1<BF16>(y, i, silu_f(ld1<BF16>(x, i)));
}

// out[b, i] = cos(t_b * f_i), out[b, half + i] = sin(t_b * f_i), f_i = exp(-ln(max_period) * i / half)
template <bool BF16>
__global__ void timestep_embedding_kernel(const float* __restrict__ t, void* __restrict__ out, int B, int dim,
                                          float neg_log_period) {
  pdl_launch_dependents();
  pdl_wait();
  const int half = dim / 2;
  const int total = B * half;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int b = i / half, k = i - b * half;
    const float f = expf(neg_log_period * (float)k / (float)half);
    const float a = t[b] * f;
    st1<BF16>(out, (size_t)b * dim + k, cosf(a));
    st1<BF16>(out, (size_t)b * dim + half + k, sinf(a));
    if ((dim & 1) && k == 0) st1<BF16>(out, (size_t)b * dim + dim - 1, 0.f);
  }
}

// x fp32 NCHW [B,C,H,W] / sqrt(sigma_b^2 + 1) -> im2col rows for the 3x3 conv_in, written `reps` times
template <bool BF16>
__global__ void unet_input_im2col_kernel(const float* __restrict__ x, const float* __restrict__ sigma,
                                         void* __restrict__ cols, int B, int C, int H, int W, int ldo, int reps) {
  pdl_launch_dependents();
  pdl_wait();
  const size_t per_rep = (size_t)B * H * W * ldo;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < per_rep; i += (size_t)gridDim.x * blockDim.x) {
    const int k = (int)(i % ldo);
    size_t t = i / ldo;
    const int w = (int)(t % W);
    t /= W;
    const int h = (int)(t % H);
    const int b = (int)(t / H);
    float v = 0.f;
    if (k < 9 * C) {
      const int tap = k / C, c = k - tap * C;
      const int ky = tap / 3, kx = tap - ky * 3;
      const int hi = h + ky - 1, wi = w + kx - 1;
      if (hi >= 0 && hi < H && wi >= 0 && wi < W) {
        const float sg = sigma[b];
        // reference: noise / (sigma ** 2 + sigma_data ** 2) ** 0.5 in fp32, then .to(fp16)
        v = x[(((size_t)b * C + c) * H + hi) * W + wi] / sqrtf(sg * sg + 1.0f);
      }
    }
    for (int r = 0; r < reps; ++r) st1<BF16>(cols, (size_t)r * per_rep + i, v);
  }
}

template <bool BF16>
__global__ void softmax_rows_kernel(void* __restrict__ x, int rows, int cols, int ld, float scale_log2, int valid,
                                    int block_rows, int block_cols) {
  pdl_launch_dependents();
  pdl_wait();
  // one CTA per row; cols up to 64K.  The row attends to the column window [lo, hi): the prefix [0, valid) when
  // block_rows == 0, else the diagonal block of its row group — (row / block_rows) * block_cols + [0, valid) — which
  // turns one big GEMM over a whole batch into per-sample attention (everything outside the window is written as 0).
  const int row = blockIdx.x;
  const int lo = block_rows > 0 ? (row / block_rows) * block_cols : 0;
  const int hi = lo + valid;
  const int c_begin = lo & ~7, c_end = (hi + 7) & ~7;
  __shared__ float red[32];
  char* base = reinterpret_cast<char*>(x) + (size_t)row * ld * 2;
  float mx = -INFINITY;
  for (int c = c_begin + threadIdx.x * 8; c < c_end; c += blockDim.x * 8) {
    float v[8];
    load8<BF16>(base, (size_t)c, v);
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (c + i >= lo && c + i < hi) mx = fmaxf(mx, v[i]);
  }
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  mx = red[0];
  for (int i = 1; i < (int)(blockDim.x >> 5); ++i) mx = fmaxf(mx, red[i]);
  __syncthreads();
  float s = 0.f;
  for (int c = c_begin + threadIdx.x * 8; c < c_end; c += blockDim.x * 8) {
    float v[8];
    load8<BF16>(base, (size_t)c, v);
#pragma unroll
    for (int i = 0; i < 8; ++i)
      if (c + i >= lo && c + i < hi) s += exp2f((v[i] - mx) * scale_log2);
  }
  for (int o = 16; o > 0; o >>= 1) s += __shfl_xor_sync(0xffffffffu, s, o);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = s;
  __syncthreads();
  s = 0.f;
  for (int i = 0; i < (int)(blockDim.x >> 5); ++i) s += red[i];
  const float inv = 1.0f / s;
  for (int c = threadIdx.x * 8; c < cols; c += blockDim.x * 8) {
    float v[8];
    if (c >= c_begin && c < c_end) {
      load8<BF16>(base, (size_t)c, v);
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = (c + i >= lo && c + i < hi) ? exp2f((v[i] - mx) * scale_log2) * inv : 0.f;
    } else {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] = 0.f;
    }
    store8<BF16>(base, (size_t)c, v);
  }
}

template <bool BF16>
__global__ void vae_post_kernel(const void* __restrict__ x, float* __restrict__ out, size_t pixels, int ldx) {
  const size_t total = pixels * 3;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const size_t px = i / 3;
    const int c = (int)(i - px * 3);
    float v = ld1<BF16>(x, px * ldx + c);
    v = fminf(fmaxf((v + 1.0f) * 0.5f, 0.f), 1.f);
    out[i] = v;
  }
}

// ------------------------------------------------------------------------------------------ tiled VAE blending
// tiled_scale_multidim (backend/patcher/vae.py:11-49): every decoded tile is multiplied by a feather mask — the first and last
// `feather` rows / columns ramp linearly ((t + 1) / feather) — and accumulated together with the mask; the result is the
// quotient.  acc is [H, W, 4] fp32 (r, g, b, mask).
__device__ __forceinline__ float feather_w(int i, int size, int feather, float inv_f) {
  float w = 1.f;
  if (i < feather) w *= inv_f * (float)(i + 1);
  if (size - 1 - i < feather) w *= inv_f * (float)(size - i);
  return w;
}

template <bool BF16>
__global__ void tile_blend_kernel(const void* __restrict__ tile, float4* __restrict__ acc, int W, int y0, int x0, int th,
                                  int tw, int ld, float bias, int feather) {
  const float inv_f = feather > 0 ? 1.0f / (float)feather : 0.f;
  const size_t total = (size_t)th * tw;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int ty = (int)(i / tw), tx = (int)(i - (size_t)ty * tw);
    const float m = feather_w(ty, th, feather, inv_f) * feather_w(tx, tw, feather, inv_f);
    float4 a = acc[(size_t)(y0 + ty) * W + (x0 + tx)];
    a.x += (ld1<BF16>(tile, i * ld + 0) + bias) * m;
    a.y += (ld1<BF16>(tile, i * ld + 1) + bias) * m;
    a.z += (ld1<BF16>(tile, i * ld + 2) + bias) * m;
    a.w += m;
    acc[(size_t)(y0 + ty) * W + (x0 + tx)] = a;
  }
}

// out[H, W, 3] (+)= acc.rgb / acc.w; the last pass scales and clamps (vae.py:109-114: clamp((A + B + C) / 3 / 2, 0, 1))
__global__ void tile_resolve_kernel(const float4* __restrict__ acc, float* __restrict__ out, size_t pixels, int accumulate,
                                    float final_scale, int finalize) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < pixels; i += (size_t)gridDim.x * blockDim.x) {
    const float4 a = acc[i];
    float r = a.x / a.w, g = a.y / a.w, b = a.z / a.w;
    if (accumulate) {
      r += out[i * 3 + 0];
      g += out[i * 3 + 1];
      b += out[i * 3 + 2];
    }
    if (finalize) {
      r = fminf(fmaxf(r * final_scale, 0.f), 1.f);
      g = fminf(fmaxf(g * final_scale, 0.f), 1.f);
      b = fminf(fmaxf(b * final_scale, 0.f), 1.f);
    }
    out[i * 3 + 0] = r;
    out[i * 3 + 1] = g;
    out[i * 3 + 2] = b;
  }
}

// fp32 images in [0, 1] -> uint8 exactly as modules/processing.py:1039-1040 does on the host (255 * x, astype(uint8) = truncation)
__global__ void images_to_u8_kernel(const float4* __restrict__ x, uchar4* __restrict__ out, size_t n4) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < n4; i += (size_t)gridDim.x * blockDim.x) {
    const float4 v = x[i];
    uchar4 o;
    o.x = (unsigned char)(255.f * v.x);
    o.y = (unsigned char)(255.f * v.y);
    o.z = (unsigned char)(255.f * v.z);
    o.w = (unsigned char)(255.f * v.w);
    out[i] = o;
  }
}

// VAE encode entry: pixels NHWC fp32 [pixels, 3] in [0, 1] -> [pixels, 8] in dtype, channels 0-2 = 2x - 1, 3-7 = 0
// (backend/patcher/vae.py:177 `2. * pixel_samples - 1.` then the cast to the VAE dtype)
template <bool BF16>
__global__ void vae_pre_kernel(const float* __restrict__ x, void* __restrict__ out, size_t pixels) {
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < pixels; i += (size_t)gridDim.x * blockDim.x) {
    const float r = 2.f * x[i * 3] - 1.f, g = 2.f * x[i * 3 + 1] - 1.f, b = 2.f * x[i * 3 + 2] - 1.f;
    uint4 o;
    o.x = pack2<BF16>(r, g);
    o.y = pack2<BF16>(b, 0.f);
    o.z = 0u;
    o.w = 0u;
    reinterpret_cast<uint4*>(out)[i] = o;
  }
}

// DiagonalGaussianDistribution (backend/nn/vae.py:16-32) on the channels-last moments [N, H, W, ld] (mean = channels
// [0, C), logvar = [C, 2C)): out NCHW fp32 = (mean + exp(0.5 * clamp(logvar, -30, 20)) * noise) * scale; noise = null -> mode()
template <bool BF16>
__global__ void vae_posterior_kernel(const void* __restrict__ mom, const float* __restrict__ noise, float* __restrict__ out,
                                     int N, int C, int HW, int ld, float scale) {
  const size_t total = (size_t)N * C * HW;
  for (size_t t = (size_t)blockIdx.x * blockDim.x + threadIdx.x; t < total; t += (size_t)gridDim.x * blockDim.x) {
    const int hw = (int)(t % HW);
    const int c = (int)((t / HW) % C);
    const int n = (int)(t / ((size_t)HW * C));
    const size_t m = ((size_t)n * HW + hw) * ld;
    float v = ld1<BF16>(mom, m + c);
    if (noise) {
      const float lv = fminf(fmaxf(ld1<BF16>(mom, m + C + c), -30.f), 20.f);
      v = fmaf(__expf(0.5f * lv), noise[t], v);
    }
    out[t] = v * scale;
  }
}

// Control residual, `h += ctrl` (backend/nn/unet.py:44-52 apply_control; cldm.py:259-262 `h += guided_hint`): h NHWC
// [N, H, W, C] (dtype) accumulates a control tensor in the reference's NCHW layout or channels-last (ctrl_nhwc), dtype or
// fp32, whose batch is N or 1 (ctrl_batch1: one image broadcast over the batch, as torch's in-place add does).  One thread
// per 8 channels of one pixel.
template <bool BF16>
__global__ void add_control_kernel(void* __restrict__ h, const void* __restrict__ ctrl, int N, int C, int H, int W,
                                   int ctrl_batch1, int ctrl_nhwc, int ctrl_is_f32) {
  const int CV = C >> 3;
  const size_t HW = (size_t)H * W;
  const size_t total = (size_t)N * HW * CV;
  for (size_t i = (size_t)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (size_t)gridDim.x * blockDim.x) {
    const int cv = (int)(i % CV);
    const size_t t = i / CV;
    const size_t hw = t % HW;
    const size_t n = ctrl_batch1 ? 0 : t / HW;  // batch index into ctrl
    float v[8];
    load8<BF16>(h, i * 8, v);
    if (ctrl_nhwc) {
      const size_t src = (n * HW + hw) * C + (size_t)cv * 8;
      float u[8];
      if (ctrl_is_f32) {
        const float4 a = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(ctrl) + src);
        const float4 b = *reinterpret_cast<const float4*>(reinterpret_cast<const float*>(ctrl) + src + 4);
        u[0] = a.x; u[1] = a.y; u[2] = a.z; u[3] = a.w; u[4] = b.x; u[5] = b.y; u[6] = b.z; u[7] = b.w;
      } else {
        load8<BF16>(ctrl, src, u);
      }
#pragma unroll
      for (int j = 0; j < 8; ++j) v[j] += u[j];
    } else {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const size_t src = (n * C + (size_t)(cv * 8 + j)) * HW + hw;
        v[j] += ctrl_is_f32 ? reinterpret_cast<const float*>(ctrl)[src] : ld1<BF16>(ctrl, src);
      }
    }
    store8<BF16>(h, i * 8, v);
  }
}

static inline int grid_for(size_t total, int block) {
  size_t g = (total + block - 1) / block;
  const size_t cap = (size_t)num_sms() * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace b200

using namespace b200;

#define DISPATCH_DTYPE(dtype, ...)                 \
  do {                                             \
    if ((dtype) == B200_BF16) {                    \
      constexpr bool BF = true;                    \
      __VA_ARGS__;                                 \
    } else {                                       \
      constexpr bool BF = false;                   \
      __VA_ARGS__;                                 \
    }                                              \
  } while (0)

static int gn_slabs(const b200_gn_desc* d, int* pix_per_slab) {
  int slabs = (4 * num_sms() + d->N - 1) / d->N;
  const int max_slabs = (d->HW + 31) / 32;
  if (slabs > max_slabs) slabs = max_slabs;
  if (slabs < 1) slabs = 1;
  *pix_per_slab = (d->HW + slabs - 1) / slabs;
  slabs = (d->HW + *pix_per_slab - 1) / *pix_per_slab;
  return slabs;
}

static int gn_check(const b200_gn_desc* d, const void* x1, const void* x2) {
  B200_CHECK_ARG(d && x1, "groupnorm: null argument");
  B200_CHECK_ARG(d->C1 > 0 && d->C1 % 8 == 0 && d->C2 >= 0 && d->C2 % 8 == 0, "groupnorm: channels %d/%d", d->C1,
                 d->C2);
  B200_CHECK_ARG((d->C2 == 0) == (x2 == nullptr), "groupnorm: x2/C2 mismatch");
  B200_CHECK_ARG(d->groups > 0 && (d->C1 + d->C2) % d->groups == 0, "groupnorm: groups");
  B200_CHECK_ARG((d->C1 + d->C2) * 8 <= 96 * 1024, "groupnorm: too many channels");
  B200_CHECK_ARG(d->N > 0 && d->N <= 65535 && d->HW > 0, "groupnorm: shape");
  return B200_OK;
}

static size_t gn_ws_tickets_bytes(int N) { return (((size_t)N * sizeof(int)) + 255) / 256 * 256; }

extern "C" size_t b200_groupnorm_ws_bytes(const b200_gn_desc* d) {
  if (!d || d->N <= 0 || d->groups <= 0 || d->HW <= 0) return 0;
  int pps;
  const int slabs = gn_slabs(d, &pps);
  return gn_ws_tickets_bytes(d->N) + (size_t)d->N * d->groups * 2 * sizeof(float) * (1 + (size_t)slabs);
}

extern "C" int b200_groupnorm_stats(const void* x1, const void* x2, void* ws, const b200_gn_desc* d, b200_stream_t s) {
  int rc = gn_check(d, x1, x2);
  if (rc) return rc;
  B200_CHECK_ARG(ws && (reinterpret_cast<uintptr_t>(ws) & 15) == 0, "groupnorm_stats: null / unaligned workspace");
  int pps;
  const int slabs = gn_slabs(d, &pps);
  const int C = d->C1 + d->C2;
  const int CV = C / 8;
  const int TX = CV < 256 ? CV : 256;
  const int RY = 256 / TX;
  const size_t smem = (size_t)C * (1 + 2 * RY) * sizeof(float);
  B200_CHECK_ARG(smem <= 200 * 1024, "groupnorm: too many channels (%d)", C);
  int* tickets = reinterpret_cast<int*>(ws);
  float* fin = reinterpret_cast<float*>(reinterpret_cast<char*>(ws) + gn_ws_tickets_bytes(d->N));
  float* part = fin + (size_t)d->N * d->groups * 2;
  dim3 grid(slabs, d->N);
  DISPATCH_DTYPE(d->dtype, {
    if (smem > 48 * 1024) cudaFuncSetAttribute(gn_stats_kernel<BF>, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);
    launch_pdl(gn_stats_kernel<BF>, dim3(grid), dim3(256), smem, (cudaStream_t)s, 1, x1, x2, tickets, fin, part, d->HW, d->C1, d->C2, d->groups, pps,
                                                               d->eps);
  });
  B200_CHECK_LAUNCH("groupnorm_stats");
  return B200_OK;
}

extern "C" int b200_groupnorm_apply(const void* x1, const void* x2, const void* ws, const void* gamma,
                                    const void* beta, void* y, const b200_gn_desc* d, b200_stream_t s) {
  int rc = gn_check(d, x1, x2);
  if (rc) return rc;
  B200_CHECK_ARG(ws && gamma && beta && y, "groupnorm_apply: null argument");
  int pps;
  const int slabs = gn_slabs(d, &pps);
  const size_t smem = (size_t)(d->C1 + d->C2) * 2 * sizeof(float);
  const float* fin = reinterpret_cast<const float*>(reinterpret_cast<const char*>(ws) + gn_ws_tickets_bytes(d->N));
  dim3 grid(slabs, d->N);
  DISPATCH_DTYPE(d->dtype, {
    if (smem > 48 * 1024) cudaFuncSetAttribute(gn_apply_kernel<BF>, cudaFuncAttributeMaxDynamicSharedMemorySize, 96 * 1024);
    launch_pdl(gn_apply_kernel<BF>, dim3(grid), dim3(256), smem, (cudaStream_t)s, 1, x1, x2, fin, gamma, beta, y, d->HW, d->C1, d->C2,
                                                               d->groups, d->silu, pps);
  });
  B200_CHECK_LAUNCH("groupnorm_apply");
  return B200_OK;
}

extern "C" int b200_layernorm(const void* x, const void* gamma, const void* beta, void* y, int rows, int C, float eps,
                              int dtype, b200_stream_t s) {
  B200_CHECK_ARG(x && y && rows > 0 && C > 0 && C % 8 == 0, "layernorm: bad arguments");
  if (C > 8 * 32 * 16) {
    set_error("layernorm: C=%d unsupported (max 4096)", C);
    return B200_EUNSUPPORTED;
  }
  const int grid = (rows + 7) / 8;
  DISPATCH_DTYPE(dtype, {
    if (C <= 8 * 32 * 5) layernorm_kernel<BF, 5><<<grid, 256, 0, (cudaStream_t)s>>>(x, gamma, beta, y, rows, C, eps);
    else layernorm_kernel<BF, 16><<<grid, 256, 0, (cudaStream_t)s>>>(x, gamma, beta, y, rows, C, eps);
  });
  B200_CHECK_LAUNCH("layernorm");
  return B200_OK;
}

extern "C" int b200_upsample2x(const void* x, void* y, int N, int H, int W, int C, int dtype, b200_stream_t s) {
  (void)dtype;
  B200_CHECK_ARG(x && y && C % 8 == 0 && N > 0 && H > 0 && W > 0, "upsample2x: bad arguments");
  const size_t total = (size_t)N * 4 * H * W * (C / 8);
  launch_pdl(upsample2x_kernel, dim3(grid_for(total, 256)), dim3(256), 0, (cudaStream_t)s, 1, (const uint4*)x, (uint4*)y, N, H, W, C / 8);
  B200_CHECK_LAUNCH("upsample2x");
  return B200_OK;
}

extern "C" int b200_im2col3x3(const void* x, void* out, int N, int H, int W, int C, int stride, int pad_lo, int Ho,
                              int Wo, int ldo, int dtype, b200_stream_t s) {
  (void)dtype;
  B200_CHECK_ARG(x && out && N > 0 && H > 0 && W > 0 && C > 0 && stride > 0 && ldo >= 9 * C && ldo % 8 == 0,
                 "im2col3x3: bad arguments");
  if (C % 8 == 0) {
    const size_t total = (size_t)N * Ho * Wo * (ldo / 8);
    launch_pdl(im2col3x3_vec_kernel, dim3(grid_for(total, 256)), dim3(256), 0, (cudaStream_t)s, 1, (const uint4*)x, (uint4*)out, N, H, W,
                                                                             C / 8, stride, pad_lo, Ho, Wo, ldo / 8);
  } else {
    const size_t total = (size_t)N * Ho * Wo * ldo;
    im2col3x3_scalar_kernel<<<grid_for(total, 256), 256, 0, (cudaStream_t)s>>>(
        (const uint16_t*)x, (uint16_t*)out, N, H, W, C, stride, pad_lo, Ho, Wo, ldo);
  }
  B200_CHECK_LAUNCH("im2col3x3");
  return B200_OK;
}

extern "C" int b200_nchw_to_nhwc(const void* x, void* y, int N, int C, int H, int W, int ldy, float scale,
                                 int in_is_f32, int dtype, b200_stream_t s) {
  B200_CHECK_ARG(x && y && N > 0 && C > 0 && H > 0 && W > 0 && ldy >= C, "nchw_to_nhwc: bad arguments");
  const size_t total = (size_t)N * ldy * H * W;
  DISPATCH_DTYPE(dtype, launch_pdl(nchw_to_nhwc_kernel<BF>, dim3(grid_for(total, 256)), dim3(256), 0, (cudaStream_t)s, 1, x, y, N, C, H, W, ldy,
                                                                                                  scale, in_is_f32));
  B200_CHECK_LAUNCH("nchw_to_nhwc");
  return B200_OK;
}

extern "C" int b200_nhwc_to_nchw(const void* x, void* y, int N, int C, int H, int W, int ldx, int out_is_f32,
                                 int dtype, b200_stream_t s) {
  B200_CHECK_ARG(x && y && N > 0 && C > 0 && H > 0 && W > 0 && ldx >= C, "nhwc_to_nchw: bad arguments");
  const size_t total = (size_t)N * C * H * W;
  DISPATCH_DTYPE(dtype, launch_pdl(nhwc_to_nchw_kernel<BF>, dim3(grid_for(total, 256)), dim3(256), 0, (cudaStream_t)s, 1, x, y, N, C, H, W, ldx,
                                                                                                  out_is_f32));
  B200_CHECK_LAUNCH("nhwc_to_nchw");
  return B200_OK;
}

extern "C" int b200_silu(const void* x, void* y, size_t n, int dtype, b200_stream_t s) {
  B200_CHECK_ARG(x && y && n > 0, "silu: bad arguments");
  DISPATCH_DTYPE(dtype, launch_pdl(silu_kernel<BF>, dim3(grid_for(n, 256)), dim3(256), 0, (cudaStream_t)s, 1, x, y, n));
  B200_CHECK_LAUNCH("silu");
  return B200_OK;
}

extern "C" int b200_softmax_rows(void* x, int rows, int cols, int valid_cols, int ld, float scale, int dtype,
                                 b200_stream_t s) {
  B200_CHECK_ARG(x && rows > 0 && cols > 0 && cols % 8 == 0 && ld % 8 == 0 && valid_cols > 0 && valid_cols <= cols,
                 "softmax_rows: bad arguments");
  DISPATCH_DTYPE(dtype, launch_pdl(softmax_rows_kernel<BF>, dim3(rows), dim3(256), 0, (cudaStream_t)s, 1, x, rows, cols, ld,
                                                                                  scale * 1.4426950408889634f, valid_cols, 0, 0));
  B200_CHECK_LAUNCH("softmax_rows");
  return B200_OK;
}

extern "C" int b200_softmax_rows_blockdiag(void* x, int rows, int cols, int ld, float scale, int block_rows, int block_cols,
                                           int valid_in_block, int dtype, b200_stream_t s) {
  B200_CHECK_ARG(x && rows > 0 && cols > 0 && cols % 8 == 0 && ld % 8 == 0 && block_rows > 0 && block_cols > 0 &&
                     valid_in_block > 0 && valid_in_block <= block_cols && rows % block_rows == 0 &&
                     (rows / block_rows - 1) * block_cols + valid_in_block <= cols,
                 "softmax_rows_blockdiag: bad arguments");
  DISPATCH_DTYPE(dtype, launch_pdl(softmax_rows_kernel<BF>, dim3(rows), dim3(256), 0, (cudaStream_t)s, 1, 
                            x, rows, cols, ld, scale * 1.4426950408889634f, valid_in_block, block_rows, block_cols));
  B200_CHECK_LAUNCH("softmax_rows_blockdiag");
  return B200_OK;
}

extern "C" int b200_timestep_embedding(const float* t, void* out, int B, int dim, float max_period, int dtype,
                                       b200_stream_t s) {
  B200_CHECK_ARG(t && out && B > 0 && dim > 1, "timestep_embedding: bad arguments");
  const float neg_log = -logf(max_period);
  DISPATCH_DTYPE(dtype, launch_pdl(timestep_embedding_kernel<BF>, dim3(grid_for((size_t)B * (dim / 2), 128)), dim3(128), 0, (cudaStream_t)s, 1, 
                            t, out, B, dim, neg_log));
  B200_CHECK_LAUNCH("timestep_embedding");
  return B200_OK;
}

extern "C" int b200_unet_input_im2col(const float* x, const float* sigma, void* cols, int B, int C, int H, int W,
                                      int ldo, int reps, int dtype, b200_stream_t s) {
  B200_CHECK_ARG(x && sigma && cols && B > 0 && C > 0 && H > 0 && W > 0 && ldo >= 9 * C && ldo % 8 == 0 && reps > 0,
                 "unet_input_im2col: bad arguments");
  const size_t total = (size_t)B * H * W * ldo;
  DISPATCH_DTYPE(dtype, launch_pdl(unet_input_im2col_kernel<BF>, dim3(grid_for(total, 256)), dim3(256), 0, (cudaStream_t)s, 1, 
                            x, sigma, cols, B, C, H, W, ldo, reps));
  B200_CHECK_LAUNCH("unet_input_im2col");
  return B200_OK;
}

extern "C" int b200_vae_postprocess(const void* x, float* out, size_t pixels, int ldx, int dtype, b200_stream_t s) {
  B200_CHECK_ARG(x && out && pixels > 0 && ldx >= 3, "vae_postprocess: bad arguments");
  DISPATCH_DTYPE(dtype, vae_post_kernel<BF><<<grid_for(pixels * 3, 256), 256, 0, (cudaStream_t)s>>>(x, out, pixels, ldx));
  B200_CHECK_LAUNCH("vae_postprocess");
  return B200_OK;
}

extern "C" int b200_tile_blend(const void* tile, float* acc, int H, int W, int y0, int x0, int th, int tw, int ld, float bias,
                               int feather, int dtype, b200_stream_t s) {
  B200_CHECK_ARG(tile && acc && th > 0 && tw > 0 && ld >= 3 && y0 >= 0 && x0 >= 0 && y0 + th <= H && x0 + tw <= W && feather >= 0,
                 "tile_blend: tile [%d,%d]+(%d,%d) outside the %dx%d image", th, tw, y0, x0, H, W);
  B200_CHECK_ARG((reinterpret_cast<uintptr_t>(acc) & 15) == 0, "tile_blend: acc must be 16-byte aligned");
  DISPATCH_DTYPE(dtype, tile_blend_kernel<BF><<<grid_for((size_t)th * tw, 256), 256, 0, (cudaStream_t)s>>>(
                            tile, reinterpret_cast<float4*>(acc), W, y0, x0, th, tw, ld, bias, feather));
  B200_CHECK_LAUNCH("tile_blend");
  return B200_OK;
}

extern "C" int b200_tile_resolve(const float* acc, float* out, size_t pixels, int accumulate, float final_scale, int finalize,
                                 b200_stream_t s) {
  B200_CHECK_ARG(acc && out && pixels > 0 && (reinterpret_cast<uintptr_t>(acc) & 15) == 0, "tile_resolve: bad arguments");
  tile_resolve_kernel<<<grid_for(pixels, 256), 256, 0, (cudaStream_t)s>>>(reinterpret_cast<const float4*>(acc), out, pixels,
                                                                           accumulate, final_scale, finalize);
  B200_CHECK_LAUNCH("tile_resolve");
  return B200_OK;
}

extern "C" int b200_images_to_u8(const float* x, unsigned char* out, size_t n, b200_stream_t s) {
  B200_CHECK_ARG(x && out && n > 0 && n % 4 == 0 && (reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(out) & 3) == 0,
                 "images_to_u8: element count must be a multiple of 4, pointers 16 / 4-byte aligned");
  images_to_u8_kernel<<<grid_for(n / 4, 256), 256, 0, (cudaStream_t)s>>>(reinterpret_cast<const float4*>(x),
                                                                           reinterpret_cast<uchar4*>(out), n / 4);
  B200_CHECK_LAUNCH("images_to_u8");
  return B200_OK;
}

extern "C" int b200_vae_preprocess(const float* x, void* out, size_t pixels, int dtype, b200_stream_t s) {
  B200_CHECK_ARG(x && out && pixels > 0, "vae_preprocess: bad arguments");
  DISPATCH_DTYPE(dtype, vae_pre_kernel<BF><<<grid_for(pixels, 256), 256, 0, (cudaStream_t)s>>>(x, out, pixels));
  B200_CHECK_LAUNCH("vae_preprocess");
  return B200_OK;
}

extern "C" int b200_vae_posterior(const void* moments, const float* noise, float* out, int N, int C, int HW, int ld,
                                  float scale, int dtype, b200_stream_t s) {
  B200_CHECK_ARG(moments && out && N > 0 && C > 0 && HW > 0 && ld >= 2 * C, "vae_posterior: bad arguments");
  DISPATCH_DTYPE(dtype, vae_posterior_kernel<BF><<<grid_for((size_t)N * C * HW, 256), 256, 0, (cudaStream_t)s>>>(
                            moments, noise, out, N, C, HW, ld, scale));
  B200_CHECK_LAUNCH("vae_posterior");
  return B200_OK;
}

extern "C" int b200_add_control(void* h, const void* ctrl, int N, int C, int H, int W, int ctrl_batch, int ctrl_nhwc,
                                int ctrl_is_f32, int dtype, b200_stream_t s) {
  B200_CHECK_ARG(h && ctrl && N > 0 && C > 0 && H > 0 && W > 0 && C % 8 == 0,
                 "add_control: bad arguments (C must be a multiple of 8)");
  B200_CHECK_ARG(ctrl_batch == N || ctrl_batch == 1, "add_control: residual batch %d must be 1 or %d", ctrl_batch, N);
  B200_CHECK_ARG(!ctrl_nhwc || (reinterpret_cast<uintptr_t>(ctrl) & 15) == 0, "add_control: NHWC residual must be 16-byte aligned");
  const size_t total = (size_t)N * H * W * (C / 8);
  DISPATCH_DTYPE(dtype, add_control_kernel<BF><<<grid_for(total, 256), 256, 0, (cudaStream_t)s>>>(
                            h, ctrl, N, C, H, W, ctrl_batch == 1 && N > 1 ? 1 : 0, ctrl_nhwc ? 1 : 0, ctrl_is_f32));
  B200_CHECK_LAUNCH("add_control");
  return B200_OK;
}

extern "C" int b200_add_nchw(void* h, const void* ctrl, int N, int C, int H, int W, int ctrl_is_f32, int dtype,
                             b200_stream_t s) {
  return b200_add_control(h, ctrl, N, C, H, W, N, 0, ctrl_is_f32, dtype, s);
}
