// nn_ops.cu — normalisation, pointwise and attention kernels shared by the s2mel / codec paths
// (channels-last fp32, see ops.h).  Reference semantics cited at each kernel.
#include "ops.h"
#include <cuda_bf16.h>
#include <cstdlib>

namespace {

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// GEMM operands of the fp16 tensor-core path are written by the kernel that produces them: every pointwise kernel
// below takes an optional fp16 destination next to (or instead of) the fp32 one.
__device__ __forceinline__ void put(float* __restrict__ y, __half* __restrict__ y16, long long i, float v) {
  if (y) y[i] = v;
  if (y16) y16[i] = __float2half_rn(v);
}

// One warp per row.  MODE 0: LayerNorm (two-pass), MODE 1: RMSNorm (gpt_fast/model.py:317-333).
template <int MODE>
__global__ void rownorm_kernel(const float* __restrict__ x, float* __restrict__ y, long long rows, int T,
                               int C, const float* __restrict__ w, const float* __restrict__ b, float eps,
                               const float* __restrict__ m0, const float* __restrict__ m1, int mod_stride,
                               __half* __restrict__ y16) {
  pdl_wait();
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const int bidx = (int)(row / T);
  const float* xr = x + row * C;
  float s = 0.f;
  for (int i = lane; i < C; i += 32) s += xr[i];
  float mean = 0.f, q = 0.f;
  if (MODE == 0) {
    mean = warp_sum(s) / C;
    for (int i = lane; i < C; i += 32) { float d = xr[i] - mean; q += d * d; }
  } else {
    for (int i = lane; i < C; i += 32) q += xr[i] * xr[i];
  }
  const float rstd = rsqrtf(warp_sum(q) / C + eps);
  for (int i = lane; i < C; i += 32) {
    float v = (xr[i] - mean) * rstd;
    if (MODE == 0) {
      if (w) v = v * w[i] + (b ? b[i] : 0.f);
      // modulate(x, shift, scale) = x * (1 + scale) + shift   (diffusion_transformer.py:11-12)
      if (m0) v = v * (1.f + m0[(long long)bidx * mod_stride + i]) + m1[(long long)bidx * mod_stride + i];
    } else {
      v *= w[i];
      // AdaptiveLayerNorm: weight * norm(x) + bias             (gpt_fast/model.py:20-39)
      if (m0) v = m0[(long long)bidx * mod_stride + i] * v + m1[(long long)bidx * mod_stride + i];
    }
    put(y, y16, row * C + i, v);
  }
}

__global__ void gn_stats_kernel(const float* __restrict__ x, double* stats, long long n_per) {
  const int b = blockIdx.y;
  const float* xb = x + (long long)b * n_per;
  double s = 0, q = 0;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_per; i += (long long)gridDim.x * blockDim.x) {
    const double v = xb[i];
    s += v; q += v * v;
  }
  __shared__ double ss[256], qq[256];
  ss[threadIdx.x] = s; qq[threadIdx.x] = q;
  __syncthreads();
  for (int o = 128; o > 0; o >>= 1) {
    if (threadIdx.x < o) { ss[threadIdx.x] += ss[threadIdx.x + o]; qq[threadIdx.x] += qq[threadIdx.x + o]; }
    __syncthreads();
  }
  if (threadIdx.x == 0) { atomicAdd(&stats[2 * b], ss[0]); atomicAdd(&stats[2 * b + 1], qq[0]); }
}
__global__ void gn_apply_mish_kernel(const float* __restrict__ x, float* __restrict__ y, const double* stats,
                                     long long n_per, int C, const float* __restrict__ w,
                                     const float* __restrict__ bb, float eps) {
  const int b = blockIdx.y;
  const double mean = stats[2 * b] / n_per;
  const double var = stats[2 * b + 1] / n_per - mean * mean;
  const float rstd = (float)(1.0 / sqrt(var + (double)eps));
  const float fm = (float)mean;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n_per; i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    float v = (x[(long long)b * n_per + i] - fm) * rstd * w[c] + bb[c];
    const float sp = (v > 20.f) ? v : log1pf(expf(v));   // F.mish = x * tanh(softplus(x))
    y[(long long)b * n_per + i] = v * tanhf(sp);
  }
}

__global__ void dwconv_kernel(const float* __restrict__ x, float* __restrict__ y, int T, int C,
                              const float* __restrict__ w, const float* __restrict__ b, int k) {
  const int bi = blockIdx.z;
  const int t = blockIdx.y;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  const float* xb = x + (long long)bi * T * C;
  float acc = b ? b[c] : 0.f;
  const int pad = (k - 1) / 2;
  for (int j = 0; j < k; ++j) {
    const int ts = t + j - pad;
    if (ts >= 0 && ts < T) acc = fmaf(xb[(long long)ts * C + c], w[c * k + j], acc);
  }
  y[((long long)bi * T + t) * C + c] = acc;
}

__global__ void nearest_kernel(const float* __restrict__ x, float* __restrict__ y, int Tin, int Tout, int C) {
  const int bi = blockIdx.z, t = blockIdx.y;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  // aten nearest_idx: scale = (float)in/out; src = min((int)floorf(dst * scale), in - 1)
  const float scale = (float)Tin / (float)Tout;
  int src = (int)floorf((float)t * scale);
  if (src > Tin - 1) src = Tin - 1;
  y[((long long)bi * Tout + t) * C + c] = x[((long long)bi * Tin + src) * C + c];
}

// ids outside [0, nrows) never index the table: the row is zero-filled and the engine flag records the position
// (torch's F.embedding raises IndexError there; the ABI call returns IDX_ERR_ARG after the stream drains)
__global__ void embedding_kernel(const float* __restrict__ table, const int* __restrict__ ids, float* out, int C,
                                 int nrows, int* bad) {
  const int t = blockIdx.y;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  const int id = ids[t];
  const bool ok = id >= 0 && id < nrows;
  if (!ok && c == 0) atomicCAS(bad, 0, t + 1);
  if (c < C) out[(long long)t * C + c] = ok ? table[(long long)id * C + c] : 0.f;
}

__global__ void swiglu_kernel(const float* __restrict__ ab, float* __restrict__ y, long long rows, int N, __half* __restrict__ y16) {
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * N) return;
  const long long r = i / N;
  const int c = (int)(i % N);
  const float a = ab[r * 2 * N + c], b = ab[r * 2 * N + N + c];
  put(y, y16, i, a / (1.f + expf(-a)) * b);   // F.silu(w1 x) * (w3 x)  (gpt_fast/model.py:311-314)
}

__global__ void wn_gate_kernel(const float* __restrict__ xin, const float* __restrict__ g, int g_stride,
                               float* __restrict__ y, int T, int N, __half* __restrict__ y16) {
  pdl_wait();
  // fused_add_tanh_sigmoid_multiply (s2mel/modules/commons.py:132-141)
  const int bi = blockIdx.z;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)T * N) return;
  const long long t = i / N;
  const int c = (int)(i % N);
  const float* xr = xin + ((long long)bi * T + t) * 2 * N;
  const float a = xr[c] + g[(long long)bi * g_stride + c];
  const float s = xr[N + c] + g[(long long)bi * g_stride + N + c];
  put(y, y16, ((long long)bi * T + t) * N + c, tanhf(a) * (1.f / (1.f + expf(-s))));
}

__global__ void copy_cols_kernel(const float* __restrict__ src, int lds, float* __restrict__ dst, int ldo,
                                 int col0, long long rows, int C, __half* __restrict__ dst16) {
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= rows * C) return;
  const long long r = i / C;
  const int c = (int)(i % C);
  put(dst, dst16, r * ldo + col0 + c, src[r * lds + c]);
}
__global__ void bcast_cols_kernel(const float* __restrict__ vec, float* __restrict__ dst, int ldo, int col0,
                                  int T, int C) {
  const int bi = blockIdx.z;
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)T * C) return;
  const long long t = i / C;
  const int c = (int)(i % C);
  dst[((long long)bi * T + t) * ldo + col0 + c] = vec[(long long)bi * C + c];
}
__global__ void silu_kernel(float* x, long long n) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) { const float v = x[i]; x[i] = v / (1.f + expf(-v)); }
}
__global__ void reflect_pad_kernel(const float* __restrict__ x, float* __restrict__ y, int T, int C, int left,
                                   int Tout, __half* __restrict__ y16) {
  pdl_wait();
  const int bi = blockIdx.z, i = blockIdx.y;
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c >= C) return;
  int t = i - left;
  if (t < 0) t = -t;
  if (t >= T) t = 2 * (T - 1) - t;
  put(y, y16, ((long long)bi * Tout + i) * C + c, x[((long long)bi * T + t) * C + c]);
}
__global__ void zero_kernel(float* x, long long n) {
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i < n) x[i] = 0.f;
}
__global__ void rope_table_kernel(float* tab, int T, int hd) {
  const int t = blockIdx.x;
  const int i = threadIdx.x;
  if (i >= hd / 2) return;
  // freqs = 1 / base^(2i/hd); angle = t * freq (fp32), cache = (cos, sin)   (model.py:336-346)
  const float freq = 1.0f / powf(10000.f, (float)(2 * i) / (float)hd);
  const float ang = (float)t * freq;
  tab[((long long)t * (hd / 2) + i) * 2] = cosf(ang);
  tab[((long long)t * (hd / 2) + i) * 2 + 1] = sinf(ang);
}
__global__ void cfg_euler_kernel(float* x, const float* vc, const float* vu, float dt, float rate, int T,
                                 int C, int P) {
  pdl_wait();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)T * C) return;
  const int t = (int)(i / C);
  // dphi = (1 + r) * dphi_cond - r * dphi_uncond ; x = x + dt * dphi ; x[:, :, :P] = 0
  // (flow_matching.py:96-113)
  const float d = (1.0f + rate) * vc[i] - rate * vu[i];
  x[i] = (t < P) ? 0.f : x[i] + dt * d;
}

// ------------------------------------------------------------------------ attention ----
// fp32 flash attention, 64 queries x 64 keys per tile, head_dim 64, RoPE applied on load
// (F.scaled_dot_product_attention with a key-padding mask, gpt_fast/model.py:293-306).
constexpr int AQ = 64, AK = 64, AD = 64;
__global__ void __launch_bounds__(256) attention_kernel(const float* __restrict__ qkv, float* __restrict__ out,
                                                        int T, int H, const float* __restrict__ rope,
                                                        const int* __restrict__ lens) {
  extern __shared__ float sm[];
  float* Qt = sm;                 // [AD][AQ]
  float* Kt = Qt + AD * AQ;       // [AD][AK]
  float* Vs = Kt + AD * AK;       // [AK][AD]
  float* Pt = Vs + AK * AD;       // [AK][AQ]
  const int b = blockIdx.z, h = blockIdx.y, q0 = blockIdx.x * AQ;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const int ld = 3 * H * AD;
  const float* base = qkv + (long long)b * T * ld;
  const int len = lens ? lens[b] : T;
  // load + rotate Q (pairs), scaled by 1/sqrt(64)
  for (int i = tid; i < AQ * (AD / 2); i += 256) {
    const int r = i / (AD / 2), pi = i % (AD / 2);
    const int t = q0 + r;
    float a = 0.f, c = 0.f;
    if (t < T) {
      const float* qp = base + (long long)t * ld + h * AD + 2 * pi;
      const float cs = rope[((long long)t * (AD / 2) + pi) * 2], sn = rope[((long long)t * (AD / 2) + pi) * 2 + 1];
      const float x0 = qp[0], x1 = qp[1];
      a = (x0 * cs - x1 * sn) * 0.125f;
      c = (x1 * cs + x0 * sn) * 0.125f;
    }
    Qt[(2 * pi) * AQ + r] = a;
    Qt[(2 * pi + 1) * AQ + r] = c;
  }
  float m[4], l[4], o[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    m[i] = -INFINITY; l[i] = 0.f;
#pragma unroll
    for (int j = 0; j < 4; ++j) o[i][j] = 0.f;
  }
  for (int k0 = 0; k0 < len; k0 += AK) {
    __syncthreads();
    for (int i = tid; i < AK * (AD / 2); i += 256) {
      const int r = i / (AD / 2), pi = i % (AD / 2);
      const int t = k0 + r;
      float a = 0.f, c = 0.f, v0 = 0.f, v1 = 0.f;
      if (t < len) {
        const float* kp = base + (long long)t * ld + H * AD + h * AD + 2 * pi;
        const float cs = rope[((long long)t * (AD / 2) + pi) * 2], sn = rope[((long long)t * (AD / 2) + pi) * 2 + 1];
        const float x0 = kp[0], x1 = kp[1];
        a = x0 * cs - x1 * sn;
        c = x1 * cs + x0 * sn;
        const float* vp = kp + H * AD;
        v0 = vp[0]; v1 = vp[1];
      }
      Kt[(2 * pi) * AK + r] = a;
      Kt[(2 * pi + 1) * AK + r] = c;
      Vs[r * AD + 2 * pi] = v0;
      Vs[r * AD + 2 * pi + 1] = v1;
    }
    __syncthreads();
    float s[4][4];
#pragma unroll
    for (int i = 0; i < 4; ++i)
#pragma unroll
      for (int j = 0; j < 4; ++j) s[i][j] = 0.f;
#pragma unroll 8
    for (int d = 0; d < AD; ++d) {
      const float4 qa = *(const float4*)(Qt + d * AQ + ty * 4);
      const float4 kb = *(const float4*)(Kt + d * AK + tx * 4);
      const float qv[4] = {qa.x, qa.y, qa.z, qa.w}, kv[4] = {kb.x, kb.y, kb.z, kb.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) s[i][j] = fmaf(qv[i], kv[j], s[i][j]);
    }
#pragma unroll
    for (int i = 0; i < 4; ++i) {
      float mx = -INFINITY;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        if (k0 + tx * 4 + j >= len) s[i][j] = -INFINITY;
        mx = fmaxf(mx, s[i][j]);
      }
#pragma unroll
      for (int xo = 1; xo <= 8; xo <<= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, xo));
      const float mn = fmaxf(m[i], mx);
      const float corr = (m[i] == -INFINITY) ? 0.f : __expf(m[i] - mn);
      float rs = 0.f;
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float p = (s[i][j] == -INFINITY) ? 0.f : __expf(s[i][j] - mn);
        s[i][j] = p;
        rs += p;
      }
#pragma unroll
      for (int xo = 1; xo <= 8; xo <<= 1) rs += __shfl_xor_sync(0xffffffffu, rs, xo);
      l[i] = l[i] * corr + rs;
      m[i] = mn;
#pragma unroll
      for (int j = 0; j < 4; ++j) o[i][j] *= corr;
#pragma unroll
      for (int j = 0; j < 4; ++j) Pt[(tx * 4 + j) * AQ + ty * 4 + i] = s[i][j];
    }
    __syncthreads();
#pragma unroll 8
    for (int k = 0; k < AK; ++k) {
      const float4 pa = *(const float4*)(Pt + k * AQ + ty * 4);
      const float4 vb = *(const float4*)(Vs + k * AD + tx * 4);
      const float pv[4] = {pa.x, pa.y, pa.z, pa.w}, vv[4] = {vb.x, vb.y, vb.z, vb.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) o[i][j] = fmaf(pv[i], vv[j], o[i][j]);
    }
  }
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int t = q0 + ty * 4 + i;
    if (t >= T) continue;
    const float inv = l[i] > 0.f ? 1.f / l[i] : 0.f;
    float4 r = make_float4(o[i][0] * inv, o[i][1] * inv, o[i][2] * inv, o[i][3] * inv);
    *(float4*)(out + ((long long)b * T + t) * H * AD + h * AD + tx * 4) = r;
  }
}

// ---- unfused tensor-core attention helpers (S = Q K^T and O = P V run on the tcgen05 GEMM) ----
__global__ void rope_split_kernel(const float* __restrict__ qkv, const float* __restrict__ rope,
                                  float* __restrict__ Qr, float* __restrict__ Kr, float* __restrict__ Vt,
                                  int T, int Tp, int H) {
  const int t = blockIdx.x, h = blockIdx.y, b = blockIdx.z, i = threadIdx.x;  // 64 threads
  const int ld = 3 * H * AD;
  const float* row = qkv + ((long long)b * T + t) * ld;
  const long long bh = (long long)b * H + h;
  if (i < AD / 2) {
    const float cs = rope[((long long)t * (AD / 2) + i) * 2], sn = rope[((long long)t * (AD / 2) + i) * 2 + 1];
    const float q0 = row[h * AD + 2 * i], q1 = row[h * AD + 2 * i + 1];
    const float k0 = row[H * AD + h * AD + 2 * i], k1 = row[H * AD + h * AD + 2 * i + 1];
    float* qo = Qr + (bh * T + t) * AD + 2 * i;
    float* ko = Kr + (bh * T + t) * AD + 2 * i;
    qo[0] = (q0 * cs - q1 * sn) * 0.125f;   // 1/sqrt(64) folded into q
    qo[1] = (q1 * cs + q0 * sn) * 0.125f;
    ko[0] = k0 * cs - k1 * sn;
    ko[1] = k1 * cs + k0 * sn;
  }
  Vt[(bh * AD + i) * Tp + t] = row[2 * H * AD + h * AD + i];
}
__global__ void softmax_rows_kernel(float* __restrict__ S, long long rows, int T, int Tp) {
  const long long row = (long long)blockIdx.x * (blockDim.x >> 5) + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float* r = S + row * Tp;
  float mx = -INFINITY;
  for (int i = lane; i < T; i += 32) mx = fmaxf(mx, r[i]);
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) mx = fmaxf(mx, __shfl_xor_sync(0xffffffffu, mx, o));
  float sum = 0.f;
  for (int i = lane; i < T; i += 32) { const float p = __expf(r[i] - mx); r[i] = p; sum += p; }
  sum = warp_sum(sum);
  const float inv = 1.f / sum;
  for (int i = lane; i < Tp; i += 32) r[i] = (i < T) ? r[i] * inv : 0.f;
}
__global__ void heads_merge_kernel(const float* __restrict__ O, float* __restrict__ out, int T, int H) {
  const int t = blockIdx.x, h = blockIdx.y, b = blockIdx.z, i = threadIdx.x;
  out[((long long)b * T + t) * H * AD + h * AD + i] = O[(((long long)b * H + h) * T + t) * AD + i];
}

// ---- fused tensor-core flash attention (mma.sync m16n8k16 fp16 for QK^T and PV, fp32 softmax/accumulate) ----
// Inputs are the rotated/split tensors of rope_split_fa_kernel: Qr, Kr, Vb fp16 [BH][T][64] (q pre-scaled by 1/8).
// fp16 since round 2: the same 10-bit mantissa as the tf32 GEMMs around it (round 1 used bf16 q/k/v/p: 8 bits, 1.2e-3 of
// DiT output error on O(1) outputs against the fp32 oracle); q, k, v of a normalised transformer stay far inside fp16 range.  One CTA = 64 queries of one (batch, head); 4 warps x 16 query rows.
// K/V tiles of 64 keys are staged in shared memory (row pitches 272 B / 144 B keep ldmatrix conflict
// free); scores, softmax statistics and the output accumulator never leave registers.
__global__ void rope_split_fa_kernel(const float* __restrict__ qkv, const float* __restrict__ rope,
                                     __half* __restrict__ Qr, __half* __restrict__ Kr,
                                     __half* __restrict__ Vb, int T, int H) {
  pdl_wait();
  const int t = blockIdx.x, h = blockIdx.y, b = blockIdx.z, i = threadIdx.x;  // 64 threads
  const int ld = 3 * H * AD;
  const float* row = qkv + ((long long)b * T + t) * ld;
  const long long bh = (long long)b * H + h;
  if (i < AD / 2) {
    const float cs = rope[((long long)t * (AD / 2) + i) * 2], sn = rope[((long long)t * (AD / 2) + i) * 2 + 1];
    const float q0 = row[h * AD + 2 * i], q1 = row[h * AD + 2 * i + 1];
    const float k0 = row[H * AD + h * AD + 2 * i], k1 = row[H * AD + h * AD + 2 * i + 1];
    *(__half2*)(Qr + (bh * T + t) * AD + 2 * i) =
        __floats2half2_rn((q0 * cs - q1 * sn) * 0.125f, (q1 * cs + q0 * sn) * 0.125f);
    *(__half2*)(Kr + (bh * T + t) * AD + 2 * i) = __floats2half2_rn(k0 * cs - k1 * sn, k1 * cs + k0 * sn);
  }
  Vb[(bh * T + t) * AD + i] = __float2half_rn(row[2 * H * AD + h * AD + i]);
}

__device__ __forceinline__ void ldsm_x4(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void ldsm_x4_trans(uint32_t addr, uint32_t& r0, uint32_t& r1, uint32_t& r2, uint32_t& r3) {
  asm volatile("ldmatrix.sync.aligned.m8n8.x4.trans.shared.b16 {%0,%1,%2,%3}, [%4];"
               : "=r"(r0), "=r"(r1), "=r"(r2), "=r"(r3) : "r"(addr));
}
__device__ __forceinline__ void mma_tf32_1688(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                              uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k8.row.col.f32.tf32.tf32.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ void mma_f16_16816_fa(float (&c)[4], uint32_t a0, uint32_t a1, uint32_t a2, uint32_t a3,
                                                  uint32_t b0, uint32_t b1) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b0), "r"(b1));
}
__device__ __forceinline__ uint32_t tf32_rn(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ uint32_t pack_h2(float lo, float hi) {
  __half2 v = __floats2half2_rn(lo, hi);
  return *(uint32_t*)&v;
}

constexpr int FQ = 64, FK = 64;
constexpr int VPITCH = 72;   // bf16 per K / V row in smem (144 B: ldmatrix rows land in distinct bank groups)
__global__ void __launch_bounds__(128) flash_attn_tc_kernel(const __half* __restrict__ Qr,
                                                            const __half* __restrict__ Kr,
                                                            const __half* __restrict__ Vb,
                                                            float* __restrict__ out, int T, int H,
                                                            __half* __restrict__ out16) {
  pdl_wait();
  // K/V tiles are double buffered: cp.async fills tile i+1 while the tensor cores work on tile i
  __shared__ __align__(16) __half Ks2[2][FK * VPITCH];
  __shared__ __align__(16) __half Vs2[2][FK * VPITCH];
  const int bh = blockIdx.y, q0 = blockIdx.x * FQ;
  const int b = bh / H, h = bh % H;
  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int g = lane >> 2, t4 = lane & 3;
  const __half* Qb = Qr + (long long)bh * T * AD;
  const __half* Kb = Kr + (long long)bh * T * AD;
  const __half* Vbb = Vb + (long long)bh * T * AD;
  // Q fragments (bf16, m16n8k16 A operand) of this warp's 16 rows: 4 k-steps of 16 dims
  uint32_t qa[4][4];
  {
    const int r0 = q0 + warp * 16 + g, r1 = r0 + 8;
#pragma unroll
    for (int ks = 0; ks < 4; ++ks) {
      const int d0 = ks * 16 + 2 * t4;
      qa[ks][0] = r0 < T ? *(const uint32_t*)(Qb + (long long)r0 * AD + d0) : 0u;
      qa[ks][1] = r1 < T ? *(const uint32_t*)(Qb + (long long)r1 * AD + d0) : 0u;
      qa[ks][2] = r0 < T ? *(const uint32_t*)(Qb + (long long)r0 * AD + d0 + 8) : 0u;
      qa[ks][3] = r1 < T ? *(const uint32_t*)(Qb + (long long)r1 * AD + d0 + 8) : 0u;
    }
  }
  float o[8][4];
#pragma unroll
  for (int j = 0; j < 8; ++j) { o[j][0] = o[j][1] = o[j][2] = o[j][3] = 0.f; }
  float m0 = -INFINITY, m1 = -INFINITY, l0 = 0.f, l1 = 0.f;
  const uint32_t ks_base0 = (uint32_t)__cvta_generic_to_shared(&Ks2[0][0]);
  const uint32_t vs_base0 = (uint32_t)__cvta_generic_to_shared(&Vs2[0][0]);

  auto stage_tile = [&](int buf, int k0) {
    // rows beyond T are zero-filled (src-size 0), so masked keys never meet NaN garbage
    for (int i = tid; i < FK * (AD / 8); i += 128) {
      const int r = i / (AD / 8), c8 = (i % (AD / 8)) * 8;
      const bool ok = k0 + r < T;
      const long long src = (long long)(ok ? k0 + r : 0) * AD + c8;
      const uint32_t kd = ks_base0 + (uint32_t)((buf * FK * VPITCH + r * VPITCH + c8) * 2);
      const uint32_t vd = vs_base0 + (uint32_t)((buf * FK * VPITCH + r * VPITCH + c8) * 2);
      const int sz = ok ? 16 : 0;
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(kd), "l"(Kb + src), "r"(sz) : "memory");
      asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"(vd), "l"(Vbb + src), "r"(sz) : "memory");
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  };
  stage_tile(0, 0);
  int buf = 0;
  for (int k0 = 0; k0 < T; k0 += FK, buf ^= 1) {
    if (k0 + FK < T) {
      stage_tile(buf ^ 1, k0 + FK);     // buffer buf^1 was released by the barrier that ended the previous tile
      asm volatile("cp.async.wait_group 1;" ::: "memory");
    } else {
      asm volatile("cp.async.wait_group 0;" ::: "memory");
    }
    __syncthreads();
    const uint32_t ks_base = ks_base0 + (uint32_t)(buf * FK * VPITCH * 2);
    const uint32_t vs_base = vs_base0 + (uint32_t)(buf * FK * VPITCH * 2);
    // S = Q K^T : 8 key tiles (n = 8 keys) x 4 k-steps (16 dims)
    float sc[8][4];
#pragma unroll
    for (int j = 0; j < 8; ++j) { sc[j][0] = sc[j][1] = sc[j][2] = sc[j][3] = 0.f; }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
#pragma unroll
      for (int kp = 0; kp < 2; ++kp) {
        // ldmatrix.x4 (non-transposed, rows = keys 8j..8j+7): matrices = d chunks 32kp + 8i .. +7, i.e. (b0,b1) of
        // k-step 2kp and (b0,b1) of k-step 2kp+1
        uint32_t b0, b1, b2, b3;
        const uint32_t addr = ks_base + (uint32_t)(((j * 8 + (lane & 7)) * VPITCH + kp * 32 + (lane >> 3) * 8) * 2);
        ldsm_x4(addr, b0, b1, b2, b3);
        mma_f16_16816_fa(sc[j], qa[2 * kp][0], qa[2 * kp][1], qa[2 * kp][2], qa[2 * kp][3], b0, b1);
        mma_f16_16816_fa(sc[j], qa[2 * kp + 1][0], qa[2 * kp + 1][1], qa[2 * kp + 1][2], qa[2 * kp + 1][3], b2, b3);
      }
    }
    // mask keys beyond T, online softmax for rows g (c0,c1) and g+8 (c2,c3)
    float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const int key = k0 + j * 8 + 2 * t4;
      if (key >= T) { sc[j][0] = -INFINITY; sc[j][2] = -INFINITY; }
      if (key + 1 >= T) { sc[j][1] = -INFINITY; sc[j][3] = -INFINITY; }
      mx0 = fmaxf(mx0, fmaxf(sc[j][0], sc[j][1]));
      mx1 = fmaxf(mx1, fmaxf(sc[j][2], sc[j][3]));
    }
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 1));
    mx0 = fmaxf(mx0, __shfl_xor_sync(0xffffffffu, mx0, 2));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 1));
    mx1 = fmaxf(mx1, __shfl_xor_sync(0xffffffffu, mx1, 2));
    const float mn0 = fmaxf(m0, mx0), mn1 = fmaxf(m1, mx1);
    const float c0 = (m0 == -INFINITY) ? 0.f : __expf(m0 - mn0);
    const float c1 = (m1 == -INFINITY) ? 0.f : __expf(m1 - mn1);
    float rs0 = 0.f, rs1 = 0.f;
    uint32_t pa[8][2];   // P as bf16 pairs: [tile j][rows g / g+8]
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const float p0 = __expf(sc[j][0] - mn0), p1 = __expf(sc[j][1] - mn0);
      const float p2 = __expf(sc[j][2] - mn1), p3 = __expf(sc[j][3] - mn1);
      rs0 += p0 + p1;
      rs1 += p2 + p3;
      pa[j][0] = pack_h2(p0, p1);
      pa[j][1] = pack_h2(p2, p3);
    }
    rs0 += __shfl_xor_sync(0xffffffffu, rs0, 1);
    rs0 += __shfl_xor_sync(0xffffffffu, rs0, 2);
    rs1 += __shfl_xor_sync(0xffffffffu, rs1, 1);
    rs1 += __shfl_xor_sync(0xffffffffu, rs1, 2);
    l0 = l0 * c0 + rs0;
    l1 = l1 * c1 + rs1;
    m0 = mn0;
    m1 = mn1;
#pragma unroll
    for (int j = 0; j < 8; ++j) { o[j][0] *= c0; o[j][1] *= c0; o[j][2] *= c1; o[j][3] *= c1; }
    // O += P V : 4 key blocks of 16 x 8 dim tiles of 8
#pragma unroll
    for (int kb = 0; kb < 4; ++kb) {
      const uint32_t a0 = pa[2 * kb][0], a1 = pa[2 * kb][1], a2 = pa[2 * kb + 1][0], a3 = pa[2 * kb + 1][1];
#pragma unroll
      for (int dp = 0; dp < 4; ++dp) {
        // ldmatrix.x4.trans: matrices (keys 16kb..+7, d 16dp..+7), (keys +8.., same d), (keys 16kb.., d +8), (keys +8, d +8)
        uint32_t v0, v1, v2, v3;
        const int mi = lane >> 3;
        const uint32_t addr = vs_base + (uint32_t)(((kb * 16 + (mi & 1) * 8 + (lane & 7)) * VPITCH + dp * 16 + (mi >> 1) * 8) * 2);
        ldsm_x4_trans(addr, v0, v1, v2, v3);
        mma_f16_16816_fa(o[2 * dp], a0, a1, a2, a3, v0, v1);
        mma_f16_16816_fa(o[2 * dp + 1], a0, a1, a2, a3, v2, v3);
      }
    }
    __syncthreads();   // every warp is done with this tile's buffer
  }
  const float i0 = l0 > 0.f ? 1.f / l0 : 0.f, i1 = l1 > 0.f ? 1.f / l1 : 0.f;
  const int r0 = q0 + warp * 16 + g, r1 = r0 + 8;
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    const int d = j * 8 + 2 * t4;
    const long long a0 = ((long long)b * T + r0) * H * AD + h * AD + d, a1 = ((long long)b * T + r1) * H * AD + h * AD + d;
    if (out) {
      if (r0 < T) *(float2*)(out + a0) = make_float2(o[j][0] * i0, o[j][1] * i0);
      if (r1 < T) *(float2*)(out + a1) = make_float2(o[j][2] * i1, o[j][3] * i1);
    }
    if (out16) {
      if (r0 < T) *(__half2*)(out16 + a0) = __floats2half2_rn(o[j][0] * i0, o[j][1] * i0);
      if (r1 < T) *(__half2*)(out16 + a1) = __floats2half2_rn(o[j][2] * i1, o[j][3] * i1);
    }
  }
}

}  // namespace

#define LAUNCH_CHECK(e)            \
  do {                             \
    IDX_CUDA(cudaGetLastError());  \
    (e)->launches++;               \
  } while (0)

void layernorm(idx_engine* e, const float* x, float* y, int B, int T, int C, const float* w, const float* b,
               float eps, const float* scale, const float* shift, int mod_stride, __half* y16) {
  const long long rows = (long long)B * T;
  launch_pdl(e, rownorm_kernel<0>, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, x, y, rows, T, C, w, b, eps, scale, shift, mod_stride, y16);
  LAUNCH_CHECK(e);
}
void rmsnorm_adaln(idx_engine* e, const float* x, float* y, int B, int T, int C, const float* nw, const float* mw,
                   const float* mb, int mod_stride, float eps, __half* y16) {
  const long long rows = (long long)B * T;
  launch_pdl(e, rownorm_kernel<1>, dim3((unsigned)((rows + 7) / 8)), dim3(256), 0, x, y, rows, T, C, nw, (const float*)nullptr, eps, mw, mb, mod_stride, y16);
  LAUNCH_CHECK(e);
}
void groupnorm1_mish(idx_engine* e, const float* x, float* y, int B, int T, int C, const float* w, const float* b,
                     float eps) {
  double* stats = (double*)e->arena.alloc(sizeof(double) * 2 * B);
  IDX_CUDA(cudaMemsetAsync(stats, 0, sizeof(double) * 2 * B, e->stream));
  const long long n_per = (long long)T * C;
  dim3 grid((unsigned)std::min<long long>(296, (n_per + 255) / 256), B);
  gn_stats_kernel<<<grid, 256, 0, e->stream>>>(x, stats, n_per);
  LAUNCH_CHECK(e);
  gn_apply_mish_kernel<<<grid, 256, 0, e->stream>>>(x, y, stats, n_per, C, w, b, eps);
  LAUNCH_CHECK(e);
}
void dwconv1d(idx_engine* e, const float* x, float* y, int B, int T, int C, const float* w, const float* b, int k) {
  dim3 grid((C + 127) / 128, T, B);
  dwconv_kernel<<<grid, 128, 0, e->stream>>>(x, y, T, C, w, b, k);
  LAUNCH_CHECK(e);
}
void nearest_interp(idx_engine* e, const float* x, float* y, int B, int Tin, int Tout, int C) {
  dim3 grid((C + 127) / 128, Tout, B);
  nearest_kernel<<<grid, 128, 0, e->stream>>>(x, y, Tin, Tout, C);
  LAUNCH_CHECK(e);
}
void embedding_rows(idx_engine* e, const float* table, const int* ids, float* out, int n, int C, int nrows) {
  dim3 grid((C + 127) / 128, n);
  embedding_kernel<<<grid, 128, 0, e->stream>>>(table, ids, out, C, nrows, e->dev_flag);
  LAUNCH_CHECK(e);
}
void swiglu(idx_engine* e, const float* ab, float* y, long long rows, int N, __half* y16) {
  launch_pdl(e, swiglu_kernel, dim3((unsigned)((rows * N + 255) / 256)), dim3(256), 0, ab, y, rows, N, y16);
  LAUNCH_CHECK(e);
}
void wn_gate(idx_engine* e, const float* xin, const float* g, int g_stride, float* y, int B, int T, int N, __half* y16) {
  dim3 grid((unsigned)(((long long)T * N + 255) / 256), 1, B);
  launch_pdl(e, wn_gate_kernel, grid, dim3(256), 0, xin, g, g_stride, y, T, N, y16);
  LAUNCH_CHECK(e);
}
void copy_cols(idx_engine* e, const float* src, int lds, float* dst, int ldo, int col0, long long rows, int C, __half* dst16) {
  launch_pdl(e, copy_cols_kernel, dim3((unsigned)((rows * C + 255) / 256)), dim3(256), 0, src, lds, dst, ldo, col0, rows, C, dst16);
  LAUNCH_CHECK(e);
}
void bcast_cols(idx_engine* e, const float* vec, float* dst, int ldo, int col0, int B, int T, int C) {
  dim3 grid((unsigned)(((long long)T * C + 255) / 256), 1, B);
  bcast_cols_kernel<<<grid, 256, 0, e->stream>>>(vec, dst, ldo, col0, T, C);
  LAUNCH_CHECK(e);
}
void silu_inplace(idx_engine* e, float* x, long long n) {
  silu_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(x, n);
  LAUNCH_CHECK(e);
}
void fill_zero(idx_engine* e, float* x, long long n) {
  launch_pdl(e, zero_kernel, dim3((unsigned)((n + 255) / 256)), dim3(256), 0, x, n);
  LAUNCH_CHECK(e);
}
void reflect_pad_rows(idx_engine* e, const float* x, float* y, int B, int T, int C, int left, int right, __half* y16) {
  const int Tout = T + left + right;
  dim3 grid((C + 127) / 128, Tout, B);
  launch_pdl(e, reflect_pad_kernel, grid, dim3(128), 0, x, y, T, C, left, Tout, y16);
  LAUNCH_CHECK(e);
}
void rope_table(idx_engine* e, float* tab, int T, int hd) {
  rope_table_kernel<<<T, 32, 0, e->stream>>>(tab, T, hd);
  LAUNCH_CHECK(e);
}
void attention_rope(idx_engine* e, const float* qkv, float* out, int B, int T, int H, const float* rope,
                    const int* lens, __half* out16) {
  static const bool unfused = getenv("IDX_ATTN_UNFUSED") != nullptr;
  if (gemm_default_backend(e) == 0 && lens == nullptr && !unfused) {
    // fused tensor-core flash attention: rotate/split once, then one kernel per layer
    const size_t mark = e->arena.off;
    const long long BH = (long long)B * H;
    __half* Qr = (__half*)e->arena.alloc((size_t)BH * T * AD * 2);
    __half* Kr = (__half*)e->arena.alloc((size_t)BH * T * AD * 2);
    __half* Vb = (__half*)e->arena.alloc((size_t)BH * T * AD * 2);
    launch_pdl(e, rope_split_fa_kernel, dim3(T, H, B), dim3(AD), 0, qkv, rope, Qr, Kr, Vb, T, H);
    LAUNCH_CHECK(e);
    flash_attention_mma(e, Qr, Kr, Vb, out, out16, B, T, H);
    e->arena.off = mark;
    return;
  }
  IDX_CHECK(out16 == nullptr, IDX_ERR_STATE, "attention_rope: an fp16 output exists only on the fused tensor-core path");
  if (gemm_default_backend(e) == 0 && lens == nullptr && T >= 128) {
    // tensor-core path: rotate/split -> S = Q K^T (tcgen05) -> row softmax -> O = P V (tcgen05) -> merge
    const size_t mark = e->arena.off;
    const int Tp = (T + 3) & ~3;
    const long long BH = (long long)B * H;
    float* Qr = e->arena.get<float>((size_t)BH * T * AD);
    float* Kr = e->arena.get<float>((size_t)BH * T * AD);
    float* Vt = e->arena.get<float>((size_t)BH * AD * Tp);
    float* S = e->arena.get<float>((size_t)BH * T * Tp);
    float* O = e->arena.get<float>((size_t)BH * T * AD);
    if (Tp != T) fill_zero(e, Vt, BH * AD * Tp);
    rope_split_kernel<<<dim3(T, H, B), AD, 0, e->stream>>>(qkv, rope, Qr, Kr, Vt, T, Tp, H);
    LAUNCH_CHECK(e);
    ConvGemm g1;
    g1.A = Qr; g1.B = (int)BH; g1.Tin = T; g1.K = AD; g1.Wk = Kr; g1.w_batch_stride = (long long)T * AD;
    g1.M = T; g1.N = T; g1.out = S; g1.ldo = Tp; g1.out_batch_stride = (long long)T * Tp;
    conv_gemm(e, g1);
    softmax_rows_kernel<<<(unsigned)((BH * T + 7) / 8), 256, 0, e->stream>>>(S, BH * T, T, Tp);
    LAUNCH_CHECK(e);
    ConvGemm g2;
    g2.A = S; g2.B = (int)BH; g2.Tin = T; g2.K = Tp; g2.Wk = Vt; g2.w_batch_stride = (long long)AD * Tp;
    g2.M = T; g2.N = AD; g2.out = O;
    conv_gemm(e, g2);
    heads_merge_kernel<<<dim3(T, H, B), AD, 0, e->stream>>>(O, out, T, H);
    LAUNCH_CHECK(e);
    e->arena.off = mark;
    return;
  }
  const int smem = 4 * AQ * AD * sizeof(float);
  if (!(e->attr_done & 8u)) {      // per engine = per device: function attributes live in the device's context
    IDX_CUDA(cudaFuncSetAttribute(attention_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, smem));
    e->attr_done |= 8u;
  }
  dim3 grid((T + AQ - 1) / AQ, H, B);
  attention_kernel<<<grid, 256, smem, e->stream>>>(qkv, out, T, H, rope, lens);
  LAUNCH_CHECK(e);
}
static bool fa5_on() {
  static const bool on = !(getenv("IDX_FA5") && atoi(getenv("IDX_FA5")) == 0);
  return on;
}
float flash_attention_q_scale() { return fa5_on() ? 0.125f * 1.4426950408889634f : 0.125f; }
void flash_attention_mma(idx_engine* e, const __half* Qr, const __half* Kr, const __half* Vb, float* out, __half* out16,
                         int B, int T, int H) {
  launch_pdl(e, flash_attn_tc_kernel, dim3((T + FQ - 1) / FQ, (unsigned)((long long)B * H)), dim3(128), 0, Qr, Kr, Vb, out, T, H, out16);
  LAUNCH_CHECK(e);
}
void flash_attention_split(idx_engine* e, const __half* Qr, const __half* Kr, const __half* Vb, float* out, __half* out16,
                           int B, int T, int H) {
  if (fa5_on()) {
    flash_attention_tc5(e, Qr, Kr, Vb, out, out16, B, T, H);
    return;
  }
  flash_attention_mma(e, Qr, Kr, Vb, out, out16, B, T, H);
}

// Diagnostic entry (tests): one flash attention over fp16 Qr | Kr | Vb [B*H][T][64] (what EPI_ROPE writes) through the
// chosen kernel: 1 = flash_attn_tc_kernel (mma.sync, scores in base e), 2 = fa5_kernel (tcgen05, scores in base 2).
extern "C" int idx_debug_flash_attention(idx_engine* e, const uint16_t* qkv16, int B, int T, int H, int kernel, float* out,
                                         uint16_t* out16) {
  IDX_API_BEGIN
  IDX_CHECK(e && qkv16 && (out || out16), IDX_ERR_ARG, "null argument");
  IDX_CHECK(B > 0 && T > 0 && H > 0, IDX_ERR_ARG, "idx_debug_flash_attention: B, T, H must be positive");
  IDX_CHECK(kernel == 1 || kernel == 2, IDX_ERR_ARG, "idx_debug_flash_attention: kernel 1 = mma.sync, 2 = tcgen05");
  IDX_CUDA(cudaSetDevice(e->device));
  const size_t n = (size_t)B * H * T * AD;       // elements of one of Qr / Kr / Vb, and of the output
  e->ensure_arena(2 * 3 * n + 4 * n + 2 * n + (4 << 10));
  e->arena.reset();
  __half* d_qkv = e->arena.get<__half>(3 * n);
  float* d_out = out ? e->arena.get<float>(n) : nullptr;
  __half* d_out16 = out16 ? e->arena.get<__half>(n) : nullptr;
  idx_to_device(e, d_qkv, qkv16, 3 * n * 2);
  if (kernel == 1) flash_attention_mma(e, d_qkv, d_qkv + n, d_qkv + 2 * n, d_out, d_out16, B, T, H);
  else flash_attention_tc5(e, d_qkv, d_qkv + n, d_qkv + 2 * n, d_out, d_out16, B, T, H);
  if (out) idx_from_device(e, out, d_out, n * 4);
  if (out16) idx_from_device(e, out16, d_out16, n * 2);
  IDX_CUDA(cudaStreamSynchronize(e->stream));
  IDX_API_END(e)
}

// Diagnostic entry (tests): attention_rope on fp32 qkv [B][T][3*H*64] with the RoPE table of the DiT; backend 1 = the SIMT
// fp32 attention_kernel (strict path), 0 = rope_split_fa_kernel + the mma.sync flash kernel (tf32-tail path).
extern "C" int idx_debug_attention_rope(idx_engine* e, const float* qkv, int B, int T, int H, int backend, float* out) {
  IDX_API_BEGIN
  IDX_CHECK(e && qkv && out, IDX_ERR_ARG, "null argument");
  IDX_CHECK(B > 0 && T > 0 && H > 0, IDX_ERR_ARG, "idx_debug_attention_rope: B, T, H must be positive");
  IDX_CHECK(backend == 0 || backend == 1, IDX_ERR_ARG, "idx_debug_attention_rope: backend 0 = tensor cores, 1 = SIMT fp32");
  IDX_CUDA(cudaSetDevice(e->device));
  const size_t nq = (size_t)B * T * 3 * H * AD, no = (size_t)B * T * H * AD, nt = (size_t)T * AD;
  // attention_rope's tensor-core path allocates Qr | Kr | Vb fp16 from the arena after these
  e->ensure_arena(4 * (nq + no + nt) + 2 * 3 * no + (8 << 10));
  e->arena.reset();
  float* d_qkv = e->arena.get<float>(nq);
  float* d_out = e->arena.get<float>(no);
  float* d_rope = e->arena.get<float>(nt);
  idx_to_device(e, d_qkv, qkv, nq * 4);
  rope_table(e, d_rope, T, AD);
  const int saved = e->gemm_backend;
  e->gemm_backend = backend;
  try {
    attention_rope(e, d_qkv, d_out, B, T, H, d_rope, nullptr);
  } catch (...) {
    e->gemm_backend = saved;
    throw;
  }
  e->gemm_backend = saved;
  idx_from_device(e, out, d_out, no * 4);
  IDX_CUDA(cudaStreamSynchronize(e->stream));
  IDX_API_END(e)
}
void cfg_euler(idx_engine* e, float* x, const float* v_cond, const float* v_uncond, float dt, float rate, int T,
               int C, int P) {
  launch_pdl(e, cfg_euler_kernel, dim3((unsigned)(((long long)T * C + 255) / 256)), dim3(256), 0, x, v_cond, v_uncond, dt, rate, T, C, P);
  LAUNCH_CHECK(e);
}
