// ops.cu — generic multi-tap GEMM (Conv1d / ConvTranspose1d / Linear on channels-last fp32) and
// layout helpers.  Two back ends behind conv_gemm():
//   * tcgen05 implicit GEMM (gemm_tc.cu): TMA-staged operands, TMEM accumulators, kind::tf32;
//   * a plain SIMT fp32 tile kernel (this file): bring-up / odd-shape path and the reference
//     the tensor-core path is tested against.  Both are CUDA; neither is a CPU fallback.
#include "ops.h"
#include <cstdlib>
#include <cstdio>

bool gemm_tc_supported(const ConvGemm& g);
void gemm_tc_launch(idx_engine* e, const ConvGemm& g);

namespace {

__device__ __forceinline__ float apply_act(float v, int act) {
  switch (act) {
    case ACT_GELU_ERF: return 0.5f * v * (1.f + erff(v * 0.70710678118654752f));
    case ACT_SILU: return v / (1.f + __expf(-v));
    case ACT_MISH: {
      float sp = (v > 20.f) ? v : log1pf(__expf(v));
      return v * tanhf(sp);
    }
    case ACT_GELU_TANH: {
      float u = 0.7978845608028654f * (v + 0.044715f * v * v * v);
      return 0.5f * v * (1.f + tanhf(u));
    }
    case ACT_RELU: return v > 0.f ? v : 0.f;
    default: return v;
  }
}

constexpr int BM = 64, BN = 64, BK = 16;

__global__ void __launch_bounds__(256) conv_gemm_simt_kernel(const ConvGemm g) {
  __shared__ float As[BK][BM + 4];
  __shared__ float Bs[BK][BN + 4];
  const int b = blockIdx.z;
  const int m0 = blockIdx.y * BM, n0 = blockIdx.x * BN;
  const int tid = threadIdx.x, tx = tid & 15, ty = tid >> 4;
  const long long abs_ = g.a_bcast ? 0 : (g.a_batch_stride ? g.a_batch_stride : (long long)g.Tin * g.K);
  const int lda = g.lda ? g.lda : g.K;
  const float* Ab = g.A + (long long)b * abs_;
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;

  const int ar = tid >> 2, ak = (tid & 3) * 4;   // A tile: row, k offset
  const int bk = tid >> 4, bn = (tid & 15) * 4;  // B tile: k, n offset
  for (int tap = 0; tap < g.taps; ++tap) {
    const int row = m0 + ar;
    int st = row + tap * g.dil - g.pad;
    if (g.reflect) {
      if (st < 0) st = -st;
      if (st >= g.Tin) st = 2 * (g.Tin - 1) - st;
    }
    const bool rvalid = row < g.M && st >= 0 && st < g.Tin;
    const float* arow = Ab + (long long)st * lda;
    for (int k0 = 0; k0 < g.K; k0 += BK) {
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const int kk = k0 + ak + i;
        As[ak + i][ar] = (rvalid && kk < g.K) ? __ldg(arow + kk) : 0.f;
      }
      if (g.W) {
        const int kk = k0 + bk;
        const float* wrow = g.W + ((long long)tap * g.K + kk) * g.N;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int n = n0 + bn + i;
          Bs[bk][bn + i] = (kk < g.K && n < g.N) ? __ldg(wrow + n) : 0.f;
        }
      } else {
        // K-major weights only (per-batch "weights" such as K / V^T of attention)
        const int kk = k0 + bk;
        const int ldw = g.ldw ? g.ldw : g.taps * g.K;
        const float* wb = g.Wk + (long long)b * g.w_batch_stride + (long long)tap * g.K + kk;
#pragma unroll
        for (int i = 0; i < 4; ++i) {
          const int n = n0 + bn + i;
          Bs[bk][bn + i] = (kk < g.K && n < g.N) ? __ldg(wb + (long long)n * ldw) : 0.f;
        }
      }
      __syncthreads();
#pragma unroll
      for (int k = 0; k < BK; ++k) {
        float a[4], w[4];
#pragma unroll
        for (int i = 0; i < 4; ++i) a[i] = As[k][ty * 4 + i];
#pragma unroll
        for (int j = 0; j < 4; ++j) w[j] = Bs[k][tx * 4 + j];
#pragma unroll
        for (int i = 0; i < 4; ++i)
#pragma unroll
          for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], w[j], acc[i][j]);
      }
      __syncthreads();
    }
  }
  const int ldo = g.ldo ? g.ldo : g.N;
  const long long obs = g.out_batch_stride ? g.out_batch_stride : (long long)g.M * g.N;
  const long long valid = g.out_valid ? g.out_valid : (long long)g.M * ldo;
  const int biasN = g.biasN ? g.biasN : g.N;
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    const int m = m0 + ty * 4 + i;
    if (m >= g.M) continue;
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int n = n0 + tx * 4 + j;
      if (n >= g.N) continue;
      const long long flat = g.out_off + (long long)m * ldo + n;
      if (flat < 0 || flat >= valid) continue;
      float v = acc[i][j];
      if (g.bias) v += __ldg(g.bias + (n % biasN));
      v = apply_act(v, g.act);
      if (g.colscale) v *= __ldg(g.colscale + n);
      if (g.rowscale) v *= __ldg(g.rowscale + (long long)b * g.M + m);
      const long long o = (long long)b * obs + flat;
      if (g.res) v += g.res[o];
      if (g.accum) v += g.out[o];
      g.out[o] = v * g.scale;
    }
  }
}

__global__ void transpose_kernel(const float* in, float* out, int R, int Cc) {
  // in [B][R][Cc] -> out [B][Cc][R]
  __shared__ float tile[32][33];
  const int b = blockIdx.z;
  const float* ib = in + (long long)b * R * Cc;
  float* ob = out + (long long)b * R * Cc;
  int c = blockIdx.x * 32 + threadIdx.x;
  for (int i = threadIdx.y; i < 32; i += 8) {
    int r = blockIdx.y * 32 + i;
    if (r < R && c < Cc) tile[i][threadIdx.x] = ib[(long long)r * Cc + c];
  }
  __syncthreads();
  int r = blockIdx.y * 32 + threadIdx.x;
  for (int i = threadIdx.y; i < 32; i += 8) {
    int cc = blockIdx.x * 32 + i;
    if (r < R && cc < Cc) ob[(long long)cc * R + r] = tile[threadIdx.x][i];
  }
}

}  // namespace


extern "C" int idx_set_option(idx_engine* e, const char* name, int value) {
  IDX_API_BEGIN
  IDX_CHECK(e && name, IDX_ERR_ARG, "null argument");
  const std::string n(name);
  if (n == "gemm_backend") {
    IDX_CHECK(value >= 0 && value <= 1, IDX_ERR_ARG, "gemm_backend: 0 = auto (tcgen05 tf32 where applicable), 1 = SIMT fp32");
    e->gemm_backend = value;       // per engine: another handle (another GPU, another thread) keeps its own
  } else if (n == "tail_f16") {
    IDX_CHECK(value >= 0 && value <= 1, IDX_ERR_ARG, "tail_f16: 1 = fp16 GEMM operands on the tensor-core path (default), 0 = tf32 over fp32 storage");
    e->tail_f16 = value;
  } else {
    throw IdxError(IDX_ERR_ARG, "unknown option: " + n);
  }
  IDX_API_END(e)
}

void conv_gemm(idx_engine* e, const ConvGemm& g) {
  IDX_CHECK((g.A || g.A16) && (g.out || g.out16) && g.M > 0 && g.N > 0 && g.K > 0, IDX_ERR_ARG, "conv_gemm: bad arguments");
  IDX_CHECK(g.epi == EPI_NONE || (g.A16 && g.Wk16), IDX_ERR_ARG, "conv_gemm: fused pair epilogues exist on the fp16 tensor-core path only");
  if (g.A16 && g.Wk16) {       // fp16 operands exist only for the tensor-core kernel
    IDX_CHECK(gemm_tc_supported(g), IDX_ERR_ARG, "conv_gemm: fp16 operands with a shape the tensor-core kernel does not take");
    gemm_tc_launch(e, g);
    return;
  }
  IDX_CHECK(g.A != nullptr, IDX_ERR_ARG, "conv_gemm: fp32 operand missing");
  static const bool force_simt = getenv("IDX_FORCE_SIMT") != nullptr;
  if (e->force_backend == 2) {
    IDX_CHECK(g.Wk && !g.reflect, IDX_ERR_ARG, "conv_gemm: tensor-core path not applicable");
    gemm_tc_launch(e, g);
    return;
  }
  if (!force_simt && e->force_backend != 1 && !(e->force_backend == 0 && e->gemm_backend == 1) && g.Wk &&
      gemm_tc_supported(g)) {
    gemm_tc_launch(e, g);
    return;
  }
  IDX_CHECK(g.W || g.Wk, IDX_ERR_ARG, "conv_gemm: weights missing");
  IDX_CHECK(g.W || true, IDX_ERR_ARG, "");
  dim3 grid((g.N + BN - 1) / BN, (g.M + BM - 1) / BM, g.B);
  conv_gemm_simt_kernel<<<grid, 256, 0, e->stream>>>(g);
  IDX_CUDA(cudaGetLastError());
  e->launches++;
}

void transpose_bct_to_btc(idx_engine* e, const float* in, float* out, int B, int C, int T) {
  dim3 grid((T + 31) / 32, (C + 31) / 32, B);
  transpose_kernel<<<grid, dim3(32, 8), 0, e->stream>>>(in, out, C, T);
  IDX_CUDA(cudaGetLastError());
  e->launches++;
}
void transpose_btc_to_bct(idx_engine* e, const float* in, float* out, int B, int T, int C) {
  dim3 grid((C + 31) / 32, (T + 31) / 32, B);
  transpose_kernel<<<grid, dim3(32, 8), 0, e->stream>>>(in, out, T, C);
  IDX_CUDA(cudaGetLastError());
  e->launches++;
}

// ------------------------------------------------------------------------ packed weights --
namespace {
__global__ void pack_conv_rows_kernel(const float* w, float* wsimt, float* wk, int Co, int Ci, int k, int row0) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  long long n = (long long)Co * Ci * k;
  if (i >= n) return;
  int kk = i % k;
  int ci = (i / k) % Ci;
  int co = i / ((long long)k * Ci);
  float v = w[(long long)row0 * Ci * k + i];
  wsimt[((long long)kk * Ci + ci) * Co + co] = v;
  wk[(long long)co * k * Ci + (long long)kk * Ci + ci] = v;
}
}  // namespace

float* WeightPool::alloc(size_t n) {
  float* p = nullptr;
  IDX_CUDA(cudaMalloc((void**)&p, n * sizeof(float)));
  owned.push_back(p);
  return p;
}
void WeightPool::release() {
  for (void* p : owned) cudaFree(p);
  owned.clear();
}

PackedW pack_conv1d(idx_engine* e, WeightPool& pool, const std::string& name, int dil, int row0, int rows) {
  const DevTensor& w = e->W(name + ".weight");
  IDX_CHECK(w.shape.size() == 3, IDX_ERR_ARG, name + ".weight must be [Co][Ci][k] (fold weight norm first)");
  PackedW p;
  const int Co = (int)w.shape[0];
  p.N = rows < 0 ? Co - row0 : rows;
  IDX_CHECK(row0 >= 0 && row0 + p.N <= Co, IDX_ERR_ARG, name + ": bad row range");
  p.K = (int)w.shape[1]; p.taps = (int)w.shape[2]; p.dil = dil;
  const size_t n = (size_t)p.N * p.K * p.taps;
  p.wsimt = pool.alloc(n);
  p.wk = pool.alloc(n);
  pack_conv_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>((const float*)w.d, p.wsimt, p.wk, p.N, p.K, p.taps, row0);
  IDX_CUDA(cudaGetLastError());
  if (e->has(name + ".bias")) p.bias = e->Wf(name + ".bias") + row0;
  return p;
}

PackedW pack_linear(idx_engine* e, WeightPool& pool, const std::string& name, int row0, int rows, bool with_bias) {
  const DevTensor& w = e->W(name + ".weight");
  IDX_CHECK(w.shape.size() == 2 || (w.shape.size() == 3 && w.shape[2] == 1), IDX_ERR_ARG, name + ".weight must be [N][K]");
  PackedW p;
  const int N = (int)w.shape[0];
  p.N = rows < 0 ? N - row0 : rows;
  IDX_CHECK(row0 >= 0 && row0 + p.N <= N, IDX_ERR_ARG, name + ": bad row range");
  p.K = (int)w.shape[1]; p.taps = 1;
  const size_t n = (size_t)p.N * p.K;
  p.wsimt = pool.alloc(n);
  p.wk = pool.alloc(n);
  pack_conv_rows_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>((const float*)w.d, p.wsimt, p.wk, p.N, p.K, 1, row0);
  IDX_CUDA(cudaGetLastError());
  if (with_bias && e->has(name + ".bias")) p.bias = e->Wf(name + ".bias") + row0;
  return p;
}

ConvGemm gemm_of(const PackedW& w, const float* A, int B, int T, float* out) {
  ConvGemm g;
  g.A = A; g.B = B; g.Tin = T; g.K = w.K;
  g.W = w.wsimt; g.Wk = w.wk;
  g.taps = w.taps; g.dil = w.dil; g.pad = (w.taps * w.dil - w.dil) / 2;
  g.M = T; g.N = w.N; g.bias = w.bias; g.out = out;
  return g;
}

ConvGemm gemm_of16(const PackedW& w, const __half* A16, int B, int T, float* out) {
  ConvGemm g = gemm_of(w, nullptr, B, T, out);
  IDX_CHECK(w.wk16, IDX_ERR_STATE, "gemm_of16: the weight has no fp16 copy (pack_half)");
  g.A16 = A16; g.Wk16 = w.wk16;
  return g;
}

namespace {
__global__ void to_half_kernel(const float* __restrict__ x, __half* __restrict__ y, long long n) {
  pdl_wait();
  long long i = ((long long)blockIdx.x * blockDim.x + threadIdx.x) * 2;
  if (i + 1 < n) *(__half2*)(y + i) = __floats2half2_rn(x[i], x[i + 1]);
  else if (i < n) y[i] = __float2half_rn(x[i]);
}
}  // namespace

void to_half(idx_engine* e, const float* x, __half* y, long long n) {
  if (n <= 0) return;
  launch_pdl(e, to_half_kernel, dim3((unsigned)((n / 2 + 256) / 256)), dim3(256), 0, x, y, n);
  e->launches++;
}

namespace {
__global__ void interleave_half_kernel(const float* __restrict__ wk, __half* __restrict__ dst, int N, long long KT) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)N * KT) return;
  const int r = (int)(i / KT);
  const long long k = i % KT;
  const int src = (r & 1) ? (N / 2 + (r >> 1)) : (r >> 1);
  dst[i] = __float2half_rn(wk[(long long)src * KT + k]);
}
__global__ void interleave_bias_kernel(const float* __restrict__ b, float* __restrict__ dst, int N) {
  const int r = blockIdx.x * blockDim.x + threadIdx.x;
  if (r < N) dst[r] = b[(r & 1) ? (N / 2 + (r >> 1)) : (r >> 1)];
}
}  // namespace

__half* pack_half_interleaved(idx_engine* e, WeightPool& pool, const PackedW& w, float** bias_out) {
  IDX_CHECK(w.wk && w.N % 2 == 0, IDX_ERR_ARG, "pack_half_interleaved: needs a K-major weight with an even row count");
  const long long KT = (long long)w.K * w.taps, n = (long long)w.N * KT;
  __half* dst = (__half*)pool.alloc((size_t)(n + 1) / 2 + 4);
  interleave_half_kernel<<<(unsigned)((n + 255) / 256), 256, 0, e->stream>>>(w.wk, dst, w.N, KT);
  IDX_CUDA(cudaGetLastError());
  if (bias_out) {
    *bias_out = nullptr;
    if (w.bias) {
      *bias_out = pool.alloc(w.N);
      interleave_bias_kernel<<<(w.N + 255) / 256, 256, 0, e->stream>>>(w.bias, *bias_out, w.N);
      IDX_CUDA(cudaGetLastError());
    }
  }
  return dst;
}

void pack_half(idx_engine* e, WeightPool& pool, PackedW& w) {
  if (w.wk16 || !w.wk) return;
  const size_t n = (size_t)w.N * w.K * w.taps;
  w.wk16 = (__half*)pool.alloc((n + 1) / 2 + 4);
  to_half(e, w.wk, w.wk16, (long long)n);
}

bool tail_half(const idx_engine* e) {
  static const bool off = getenv("IDX_TAIL_F16") && atoi(getenv("IDX_TAIL_F16")) == 0;
  return !off && e->tail_f16 && e->gemm_backend == 0 && e->force_backend == 0;
}

namespace {
__global__ void kmajor_to_simt_kernel(const float* wk, float* ws, int N, int KT) {
  long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)N * KT) return;
  int n = (int)(i / KT), k = (int)(i % KT);
  ws[(long long)k * N + n] = wk[i];
}
}  // namespace

// Diagnostic entry (tests): run one multi-tap GEMM through a chosen back end.
// wk is the K-major weight [N][taps*K]; out is [B][out_rows][ldo]-shaped via (out_off, ldo, out_valid).
extern "C" int idx_debug_conv_gemm(idx_engine* e, const float* A, int B, int Tin, int K, const float* wk, int taps,
                                   int dil, int pad, int M, int N, const float* bias, int biasN, int act,
                                   const float* res, int accum, float scale, long long out_off, int ldo,
                                   long long out_valid, long long out_elems_per_batch, int backend, float* out) {
  IDX_API_BEGIN
  IDX_CHECK(e && A && wk && out, IDX_ERR_ARG, "null argument");
  IDX_CUDA(cudaSetDevice(e->device));
  const size_t na = (size_t)B * Tin * K, nw = (size_t)N * taps * K, no = (size_t)B * out_elems_per_batch;
  e->ensure_arena(4 * (2 * na + 3 * nw + 2 * no + (size_t)N) + (1 << 20));
  e->arena.reset();
  float* dA = e->arena.get<float>(na);
  float* dWk = e->arena.get<float>(nw);
  float* dWs = e->arena.get<float>(nw);
  float* dOut = e->arena.get<float>(no);
  float* dRes = res ? e->arena.get<float>(no) : nullptr;
  float* dBias = bias ? e->arena.get<float>(biasN ? biasN : N) : nullptr;
  idx_to_device(e, dA, A, na * 4);
  idx_to_device(e, dWk, wk, nw * 4);
  idx_to_device(e, dOut, out, no * 4);   // initial contents matter for accum
  if (res) idx_to_device(e, dRes, res, no * 4);
  if (bias) idx_to_device(e, dBias, bias, (size_t)(biasN ? biasN : N) * 4);
  kmajor_to_simt_kernel<<<(unsigned)((nw + 255) / 256), 256, 0, e->stream>>>(dWk, dWs, N, taps * K);
  IDX_CUDA(cudaGetLastError());
  ConvGemm g;
  g.A = dA; g.B = B; g.Tin = Tin; g.K = K; g.W = dWs; g.Wk = dWk; g.taps = taps; g.dil = dil; g.pad = pad;
  g.M = M; g.N = N; g.bias = dBias; g.biasN = biasN; g.act = act; g.res = dRes; g.accum = accum; g.scale = scale;
  g.out = dOut; g.out_off = out_off; g.ldo = ldo; g.out_valid = out_valid; g.out_batch_stride = out_elems_per_batch;
  if (backend == 3) {          // fp16 operands on the tensor cores: convert A and the K-major weights on the device
    __half* dA16 = (__half*)e->arena.get<float>(na / 2 + 4);
    __half* dW16 = (__half*)e->arena.get<float>(nw / 2 + 4);
    to_half(e, dA, dA16, (long long)na);
    to_half(e, dWk, dW16, (long long)nw);
    g.A16 = dA16; g.Wk16 = dW16;
    backend = 0;
  }
  e->force_backend = backend;
  try {
    conv_gemm(e, g);
    // timing loop (diagnostics): env IDX_GEMM_REPS=n repeats the launch between CUDA events
    static const int reps = getenv("IDX_GEMM_REPS") ? atoi(getenv("IDX_GEMM_REPS")) : 0;
    if (reps > 0) {
      cudaEvent_t a, b2;
      IDX_CUDA(cudaEventCreate(&a)); IDX_CUDA(cudaEventCreate(&b2));
      IDX_CUDA(cudaEventRecord(a, e->stream));
      for (int i = 0; i < reps; ++i) conv_gemm(e, g);
      IDX_CUDA(cudaEventRecord(b2, e->stream));
      IDX_CUDA(cudaEventSynchronize(b2));
      float ms = 0; IDX_CUDA(cudaEventElapsedTime(&ms, a, b2));
      fprintf(stderr, "[idx_debug_conv_gemm] backend %d B=%d M=%d N=%d K=%d taps=%d: %.2f us/launch, %.1f TFLOP/s\n", backend, B,
              M, N, K, taps, ms * 1000.0 / reps, 2.0 * B * M * (double)N * K * taps / (ms / reps * 1e-3) / 1e12);
      cudaEventDestroy(a); cudaEventDestroy(b2);
    }
  } catch (...) {
    e->force_backend = 0;
    throw;
  }
  e->force_backend = 0;
  idx_from_device(e, out, dOut, no * 4);
  IDX_CUDA(cudaStreamSynchronize(e->stream));
  IDX_API_END(e)
}

// Diagnostic entry (tests): one fp16 tensor-core GEMM with a fused pair epilogue, prepared the way the DiT / WaveNet
// prepare theirs: fp16 images by to_half, SwiGLU / gate weights and bias interleaved by pack_half_interleaved, the RoPE
// table by rope_table.  wk [N][taps*K] and bias [N] are in the module's row order (w1 | w3, a | c, q | k | v).
extern "C" int idx_debug_gemm_pair_epilogue(idx_engine* e, const float* A, int B, int Tin, int K, const float* wk, int taps,
                                            int dil, int pad, int M, int N, const float* bias, int epi, const float* aux,
                                            int aux_stride, float scale, uint16_t* out16) {
  IDX_API_BEGIN
  IDX_CHECK(e && A && wk && out16, IDX_ERR_ARG, "null argument");
  IDX_CHECK(B > 0 && Tin > 0 && K > 0 && taps > 0 && M > 0 && N > 0, IDX_ERR_ARG, "idx_debug_gemm_pair_epilogue: bad sizes");
  IDX_CHECK(epi == EPI_SWIGLU || epi == EPI_WNGATE || epi == EPI_ROPE, IDX_ERR_ARG,
            "idx_debug_gemm_pair_epilogue: epi 1 = SwiGLU, 2 = WaveNet gate, 3 = RoPE");
  if (epi == EPI_ROPE)
    IDX_CHECK(aux_stride > 0 && N == 3 * 64 * aux_stride, IDX_ERR_ARG, "EPI_ROPE: N must be 3 * 64 * heads (aux_stride = heads)");
  if (epi == EPI_WNGATE)
    IDX_CHECK(aux && (aux_stride == 0 || aux_stride >= N), IDX_ERR_ARG,
              "EPI_WNGATE: needs the gate g [N] (aux_stride 0: shared by every batch entry) or [B][aux_stride >= N]");
  IDX_CUDA(cudaSetDevice(e->device));
  const size_t na = (size_t)B * Tin * K, nw = (size_t)N * taps * K;
  const size_t no = (epi == EPI_ROPE) ? (size_t)B * M * N : (size_t)B * M * (N / 2);
  const size_t ng = (epi == EPI_WNGATE) ? (size_t)(B - 1) * aux_stride + N : 0;
  const size_t nt = (epi == EPI_ROPE) ? (size_t)M * 64 : 0;
  e->ensure_arena(4 * (na + nw + N + ng + nt) + 2 * (na + nw + no) + (8 << 10));
  e->arena.reset();
  float* dA = e->arena.get<float>(na);
  float* dWk = e->arena.get<float>(nw);
  float* dBias = bias ? e->arena.get<float>(N) : nullptr;
  __half* dA16 = e->arena.get<__half>(na);
  __half* dOut = e->arena.get<__half>(no);
  idx_to_device(e, dA, A, na * 4);
  idx_to_device(e, dWk, wk, nw * 4);
  if (bias) idx_to_device(e, dBias, bias, (size_t)N * 4);
  to_half(e, dA, dA16, (long long)na);
  ConvGemm g;
  g.A16 = dA16; g.B = B; g.Tin = Tin; g.K = K; g.taps = taps; g.dil = dil; g.pad = pad; g.M = M; g.N = N;
  g.epi = epi; g.out16 = dOut; g.aux_stride = aux_stride; g.scale = scale;
  struct PoolGuard {           // the interleaved weights live outside the arena, like the model's
    WeightPool p;
    ~PoolGuard() { cudaDeviceSynchronize(); p.release(); }
  } pool;
  if (epi == EPI_ROPE) {
    __half* dW16 = e->arena.get<__half>(nw);
    to_half(e, dWk, dW16, (long long)nw);
    float* tab = e->arena.get<float>(nt);
    rope_table(e, tab, M, 64);
    g.Wk16 = dW16; g.bias = dBias; g.aux = tab;
  } else {
    PackedW w;
    w.wk = dWk; w.N = N; w.K = K; w.taps = taps; w.dil = dil; w.bias = dBias;
    float* bias_i = nullptr;
    g.Wk16 = pack_half_interleaved(e, pool.p, w, &bias_i);
    g.bias = bias_i;
    if (epi == EPI_WNGATE) {
      float* dG = e->arena.get<float>(ng);
      idx_to_device(e, dG, aux, ng * 4);
      g.aux = dG;
    }
  }
  conv_gemm(e, g);
  idx_from_device(e, out16, dOut, no * 2);
  IDX_CUDA(cudaStreamSynchronize(e->stream));
  IDX_API_END(e)
}
