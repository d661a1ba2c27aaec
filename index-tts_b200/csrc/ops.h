// ops.h — generic building blocks shared by the vocoder / s2mel / codec paths.
// Activations are channels-last fp32: a [B][T][C] tensor is a row-major [B*T, C] matrix whose
// rows are time steps, so every Conv1d / Linear is a (multi-tap) GEMM with K = C contiguous.
#pragma once
#include "engine.h"
#include <cuda_fp16.h>
#include <cstdlib>
#include <string>
#include <utility>
#include <vector>

enum { EPI_NONE = 0, EPI_SWIGLU = 1, EPI_WNGATE = 2, EPI_ROPE = 3 };
enum { ACT_NONE = 0, ACT_GELU_ERF = 1, ACT_SILU = 2, ACT_MISH = 3, ACT_GELU_TANH = 4, ACT_RELU = 5 };

// D[b][m][j] = epi( sum_{tap} sum_{k} A[b][m + tap*dil - pad][k] * W[tap][k][j] )
// rows of A outside [0, Tin) read as zero (Conv1d zero padding) or are reflected (SConv1d).
struct ConvGemm {
  const float* A = nullptr;   // [B][Tin][K]
  int B = 1, Tin = 0, K = 0;
  long long a_batch_stride = 0;  // elements; 0 → Tin*K
  int a_bcast = 0;               // 1 → every batch entry reads the same A (stride 0)
  int lda = 0;                   // row stride of A in elements; 0 → K
  const float* W = nullptr;   // [taps][K][N]  (N contiguous)  — SIMT layout
  const float* Wk = nullptr;  // [N][taps*K]   (K contiguous)  — tensor-core layout (optional)
  // fp16 operand path (tcgen05 kind::f16): both set -> the tensor-core kernel reads these instead of A / Wk (same shapes,
  // strides given in ELEMENTS as for the fp32 operands).  Written by the producing kernel of A / converted once at init.
  const __half* A16 = nullptr;
  const __half* Wk16 = nullptr;
  // fused pair epilogues of the tensor-core kernel (fp16 results straight into the operand of the next GEMM / the attention):
  //   EPI_SWIGLU : columns (2j, 2j+1) = (w1 x, w3 x)_j (weight rows interleaved at pack time) -> out16[row][j] = silu(a) * b
  //   EPI_WNGATE : columns (2j, 2j+1) = (a_j, c_j) of the WaveNet in_layer -> out16[row][j] = tanh(a + g[b][j]) * sigmoid(c + g[b][N/2 + j])
  //   EPI_ROPE   : columns = q | k | v of the fused wqkv: interleaved-pair RoPE (table aux [T][32][2]) on q (x 1/8) and k, v as is,
  //                written head-major as fp16 Qr | Kr | Vb [B*H][T][64] (out16 = Qr; the three tensors are contiguous)
  int epi = 0;
  __half* out16 = nullptr;
  const float* aux = nullptr;      // EPI_WNGATE: g [B][aux_stride] ; EPI_ROPE: rope table
  int aux_stride = 0;              // EPI_WNGATE: floats per batch entry of g ; EPI_ROPE: heads
  long long w_batch_stride = 0;  // elements between the Wk matrices of consecutive batch entries (0: shared)
  int ldw = 0;                   // row stride of Wk in elements; 0 → taps*K
  int taps = 1, dil = 1, pad = 0, reflect = 0;
  int M = 0;                  // output rows per batch
  int N = 0;
  const float* bias = nullptr;
  int biasN = 0;              // bias index = j % biasN (0 → N)
  int act = ACT_NONE;
  const float* res = nullptr;   // optional residual, indexed like out
  const float* rowscale = nullptr;  // optional per-(b,m) multiplier (masks), [B][M]
  const float* colscale = nullptr;  // optional per-column multiplier applied to (acc+bias) (layer scale)
  int accum = 0;              // out = scale * (v + out_old)
  float scale = 1.f;
  float* out = nullptr;
  long long out_batch_stride = 0;  // elements; 0 → M*N
  long long out_off = 0;           // flat offset added to m*ldo + j (may be negative: ConvTranspose)
  long long out_valid = 0;         // writes only where 0 <= flat < out_valid (0 → M*ldo)
  int ldo = 0;                     // 0 → N
};

void conv_gemm(idx_engine* e, const ConvGemm& g);
inline int gemm_default_backend(const idx_engine* e) { return e->gemm_backend; }   // 0 auto (tcgen05), 1 SIMT fp32

// [B][C][T] <-> [B][T][C]
void transpose_bct_to_btc(idx_engine* e, const float* in, float* out, int B, int C, int T);
void transpose_btc_to_bct(idx_engine* e, const float* in, float* out, int B, int T, int C);

// ------------------------------------------------------------- programmatic dependent launch --
// The tail is ~4000 short kernels per utterance.  Kernels launched through launch_pdl() carry the programmatic-stream-
// serialization attribute: their CTAs may be scheduled while the previous kernel of the stream is still draining, so launch
// latency and the kernel's own prologue (barrier init, TMEM allocation, descriptor prefetch) overlap with it.  Such a kernel
// executes pdl_wait() — every thread — before it touches global memory, and pdl_trigger() as soon as it has nothing left that
// the NEXT kernel could disturb (the next kernel's own pdl_wait still waits for this grid to finish completely).
#ifdef __CUDACC__
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }
__device__ __forceinline__ void pdl_trigger() { asm volatile("griddepcontrol.launch_dependents;" ::: "memory"); }
template <typename... KArgs, typename... Args>
inline void launch_pdl(idx_engine* e, void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, Args&&... args) {
  static const bool off = getenv("IDX_PDL") && atoi(getenv("IDX_PDL")) == 0;
  cudaLaunchConfig_t cfg = {};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = e->stream;
  cudaLaunchAttribute attr[1];
  attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
  attr[0].val.programmaticStreamSerializationAllowed = 1;
  cfg.attrs = attr; cfg.numAttrs = off ? 0 : 1;
  IDX_CUDA(cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...));
}
#endif

// ---------------------------------------------------------------- normalisation / pointwise --
// y = LayerNorm(x) [* w + b] [ * (1 + scale[b]) + shift[b] ]   rows of C, x/y [B][T][C]
void layernorm(idx_engine* e, const float* x, float* y, int B, int T, int C, const float* w,
               const float* b, float eps, const float* scale, const float* shift, int mod_stride, __half* y16 = nullptr);
// y = mw[b] * (x * rsqrt(mean(x^2)+eps) * nw) + mb[b]          (AdaptiveLayerNorm over RMSNorm)
void rmsnorm_adaln(idx_engine* e, const float* x, float* y, int B, int T, int C, const float* nw,
                   const float* mw, const float* mb, int mod_stride, float eps, __half* y16 = nullptr);
// GroupNorm(1 group) over each sample's [T][C] block, affine per channel, followed by Mish
void groupnorm1_mish(idx_engine* e, const float* x, float* y, int B, int T, int C, const float* w,
                     const float* b, float eps);
// depthwise Conv1d (groups = C), zero padding (k-1)/2; w [C][k]
void dwconv1d(idx_engine* e, const float* x, float* y, int B, int T, int C, const float* w,
              const float* b, int k);
// y[b][t][:] = x[b][src(t)][:], src(t) = min(floor(t * Tin/Tout), Tin-1)  (F.interpolate nearest)
void nearest_interp(idx_engine* e, const float* x, float* y, int B, int Tin, int Tout, int C);
// out[t][:] = table[ids[t]][:]
void embedding_rows(idx_engine* e, const float* table, const int* ids, float* out, int n, int C, int nrows);
// y = silu(a) * b where ab [rows][2*N] holds a | b side by side
void swiglu(idx_engine* e, const float* ab, float* y, long long rows, int N, __half* y16 = nullptr);
// y = tanh(a + ga[b]) * sigmoid(c + gc[b]),  xin [B][T][2N] = a | c ; g [B][*] with stride
void wn_gate(idx_engine* e, const float* xin, const float* g, int g_stride, float* y, int B, int T, int N, __half* y16 = nullptr);
// copy a [rows][C] block into columns [col0, col0+C) of a [rows][ldo] matrix (concat by columns)
void copy_cols(idx_engine* e, const float* src, int lds, float* dst, int ldo, int col0, long long rows, int C, __half* dst16 = nullptr);
// broadcast a per-batch vector [B][C] over T rows into columns of dst
void bcast_cols(idx_engine* e, const float* vec, float* dst, int ldo, int col0, int B, int T, int C);
// y = silu(x)
void silu_inplace(idx_engine* e, float* x, long long n);
// RoPE table [T][hd/2][2] (cos, sin), base 1e4 (gpt_fast/model.py:336-346)
void rope_table(idx_engine* e, float* tab, int T, int hd);
// full (non-causal) attention with key-length mask and interleaved-pair RoPE on q,k.
// qkv [B][T][3*H*64] (q | k | v), out [B][T][H*64]; lens [B] valid keys (device ints) or null
// out16 (tensor-core flash path only): the result as fp16 (the operand of the output projection); out may then be null
void attention_rope(idx_engine* e, const float* qkv, float* out, int B, int T, int H, const float* rope,
                    const int* lens, __half* out16 = nullptr);
// x[b][t][c] (+)= ... CFG + Euler: x += dt * ((1+r) * v[0] - r * v[1]); rows t < P zeroed. x,v: [T][C]
void cfg_euler(idx_engine* e, float* x, const float* v_cond, const float* v_uncond, float dt, float rate,
               int T, int C, int P);
void fill_zero(idx_engine* e, float* x, long long n);
// y[b][i][:] = x[b][reflect(i - left)][:], i in [0, T + left + right)   (F.pad mode='reflect')
void reflect_pad_rows(idx_engine* e, const float* x, float* y, int B, int T, int C, int left, int right, __half* y16 = nullptr);

// ------------------------------------------------------------------------ packed weights --
struct PackedW {
  float* wsimt = nullptr;  // [taps][K][N]
  float* wk = nullptr;     // [N][taps*K]
  __half* wk16 = nullptr;  // [N][taps*K] fp16 copy of wk (made on demand by pack_half)
  const float* bias = nullptr;
  int N = 0, K = 0, taps = 1, dil = 1;
};
struct WeightPool {
  std::vector<void*> owned;
  float* alloc(size_t n);
  void release();
};
// nn.Linear weight [N][K] (optionally only rows [row0, row0+rows))
PackedW pack_linear(idx_engine* e, WeightPool& pool, const std::string& name, int row0 = 0, int rows = -1,
                    bool with_bias = true);
// nn.Conv1d weight [Co][Ci][k] (optionally only output rows [row0, row0+rows))
PackedW pack_conv1d(idx_engine* e, WeightPool& pool, const std::string& name, int dil = 1, int row0 = 0,
                    int rows = -1);
// convenience: D = A·W^T (+bias) for a channels-last activation with optional epilogue fields preset in g
ConvGemm gemm_of(const PackedW& w, const float* A, int B, int T, float* out);
// same GEMM with fp16 operands: A16 is the fp16 image of the activation (the fp32 pointer may be null)
ConvGemm gemm_of16(const PackedW& w, const __half* A16, int B, int T, float* out);
// fp16 copy of a K-major weight matrix (w.wk must exist); idempotent
void pack_half(idx_engine* e, WeightPool& pool, PackedW& w);
// fp16 K-major copy of w.wk with the two halves of the output rows interleaved (row 2j = row j, row 2j+1 = row N/2 + j): the
// weight layout of the EPI_SWIGLU / EPI_WNGATE pair epilogues; bias_out (optional) receives the bias interleaved the same way
__half* pack_half_interleaved(idx_engine* e, WeightPool& pool, const PackedW& w, float** bias_out);
// the fused flash attention on already rotated / split fp16 tensors Qr | Kr | Vb [B*H][T][64] (what EPI_ROPE writes)
void flash_attention_split(idx_engine* e, const __half* Qr, const __half* Kr, const __half* Vb, float* out, __half* out16,
                           int B, int T, int H);
// scale EPI_ROPE must apply to q for flash_attention_split: 1/8, times log2(e) when the tcgen05 kernel (exp2 softmax) is on
float flash_attention_q_scale();
// the same on mma.sync (nn_ops.cu: flash_attn_tc_kernel, scores in base e: q pre-scaled by 1/8 only)
void flash_attention_mma(idx_engine* e, const __half* Qr, const __half* Kr, const __half* Vb, float* out, __half* out16,
                         int B, int T, int H);
// the same on tcgen05 (gemm_tc.cu: S and O in tensor memory, P fed back as a tensor-memory operand)
void flash_attention_tc5(idx_engine* e, const __half* Qr, const __half* Kr, const __half* Vb, float* out, __half* out16,
                         int B, int T, int H);
// fp32 -> fp16 (round to nearest), n elements
void to_half(idx_engine* e, const float* x, __half* y, long long n);
// true when the engine runs the tail with fp16 GEMM operands (tensor-core back end and not disabled by IDX_TAIL_F16=0)
bool tail_half(const idx_engine* e);
