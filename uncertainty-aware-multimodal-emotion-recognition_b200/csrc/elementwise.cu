// Memory-bound helpers: activation backward + bias gradient, dropout, scorer dot, layout moves, small combiners.
// All are streaming kernels: coalesced along the innermost dimension, float4 where the shape allows,
// grids sized from the data (>= 2 waves of 148 SMs at the benchmark shapes).
#include <cuda_bf16.h>
#include <cuda_fp16.h>

#include "common.cuh"

namespace deer {

// ------------------------------------------------------------------ bias/act backward
__global__ void __launch_bounds__(256) bias_act_bwd_kernel(const float* __restrict__ dy, long long ld_dy,
                                                           const float* __restrict__ y, long long ld_y,
                                                           float* __restrict__ dz, long long ld_dz,
                                                           float* __restrict__ dbias, int M, int N, int act,
                                                           int rows_per_block) {
  DEER_PDL_ENTRY();
  __shared__ float red[8][33];
  const int n = blockIdx.x * 32 + threadIdx.x;
  const int r0 = blockIdx.y * rows_per_block;
  const int r1 = min(M, r0 + rows_per_block);
  float s = 0.f;
  if (n < N) {
    for (int m = r0 + threadIdx.y; m < r1; m += 8) {
      float g = dy[(long long)m * ld_dy + n];
      if (act != DEER_ACT_NONE) g *= act_grad_from_out(y[(long long)m * ld_y + n], act);
      if (dz) dz[(long long)m * ld_dz + n] = g;
      s += g;
    }
  }
  if (dbias) {
    red[threadIdx.y][threadIdx.x] = s;
    __syncthreads();
    if (threadIdx.y == 0 && n < N) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; i++) t += red[i][threadIdx.x];
      atomicAdd(dbias + n, t);
    }
  }
}

// ------------------------------------------------------------------ attention-scorer backward (Linear-Tanh-Linear(1))
// s[m] = w2 . hidden[m,:] + b2 with hidden = tanh(.): from ds [M] in ONE pass over hidden
//   dz[m,j] = ds[m] w2[j] (1 - hidden[m,j]^2)   (gradient at the first Linear's output; may overwrite `hidden`)
//   dw2[j] += sum_m ds[m] hidden[m,j],  db1[j] += sum_m dz[m,j],  db2 += sum_m ds[m]
// (as rowdot_bwd followed by bias_act_bwd the [M,Hd] intermediate was written and read once more).
__global__ void __launch_bounds__(256) scorer_bwd_kernel(const float* __restrict__ ds, const float* __restrict__ hidden,
                                                         const float* __restrict__ w2, float* __restrict__ dz,
                                                         float* __restrict__ dw2, float* __restrict__ db1,
                                                         float* __restrict__ db2, const float* __restrict__ dz_row_scale,
                                                         int M, int N, int rows_per_block) {
  DEER_PDL_ENTRY();
  __shared__ float red[2][8][33];
  const int n = blockIdx.x * 32 + threadIdx.x;
  const int r0 = blockIdx.y * rows_per_block;
  const int r1 = min(M, r0 + rows_per_block);
  float sw = 0.f, sb = 0.f, sd = 0.f;
  if (n < N) {
    const float w = w2[n];
    for (int m = r0 + threadIdx.y; m < r1; m += 8) {
      const float d = ds[m];
      const float h = hidden[(long long)m * N + n];
      const float g = d * w * (1.f - h * h);
      // dz_row_scale: the Linear's input was row_scale[m] * x[m] (masked text embeddings): dW1 = dz^T (scale x) is taken as
      // (scale dz)^T x, so the stored rows carry the factor while db1 sums the unscaled gradient
      dz[(long long)m * N + n] = dz_row_scale ? g * __ldg(dz_row_scale + m) : g;
      sw = fmaf(d, h, sw);
      sb += g;
      if (blockIdx.x == 0 && threadIdx.x == 0) sd += d;
    }
  }
  red[0][threadIdx.y][threadIdx.x] = sw;
  red[1][threadIdx.y][threadIdx.x] = sb;
  __syncthreads();
  if (threadIdx.y == 0 && n < N) {
    float tw = 0.f, tb = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      tw += red[0][i][threadIdx.x];
      tb += red[1][i][threadIdx.x];
    }
    atomicAdd(dw2 + n, tw);
    atomicAdd(db1 + n, tb);
  }
  if (blockIdx.x == 0 && threadIdx.x == 0) atomicAdd(db2, sd);   // one column of blocks sums ds
}

__global__ void __launch_bounds__(256) dropout_kernel(const float* __restrict__ x, float* __restrict__ y, long long n,
                                                      float p, float scale, unsigned long long seed,
                                                      unsigned long long offset,
                                                      const unsigned long long* __restrict__ step_ptr, int vec) {
  DEER_PDL_ENTRY();
  const unsigned long long st = step_ptr ? *step_ptr : 0ull;  // device-side step counter: new mask per graph replay
  const uint32_t thr = (uint32_t)fminf(p * 4294967296.f, 4294967040.f);
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  const long long groups = (n + 3) >> 2;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < groups;
       q += (long long)gridDim.x * blockDim.x) {  // group of 4 elements = one Philox block
    const long long i = q * 4;
    const unsigned long long c = (unsigned long long)q + offset;
    const uint4 r = philox4x32_10(make_uint4((uint32_t)c, (uint32_t)(c >> 32), (uint32_t)st, (uint32_t)(st >> 32)), key);
    if (vec && i + 3 < n) {  // 16-byte aligned buffers: one 128-bit load and store per Philox block
      const float4 v = __ldcs(reinterpret_cast<const float4*>(x + i));
      float4 o;
      o.x = r.x >= thr ? v.x * scale : 0.f;
      o.y = r.y >= thr ? v.y * scale : 0.f;
      o.z = r.z >= thr ? v.z * scale : 0.f;
      o.w = r.w >= thr ? v.w * scale : 0.f;
      __stcs(reinterpret_cast<float4*>(y + i), o);
    } else {
      const uint32_t rr[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
      for (int j = 0; j < 4; j++)
        if (i + j < n) y[i + j] = rr[j] >= thr ? x[i + j] * scale : 0.f;
    }
  }
}

// dropout of a row-major fp32 matrix fused with its 16-bit casts: the LSTM layer-1 input is consumed only as FP16
// (input projection) and BF16 (dW_ih) GEMM operands, so the dropped fp32 tensor is never materialised.
// Same Philox stream as dropout_kernel over the flattened [rows, cols] index (cols % 4 == 0).
__global__ void __launch_bounds__(256) dropout_cast16_kernel(const float* __restrict__ x, uint16_t* __restrict__ y_h,
                                                             uint16_t* __restrict__ y_b, long long n, float p,
                                                             float scale, unsigned long long seed,
                                                             unsigned long long offset,
                                                             const unsigned long long* __restrict__ step_ptr,
                                                             uint32_t* __restrict__ mask_out) {
  DEER_PDL_ENTRY();
  const unsigned long long st = step_ptr ? *step_ptr : 0ull;
  const uint32_t thr = (uint32_t)fminf(p * 4294967296.f, 4294967040.f);
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  const long long groups = n >> 2;
  for (long long q = (long long)blockIdx.x * blockDim.x + threadIdx.x; q < groups;
       q += (long long)gridDim.x * blockDim.x) {
    const long long i = q * 4;
    float4 v = __ldcs(reinterpret_cast<const float4*>(x + i));
    uint32_t keep = 0xFu;
    if (p > 0.f) {
      const unsigned long long c = (unsigned long long)q + offset;
      const uint4 r =
          philox4x32_10(make_uint4((uint32_t)c, (uint32_t)(c >> 32), (uint32_t)st, (uint32_t)(st >> 32)), key);
      v.x = r.x >= thr ? v.x * scale : 0.f;
      v.y = r.y >= thr ? v.y * scale : 0.f;
      v.z = r.z >= thr ? v.z * scale : 0.f;
      v.w = r.w >= thr ? v.w * scale : 0.f;
      keep = (r.x >= thr ? 1u : 0u) | (r.y >= thr ? 2u : 0u) | (r.z >= thr ? 4u : 0u) | (r.w >= thr ? 8u : 0u);
    }
    if (mask_out) {
      // keep bits of 32 consecutive elements as one word (bit j = element 32 w + j): 8 lanes x 4 bits; the host
      // guarantees n % 128 == 0, so every warp is complete here.  Read back by the epilogue of the backward's
      // input-gradient GEMM (deer_gemm_h16_dropmask) instead of a Philox pass over dx.
      uint32_t w = keep << (4 * (threadIdx.x & 7));
      w |= __shfl_xor_sync(0xffffffffu, w, 1);
      w |= __shfl_xor_sync(0xffffffffu, w, 2);
      w |= __shfl_xor_sync(0xffffffffu, w, 4);
      if ((threadIdx.x & 7) == 0) mask_out[q >> 3] = w;
    }
    if (y_h) {
      __half2 a = __floats2half2_rn(v.x, v.y), b = __floats2half2_rn(v.z, v.w);
      uint2 o = make_uint2(*reinterpret_cast<uint32_t*>(&a), *reinterpret_cast<uint32_t*>(&b));
      *reinterpret_cast<uint2*>(y_h + i) = o;
    }
    if (y_b) {
      __nv_bfloat162 a = __floats2bfloat162_rn(v.x, v.y), b = __floats2bfloat162_rn(v.z, v.w);
      uint2 o = make_uint2(*reinterpret_cast<uint32_t*>(&a), *reinterpret_cast<uint32_t*>(&b));
      *reinterpret_cast<uint2*>(y_b + i) = o;
    }
  }
}

// ------------------------------------------------------------------ scorer head: s[m] = h[m,:].w + b
__global__ void __launch_bounds__(256) rowdot_fwd_kernel(const float* __restrict__ h, const float* __restrict__ w,
                                                         const float* __restrict__ b, float* __restrict__ s,
                                                         long long M, int N) {
  DEER_PDL_ENTRY();
  const long long row = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float* hr = h + row * N;
  float acc = 0.f;
  for (int j = lane; j < N; j += 32) acc = fmaf(hr[j], w[j], acc);
  acc = warp_sum(acc);
  if (lane == 0) s[row] = acc + b[0];
}

// dh[m,j] = ds[m]*w[j]; dw[j] += sum_m ds[m]*h[m,j]; db += sum_m ds[m]
__global__ void __launch_bounds__(256) rowdot_bwd_kernel(const float* __restrict__ ds, const float* __restrict__ h,
                                                         const float* __restrict__ w, float* __restrict__ dh,
                                                         float* __restrict__ dw, float* __restrict__ db, long long M,
                                                         int N, int rows_per_block) {
  DEER_PDL_ENTRY();
  __shared__ float red[8][33];
  const int n = blockIdx.x * 32 + threadIdx.x;
  const long long r0 = (long long)blockIdx.y * rows_per_block;
  const long long r1 = min(M, r0 + (long long)rows_per_block);
  float s = 0.f, sb = 0.f;
  const float wn = n < N ? w[n] : 0.f;
  for (long long m = r0 + threadIdx.y; m < r1; m += 8) {
    const float d = ds[m];
    if (n < N) {
      s = fmaf(d, h[m * N + n], s);
      if (dh) dh[m * N + n] = d * wn;
    }
    sb += d;
  }
  red[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && n < N) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) t += red[i][threadIdx.x];
    atomicAdd(dw + n, t);
  }
  if (blockIdx.x == 0) {  // block-uniform: one column-block also reduces db = sum_m ds[m]
    __syncthreads();
    red[threadIdx.y][threadIdx.x] = (threadIdx.x == 0) ? sb : 0.f;
    __syncthreads();
    if (threadIdx.y == 0 && threadIdx.x == 0) {
      float t = 0.f;
#pragma unroll
      for (int i = 0; i < 8; i++) t += red[i][0];
      atomicAdd(db, t);
    }
  }
}

// ------------------------------------------------------------------ layout moves
// y[t,b,:] = x[b,t,:]
__global__ void __launch_bounds__(256) permute_bt_kernel(const float* __restrict__ x, float* __restrict__ y, int B,
                                                         int T, int D) {
  DEER_PDL_ENTRY();
  const long long total = (long long)B * T * D;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int d = (int)(i % D);
    const long long r = i / D;  // output row = t*B + b
    const int b = (int)(r % B);
    const int t = (int)(r / B);
    y[i] = x[((long long)b * T + t) * D + d];
  }
}

// [B,T,D] fp32 -> time-major 16-bit rows [T*B, Dp] (columns D..Dp-1 zero): the first LSTM layer's A operand (FP16) and,
// for training, the BF16 copy its weight-gradient GEMM reads -- one pass over the input instead of permute_bt (fp32
// time-major copy) + cast16 forward + cast16 backward.
// kLengths: the padded frames t >= L_b are written as zeros (never read), so the 16-bit operand copies carry no NaN / Inf
// from the padding into the projection or into dW_ih = dpre^T x (0 * NaN); x_time_major: x is already [T,B,D] (the layer
// input that needs a gradient went through to_time_major).
template <bool kLengths>
__global__ void __launch_bounds__(256) permute_bt_cast16_kernel(const float* __restrict__ x, __half* __restrict__ y16,
                                                                __nv_bfloat16* __restrict__ yb16, int B, int T, int D,
                                                                int Dp, const void* lengths, int lengths_i64,
                                                                int x_time_major) {
  DEER_PDL_ENTRY();
  const int pairs = Dp >> 1;
  const long long total = (long long)B * T * pairs;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int d = (int)(i % pairs) * 2;
    const long long r = i / pairs;  // output row = t*B + b
    const int b = (int)(r % B);
    const int t = (int)(r / B);
    float v0 = 0.f, v1 = 0.f;
    if (!kLengths || t < seq_length(lengths, lengths_i64, b, T)) {
      const float* src = x + (kLengths && x_time_major ? r : (long long)b * T + t) * D + d;
      v0 = d < D ? __ldcs(src) : 0.f;
      v1 = d + 1 < D ? __ldcs(src + 1) : 0.f;
    }
    if (y16) *reinterpret_cast<__half2*>(y16 + r * Dp + d) = __floats2half2_rn(v0, v1);
    if (yb16) *reinterpret_cast<__nv_bfloat162*>(yb16 + r * Dp + d) = __floats2bfloat162_rn(v0, v1);
  }
}

// Gate saturation of the padded rows of the gate-interleaved LSTM pre-activations [T, B, 2 directions, H units, 4 gates]
// (gate order i, f, g, o): i, f and o of rows t >= L_b are set to -65504 (the most negative finite FP16), so the recurrence
// kernels' sigmoid gives 2^-60 and the state collapses to ~0 at every padded step -- the reverse direction then starts at
// L_b - 1 from a zero state, as nn.LSTM does on a packed sequence, and the FP16 gates / cell states kept for BPTT underflow
// to exactly 0 there (every pre-activation gradient of a padded step is 0).  g is left as it is.
// grid (B, ny): block (b, y) takes the padded rows L_b + y, L_b + y + ny, ...: the work is that of the padded rows only.
template <typename Unit>
__global__ void __launch_bounds__(256) lstm_mask_pre_kernel(Unit* __restrict__ pre, const void* lengths,
                                                            int lengths_i64, int T, int B, int H) {
  DEER_PDL_ENTRY();
  const int b = blockIdx.x;
  const int units = 2 * H;  // both directions
  for (int t = seq_length(lengths, lengths_i64, b, T) + blockIdx.y; t < T; t += gridDim.y) {
    Unit* row = pre + ((long long)t * B + b) * units;
    for (int u = threadIdx.x; u < units; u += blockDim.x) {
      Unit v = row[u];
      if constexpr (sizeof(Unit) == 16) {  // fp32 gates
        v.x = v.y = v.w = -65504.f;
      } else {                             // FP16 gates: 0xFBFF = -65504 in the two low halves and the top one
        v.x = 0xFBFFFBFFu;
        v.y = (v.y & 0x0000FFFFu) | 0xFBFF0000u;
      }
      row[u] = v;
    }
  }
}

// kLengths: the row mask comes from per-utterance lengths (rows m = b*T + t of a [B,T,D] tensor): y = x at t < L_b and y = 0
// at padded rows, which are not read (x * 0 would keep a NaN) -- the masked copy of a length-aware layer's input
template <bool kLengths>
__global__ void __launch_bounds__(256) rowscale_kernel(const float* __restrict__ x, const float* __restrict__ mask,
                                                       float* __restrict__ y, long long M, int D, const void* lengths,
                                                       int lengths_i64, int T) {
  DEER_PDL_ENTRY();
  const long long total = M * D;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    if constexpr (kLengths)
      y[i] = seq_row_valid(i / D, lengths, lengths_i64, T) ? x[i] : 0.f;
    else
      y[i] = x[i] * mask[i / D];
  }
}

// col[(b,t), k*C + c] = x[b, t+k-1, c]
__global__ void __launch_bounds__(256) im2col3_kernel(const float* __restrict__ x, float* __restrict__ col, int B, int T,
                                                      int C) {
  DEER_PDL_ENTRY();
  const long long total = (long long)B * T * 3 * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    long long r = i / C;
    const int k = (int)(r % 3);
    r /= 3;
    const int t = (int)(r % T);
    const int b = (int)(r / T);
    const int ts = t + k - 1;
    col[i] = (ts >= 0 && ts < T) ? x[((long long)b * T + ts) * C + c] : 0.f;
  }
}
// ------------------------------------------------------------------ zero-row padding for the sliding-window Conv1d
// padded layout: [lead zero rows][sample 0: T rows][1 zero row][sample 1: T rows][1 zero row] ...  (one shared pad row
// between samples; with lead = 1 a row view of 3*C contiguous floats starting at padded row q is exactly the k=3
// im2col row centred on padded row q+1).  dir 0: x [B,T,C] -> xp (pad rows written as zeros); dir 1: xp -> x.
__global__ void __launch_bounds__(256) rows_pad_kernel(const float* __restrict__ src, float* __restrict__ dst, int B,
                                                       int T, int C4, int lead, int dir, long long pad_rows_total) {
  DEER_PDL_ENTRY();
  const long long per_sample = (long long)(T + 1) * C4;
  const long long total = (dir == 0) ? pad_rows_total * C4 : (long long)B * T * C4;   // in float4 units
  const float4* s4 = reinterpret_cast<const float4*>(src);
  float4* d4 = reinterpret_cast<float4*>(dst);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    if (dir == 0) {   // iterate over PADDED elements: copy or zero
      const long long r = i / C4;
      const int c = (int)(i % C4);
      const long long q = r - lead;
      float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
      if (q >= 0) {
        const long long b = q / (T + 1);
        const int t = (int)(q % (T + 1));
        if (b < B && t < T) v = __ldcs(s4 + (b * T + t) * C4 + c);
      }
      d4[i] = v;
    } else {          // iterate over compact elements
      const long long r = i / C4;
      const int c = (int)(i % C4);
      const long long b = r / T;
      const int t = (int)(r % T);
      __stcs(d4 + i, s4[(lead + b * (T + 1) + t) * C4 + c]);
    }
  }
  (void)per_sample;
}

// rows_pad with the neighbouring elementwise passes of the video encoder's Conv1d stack folded in (encoders.py:450-459:
// Dropout -> Conv1d): dir 0 reads x [B,T,C] once, applies inverted dropout (the Philox stream of deer_dropout over the flat
// index of x, so the fused and the separate path draw identical masks), writes the padded fp32 copy (kept for the weight
// gradient) and, optionally, its FP16 hi / lo split in the same geometry (the A operand of the split-precision forward
// GEMM); dir 1 (backward) drops the pad rows of dx_p and applies the same mask.  Replaces dropout + rows_pad +
// cast_split16 (three passes over the tensor) forward and rows_pad + dropout backward.
// kLengths (per-utterance lengths): frames t >= L_b count as pad rows.  dir 0 writes zeros for them (their source rows are
// not read), so the convolution sees each clip zero-padded at both ends; dir 1 writes dx = 0 for them -- dx_p row L_b holds
// the tap dy[L_b - 1] W, which would otherwise leak into the padded rows' gradient.
template <bool kLengths>
__global__ void __launch_bounds__(256) rows_pad_fused_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                             uint16_t* __restrict__ hi, uint16_t* __restrict__ lo, int B,
                                                             int T, int C4, int lead, int dir, long long pad_rows_total,
                                                             float p, float scale, unsigned long long seed,
                                                             unsigned long long offset,
                                                             const unsigned long long* __restrict__ step_ptr,
                                                             const void* lengths, int lengths_i64) {
  DEER_PDL_ENTRY();
  const unsigned long long st = step_ptr ? *step_ptr : 0ull;
  const uint32_t thr = (uint32_t)fminf(p * 4294967296.f, 4294967040.f);
  const uint2 key = make_uint2((uint32_t)seed, (uint32_t)(seed >> 32));
  const bool drop = p > 0.f;
  const long long total = (dir == 0) ? pad_rows_total * C4 : (long long)B * T * C4;   // in float4 units
  const float4* s4 = reinterpret_cast<const float4*>(src);
  float4* d4 = reinterpret_cast<float4*>(dst);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long r = i / C4;
    const int c = (int)(i % C4);
    long long ci;          // float4 index into the compact [B,T,C] tensor, < 0: a pad row
    if (dir == 0) {
      const long long q = r - lead;
      ci = -1;
      if (q >= 0) {
        const long long b = q / (T + 1);
        const int t = (int)(q % (T + 1));
        if (b < B && t < T && (!kLengths || t < seq_length(lengths, lengths_i64, (int)b, T))) ci = (b * T + t) * C4 + c;
      }
    } else {
      ci = (!kLengths || seq_row_valid(r, lengths, lengths_i64, T)) ? i : -1;
    }
    float4 v = make_float4(0.f, 0.f, 0.f, 0.f);
    if (ci >= 0) {
      if (dir == 0) {
        v = __ldcs(s4 + ci);
      } else {
        const long long b = r / T;
        const int t = (int)(r % T);
        v = __ldcs(s4 + (lead + b * (T + 1) + t) * C4 + c);
      }
      if (drop) {
        const unsigned long long cnt = (unsigned long long)ci + offset;
        const uint4 rr = philox4x32_10(make_uint4((uint32_t)cnt, (uint32_t)(cnt >> 32), (uint32_t)st, (uint32_t)(st >> 32)), key);
        v.x = rr.x >= thr ? v.x * scale : 0.f;
        v.y = rr.y >= thr ? v.y * scale : 0.f;
        v.z = rr.z >= thr ? v.z * scale : 0.f;
        v.w = rr.w >= thr ? v.w * scale : 0.f;
      }
    }
    if (dir == 0) {
      d4[i] = v;            // re-read by the GEMMs: default caching
      if (hi) {
        const float f[4] = {v.x, v.y, v.z, v.w};
        __half h[4], l[4];
#pragma unroll
        for (int j = 0; j < 4; j++) {
          h[j] = __float2half_rn(f[j]);
          l[j] = __float2half_rn(f[j] - __half2float(h[j]));
        }
        *reinterpret_cast<uint2*>(hi + i * 4) = *reinterpret_cast<const uint2*>(h);
        *reinterpret_cast<uint2*>(lo + i * 4) = *reinterpret_cast<const uint2*>(l);
      }
    } else {
      __stcs(d4 + i, v);
    }
  }
}

// Backward entry of the sliding-window Conv1d: dy [B,T,C] -> dy_big [B*(T+1), C] (one zero row behind every sample: the
// rows centred on a pad row) AND the bias gradient db[c] += sum_rows dy[., c] in the same pass (it was a second pass over
// dy: deer_bias_act_bwd).  grid (ceil(C4/32), row chunks), block (32, 8): lane x owns one float4 column group, the 8 rows
// of threads stride over the chunk's rows; column sums folded through shared memory, one atomicAdd per column and block.
__global__ void __launch_bounds__(256) rows_pad_colsum_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                              float* __restrict__ colsum, int B, int T, int C4,
                                                              int rows_per_block) {
  DEER_PDL_ENTRY();
  __shared__ float4 red[8][33];
  const int c4 = blockIdx.x * 32 + threadIdx.x;
  const long long M = (long long)B * T;
  const long long r0 = (long long)blockIdx.y * rows_per_block;
  const long long r1 = min(M, r0 + (long long)rows_per_block);
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c4 < C4) {
    const float4* s4 = reinterpret_cast<const float4*>(src);
    float4* d4 = reinterpret_cast<float4*>(dst);
    for (long long m = r0 + threadIdx.y; m < r1; m += 8) {
      const float4 v = __ldcs(s4 + m * C4 + c4);
      const long long b = m / T;
      const int t = (int)(m - b * T);
      const long long q = b * (T + 1) + t;
      d4[q * C4 + c4] = v;                                                      // re-read by two GEMMs: default caching
      if (t == T - 1) d4[(q + 1) * C4 + c4] = make_float4(0.f, 0.f, 0.f, 0.f);  // the sample's pad row
      acc.x += v.x; acc.y += v.y; acc.z += v.z; acc.w += v.w;
    }
  }
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && c4 < C4 && colsum != nullptr) {
    float4 t4 = red[0][threadIdx.x];
#pragma unroll
    for (int i = 1; i < 8; i++) {
      const float4 u = red[i][threadIdx.x];
      t4.x += u.x; t4.y += u.y; t4.z += u.z; t4.w += u.w;
    }
    atomicAdd(colsum + 4 * c4 + 0, t4.x);
    atomicAdd(colsum + 4 * c4 + 1, t4.y);
    atomicAdd(colsum + 4 * c4 + 2, t4.z);
    atomicAdd(colsum + 4 * c4 + 3, t4.w);
  }
}

// dx[b,t,c] = sum_k dcol[(b,t-k+1), k*C + c]
__global__ void __launch_bounds__(256) col2im3_kernel(const float* __restrict__ dcol, float* __restrict__ dx, int B,
                                                      int T, int C) {
  DEER_PDL_ENTRY();
  const long long total = (long long)B * T * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int c = (int)(i % C);
    const long long r = i / C;
    const int t = (int)(r % T);
    const int b = (int)(r / T);
    float s = 0.f;
#pragma unroll
    for (int k = 0; k < 3; k++) {
      const int tt = t - k + 1;
      if (tt >= 0 && tt < T) s += dcol[(((long long)b * T + tt) * 3 + k) * C + c];
    }
    dx[i] = s;
  }
}
// dir 0: wk[o,k,i] = w[o,i,k];  dir 1: w[o,i,k] += wk[o,k,i]
__global__ void __launch_bounds__(256) conv3_pack_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                         int Cout, int Cin, int dir) {
  DEER_PDL_ENTRY();
  const long long total = (long long)Cout * Cin * 3;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    if (dir == 0) {  // i indexes wk [o,k,ci]
      const int ci = (int)(i % Cin);
      const int k = (int)((i / Cin) % 3);
      const long long o = i / (3LL * Cin);
      dst[i] = src[(o * Cin + ci) * 3 + k];
    } else {  // i indexes w [o,ci,k]
      const int k = (int)(i % 3);
      const int ci = (int)((i / 3) % Cin);
      const long long o = i / (3LL * Cin);
      dst[i] += src[(o * 3 + k) * Cin + ci];
    }
  }
}

// ------------------------------------------------------------------ small combiners (pooled model)
__global__ void __launch_bounds__(256) axpby_kernel(const float* __restrict__ x1, const float* __restrict__ x2,
                                                    float* __restrict__ y, long long n, float a, float b) {
  DEER_PDL_ENTRY();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    y[i] = a * x1[i] + (x2 ? b * x2[i] : 0.f);
}

__global__ void __launch_bounds__(256) mix_fwd_kernel(const float* __restrict__ w, long long ldw,
                                                      const float* __restrict__ u, long long ldu,
                                                      const float* __restrict__ s, const float* __restrict__ c,
                                                      float* __restrict__ out, long long M, int N) {
  DEER_PDL_ENTRY();
  const long long total = M * N;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const long long m = i / N;
    out[i] = w[m * ldw] * s[i] + (1.f - u[m * ldu]) * c[i];
  }
}
// one warp per row
__global__ void __launch_bounds__(256) mix_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ w,
                                                      long long ldw, const float* __restrict__ u, long long ldu,
                                                      const float* __restrict__ s, const float* __restrict__ c,
                                                      float* __restrict__ dw, long long lddw, float* __restrict__ du,
                                                      long long lddu, float* __restrict__ ds, float* __restrict__ dc,
                                                      long long M, int N) {
  DEER_PDL_ENTRY();
  const long long m = (long long)blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (m >= M) return;
  const float wm = w[m * ldw], um = u[m * ldu];
  float aw = 0.f, au = 0.f;
  for (int j = lane; j < N; j += 32) {
    const long long i = m * N + j;
    const float g = dout[i];
    aw = fmaf(g, s[i], aw);
    au = fmaf(g, c[i], au);
    ds[i] = g * wm;
    dc[i] = g * (1.f - um);
  }
  aw = warp_sum(aw);
  au = warp_sum(au);
  if (lane == 0) {
    dw[m * lddw] = aw;
    du[m * lddu] = -au;
  }
}

__global__ void __launch_bounds__(256) gate_fwd_kernel(const float* __restrict__ g, const float* __restrict__ a,
                                                       const float* __restrict__ b, float* __restrict__ out,
                                                       long long n) {
  DEER_PDL_ENTRY();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x)
    out[i] = g[i] * a[i] + (1.f - g[i]) * b[i];
}
__global__ void __launch_bounds__(256) gate_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ g,
                                                       const float* __restrict__ a, const float* __restrict__ b,
                                                       float* __restrict__ dg, float* __restrict__ da,
                                                       float* __restrict__ db, long long n) {
  DEER_PDL_ENTRY();
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    const float d = dout[i], gi = g[i];
    dg[i] = d * (a[i] - b[i]);
    da[i] = d * gi;
    db[i] = d * (1.f - gi);
  }
}

__global__ void __launch_bounds__(256) softmax_rows_fwd_kernel(const float* __restrict__ x, float* __restrict__ y,
                                                               long long M, int N) {
  DEER_PDL_ENTRY();
  const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  float mx = -INFINITY;
  for (int j = 0; j < N; j++) mx = fmaxf(mx, x[m * N + j]);
  float s = 0.f;
  for (int j = 0; j < N; j++) s += expf(x[m * N + j] - mx);
  const float inv = 1.f / s;
  for (int j = 0; j < N; j++) y[m * N + j] = expf(x[m * N + j] - mx) * inv;
}
__global__ void __launch_bounds__(256) softmax_rows_bwd_kernel(const float* __restrict__ dy,
                                                               const float* __restrict__ y, float* __restrict__ dx,
                                                               long long M, int N) {
  DEER_PDL_ENTRY();
  const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= M) return;
  float dot = 0.f;
  for (int j = 0; j < N; j++) dot = fmaf(dy[m * N + j], y[m * N + j], dot);
  for (int j = 0; j < N; j++) dx[m * N + j] = y[m * N + j] * (dy[m * N + j] - dot);
}

static inline int grid_for(long long n, int per_block = 256, int max_blocks = kNumSMs * 16) {
  long long g = cdiv(n, per_block);
  if (g > max_blocks) g = max_blocks;
  if (g < 1) g = 1;
  return (int)g;
}

// y[m,n] = x[m,n] / t[n]   (temperature scaling, complete_project.py:449) and its backward
__global__ void __launch_bounds__(256) coldiv_fwd_kernel(const float* __restrict__ x, const float* __restrict__ t,
                                                         float* __restrict__ y, long long M, int N) {
  DEER_PDL_ENTRY();
  const long long total = M * N;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x)
    y[i] = x[i] / t[i % N];
}
// dx = dy / t;  dt[n] += -sum_m dy[m,n] x[m,n] / t[n]^2   (one block per column; N is tiny)
__global__ void __launch_bounds__(256) coldiv_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                         const float* __restrict__ t, float* __restrict__ dx,
                                                         float* __restrict__ dt, long long M, int N) {
  DEER_PDL_ENTRY();
  __shared__ float red[32];
  const int n = blockIdx.x;
  const float tn = t[n];
  float acc = 0.f;
  for (long long m = threadIdx.x; m < M; m += blockDim.x) {
    const float g = dy[m * N + n];
    dx[m * N + n] = g / tn;
    acc += g * x[m * N + n];
  }
  acc = block_sum(acc, red);
  if (threadIdx.x == 0 && dt) dt[n] += -acc / (tn * tn);
}

// nn.LSTM gate rows (row g*H+u of a [4H,K] matrix) <-> gate-interleaved rows (4u+g) used by the persistent LSTM
// kernels; inverse=1 maps interleaved -> natural; accumulate adds into dst (gradient un-permutation into .grad)
__global__ void __launch_bounds__(256) gate_rows_interleave_kernel(const float* __restrict__ src, float* __restrict__ dst,
                                                                   int H, int K, int inverse, int accumulate) {
  DEER_PDL_ENTRY();
  const long long total = 4LL * H * K;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int k = (int)(i % K);
    const int row = (int)(i / K);             // index in the SOURCE row order
    int drow;
    if (!inverse) {                           // src natural (g*H+u) -> dst interleaved (4u+g)
      const int g = row / H, u = row % H;
      drow = 4 * u + g;
    } else {                                  // src interleaved -> dst natural
      const int u = row >> 2, g = row & 3;
      drow = g * H + u;
    }
    const float v = src[i];
    float* d = dst + (long long)drow * K + k;
    *d = accumulate ? *d + v : v;
  }
}

}  // namespace deer

using namespace deer;

extern "C" {

int deer_coldiv_fwd(const float* x, const float* t, float* y, long long M, int N, void* stream) {
  DEER_CHECK_ARG(x && t && y && M > 0 && N > 0, "coldiv_fwd: bad args");
  DEER_LAUNCH(coldiv_fwd_kernel, grid_for(M * N), 256, 0, stream, x, t, y, M, N);
  return DEER_OK;
}

int deer_coldiv_bwd(const float* dy, const float* x, const float* t, float* dx, float* dt, long long M, int N,
                    void* stream) {
  DEER_CHECK_ARG(dy && x && t && dx && M > 0 && N > 0, "coldiv_bwd: bad args");
  DEER_LAUNCH(coldiv_bwd_kernel, (unsigned)N, 256, 0, stream, dy, x, t, dx, dt, M, N);
  return DEER_OK;
}

int deer_gate_rows_interleave(const float* src, float* dst, int H, int K, int inverse, int accumulate, void* stream) {
  DEER_CHECK_ARG(src && dst && H > 0 && K > 0 && src != dst, "gate_rows_interleave: bad args");
  DEER_LAUNCH(gate_rows_interleave_kernel, grid_for(4LL * H * K), 256, 0, stream, src, dst, H, K, inverse, accumulate);
  return DEER_OK;
}


int deer_bias_act_bwd(const float* dy, long long ld_dy, const float* y, long long ld_y, float* dz, long long ld_dz,
                      float* dbias, int M, int N, int act, void* stream) {
  DEER_CHECK_ARG(dy && M > 0 && N > 0, "bias_act_bwd: null/empty");
  DEER_CHECK_ARG(act == DEER_ACT_NONE || y, "bias_act_bwd: act needs y");
  // rows per block: enough blocks for ~4 per SM even when N is a few hundred columns (the post-pooling layers)
  const long long gx = cdiv(N, 32);
  long long want_gy = cdiv(4 * kNumSMs, gx);
  int rpb = (int)cdiv(M, want_gy);
  rpb = ((rpb + 7) / 8) * 8;
  if (rpb < 8) rpb = 8;
  dim3 grid((unsigned)gx, (unsigned)cdiv(M, rpb));
  DEER_LAUNCH(bias_act_bwd_kernel, grid, dim3(32, 8), 0, stream, dy, ld_dy, y, ld_y, dz, ld_dz, dbias, M, N, act, rpb);
  return DEER_OK;
}

static int dropout_grid(long long groups) {
  long long g = cdiv(groups, 256);
  const long long cap = (long long)kNumSMs * 16;
  if (g > cap) g = cap;
  return (int)(g < 1 ? 1 : g);
}

int deer_dropout(const float* x, float* y, long long n, float p, unsigned long long seed, unsigned long long offset,
                 const unsigned long long* step_ptr, void* stream) {
  DEER_CHECK_ARG(x && y && n > 0 && p >= 0.f && p < 1.f, "dropout: bad args");
  const long long groups = cdiv(n, 4);
  const int vec = ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(y)) & 15) == 0;
  DEER_LAUNCH(dropout_kernel, dropout_grid(groups), 256, 0, stream, x, y, n, p, 1.f / (1.f - p), seed, offset, step_ptr,
              vec);
  return DEER_OK;
}

int deer_dropout_cast16(const float* x, void* y_fp16, void* y_bf16, long long n, float p, unsigned long long seed,
                        unsigned long long offset, const unsigned long long* step_ptr, void* keep_mask, void* stream) {
  DEER_CHECK_ARG(x && (y_fp16 || y_bf16) && n > 0 && (n & 3) == 0 && p >= 0.f && p < 1.f && (!keep_mask || (n & 127) == 0),
                 "dropout_cast16: bad args");
  DEER_CHECK_ARG((reinterpret_cast<uintptr_t>(x) & 15) == 0 && (reinterpret_cast<uintptr_t>(y_fp16) & 7) == 0 &&
                     (reinterpret_cast<uintptr_t>(y_bf16) & 7) == 0,
                 "dropout_cast16: alignment");
  DEER_LAUNCH(dropout_cast16_kernel, dropout_grid(n >> 2), 256, 0, stream, x, reinterpret_cast<uint16_t*>(y_fp16),
              reinterpret_cast<uint16_t*>(y_bf16), n, p, 1.f / (1.f - p), seed, offset, step_ptr,
              reinterpret_cast<uint32_t*>(keep_mask));
  return DEER_OK;
}

int deer_scorer_bwd(const float* ds, const float* hidden, const float* w2, float* dz, float* dw2, float* db1, float* db2,
                    const float* dz_row_scale, long long M, int N, void* stream) {
  DEER_CHECK_ARG(ds && hidden && w2 && dz && dw2 && db1 && db2 && M > 0 && M < (1ll << 31) && N > 0,
                 "scorer_bwd: bad args");
  const long long gx = cdiv(N, 32);
  long long want_gy = cdiv(6 * kNumSMs, gx);
  int rpb = (int)cdiv(M, want_gy);
  rpb = ((rpb + 7) / 8) * 8;
  if (rpb < 8) rpb = 8;
  dim3 grid((unsigned)gx, (unsigned)cdiv(M, rpb));
  DEER_LAUNCH(scorer_bwd_kernel, grid, dim3(32, 8), 0, stream, ds, hidden, w2, dz, dw2, db1, db2, dz_row_scale, (int)M, N, rpb);
  return DEER_OK;
}

int deer_rowdot_fwd(const float* h, const float* w, const float* b, float* s, long long M, int N, void* stream) {
  DEER_CHECK_ARG(h && w && b && s && M > 0 && N > 0, "rowdot_fwd: bad args");
  DEER_LAUNCH(rowdot_fwd_kernel, (unsigned)cdiv(M, 8), 256, 0, stream, h, w, b, s, M, N);
  return DEER_OK;
}

int deer_rowdot_bwd(const float* ds, const float* h, const float* w, float* dh, float* dw, float* db, long long M,
                    int N, void* stream) {
  DEER_CHECK_ARG(ds && h && w && dw && db && M > 0 && N > 0, "rowdot_bwd: bad args");
  const int rpb = 256;
  dim3 grid((unsigned)cdiv(N, 32), (unsigned)cdiv(M, rpb));
  DEER_LAUNCH(rowdot_bwd_kernel, grid, dim3(32, 8), 0, stream, ds, h, w, dh, dw, db, M, N, rpb);
  return DEER_OK;
}

int deer_permute_bt(const float* x, float* y, int B, int T, int D, void* stream) {
  DEER_CHECK_ARG(x && y && B > 0 && T > 0 && D > 0, "permute_bt: bad args");
  DEER_LAUNCH(permute_bt_kernel, grid_for((long long)B * T * D), 256, 0, stream, x, y, B, T, D);
  return DEER_OK;
}

int deer_permute_bt_cast16(const float* x, void* y_fp16, void* y_bf16, int B, int T, int D, int Dp, void* stream) {
  DEER_CHECK_ARG(x && (y_fp16 || y_bf16) && B > 0 && T > 0 && D > 0 && Dp >= D && (Dp & 1) == 0, "permute_bt_cast16: bad args");
  DEER_LAUNCH(permute_bt_cast16_kernel<false>, grid_for((long long)B * T * (Dp / 2)), 256, 0, stream, x,
              reinterpret_cast<__half*>(y_fp16), reinterpret_cast<__nv_bfloat16*>(y_bf16), B, T, D, Dp, nullptr, 0, 0);
  return DEER_OK;
}

int deer_permute_bt_cast16_len(const float* x, void* y_fp16, void* y_bf16, const void* lengths, int lengths_i64, int B,
                               int T, int D, int Dp, int x_time_major, void* stream) {
  DEER_CHECK_ARG(x && (y_fp16 || y_bf16) && lengths && B > 0 && T > 0 && D > 0 && Dp >= D && (Dp & 1) == 0,
                 "permute_bt_cast16_len: bad args");
  DEER_LAUNCH(permute_bt_cast16_kernel<true>, grid_for((long long)B * T * (Dp / 2)), 256, 0, stream, x,
              reinterpret_cast<__half*>(y_fp16), reinterpret_cast<__nv_bfloat16*>(y_bf16), B, T, D, Dp, lengths,
              lengths_i64, x_time_major);
  return DEER_OK;
}

int deer_lstm_mask_pre(void* pre, int pre_fp16, const void* lengths, int lengths_i64, int T, int B, int H, void* stream) {
  DEER_CHECK_ARG(pre && lengths && T > 0 && B > 0 && H > 0 && (reinterpret_cast<uintptr_t>(pre) & 15) == 0,
                 "lstm_mask_pre: bad args");
  // up to 8 blocks per sample share its padded rows (one 8 KB FP16 / 16 KB fp32 row per block and trip)
  const dim3 grid((unsigned)B, (unsigned)(T < 8 ? T : 8));
  const int threads = 2 * H < 256 ? 2 * H : 256;
  if (pre_fp16)
    DEER_LAUNCH(lstm_mask_pre_kernel<uint2>, grid, threads, 0, stream, reinterpret_cast<uint2*>(pre), lengths,
                lengths_i64, T, B, H);
  else
    DEER_LAUNCH(lstm_mask_pre_kernel<float4>, grid, threads, 0, stream, reinterpret_cast<float4*>(pre), lengths,
                lengths_i64, T, B, H);
  return DEER_OK;
}

int deer_rowscale(const float* x, const float* mask, float* y, long long M, int D, void* stream) {
  DEER_CHECK_ARG(x && mask && y && M > 0 && D > 0, "rowscale: bad args");
  DEER_LAUNCH(rowscale_kernel<false>, grid_for(M * D), 256, 0, stream, x, mask, y, M, D, nullptr, 0, 1);
  return DEER_OK;
}

int deer_rowscale_len(const float* x, float* y, const void* lengths, int lengths_i64, int B, int T, int D, void* stream) {
  DEER_CHECK_ARG(x && y && lengths && B > 0 && T > 0 && D > 0, "rowscale_len: bad args");
  const long long M = (long long)B * T;
  DEER_LAUNCH(rowscale_kernel<true>, grid_for(M * D), 256, 0, stream, x, nullptr, y, M, D, lengths, lengths_i64, T);
  return DEER_OK;
}

int deer_im2col3(const float* x, float* col, int B, int T, int C, void* stream) {
  DEER_CHECK_ARG(x && col && B > 0 && T > 0 && C > 0, "im2col3: bad args");
  DEER_LAUNCH(im2col3_kernel, grid_for((long long)B * T * 3 * C), 256, 0, stream, x, col, B, T, C);
  return DEER_OK;
}

int deer_rows_pad(const float* src, float* dst, int B, int T, int C, int lead, int tail, int dir, void* stream) {
  DEER_CHECK_ARG(src && dst && B > 0 && T > 0 && C > 0 && (C & 3) == 0 && lead >= 0 && tail >= 0 && (dir == 0 || dir == 1),
                 "rows_pad: bad args");
  DEER_CHECK_ARG(((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0, "rows_pad: alignment");
  const long long pad_rows = (long long)lead + (long long)B * (T + 1) + tail;
  const long long n4 = (dir == 0 ? pad_rows : (long long)B * T) * (C / 4);
  DEER_LAUNCH(rows_pad_kernel, grid_for(n4), 256, 0, stream, src, dst, B, T, C / 4, lead, dir, pad_rows);
  return DEER_OK;
}

static int rows_pad_fused(const float* src, float* dst, void* hi, void* lo, int B, int T, int C, int lead, int tail,
                          int dir, float drop_p, unsigned long long seed, unsigned long long offset,
                          const unsigned long long* step_ptr, const void* lengths, int lengths_i64, void* stream) {
  DEER_CHECK_ARG(src && dst && B > 0 && T > 0 && C > 0 && (C & 3) == 0 && lead >= 0 && tail >= 0 && (dir == 0 || dir == 1) &&
                     drop_p >= 0.f && drop_p < 1.f && ((hi == nullptr) == (lo == nullptr)) && (dir == 0 || hi == nullptr),
                 "rows_pad_fused: bad args");
  DEER_CHECK_ARG(((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0 &&
                     ((reinterpret_cast<uintptr_t>(hi) | reinterpret_cast<uintptr_t>(lo)) & 7) == 0,
                 "rows_pad_fused: alignment");
  const long long pad_rows = (long long)lead + (long long)B * (T + 1) + tail;
  const long long n4 = (dir == 0 ? pad_rows : (long long)B * T) * (C / 4);
  DEER_LAUNCH(lengths ? rows_pad_fused_kernel<true> : rows_pad_fused_kernel<false>, grid_for(n4), 256, 0, stream, src,
              dst, reinterpret_cast<uint16_t*>(hi), reinterpret_cast<uint16_t*>(lo), B, T, C / 4, lead, dir, pad_rows,
              drop_p, 1.f / (1.f - drop_p), seed, offset, step_ptr, lengths, lengths_i64);
  return DEER_OK;
}

int deer_rows_pad_fused(const float* src, float* dst, void* hi, void* lo, int B, int T, int C, int lead, int tail, int dir,
                        float drop_p, unsigned long long seed, unsigned long long offset, const unsigned long long* step_ptr,
                        void* stream) {
  return rows_pad_fused(src, dst, hi, lo, B, T, C, lead, tail, dir, drop_p, seed, offset, step_ptr, nullptr, 0, stream);
}

int deer_rows_pad_fused_len(const float* src, float* dst, void* hi, void* lo, const void* lengths, int lengths_i64, int B,
                            int T, int C, int lead, int tail, int dir, float drop_p, unsigned long long seed,
                            unsigned long long offset, const unsigned long long* step_ptr, void* stream) {
  DEER_CHECK_ARG(lengths, "rows_pad_fused_len: bad args");
  return rows_pad_fused(src, dst, hi, lo, B, T, C, lead, tail, dir, drop_p, seed, offset, step_ptr, lengths, lengths_i64,
                        stream);
}

int deer_rows_pad_colsum(const float* src, float* dst, float* colsum, int B, int T, int C, void* stream) {
  DEER_CHECK_ARG(src && dst && B > 0 && T > 0 && C > 0 && (C & 3) == 0, "rows_pad_colsum: bad args");   // colsum may be NULL
  DEER_CHECK_ARG(((reinterpret_cast<uintptr_t>(src) | reinterpret_cast<uintptr_t>(dst)) & 15) == 0, "rows_pad_colsum: alignment");
  const long long M = (long long)B * T;
  const int gx = (int)cdiv(C / 4, 32);
  long long want_gy = cdiv(8 * kNumSMs, gx);
  long long rpb = cdiv(M, want_gy);
  rpb = ((rpb + 7) / 8) * 8;
  if (rpb < 8) rpb = 8;
  dim3 grid((unsigned)gx, (unsigned)cdiv(M, rpb));
  DEER_LAUNCH(rows_pad_colsum_kernel, grid, dim3(32, 8), 0, stream, src, dst, colsum, B, T, C / 4, (int)rpb);
  return DEER_OK;
}

int deer_col2im3(const float* dcol, float* dx, int B, int T, int C, void* stream) {
  DEER_CHECK_ARG(dcol && dx && B > 0 && T > 0 && C > 0, "col2im3: bad args");
  DEER_LAUNCH(col2im3_kernel, grid_for((long long)B * T * C), 256, 0, stream, dcol, dx, B, T, C);
  return DEER_OK;
}

int deer_conv3_weight_pack(const float* w, float* wk, int Cout, int Cin, int dir, void* stream) {
  DEER_CHECK_ARG(w && wk && Cout > 0 && Cin > 0, "conv3_weight_pack: bad args");
  DEER_LAUNCH(conv3_pack_kernel, grid_for((long long)Cout * Cin * 3), 256, 0, stream, w, wk, Cout, Cin, dir);
  return DEER_OK;
}

int deer_axpby(const float* x1, const float* x2, float* y, long long n, float a, float b, void* stream) {
  DEER_CHECK_ARG(x1 && y && n > 0, "axpby: bad args");
  DEER_LAUNCH(axpby_kernel, grid_for(n), 256, 0, stream, x1, x2, y, n, a, b);
  return DEER_OK;
}

int deer_mix_fwd(const float* w, long long ldw, const float* u, long long ldu, const float* s, const float* c,
                 float* out, long long M, int N, void* stream) {
  DEER_CHECK_ARG(w && u && s && c && out && M > 0 && N > 0, "mix_fwd: bad args");
  DEER_LAUNCH(mix_fwd_kernel, grid_for(M * N), 256, 0, stream, w, ldw, u, ldu, s, c, out, M, N);
  return DEER_OK;
}

int deer_mix_bwd(const float* dout, const float* w, long long ldw, const float* u, long long ldu, const float* s,
                 const float* c, float* dw, long long lddw, float* du, long long lddu, float* ds, float* dc,
                 long long M, int N, void* stream) {
  DEER_CHECK_ARG(dout && w && u && s && c && dw && du && ds && dc && M > 0 && N > 0, "mix_bwd: bad args");
  DEER_LAUNCH(mix_bwd_kernel, (unsigned)cdiv(M, 8), 256, 0, stream, dout, w, ldw, u, ldu, s, c, dw, lddw, du, lddu, ds,
              dc, M, N);
  return DEER_OK;
}

int deer_gate_fwd(const float* g, const float* a, const float* b, float* out, long long n, void* stream) {
  DEER_CHECK_ARG(g && a && b && out && n > 0, "gate_fwd: bad args");
  DEER_LAUNCH(gate_fwd_kernel, grid_for(n), 256, 0, stream, g, a, b, out, n);
  return DEER_OK;
}

int deer_gate_bwd(const float* dout, const float* g, const float* a, const float* b, float* dg, float* da, float* db,
                  long long n, void* stream) {
  DEER_CHECK_ARG(dout && g && a && b && dg && da && db && n > 0, "gate_bwd: bad args");
  DEER_LAUNCH(gate_bwd_kernel, grid_for(n), 256, 0, stream, dout, g, a, b, dg, da, db, n);
  return DEER_OK;
}

int deer_softmax_rows_fwd(const float* x, float* y, long long M, int N, void* stream) {
  DEER_CHECK_ARG(x && y && M > 0 && N > 0 && N <= 32, "softmax_rows_fwd: bad args");
  DEER_LAUNCH(softmax_rows_fwd_kernel, (unsigned)cdiv(M, 256), 256, 0, stream, x, y, M, N);
  return DEER_OK;
}

int deer_softmax_rows_bwd(const float* dy, const float* y, float* dx, long long M, int N, void* stream) {
  DEER_CHECK_ARG(dy && y && dx && M > 0 && N > 0 && N <= 32, "softmax_rows_bwd: bad args");
  DEER_LAUNCH(softmax_rows_bwd_kernel, (unsigned)cdiv(M, 256), 256, 0, stream, dy, y, dx, M, N);
  return DEER_OK;
}

}  // extern "C"
