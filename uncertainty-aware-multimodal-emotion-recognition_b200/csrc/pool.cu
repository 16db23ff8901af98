// Attention pooling over time: softmax over T of per-step scores (optionally masked + renormalised) and the
// weighted sum of the [B,T,D] activations.  HBM-bound: x is read exactly once per direction (fwd: once;
// bwd: once, dx written once), float4-vectorised along D, strides generic so the time-major LSTM output
// [T,B,D] and batch-first [B,T,D] tensors use the same kernel.
#include "common.cuh"

namespace deer {

constexpr int POOL_MAX_T = 2048;

// softmax (and optional mask/renorm) of one row of scores into shared memory p[T]; returns nothing, syncs.
__device__ void row_softmax_to_smem(const float* s, long long ss_t, const float* mask_row, int T, float* p,
                                    float* red) {
  float mx = -INFINITY;
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    const float v = s[t * ss_t];
    p[t] = v;
    mx = fmaxf(mx, v);
  }
  // block max
  mx = warp_max(mx);
  __syncthreads();
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = mx;
  __syncthreads();
  {
    const int nw = (blockDim.x + 31) >> 5;
    float r = (threadIdx.x & 31) < nw ? red[threadIdx.x & 31] : -INFINITY;
    mx = warp_max(r);
  }
  float sum = 0.f;
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    const float e = expf(p[t] - mx);
    p[t] = e;
    sum += e;
  }
  sum = block_sum(sum, red);
  const float inv = 1.f / sum;
  if (mask_row == nullptr) {
    for (int t = threadIdx.x; t < T; t += blockDim.x) p[t] *= inv;
    __syncthreads();
  } else {
    float z = 0.f;
    for (int t = threadIdx.x; t < T; t += blockDim.x) {
      const float u = p[t] * inv * mask_row[t];
      p[t] = u;
      z += u;
    }
    z = block_sum(z, red) + 1e-10f;
    const float iz = 1.f / z;
    for (int t = threadIdx.x; t < T; t += blockDim.x) p[t] *= iz;
    __syncthreads();
  }
}

// grid (B, ceil(D/128)); block 256 = 8 warps x 32 lanes; lane owns one float4 column of the 128-wide D chunk,
// warp w takes t = w, w+8, ...
// kLengths (lengths set, mask not): softmax and weighted sum over each sample's own frames t < L_b only -- padded rows of
// x and s are never read (the bytes read scale with sum_b L_b) and wts is 0 there.
template <bool kLengths>
__global__ void __launch_bounds__(256) attn_pool_fwd_kernel(const float* __restrict__ x, long long xs_b,
                                                            long long xs_t, const float* __restrict__ s,
                                                            long long ss_b, long long ss_t,
                                                            const float* __restrict__ mask, const void* lengths,
                                                            int lengths_i64, float* __restrict__ out,
                                                            float* __restrict__ wts, int B, int T, int D, int premask) {
  DEER_PDL_ENTRY();
  __shared__ float p[POOL_MAX_T];
  __shared__ float red[32];
  __shared__ float4 part[8][32];
  if constexpr (kLengths) {  // lengths exclude a mask: constants here, so this instantiation carries none of its code
    mask = nullptr;
    premask = 0;
  }
  const int b = blockIdx.x;
  const int L = kLengths ? seq_length(lengths, lengths_i64, b, T) : T;
  row_softmax_to_smem(s + b * ss_b, ss_t, mask ? mask + (long long)b * T : nullptr, L, p, red);
  if (blockIdx.y == 0 && wts)
    for (int t = threadIdx.x; t < T; t += blockDim.x) wts[(long long)b * T + t] = t < L ? p[t] : 0.f;
  if (premask) {
    // the pooled rows are x~[b,t] = mask[b,t] x[b,t] (encoders.py:733-735): fold the factor into the weights of the sum
    // instead of materialising x~ (a read + write of the whole [B,T,D] tensor)
    __syncthreads();
    for (int t = threadIdx.x; t < T; t += blockDim.x) p[t] *= mask[(long long)b * T + t];
    __syncthreads();
  }
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int c4 = blockIdx.y * 32 + lane;  // float4 column
  float4 acc = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c4 * 4 < D) {
    const float* xb = x + b * xs_b + c4 * 4;
    int t = w;
    for (; t + 24 < L; t += 32) {  // 4 independent loads in flight
      const float4 v0 = *reinterpret_cast<const float4*>(xb + (long long)t * xs_t);
      const float4 v1 = *reinterpret_cast<const float4*>(xb + (long long)(t + 8) * xs_t);
      const float4 v2 = *reinterpret_cast<const float4*>(xb + (long long)(t + 16) * xs_t);
      const float4 v3 = *reinterpret_cast<const float4*>(xb + (long long)(t + 24) * xs_t);
      const float p0 = p[t], p1 = p[t + 8], p2 = p[t + 16], p3 = p[t + 24];
      acc.x += p0 * v0.x + p1 * v1.x + p2 * v2.x + p3 * v3.x;
      acc.y += p0 * v0.y + p1 * v1.y + p2 * v2.y + p3 * v3.y;
      acc.z += p0 * v0.z + p1 * v1.z + p2 * v2.z + p3 * v3.z;
      acc.w += p0 * v0.w + p1 * v1.w + p2 * v2.w + p3 * v3.w;
    }
    for (; t < L; t += 8) {
      const float4 v = *reinterpret_cast<const float4*>(xb + (long long)t * xs_t);
      const float pt = p[t];
      acc.x += pt * v.x;
      acc.y += pt * v.y;
      acc.z += pt * v.z;
      acc.w += pt * v.w;
    }
  }
  part[w][lane] = acc;
  __syncthreads();
  if (w == 0 && c4 * 4 < D) {
    float4 r = part[0][lane];
#pragma unroll
    for (int k = 1; k < 8; k++) {
      const float4 q = part[k][lane];
      r.x += q.x;
      r.y += q.y;
      r.z += q.z;
      r.w += q.w;
    }
    *reinterpret_cast<float4*>(out + (long long)b * D + c4 * 4) = r;
  }
}

// one block per b. warp per t: dw_t = x_t . dout ; dx_t (+)= w_t * dout ; then softmax(/mask) backward -> ds.
// kLengths (lengths set; mask, premask and accumulate not): the same over t < L_b, with dx = 0 (overwritten) and ds = 0
// at padded rows -- that dx is the dh the BPTT kernel reads, where uninitialised memory would turn into NaN through
// 0 * NaN.
template <bool kLengths>
__global__ void __launch_bounds__(256) attn_pool_bwd_kernel(const float* __restrict__ dout, const float* __restrict__ x,
                                                            long long xs_b, long long xs_t,
                                                            const float* __restrict__ s, long long ss_b,
                                                            long long ss_t, const float* __restrict__ mask,
                                                            const void* lengths, int lengths_i64,
                                                            const float* __restrict__ wts, float* __restrict__ dx,
                                                            float* __restrict__ ds, int B, int T, int D,
                                                            int accumulate, int premask) {
  DEER_PDL_ENTRY();
  __shared__ float dw[POOL_MAX_T];
  __shared__ float p[POOL_MAX_T];
  __shared__ float red[32];
  if constexpr (kLengths) {  // lengths exclude a mask and accumulate, as in forward
    mask = nullptr;
    premask = 0;
    accumulate = 0;
  }
  const int b = blockIdx.x;
  const int L = kLengths ? seq_length(lengths, lengths_i64, b, T) : T;
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const float* dob = dout + (long long)b * D;
  const float* xb = x + b * xs_b;
  float* dxb = dx + b * xs_b;
  const float* wb = wts + (long long)b * T;
  for (int t = w; t < L; t += 8) {
    // premask: the pooled rows are x~ = mask x, so dw_t = mask_t (x_t . dout) and dx_t = mask_t w_t dout
    const float mt = premask ? mask[(long long)b * T + t] : 1.f;
    const float wt = wb[t] * mt;
    float acc = 0.f;
    for (int c = lane * 4; c < D; c += 128) {
      const float4 g = *reinterpret_cast<const float4*>(dob + c);
      const float4 v = *reinterpret_cast<const float4*>(xb + (long long)t * xs_t + c);
      acc += g.x * v.x + g.y * v.y + g.z * v.z + g.w * v.w;
      if (dx == nullptr) continue;           // x needs no gradient (an input tensor): only ds is produced
      float4* dp = reinterpret_cast<float4*>(dxb + (long long)t * xs_t + c);
      float4 o = make_float4(wt * g.x, wt * g.y, wt * g.z, wt * g.w);
      if (accumulate) {
        const float4 old = *dp;
        o.x += old.x;
        o.y += old.y;
        o.z += old.z;
        o.w += old.w;
      }
      *dp = o;
    }
    acc = warp_sum(acc) * mt;
    if (lane == 0) dw[t] = acc;
  }
  if (dx != nullptr)
    for (int t = L + w; t < T; t += 8)
      for (int c = lane * 4; c < D; c += 128)
        *reinterpret_cast<float4*>(dxb + (long long)t * xs_t + c) = make_float4(0.f, 0.f, 0.f, 0.f);
  __syncthreads();
  // dot = sum_t w_t dw_t
  float d = 0.f;
  for (int t = threadIdx.x; t < L; t += blockDim.x) d = fmaf(wb[t], dw[t], d);
  d = block_sum(d, red);
  float* dsb = ds + b * ss_b;
  if (mask == nullptr) {
    for (int t = threadIdx.x; t < T; t += blockDim.x) dsb[t * ss_t] = t < L ? wb[t] * (dw[t] - d) : 0.f;
    return;
  }
  // masked: p = softmax(s); u = p*m; Z = sum u + 1e-10; w = u/Z
  const float* mb = mask + (long long)b * T;
  __syncthreads();
  row_softmax_to_smem(s + b * ss_b, ss_t, nullptr, T, p, red);
  float z = 0.f;
  for (int t = threadIdx.x; t < T; t += blockDim.x) z = fmaf(p[t], mb[t], z);
  z = block_sum(z, red) + 1e-10f;
  const float iz = 1.f / z;
  // dp_t = (dw_t - d) * m_t / Z ; ds_t = p_t (dp_t - sum_j p_j dp_j)
  float e = 0.f;
  for (int t = threadIdx.x; t < T; t += blockDim.x) {
    const float dpt = (dw[t] - d) * mb[t] * iz;
    dw[t] = dpt;
    e = fmaf(p[t], dpt, e);
  }
  e = block_sum(e, red);
  for (int t = threadIdx.x; t < T; t += blockDim.x) dsb[t * ss_t] = p[t] * (dw[t] - e);
}

// Host side of the plain and the per-utterance-length entries: one kernel source each way, instantiated with and without
// lengths (compile-time, DESIGN.md 4.12: a run-time bound in place of T slowed the forward's load loop).  Lengths exclude
// mask (a mask renormalises after the full softmax) and accumulate (the lengths backward overwrites dx at padded rows).
static int pool_fwd(const char* what, const float* x, long long xs_b, long long xs_t, const float* s, long long ss_b,
                    long long ss_t, const float* mask, const void* lengths, int lengths_i64, float* out, float* wts,
                    int B, int T, int D, int premask, void* stream) {
  DEER_CHECK_ARG(!(lengths && mask), "attn_pool: mask and lengths together");
  if (T > POOL_MAX_T || (D & 3) || (xs_b & 3) || (xs_t & 3)) {
    set_error("%s: need T<=%d and D, strides multiples of 4 (T=%d D=%d)", what, POOL_MAX_T, T, D);
    return DEER_ERR_UNSUPPORTED;
  }
  dim3 grid(B, (unsigned)cdiv(D, 128));
  DEER_LAUNCH(lengths ? attn_pool_fwd_kernel<true> : attn_pool_fwd_kernel<false>, grid, 256, 0, stream, x, xs_b, xs_t,
              s, ss_b, ss_t, mask, lengths, lengths_i64, out, wts, B, T, D, premask);
  return DEER_OK;
}

static int pool_bwd(const char* what, const float* dout, const float* x, long long xs_b, long long xs_t, const float* s,
                    long long ss_b, long long ss_t, const float* mask, const void* lengths, int lengths_i64,
                    const float* wts, float* dx, float* ds, int B, int T, int D, int accumulate, int premask,
                    void* stream) {
  DEER_CHECK_ARG(!(lengths && (mask || accumulate)), "attn_pool: lengths with mask or accumulate");
  if (T > POOL_MAX_T || (D & 3) || (xs_b & 3) || (xs_t & 3)) {
    set_error("%s: need T<=%d and D, strides multiples of 4 (T=%d D=%d)", what, POOL_MAX_T, T, D);
    return DEER_ERR_UNSUPPORTED;
  }
  DEER_LAUNCH(lengths ? attn_pool_bwd_kernel<true> : attn_pool_bwd_kernel<false>, B, 256, 0, stream, dout, x, xs_b,
              xs_t, s, ss_b, ss_t, mask, lengths, lengths_i64, wts, dx, ds, B, T, D, accumulate, premask);
  return DEER_OK;
}

}  // namespace deer

using namespace deer;

extern "C" {

int deer_attn_pool_fwd(const float* x, long long xs_b, long long xs_t, const float* s, long long ss_b, long long ss_t,
                       const float* mask, float* out, float* wts, int B, int T, int D, int premask, void* stream) {
  DEER_CHECK_ARG(x && s && out && B > 0 && T > 0 && D > 0 && (!premask || mask), "attn_pool_fwd: bad args");
  return pool_fwd("attn_pool_fwd", x, xs_b, xs_t, s, ss_b, ss_t, mask, nullptr, 0, out, wts, B, T, D, premask, stream);
}

int deer_attn_pool_bwd(const float* dout, const float* x, long long xs_b, long long xs_t, const float* s, long long ss_b,
                       long long ss_t, const float* mask, const float* wts, float* dx, float* ds, int B, int T, int D,
                       int accumulate, int premask, void* stream) {
  DEER_CHECK_ARG(dout && x && s && wts && ds && B > 0 && T > 0 && D > 0 && (!premask || mask), "attn_pool_bwd: bad args");
  return pool_bwd("attn_pool_bwd", dout, x, xs_b, xs_t, s, ss_b, ss_t, mask, nullptr, 0, wts, dx, ds, B, T, D,
                  accumulate, premask, stream);
}

int deer_attn_pool_len_fwd(const float* x, long long xs_b, long long xs_t, const float* s, long long ss_b, long long ss_t,
                           const void* lengths, int lengths_i64, float* out, float* wts, int B, int T, int D,
                           void* stream) {
  DEER_CHECK_ARG(x && s && lengths && out && B > 0 && T > 0 && D > 0, "attn_pool_len_fwd: bad args");
  return pool_fwd("attn_pool_len_fwd", x, xs_b, xs_t, s, ss_b, ss_t, nullptr, lengths, lengths_i64, out, wts, B, T, D,
                  0, stream);
}

int deer_attn_pool_len_bwd(const float* dout, const float* x, long long xs_b, long long xs_t, long long ss_b,
                           long long ss_t, const void* lengths, int lengths_i64, const float* wts, float* dx, float* ds,
                           int B, int T, int D, void* stream) {
  DEER_CHECK_ARG(dout && x && lengths && wts && ds && B > 0 && T > 0 && D > 0, "attn_pool_len_bwd: bad args");
  return pool_bwd("attn_pool_len_bwd", dout, x, xs_b, xs_t, nullptr, ss_b, ss_t, nullptr, lengths, lengths_i64, wts, dx,
                  ds, B, T, D, 0, 0, stream);
}

}  // extern "C"
