// LayerNorm (row-wise, one warp per row, row held in registers) and BatchNorm1d+ReLU on channels-last rows.
#include "common.cuh"

namespace deer {

constexpr int LN_MAX_PER_LANE = 32;  // N <= 1024 (kernels templated on 8/16/32 elements per lane)

template <int PL>
__global__ void __launch_bounds__(256) layernorm_fwd_kernel(const float* __restrict__ x,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ beta, float* __restrict__ y,
                                                            float* __restrict__ mean, float* __restrict__ rstd, int M,
                                                            int N, float eps) {
  DEER_PDL_ENTRY();
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float* xr = x + (long long)row * N;
  float v[PL];
  float s = 0.f;
#pragma unroll
  for (int i = 0; i < PL; i++) {
    const int j = lane + 32 * i;
    v[i] = j < N ? xr[j] : 0.f;
    s += v[i];
  }
  const float mu = warp_sum(s) / N;
  float q = 0.f;
#pragma unroll
  for (int i = 0; i < PL; i++) {
    const int j = lane + 32 * i;
    const float d = j < N ? v[i] - mu : 0.f;
    q = fmaf(d, d, q);
  }
  const float rs = rsqrtf(warp_sum(q) / N + eps);
  float* yr = y + (long long)row * N;
#pragma unroll
  for (int i = 0; i < PL; i++) {
    const int j = lane + 32 * i;
    if (j < N) yr[j] = (v[i] - mu) * rs * gamma[j] + beta[j];
  }
  if (lane == 0) {
    mean[row] = mu;
    rstd[row] = rs;
  }
}

// dx = rstd*(g - mean(g) - xhat*mean(g*xhat)), g = dy*gamma;  dgamma += sum_m dy*xhat;  dbeta += sum_m dy
template <int PL>
__global__ void __launch_bounds__(256) layernorm_bwd_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                            const float* __restrict__ gamma,
                                                            const float* __restrict__ mean,
                                                            const float* __restrict__ rstd, float* __restrict__ dx,
                                                            float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                            int M, int N, int rows_per_block) {
  DEER_PDL_ENTRY();
  extern __shared__ float sm[];  // [8][N] dgamma partials, [8][N] dbeta partials
  const int w = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int r0 = blockIdx.x * rows_per_block;
  const int r1 = min(M, r0 + rows_per_block);
  float ag[PL], ab[PL];
#pragma unroll
  for (int i = 0; i < PL; i++) ag[i] = ab[i] = 0.f;
  for (int row = r0 + w; row < r1; row += 8) {
    const float mu = mean[row], rs = rstd[row];
    const float* xr = x + (long long)row * N;
    const float* dr = dy + (long long)row * N;
    float xh[PL], g[PL];
    float s1 = 0.f, s2 = 0.f;
#pragma unroll
    for (int i = 0; i < PL; i++) {
      const int j = lane + 32 * i;
      if (j < N) {
        const float d = dr[j];
        xh[i] = (xr[j] - mu) * rs;
        g[i] = d * gamma[j];
        ag[i] = fmaf(d, xh[i], ag[i]);
        ab[i] += d;
        s1 += g[i];
        s2 = fmaf(g[i], xh[i], s2);
      } else {
        xh[i] = g[i] = 0.f;
      }
    }
    s1 = warp_sum(s1) / N;
    s2 = warp_sum(s2) / N;
    float* dxr = dx + (long long)row * N;
#pragma unroll
    for (int i = 0; i < PL; i++) {
      const int j = lane + 32 * i;
      if (j < N) dxr[j] = rs * (g[i] - s1 - xh[i] * s2);
    }
  }
  if (dgamma == nullptr) return;
  float* sg = sm;
  float* sb = sm + 8 * N;
#pragma unroll
  for (int i = 0; i < PL; i++) {
    const int j = lane + 32 * i;
    if (j < N) {
      sg[w * N + j] = ag[i];
      sb[w * N + j] = ab[i];
    }
  }
  __syncthreads();
  for (int j = threadIdx.x; j < N; j += blockDim.x) {
    float tg = 0.f, tb = 0.f;
#pragma unroll
    for (int k = 0; k < 8; k++) {
      tg += sg[k * N + j];
      tb += sb[k * N + j];
    }
    atomicAdd(dgamma + j, tg);
    atomicAdd(dbeta + j, tb);
  }
}

// ----------------------------------------------------------------------------- BatchNorm1d (channels-last rows)
// kLengths (per-utterance lengths, lengths [B] int32 / int64, rows m = b*T + t): the statistics cover the N = sum_b L_b valid
// rows only.  Padded rows (seq_row_valid false) are neither read nor counted, N is counted on the device into stats[2C]
// (stats [2C+1]: mean, biased var, N) and takes the place of M, the forward writes 0 and the backward dx = 0 at padded rows.
// Without lengths every row is valid and the kernels compile as they did before the flag.

// valid rows among [r0, r1)
__device__ long long seq_valid_rows(long long r0, long long r1, const void* lengths, int i64, int T) {
  long long n = 0;
  for (long long b = r0 / T; b * T < r1; b++) {
    const long long lo = max(r0, b * T), hi = min(r1, b * T + seq_length(lengths, i64, (int)b, T));
    if (hi > lo) n += hi - lo;
  }
  return n;
}

// mode 0: out[c] += sum_m x[m,c];  mode 1: out[c] += sum_m (x[m,c]-sum[c]/M)^2
// kLengths: mode 0 (out = stats) also adds the block's valid-row count to out[2C] (blocks of the first column group);
// mode 1 divides by that count (sum = stats)
template <bool kLengths>
__global__ void __launch_bounds__(256) bn_colreduce_kernel(const float* __restrict__ x, const float* __restrict__ sum,
                                                           float* __restrict__ out, long long M, int C, int mode,
                                                           int rows_per_block, const void* lengths, int lengths_i64,
                                                           int T) {
  DEER_PDL_ENTRY();
  __shared__ float red[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const long long r0 = (long long)blockIdx.y * rows_per_block;
  const long long r1 = min(M, r0 + (long long)rows_per_block);
  float s = 0.f;
  if (c < C) {
    const float mu = mode ? sum[c] / (kLengths ? sum[2 * C] : (float)M) : 0.f;
    for (long long m = r0 + threadIdx.y; m < r1; m += 8) {
      if (kLengths && !seq_row_valid(m, lengths, lengths_i64, T)) continue;
      const float d = x[m * C + c] - mu;
      s += mode ? d * d : d;
    }
  }
  if (kLengths && mode == 0 && blockIdx.x == 0 && threadIdx.x == 0 && threadIdx.y == 0)
    atomicAdd(out + 2 * C, (float)seq_valid_rows(r0, r1, lengths, lengths_i64, T));
  red[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) t += red[i][threadIdx.x];
    atomicAdd(out + c, t);
  }
}
template <bool kLengths>
__global__ void bn_finalize_kernel(float* stats, long long M, int C) {
  DEER_PDL_ENTRY();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    const float n = kLengths ? stats[2 * C] : (float)M;
    stats[c] /= n;
    stats[C + c] /= n;
  }
}
template <bool kLengths>
__global__ void bn_running_kernel(const float* __restrict__ stats, float* __restrict__ rm, float* __restrict__ rv,
                                  long long* __restrict__ nbt, long long M, int C, float momentum) {
  DEER_PDL_ENTRY();
  const int c = blockIdx.x * blockDim.x + threadIdx.x;
  if (c < C) {
    float unb = stats[C + c];
    if constexpr (kLengths) {
      const float n = stats[2 * C];
      if (n > 1.f) unb *= n / (n - 1.f);
    } else {
      unb = M > 1 ? stats[C + c] * ((float)M / (float)(M - 1)) : stats[C + c];
    }
    rm[c] = (1.f - momentum) * rm[c] + momentum * stats[c];
    rv[c] = (1.f - momentum) * rv[c] + momentum * unb;
  }
  if (c == 0 && nbt) *nbt += 1;
}

template <bool kLengths>
__global__ void __launch_bounds__(256) bn_relu_fwd_kernel(const float* __restrict__ x, const float* __restrict__ mean,
                                                          const float* __restrict__ var,
                                                          const float* __restrict__ gamma,
                                                          const float* __restrict__ beta, float* __restrict__ y,
                                                          long long M, int C, float eps, const void* lengths,
                                                          int lengths_i64, int T) {
  DEER_PDL_ENTRY();
  const long long total = M * C;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    if (kLengths && !seq_row_valid(i / C, lengths, lengths_i64, T)) {
      y[i] = 0.f;
      continue;
    }
    const int c = (int)(i % C);
    const float v = (x[i] - mean[c]) * rsqrtf(var[c] + eps) * gamma[c] + beta[c];
    y[i] = fmaxf(v, 0.f);
  }
}

// scratch[0][c] += sum_m g ; scratch[1][c] += sum_m g*xhat   with g = dy*(y>0)
// kLengths: padded rows are skipped, not read.  (Their g is 0 anyway, y being 0 there, but g*xhat would be 0*NaN for a
// NaN x: the reduction must not depend on the content of padded rows.)
template <bool kLengths>
__global__ void __launch_bounds__(256) bn_bwd_reduce_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                            const float* __restrict__ y,
                                                            const float* __restrict__ mean,
                                                            const float* __restrict__ var, float* __restrict__ scratch,
                                                            long long M, int C, float eps, int rows_per_block,
                                                            const void* lengths, int lengths_i64, int T) {
  DEER_PDL_ENTRY();
  __shared__ float r1s[8][33], r2s[8][33];
  const int c = blockIdx.x * 32 + threadIdx.x;
  const long long r0 = (long long)blockIdx.y * rows_per_block;
  const long long r1 = min(M, r0 + (long long)rows_per_block);
  float s1 = 0.f, s2 = 0.f;
  if (c < C) {
    const float mu = mean[c], rs = rsqrtf(var[c] + eps);
    for (long long m = r0 + threadIdx.y; m < r1; m += 8) {
      if (kLengths && !seq_row_valid(m, lengths, lengths_i64, T)) continue;
      const float g = y[m * C + c] > 0.f ? dy[m * C + c] : 0.f;
      s1 += g;
      s2 = fmaf(g, (x[m * C + c] - mu) * rs, s2);
    }
  }
  r1s[threadIdx.y][threadIdx.x] = s1;
  r2s[threadIdx.y][threadIdx.x] = s2;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    float t1 = 0.f, t2 = 0.f;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      t1 += r1s[i][threadIdx.x];
      t2 += r2s[i][threadIdx.x];
    }
    atomicAdd(scratch + c, t1);
    atomicAdd(scratch + C + c, t2);
  }
}
// kLengths: dx = 0 at padded rows; with batch_stats the count is N = mean[2C] (mean is the [2C+1] stats buffer)
template <bool kLengths>
__global__ void __launch_bounds__(256) bn_bwd_apply_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                           const float* __restrict__ y,
                                                           const float* __restrict__ mean,
                                                           const float* __restrict__ var,
                                                           const float* __restrict__ gamma,
                                                           const float* __restrict__ scratch, float* __restrict__ dx,
                                                           float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                           long long M, int C, float eps, int batch_stats,
                                                           const void* lengths, int lengths_i64, int T) {
  DEER_PDL_ENTRY();
  const long long total = M * C;
  const float invM = 1.f / (kLengths && batch_stats ? mean[2 * C] : (float)M);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    if (kLengths && !seq_row_valid(i / C, lengths, lengths_i64, T)) {
      dx[i] = 0.f;
      continue;
    }
    const int c = (int)(i % C);
    const float rs = rsqrtf(var[c] + eps);
    const float g = y[i] > 0.f ? dy[i] : 0.f;
    float v = g;
    if (batch_stats) v -= scratch[c] * invM + (x[i] - mean[c]) * rs * scratch[C + c] * invM;
    dx[i] = gamma[c] * rs * v;
  }
  if (blockIdx.x == 0) {
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      dbeta[c] += scratch[c];
      dgamma[c] += scratch[C + c];
    }
  }
}

// ---- 128-bit variants (C % 4 == 0, 16-byte aligned rows): four channels per thread, two rows in flight per trip.  The
// scalar kernels above moved 1.1-2 TB/s (one 4-byte load per tensor and trip in flight per thread).
__device__ __forceinline__ float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }

template <bool kLengths>
__global__ void __launch_bounds__(256) bn_colreduce_v4_kernel(const float* __restrict__ x, const float* __restrict__ sum,
                                                              float* __restrict__ out, long long M, int C, int mode,
                                                              int rows_per_block, const void* lengths, int lengths_i64,
                                                              int T) {
  DEER_PDL_ENTRY();
  __shared__ float4 red[8][33];
  const int c = (blockIdx.x * 32 + threadIdx.x) * 4;
  const long long r0 = (long long)blockIdx.y * rows_per_block;
  const long long r1 = min(M, r0 + (long long)rows_per_block);
  float4 s = make_float4(0.f, 0.f, 0.f, 0.f);
  if (c < C) {
    float4 mu = make_float4(0.f, 0.f, 0.f, 0.f);
    if (mode) {
      const float4 t = ld4(sum + c);
      const float inv = 1.f / (kLengths ? sum[2 * C] : (float)M);
      mu = make_float4(t.x * inv, t.y * inv, t.z * inv, t.w * inv);
    }
    // a padded row reads as mu: it adds 0 in both modes
    auto row = [&](long long m) {
      return kLengths && !seq_row_valid(m, lengths, lengths_i64, T) ? mu : ld4(x + m * C + c);
    };
    long long m = r0 + threadIdx.y;
    for (; m + 8 < r1; m += 16) {
      const float4 a = row(m), b = row(m + 8);
      const float4 da = make_float4(a.x - mu.x, a.y - mu.y, a.z - mu.z, a.w - mu.w);
      const float4 db = make_float4(b.x - mu.x, b.y - mu.y, b.z - mu.z, b.w - mu.w);
      if (mode) {
        s.x += da.x * da.x + db.x * db.x; s.y += da.y * da.y + db.y * db.y;
        s.z += da.z * da.z + db.z * db.z; s.w += da.w * da.w + db.w * db.w;
      } else {
        s.x += da.x + db.x; s.y += da.y + db.y; s.z += da.z + db.z; s.w += da.w + db.w;
      }
    }
    for (; m < r1; m += 8) {
      const float4 a = row(m);
      const float4 da = make_float4(a.x - mu.x, a.y - mu.y, a.z - mu.z, a.w - mu.w);
      if (mode) { s.x += da.x * da.x; s.y += da.y * da.y; s.z += da.z * da.z; s.w += da.w * da.w; }
      else { s.x += da.x; s.y += da.y; s.z += da.z; s.w += da.w; }
    }
  }
  if (kLengths && mode == 0 && blockIdx.x == 0 && threadIdx.x == 0 && threadIdx.y == 0)
    atomicAdd(out + 2 * C, (float)seq_valid_rows(r0, r1, lengths, lengths_i64, T));
  red[threadIdx.y][threadIdx.x] = s;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    float4 t = make_float4(0.f, 0.f, 0.f, 0.f);
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const float4 v = red[i][threadIdx.x];
      t.x += v.x; t.y += v.y; t.z += v.z; t.w += v.w;
    }
    atomicAdd(out + c, t.x); atomicAdd(out + c + 1, t.y); atomicAdd(out + c + 2, t.z); atomicAdd(out + c + 3, t.w);
  }
}

template <bool kLengths>
__global__ void __launch_bounds__(256) bn_relu_fwd_v4_kernel(const float* __restrict__ x, const float* __restrict__ mean,
                                                             const float* __restrict__ var,
                                                             const float* __restrict__ gamma,
                                                             const float* __restrict__ beta, float* __restrict__ y,
                                                             long long M, int C, float eps, const void* lengths,
                                                             int lengths_i64, int T) {
  DEER_PDL_ENTRY();
  const int C4 = C >> 2;
  const long long total = M * C4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    if (kLengths && !seq_row_valid(i / C4, lengths, lengths_i64, T)) {
      *reinterpret_cast<float4*>(y + i * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
      continue;
    }
    const int c = (int)(i % C4) * 4;
    const float4 v = ld4(x + i * 4), mu = ld4(mean + c), va = ld4(var + c), g = ld4(gamma + c), b = ld4(beta + c);
    float4 o;
    o.x = fmaxf((v.x - mu.x) * rsqrtf(va.x + eps) * g.x + b.x, 0.f);
    o.y = fmaxf((v.y - mu.y) * rsqrtf(va.y + eps) * g.y + b.y, 0.f);
    o.z = fmaxf((v.z - mu.z) * rsqrtf(va.z + eps) * g.z + b.z, 0.f);
    o.w = fmaxf((v.w - mu.w) * rsqrtf(va.w + eps) * g.w + b.w, 0.f);
    *reinterpret_cast<float4*>(y + i * 4) = o;
  }
}

template <bool kLengths>
__global__ void __launch_bounds__(256) bn_bwd_reduce_v4_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                               const float* __restrict__ y,
                                                               const float* __restrict__ mean,
                                                               const float* __restrict__ var, float* __restrict__ scratch,
                                                               long long M, int C, float eps, int rows_per_block,
                                                               const void* lengths, int lengths_i64, int T) {
  DEER_PDL_ENTRY();
  __shared__ float4 r1s[8][33], r2s[8][33];
  const int c = (blockIdx.x * 32 + threadIdx.x) * 4;
  const long long r0 = (long long)blockIdx.y * rows_per_block;
  const long long r1 = min(M, r0 + (long long)rows_per_block);
  float4 s1 = make_float4(0.f, 0.f, 0.f, 0.f), s2 = s1;
  if (c < C) {
    const float4 mu = ld4(mean + c), va = ld4(var + c);
    const float4 rs = make_float4(rsqrtf(va.x + eps), rsqrtf(va.y + eps), rsqrtf(va.z + eps), rsqrtf(va.w + eps));
    auto acc = [&](const float4& yy, const float4& dd, const float4& xx) {
      const float gx = yy.x > 0.f ? dd.x : 0.f, gy = yy.y > 0.f ? dd.y : 0.f;
      const float gz = yy.z > 0.f ? dd.z : 0.f, gw = yy.w > 0.f ? dd.w : 0.f;
      s1.x += gx; s1.y += gy; s1.z += gz; s1.w += gw;
      s2.x = fmaf(gx, (xx.x - mu.x) * rs.x, s2.x); s2.y = fmaf(gy, (xx.y - mu.y) * rs.y, s2.y);
      s2.z = fmaf(gz, (xx.z - mu.z) * rs.z, s2.z); s2.w = fmaf(gw, (xx.w - mu.w) * rs.w, s2.w);
    };
    // kLengths: a padded row is skipped (as in the scalar kernel), not read
    auto valid = [&](long long m) { return !kLengths || seq_row_valid(m, lengths, lengths_i64, T); };
    long long m = r0 + threadIdx.y;
    for (; m + 8 < r1; m += 16) {   // two rows (six 128-bit loads) in flight per trip
      const long long o0 = m * C + c, o1 = (m + 8) * C + c;
      if constexpr (kLengths) {
        const bool v0 = valid(m), v1 = valid(m + 8);
        if (v0) acc(ld4(y + o0), ld4(dy + o0), ld4(x + o0));
        if (v1) acc(ld4(y + o1), ld4(dy + o1), ld4(x + o1));
      } else {
        const float4 y0 = ld4(y + o0), d0 = ld4(dy + o0), x0 = ld4(x + o0);
        const float4 y1 = ld4(y + o1), d1 = ld4(dy + o1), x1 = ld4(x + o1);
        acc(y0, d0, x0);
        acc(y1, d1, x1);
      }
    }
    for (; m < r1; m += 8) {
      const long long o0 = m * C + c;
      if (valid(m)) acc(ld4(y + o0), ld4(dy + o0), ld4(x + o0));
    }
  }
  r1s[threadIdx.y][threadIdx.x] = s1;
  r2s[threadIdx.y][threadIdx.x] = s2;
  __syncthreads();
  if (threadIdx.y == 0 && c < C) {
    float4 t1 = make_float4(0.f, 0.f, 0.f, 0.f), t2 = t1;
#pragma unroll
    for (int i = 0; i < 8; i++) {
      const float4 a = r1s[i][threadIdx.x], b = r2s[i][threadIdx.x];
      t1.x += a.x; t1.y += a.y; t1.z += a.z; t1.w += a.w;
      t2.x += b.x; t2.y += b.y; t2.z += b.z; t2.w += b.w;
    }
    atomicAdd(scratch + c, t1.x); atomicAdd(scratch + c + 1, t1.y);
    atomicAdd(scratch + c + 2, t1.z); atomicAdd(scratch + c + 3, t1.w);
    atomicAdd(scratch + C + c, t2.x); atomicAdd(scratch + C + c + 1, t2.y);
    atomicAdd(scratch + C + c + 2, t2.z); atomicAdd(scratch + C + c + 3, t2.w);
  }
}

template <bool kLengths>
__global__ void __launch_bounds__(256) bn_bwd_apply_v4_kernel(const float* __restrict__ dy, const float* __restrict__ x,
                                                              const float* __restrict__ y,
                                                              const float* __restrict__ mean,
                                                              const float* __restrict__ var,
                                                              const float* __restrict__ gamma,
                                                              const float* __restrict__ scratch, float* __restrict__ dx,
                                                              float* __restrict__ dgamma, float* __restrict__ dbeta,
                                                              long long M, int C, float eps, int batch_stats,
                                                              const void* lengths, int lengths_i64, int T) {
  DEER_PDL_ENTRY();
  const int C4 = C >> 2;
  const long long total = M * C4;
  const float invM = 1.f / (kLengths && batch_stats ? mean[2 * C] : (float)M);
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    if (kLengths && !seq_row_valid(i / C4, lengths, lengths_i64, T)) {
      *reinterpret_cast<float4*>(dx + i * 4) = make_float4(0.f, 0.f, 0.f, 0.f);
      continue;
    }
    const int c = (int)(i % C4) * 4;
    const float4 va = ld4(var + c), mu = ld4(mean + c), ga = ld4(gamma + c);
    const float4 yy = ld4(y + i * 4), dd = ld4(dy + i * 4);
    const float4 rs = make_float4(rsqrtf(va.x + eps), rsqrtf(va.y + eps), rsqrtf(va.z + eps), rsqrtf(va.w + eps));
    float4 v = make_float4(yy.x > 0.f ? dd.x : 0.f, yy.y > 0.f ? dd.y : 0.f, yy.z > 0.f ? dd.z : 0.f,
                           yy.w > 0.f ? dd.w : 0.f);
    if (batch_stats) {
      const float4 xx = ld4(x + i * 4), sa = ld4(scratch + c), sb = ld4(scratch + C + c);
      v.x -= sa.x * invM + (xx.x - mu.x) * rs.x * sb.x * invM;
      v.y -= sa.y * invM + (xx.y - mu.y) * rs.y * sb.y * invM;
      v.z -= sa.z * invM + (xx.z - mu.z) * rs.z * sb.z * invM;
      v.w -= sa.w * invM + (xx.w - mu.w) * rs.w * sb.w * invM;
    }
    *reinterpret_cast<float4*>(dx + i * 4) = make_float4(ga.x * rs.x * v.x, ga.y * rs.y * v.y, ga.z * rs.z * v.z,
                                                         ga.w * rs.w * v.w);
  }
  if (blockIdx.x == 0) {
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      dbeta[c] += scratch[c];
      dgamma[c] += scratch[C + c];
    }
  }
}

static bool bn_vec4_ok(int C, const void* a, const void* b, const void* c, const void* d) {
  auto al = [](const void* q) { return q == nullptr || (reinterpret_cast<uintptr_t>(q) & 15) == 0; };
  return (C & 3) == 0 && al(a) && al(b) && al(c) && al(d);
}

// Host side of the plain and the per-utterance-length BatchNorm entries: one kernel source each, instantiated with and
// without lengths (lengths == nullptr: every row of the M = B*T is valid; T is then unused).
static int bn_stats(const float* x, float* stats, long long M, int C, const void* lengths, int lengths_i64, int T,
                    void* stream) {
  cudaError_t e = cudaMemsetAsync(stats, 0, sizeof(float) * (2 * C + (lengths ? 1 : 0)), (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_status(e, "bn_stats memset");
  const int rpb = 128;
  if (bn_vec4_ok(C, x, stats, nullptr, nullptr)) {
    auto k = lengths ? bn_colreduce_v4_kernel<true> : bn_colreduce_v4_kernel<false>;
    dim3 grid4((unsigned)cdiv(C, 128), (unsigned)cdiv(M, rpb));
    DEER_LAUNCH(k, grid4, dim3(32, 8), 0, stream, x, stats, stats, M, C, 0, rpb, lengths, lengths_i64, T);
    DEER_LAUNCH(k, grid4, dim3(32, 8), 0, stream, x, stats, stats + C, M, C, 1, rpb, lengths, lengths_i64, T);
  } else {
    auto k = lengths ? bn_colreduce_kernel<true> : bn_colreduce_kernel<false>;
    dim3 grid((unsigned)cdiv(C, 32), (unsigned)cdiv(M, rpb));
    DEER_LAUNCH(k, grid, dim3(32, 8), 0, stream, x, stats, stats, M, C, 0, rpb, lengths, lengths_i64, T);
    DEER_LAUNCH(k, grid, dim3(32, 8), 0, stream, x, stats, stats + C, M, C, 1, rpb, lengths, lengths_i64, T);
  }
  DEER_LAUNCH(lengths ? bn_finalize_kernel<true> : bn_finalize_kernel<false>, (unsigned)cdiv(C, 256), 256, 0, stream,
              stats, M, C);
  return DEER_OK;
}

static int bn_relu_fwd(const float* x, const float* mean, const float* var, const float* gamma, const float* beta,
                       float* y, long long M, int C, float eps, const void* lengths, int lengths_i64, int T,
                       void* stream) {
  if (bn_vec4_ok(C, x, y, mean, var) && bn_vec4_ok(C, gamma, beta, nullptr, nullptr)) {
    long long g4 = cdiv(M * (C / 4), 256);
    if (g4 > kNumSMs * 8) g4 = kNumSMs * 8;
    DEER_LAUNCH(lengths ? bn_relu_fwd_v4_kernel<true> : bn_relu_fwd_v4_kernel<false>, (unsigned)g4, 256, 0, stream, x,
                mean, var, gamma, beta, y, M, C, eps, lengths, lengths_i64, T);
    return DEER_OK;
  }
  long long g = cdiv(M * C, 256);
  if (g > kNumSMs * 16) g = kNumSMs * 16;
  DEER_LAUNCH(lengths ? bn_relu_fwd_kernel<true> : bn_relu_fwd_kernel<false>, (unsigned)g, 256, 0, stream, x, mean, var,
              gamma, beta, y, M, C, eps, lengths, lengths_i64, T);
  return DEER_OK;
}

static int bn_relu_bwd(const float* dy, const float* x, const float* y, const float* mean, const float* var,
                       const float* gamma, float* dx, float* dgamma, float* dbeta, float* scratch, long long M, int C,
                       float eps, int batch_stats, const void* lengths, int lengths_i64, int T, void* stream) {
  cudaError_t e = cudaMemsetAsync(scratch, 0, sizeof(float) * 2 * C, (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_status(e, "bn_relu_bwd memset");
  const int rpb = 128;
  if (bn_vec4_ok(C, dy, x, y, dx) && bn_vec4_ok(C, mean, var, gamma, scratch)) {
    dim3 grid4((unsigned)cdiv(C, 128), (unsigned)cdiv(M, rpb));
    DEER_LAUNCH(lengths ? bn_bwd_reduce_v4_kernel<true> : bn_bwd_reduce_v4_kernel<false>, grid4, dim3(32, 8), 0, stream,
                dy, x, y, mean, var, scratch, M, C, eps, rpb, lengths, lengths_i64, T);
    long long g4 = cdiv(M * (C / 4), 256);
    if (g4 > kNumSMs * 8) g4 = kNumSMs * 8;
    DEER_LAUNCH(lengths ? bn_bwd_apply_v4_kernel<true> : bn_bwd_apply_v4_kernel<false>, (unsigned)g4, 256, 0, stream, dy,
                x, y, mean, var, gamma, scratch, dx, dgamma, dbeta, M, C, eps, batch_stats, lengths, lengths_i64, T);
    return DEER_OK;
  }
  dim3 grid((unsigned)cdiv(C, 32), (unsigned)cdiv(M, rpb));
  DEER_LAUNCH(lengths ? bn_bwd_reduce_kernel<true> : bn_bwd_reduce_kernel<false>, grid, dim3(32, 8), 0, stream, dy, x, y,
              mean, var, scratch, M, C, eps, rpb, lengths, lengths_i64, T);
  long long g = cdiv(M * C, 256);
  if (g > kNumSMs * 16) g = kNumSMs * 16;
  DEER_LAUNCH(lengths ? bn_bwd_apply_kernel<true> : bn_bwd_apply_kernel<false>, (unsigned)g, 256, 0, stream, dy, x, y,
              mean, var, gamma, scratch, dx, dgamma, dbeta, M, C, eps, batch_stats, lengths, lengths_i64, T);
  return DEER_OK;
}

}  // namespace deer

using namespace deer;

extern "C" {

int deer_layernorm_fwd(const float* x, const float* gamma, const float* beta, float* y, float* mean, float* rstd,
                       int M, int N, float eps, void* stream) {
  DEER_CHECK_ARG(x && gamma && beta && y && mean && rstd && M > 0 && N > 0, "layernorm_fwd: bad args");
  if (N > 32 * LN_MAX_PER_LANE) {
    set_error("layernorm_fwd: N=%d > %d unsupported", N, 32 * LN_MAX_PER_LANE);
    return DEER_ERR_UNSUPPORTED;
  }
  if (N <= 256) DEER_LAUNCH(layernorm_fwd_kernel<8>, (unsigned)cdiv(M, 8), 256, 0, stream, x, gamma, beta, y, mean, rstd, M, N, eps);
  else if (N <= 512) DEER_LAUNCH(layernorm_fwd_kernel<16>, (unsigned)cdiv(M, 8), 256, 0, stream, x, gamma, beta, y, mean, rstd, M, N, eps);
  else DEER_LAUNCH(layernorm_fwd_kernel<32>, (unsigned)cdiv(M, 8), 256, 0, stream, x, gamma, beta, y, mean, rstd, M, N, eps);
  return DEER_OK;
}

int deer_layernorm_bwd(const float* dy, const float* x, const float* gamma, const float* mean, const float* rstd,
                       float* dx, float* dgamma, float* dbeta, int M, int N, void* stream) {
  DEER_CHECK_ARG(dy && x && gamma && mean && rstd && dx && M > 0 && N > 0, "layernorm_bwd: bad args");
  DEER_CHECK_ARG((dgamma == nullptr) == (dbeta == nullptr), "layernorm_bwd: dgamma/dbeta together");
  if (N > 32 * LN_MAX_PER_LANE) {
    set_error("layernorm_bwd: N=%d unsupported", N);
    return DEER_ERR_UNSUPPORTED;
  }
  // rows per block: one row per warp for the post-pooling layers (M = batch rows: 8 blocks of 32 rows left 140 SMs
  // idle and took 11 us), more rows per block as M grows so that the 2N atomics per block stay negligible
  const int rpb = M <= 1024 ? 8 : (M <= 4096 ? 16 : 32);
  const size_t smem = (size_t)16 * N * sizeof(float);
  static bool attr_set = false;
  if (!attr_set) {
    cudaFuncSetAttribute(layernorm_bwd_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 16 * 1024 * 4);
    attr_set = true;
  }
  if (N <= 256) DEER_LAUNCH(layernorm_bwd_kernel<8>, (unsigned)cdiv(M, rpb), 256, smem, stream, dy, x, gamma, mean, rstd, dx, dgamma, dbeta, M, N, rpb);
  else if (N <= 512) DEER_LAUNCH(layernorm_bwd_kernel<16>, (unsigned)cdiv(M, rpb), 256, smem, stream, dy, x, gamma, mean, rstd, dx, dgamma, dbeta, M, N, rpb);
  else DEER_LAUNCH(layernorm_bwd_kernel<32>, (unsigned)cdiv(M, rpb), 256, smem, stream, dy, x, gamma, mean, rstd, dx, dgamma, dbeta, M, N, rpb);
  return DEER_OK;
}

int deer_bn_stats(const float* x, float* stats, long long M, int C, void* stream) {
  DEER_CHECK_ARG(x && stats && M > 0 && C > 0, "bn_stats: bad args");
  return bn_stats(x, stats, M, C, nullptr, 0, 1, stream);
}

int deer_bn_stats_len(const float* x, float* stats, const void* lengths, int lengths_i64, int B, int T, int C,
                      void* stream) {
  DEER_CHECK_ARG(x && stats && lengths && B > 0 && T > 0 && C > 0, "bn_stats_len: bad args");
  return bn_stats(x, stats, (long long)B * T, C, lengths, lengths_i64, T, stream);
}

int deer_bn_update_running(const float* stats, float* running_mean, float* running_var, long long* num_batches_tracked,
                           long long M, int C, float momentum, void* stream) {
  DEER_CHECK_ARG(stats && running_mean && running_var && M > 0 && C > 0, "bn_update_running: bad args");
  DEER_LAUNCH(bn_running_kernel<false>, (unsigned)cdiv(C, 256), 256, 0, stream, stats, running_mean, running_var,
              num_batches_tracked, M, C, momentum);
  return DEER_OK;
}

int deer_bn_update_running_len(const float* stats, float* running_mean, float* running_var,
                               long long* num_batches_tracked, int C, float momentum, void* stream) {
  DEER_CHECK_ARG(stats && running_mean && running_var && C > 0, "bn_update_running_len: bad args");
  DEER_LAUNCH(bn_running_kernel<true>, (unsigned)cdiv(C, 256), 256, 0, stream, stats, running_mean, running_var,
              num_batches_tracked, 0LL, C, momentum);
  return DEER_OK;
}

int deer_bn_relu_fwd(const float* x, const float* mean, const float* var, const float* gamma, const float* beta,
                     float* y, long long M, int C, float eps, void* stream) {
  DEER_CHECK_ARG(x && mean && var && gamma && beta && y && M > 0 && C > 0, "bn_relu_fwd: bad args");
  return bn_relu_fwd(x, mean, var, gamma, beta, y, M, C, eps, nullptr, 0, 1, stream);
}

int deer_bn_relu_fwd_len(const float* x, const float* mean, const float* var, const float* gamma, const float* beta,
                         float* y, const void* lengths, int lengths_i64, int B, int T, int C, float eps, void* stream) {
  DEER_CHECK_ARG(x && mean && var && gamma && beta && y && lengths && B > 0 && T > 0 && C > 0,
                 "bn_relu_fwd_len: bad args");
  return bn_relu_fwd(x, mean, var, gamma, beta, y, (long long)B * T, C, eps, lengths, lengths_i64, T, stream);
}

int deer_bn_relu_bwd(const float* dy, const float* x, const float* y, const float* mean, const float* var,
                     const float* gamma, float* dx, float* dgamma, float* dbeta, float* scratch, long long M, int C,
                     float eps, int batch_stats, void* stream) {
  DEER_CHECK_ARG(dy && x && y && mean && var && gamma && dx && dgamma && dbeta && scratch && M > 0 && C > 0,
                 "bn_relu_bwd: bad args");
  return bn_relu_bwd(dy, x, y, mean, var, gamma, dx, dgamma, dbeta, scratch, M, C, eps, batch_stats, nullptr, 0, 1,
                     stream);
}

int deer_bn_relu_bwd_len(const float* dy, const float* x, const float* y, const float* mean, const float* var,
                         const float* gamma, float* dx, float* dgamma, float* dbeta, float* scratch, const void* lengths,
                         int lengths_i64, int B, int T, int C, float eps, int batch_stats, void* stream) {
  DEER_CHECK_ARG(dy && x && y && mean && var && gamma && dx && dgamma && dbeta && scratch && lengths && B > 0 && T > 0 &&
                     C > 0 && (!batch_stats || var == mean + C),
                 "bn_relu_bwd_len: bad args");
  return bn_relu_bwd(dy, x, y, mean, var, gamma, dx, dgamma, dbeta, scratch, (long long)B * T, C, eps, batch_stats,
                     lengths, lengths_i64, T, stream);
}

}  // extern "C"
