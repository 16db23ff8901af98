// Normal-Inverse-Gamma head + DEER loss, fused.
//
//   head   (deer.py:90-98, complete_project.py:399-407): gamma=e0, nu=softplus(e1)+1e-6, alpha=softplus(e2)+1,
//          beta=softplus(e3)+1e-6, aleatoric=beta/(alpha-1), epistemic=beta/(nu(alpha-1)).
//   loss   (losses.py:72-348): per dimension  nll + reg_w*reg + kl_w*kl + ece_w*ece, cross-dimension consistency,
//          divided by the number of dimensions.  Exact formulas: SURVEY.md appendix A.
//
// Two streaming phases over flat (sample,dim) elements, element e = b*D + d, one float4 of evidence each:
//   phase 1 (deer_nig_loss_stats)  reads 16 B evidence + 4 B target, optionally writes 7x4 B NIG outputs, and
//           reduces 35 statistics per dimension (sums for nll/reg/kl/mean-u, 10 ECE bins x {count, sum conf,
//           sum |err|}).  Scalar sums live in registers across the grid-stride loop; ECE bins live in
//           per-thread-private shared-memory columns (no atomics in the loop); one block reduction and
//           35*D global atomics per block at the end.
//   phase 2 (deer_nig_loss_finish) turns the statistics into the loss scalars (block 0) and streams the
//           analytic gradient: reads 16+4 B, writes 16 B per element.
// A data-parallel caller all-reduces `stats` between the phases (B_global = global batch).
//
// Partially labelled batches (kMask, deer_nig_loss_*_mask): one more byte per element, target_mask[e] != 0 = labelled.
// Phase 1 substitutes gamma for the target of an unlabelled element (err = 0: every intermediate stays finite whatever
// the target holds) and SELECTS its statistic contributions and ECE bin update to nothing (0 * NaN would be NaN); it
// counts the labelled elements of each dimension into statistic 35.  Phase 2 divides by that per-dimension N_d instead
// of B_global, forms the cross-dimension term over the dimensions with N_d > 0 and stores a zero gradient at
// unlabelled elements.  The kMask = false instantiations are the kernels of the plain entries, unchanged.
#include "common.cuh"

namespace deer {

constexpr int NSTAT = DEER_LOSS_NSTAT;  // 0 nll,1 reg,2 kl_alpha,3 kl_beta,4 sum u, 5..14 cnt, 15..24 conf, 25..34 err,
                                        // 35 labelled count (mask entries only)
constexpr int LOSS_THREADS = 192;       // multiple of every supported D (1,2,3,4,6,8)
constexpr int LOSS_MIN_BLOCKS = 5;      // 64 registers: two P2 pairs in flight per thread without spills
constexpr int LOSS_MIN_BLOCKS_PIPE = 4; // 80 registers: + the next trip's operands (software-pipelined loads)
constexpr int NBINS = 10;
constexpr long long DEER_NIG_MAX_ELEMENTS = (1ll << 31) - (1ll << 24);  // 32-bit element indices + unroll slack
constexpr long long DEER_NIG_L2_KEEP_BYTES = 72ll << 20;  // operand footprint up to which pass 1 pins its loads in L2

// ------------------------------------------------------------------------------------------------------------------
// Value types.  The loss passes are instruction-ISSUE bound (ncu: 60-73 % issue-active, DRAM at 45-55 %), and two thirds
// of what they issue is fp32 add / mul / fma.  Blackwell's packed fp32 instructions (add/mul/fma.f32x2 -> FADD2 /
// FMUL2 / FFMA2) do two lanes' worth of that arithmetic per issue slot, so every thread processes its elements in
// PAIRS: P2 holds the same quantity of two independent (sample, dim) elements, arithmetic goes through the packed
// instructions, and the per-component work (MUFU, selects, compares, bin updates) stays scalar.  The math below is
// written once, templated on the value type V = float (tail elements) or P2 (pairs): identical numerics.
struct P2 {
  float x, y;
  __device__ __forceinline__ P2() {}
  __device__ __forceinline__ P2(float a) : x(a), y(a) {}
  __device__ __forceinline__ P2(float a, float b) : x(a), y(b) {}
};
#define DEER_P2_BIN(NAME, PTX)                                                                                          \
  __device__ __forceinline__ P2 NAME(P2 a, P2 b) {                                                                      \
    P2 o;                                                                                                               \
    asm("{\n\t.reg .b64 ra, rb, ro;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\t" PTX                          \
        " ro, ra, rb;\n\tmov.b64 {%0, %1}, ro;\n\t}"                                                                    \
        : "=f"(o.x), "=f"(o.y)                                                                                          \
        : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y));                                                                      \
    return o;                                                                                                           \
  }
DEER_P2_BIN(operator+, "add.f32x2")
DEER_P2_BIN(operator-, "sub.f32x2")
DEER_P2_BIN(operator*, "mul.f32x2")
#undef DEER_P2_BIN
__device__ __forceinline__ P2 vfma(P2 a, P2 b, P2 c) {
  P2 o;
  asm("{\n\t.reg .b64 ra, rb, rc, ro;\n\tmov.b64 ra, {%2, %3};\n\tmov.b64 rb, {%4, %5};\n\tmov.b64 rc, {%6, %7};\n\t"
      "fma.rn.f32x2 ro, ra, rb, rc;\n\tmov.b64 {%0, %1}, ro;\n\t}"
      : "=f"(o.x), "=f"(o.y)
      : "f"(a.x), "f"(a.y), "f"(b.x), "f"(b.y), "f"(c.x), "f"(c.y));
  return o;
}
__device__ __forceinline__ float vfma(float a, float b, float c) { return fmaf(a, b, c); }
struct M2 {
  bool x, y;
};
// single MUFU instructions with flush-to-zero semantics (no denormal pre/post-scaling around ex2/lg2/rcp); relative
// error ~1e-6, far inside the 1e-3 gate
__device__ __forceinline__ float fex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float flg2(float x) {
  float y;
  asm("lg2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float frcp(float x) {
  float y;
  asm("rcp.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ float vrcp(float x) { return frcp(x); }
__device__ __forceinline__ P2 vrcp(P2 a) { return P2(frcp(a.x), frcp(a.y)); }
__device__ __forceinline__ float vlog(float x) { return flg2(x) * 0.6931471805599453f; }
__device__ __forceinline__ P2 vlog(P2 a) { return P2(flg2(a.x), flg2(a.y)) * P2(0.6931471805599453f); }
// exp(-|x|): the -|.| is an operand modifier of the MUFU instruction
__device__ __forceinline__ float vexp_negabs(float x) { return fex2(-fabsf(x * 1.4426950408889634f)); }
__device__ __forceinline__ P2 vexp_negabs(P2 a) {
  const P2 t = a * P2(1.4426950408889634f);
  return P2(fex2(-fabsf(t.x)), fex2(-fabsf(t.y)));
}
__device__ __forceinline__ float vmax0(float x) { return fmaxf(x, 0.f); }
__device__ __forceinline__ P2 vmax0(P2 a) { return P2(fmaxf(a.x, 0.f), fmaxf(a.y, 0.f)); }
__device__ __forceinline__ float vmin(float x, float c) { return fminf(x, c); }
__device__ __forceinline__ P2 vmin(P2 a, float c) { return P2(fminf(a.x, c), fminf(a.y, c)); }
__device__ __forceinline__ float vabs(float x) { return fabsf(x); }
__device__ __forceinline__ P2 vabs(P2 a) { return P2(fabsf(a.x), fabsf(a.y)); }
__device__ __forceinline__ bool vgt(float a, float c) { return a > c; }
__device__ __forceinline__ M2 vgt(P2 a, float c) { return M2{a.x > c, a.y > c}; }
__device__ __forceinline__ bool vlt(float a, float c) { return a < c; }
__device__ __forceinline__ M2 vlt(P2 a, float c) { return M2{a.x < c, a.y < c}; }
__device__ __forceinline__ bool vge(float a, float c) { return a >= c; }
__device__ __forceinline__ M2 vge(P2 a, float c) { return M2{a.x >= c, a.y >= c}; }
__device__ __forceinline__ float vsel(bool m, float a, float b) { return m ? a : b; }
__device__ __forceinline__ P2 vsel(M2 m, P2 a, P2 b) { return P2(m.x ? a.x : b.x, m.y ? a.y : b.y); }
// sign(err) * s  (0 at err == 0)
__device__ __forceinline__ float vsignmul(float err, float s) { return err > 0.f ? s : (err < 0.f ? -s : 0.f); }
__device__ __forceinline__ P2 vsignmul(P2 err, P2 s) { return P2(vsignmul(err.x, s.x), vsignmul(err.y, s.y)); }
__device__ __forceinline__ float hsum(float a) { return a; }
__device__ __forceinline__ float hsum(P2 a) { return a.x + a.y; }

template <class V>
struct NigT {
  V gamma, nu, alpha, beta;
  V sn, sa, sb;  // softplus'(raw) of nu / alpha / beta (chain rule back to the evidence)
};

// softplus(x) (torch: beta=1, threshold=20) and its derivative sigmoid(x) from ONE exponential e = exp(-|x|):
//   softplus = max(x,0) + log1p(e),  log1p(e) = log(u) + (e - (u - 1)) / u with u = fl(1 + e): the first-order
//   correction of the rounding of 1 + e (both differences are exact in fp32), reusing the reciprocal sigmoid needs
template <class V>
__device__ __forceinline__ void softplus_fast(V x, V& sp, V& sg) {
  const V e = vexp_negabs(x);
  const V u = V(1.f) + e;
  const V r = vrcp(u);
  const V l = vfma(e - (u - V(1.f)), r, vlog(u));
  // torch's linear branch (x > 20 -> x, derivative 1) needs no select in fp32: there log1p(e) < 2.1e-9 is below half an
  // ulp of x (>= 9.5e-7), so x + l == x, and r = 1 / (1 + e) rounds to exactly 1
  sp = vmax0(x) + l;
  sg = vsel(vge(x, 0.f), r, e * r);
}
// lgamma(a), a >= 1: shift a < 5 by 4 with one product, then Stirling through a^-7 (truncation < 5e-10 at a = 5;
// fp32 rounding of (a-1/2) ln a dominates: < 1e-6 absolute for a in [1, 1e5])
template <class V>
__device__ __forceinline__ V lgamma_ge1_fast(V a) {
  const auto sh = vlt(a, 5.f);
  const V as = vsel(sh, a, V(1.f));
  const V lp = vsel(sh, vlog((as * (as + V(1.f))) * ((as + V(2.f)) * (as + V(3.f)))), V(0.f));
  a = vsel(sh, a + V(4.f), a);
  const V r = vrcp(a), r2 = r * r;
  // r * (1/12 - r2 (1/360 - r2 (1/1260 - r2/1680))), Horner with signed coefficients
  const V s = r * vfma(r2, vfma(r2, vfma(r2, V(-0.000595238095f), V(0.000793650794f)), V(-0.00277777778f)),
                       V(0.0833333333f));
  return vfma(a - V(0.5f), vlog(a), V(0.918938533f) - a) + (s - lp);
}
// digamma(x), x >= 1: psi(x) = psi(x+4) - sum_{i<4} 1/(x+i), the sum as ONE quotient p'(x)/p(x); series through (x+4)^-8
template <class V>
__device__ __forceinline__ V digamma_ge1_fast(V x) {
  // the shift is applied for every x (it is exact); the shift terms use min(x, 1e6) so that p * x cannot overflow:
  // beyond 1e6 that changes psi by < 4e-6 absolute (psi > 13.8 there)
  const V t0 = vmin(x, 1e6f), t1 = t0 + V(1.f), t2 = t0 + V(2.f), t3 = t0 + V(3.f);
  const V p01 = t0 * t1, p23 = t2 * t3;
  // d/dx [t0 t1 t2 t3] = (t0 + t1) p23 + (t2 + t3) p01
  const V p = p01 * p23;
  x = x + V(4.f);
  const V R = vrcp(p * x);  // one MUFU for both 1/p and 1/x
  const V corr = vfma(t0 + t1, p23, (t2 + t3) * p01) * (x * R);
  const V r = p * R, r2 = r * r;
  // r2 (1/12 - r2 (1/120 - r2 (1/252 - r2/240))), Horner with signed coefficients
  const V ser = r2 * vfma(r2, vfma(r2, vfma(r2, V(-0.00416666667f), V(0.00396825397f)), V(-0.00833333333f)),
                          V(0.0833333333f));
  return vfma(r, V(-0.5f), vlog(x)) - ser - corr;
}

// raw operands of one (sample, dim) element; fetched for several elements before any of them is processed so that
// each thread keeps LOSS_UNROLL independent 128-bit loads in flight (the kernels are otherwise latency-bound)
struct RawNig {
  float4 v;  // evidence, or (gamma, nu, alpha, beta)
  float y;   // target (gamma when unlabelled)
  bool lab;  // labelled (always true without a mask)
};
// L2 residency control.  The loss is two passes over the same 20 B per element; when the operands fit in L2 the first
// pass loads them with an evict_last policy so that the second pass (streaming loads, which demote the lines again) is
// served from L2 and HBM sees each operand once.
__device__ __forceinline__ unsigned long long l2_evict_last_policy() {
  unsigned long long pol;
  asm volatile("createpolicy.fractional.L2::evict_last.b64 %0, 1.0;" : "=l"(pol));
  return pol;
}
__device__ __forceinline__ float4 ld_keep_f4(const float4* p, unsigned long long pol) {
  float4 v;
  asm volatile("ld.global.L2::cache_hint.v4.f32 {%0, %1, %2, %3}, [%4], %5;"
               : "=f"(v.x), "=f"(v.y), "=f"(v.z), "=f"(v.w)
               : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ float ld_keep_f(const float* p, unsigned long long pol) {
  float v;
  asm volatile("ld.global.L2::cache_hint.f32 %0, [%1], %2;" : "=f"(v) : "l"(p), "l"(pol));
  return v;
}
__device__ __forceinline__ unsigned ld_keep_u8(const unsigned char* p, unsigned long long pol) {
  unsigned v;
  asm volatile("ld.global.L2::cache_hint.u8 %0, [%1], %2;" : "=r"(v) : "l"(p), "l"(pol));
  return v;
}
template <bool KEEP, bool from_evidence, bool kMask>
__device__ __forceinline__ RawNig fetch_nig(const float* __restrict__ evidence, const float* __restrict__ gamma,
                                            const float* __restrict__ nu, const float* __restrict__ alpha,
                                            const float* __restrict__ beta, const float* __restrict__ targets,
                                            const unsigned char* __restrict__ mask, int e, unsigned long long pol) {
  RawNig r;
  r.lab = true;
  if (KEEP) {
    if (from_evidence) r.v = ld_keep_f4(reinterpret_cast<const float4*>(evidence) + e, pol);
    else r.v = make_float4(ld_keep_f(gamma + e, pol), ld_keep_f(nu + e, pol), ld_keep_f(alpha + e, pol),
                           ld_keep_f(beta + e, pol));
    r.y = ld_keep_f(targets + e, pol);
  } else {
    if (from_evidence) r.v = __ldcs(reinterpret_cast<const float4*>(evidence) + e);
    else r.v = make_float4(__ldcs(gamma + e), __ldcs(nu + e), __ldcs(alpha + e), __ldcs(beta + e));
    r.y = __ldcs(targets + e);
  }
  if (kMask) {
    r.lab = (KEEP ? ld_keep_u8(mask + e, pol) : (unsigned)__ldcs(mask + e)) != 0u;
    r.y = r.lab ? r.y : r.v.x;   // a select: the unlabelled target value never enters the math
  }
  return r;
}
// (e0, e1, e2, e3) of one element (V = float) or of two elements side by side (V = P2)
template <bool from_evidence, class V>
__device__ __forceinline__ NigT<V> derive_nig(V e0, V e1, V e2, V e3) {
  NigT<V> p;
  p.sn = p.sa = p.sb = V(1.f);
  p.gamma = e0;
  if (from_evidence) {
    V sp;
    softplus_fast(e1, sp, p.sn);
    p.nu = sp + V(1e-6f);
    softplus_fast(e2, sp, p.sa);
    p.alpha = sp + V(1.0f);
    softplus_fast(e3, sp, p.sb);
    p.beta = sp + V(1e-6f);
  } else {
    p.nu = e1;
    p.alpha = e2;
    p.beta = e3;
  }
  return p;
}
constexpr int LOSS_UNROLL = 4;   // elements in flight per thread = two P2 pairs

__device__ __forceinline__ int ece_bin(float conf, const float* __restrict__ edges) {
  // (edges[k], edges[k+1]]  (losses.py:207-215); -1 when outside every bin (NaN / conf <= 0 / conf > 1)
  // closed-form guess, then at most one step against the exact fp32 edges (torch.linspace(0,1,11), losses.py:207)
  int k = min(max(__float2int_ru(conf * 10.f) - 1, 0), NBINS - 1);
  k += (int)(conf > edges[k + 1]) - (int)!(conf > edges[k]);
  return (conf > 0.f && conf <= 1.f) ? k : -1;
}

struct NigPlanes {
  float* p[7];  // gamma, nu, alpha, beta, aleatoric, epistemic, total: [B*D] each
};

// ---- phase 1, per-value math (everything that is plain arithmetic); the bin update / stores stay per component
template <class V>
struct StatsOut {
  V nll, reg, kla, klb, u, conf, aerr;   // contributions to the five sums; confidence and |err| for the ECE bins
  V alea, epis;                          // head outputs (when requested)
};
template <class V>
__device__ __forceinline__ StatsOut<V> stats_math(const NigT<V>& p, V y, float eps, float inv_two_pi_eps, float log1eps,
                                                  bool eps_is_1e8, int nig_out) {
  StatsOut<V> o;
  const V err = y - p.gamma;
  const V e2 = err * err;
  const V S = vfma(p.nu * V(0.5f), e2, p.beta + V(eps));
  const V lb = vlog(p.beta + V(eps));
  const V lp = vfma(vlog(p.nu * V(inv_two_pi_eps)), V(0.5f), p.alpha * lb) - lgamma_ge1_fast(p.alpha + V(eps)) -
               (p.alpha + V(0.5f)) * vlog(S);
  o.nll = V(0.f) - lp;
  o.reg = e2 * vfma(p.nu, e2, p.beta + p.beta);
  const V am1 = p.alpha - V(1.f);
  o.kla = am1 * am1;
  const V dl = lb - V(log1eps);
  o.klb = dl * dl;
  const V den = am1 + V(eps);
  const V dpb = den + p.beta;
  const V rdc = vrcp(den * dpb);  // 1/den and conf = 1/(1+u) = den/(den+beta) from one reciprocal
  const V u = p.beta * (dpb * rdc);
  o.u = eps_is_1e8 ? u : p.beta * vrcp(am1 + V(1e-8f));
  o.conf = den * (den * rdc);
  o.aerr = vabs(err);
  if (nig_out) {
    const V ran = vrcp(am1 * p.nu);
    o.alea = p.beta * (p.nu * ran);
    o.epis = p.beta * ran;
  }
  return o;
}

// element indices are 32-bit inside the kernels (the entry points reject B*D >= 2^31 - grid slack)
// from_evidence is a template parameter: as a runtime flag both load variants were emitted predicated, and the
// predicated-off half still took ~10 issue slots per element
// kMask: partially labelled batch (mask appended to the parameter list, so the plain instantiations keep their layout)
template <bool KEEP, bool from_evidence, bool PIPE, bool kMask>
__global__ void __launch_bounds__(LOSS_THREADS, PIPE ? LOSS_MIN_BLOCKS_PIPE : LOSS_MIN_BLOCKS) nig_loss_stats_kernel(
    const float* __restrict__ evidence, const float* __restrict__ gamma, const float* __restrict__ nu,
    const float* __restrict__ alpha, const float* __restrict__ beta, const float* __restrict__ targets,
    const float* __restrict__ bin_edges, float* __restrict__ stats, const NigPlanes planes, int nig_out, int total, int D,
    float eps, const unsigned char* __restrict__ mask) {
  DEER_PDL_ENTRY();
  constexpr int NRED = kMask ? 6 : 5;     // register sums reduced through shared memory (+ the labelled count)
  constexpr int NRS = 30 + NRED;          // statistics written per dimension
  __shared__ float bins[3 * NBINS][LOSS_THREADS];  // private column per thread: conflict-free, no atomics
  __shared__ float sedges[NBINS + 1];
  __shared__ float red[NRED][LOSS_THREADS];
  const int tid = threadIdx.x;
  if (tid <= NBINS) sedges[tid] = bin_edges[tid];
#pragma unroll
  for (int i = 0; i < 3 * NBINS; i++) bins[i][tid] = 0.f;
  __syncthreads();
  const float inv_two_pi_eps = (float)(1.0 / (6.283185307179586 + (double)eps));
  const float log1eps = logf(1.f + eps);
  const bool eps_is_1e8 = eps == 1e-8f;
  P2 a_nll(0.f), a_reg(0.f), a_kla(0.f), a_klb(0.f), a_u(0.f);   // per-component partial sums, folded at the end
  float a_n = 0.f;                                                 // kMask: labelled elements seen by this thread
  const unsigned long long pol = KEEP ? l2_evict_last_policy() : 0ull;
  const int stride = (int)gridDim.x * LOSS_THREADS;  // multiple of D -> dimension fixed per thread
  // a statistic contribution, selected to 0 at an unlabelled element
  auto keep = [&](auto v, auto m) {
    if constexpr (kMask) return vsel(m, v, decltype(v)(0.f));
    else return v;
  };
  auto tail = [&](float conf, float aerr, const NigT<float>& p, float alea, float epis, int e, bool lab) {
    const int k = ece_bin(conf, sedges);
    if (k >= 0 && lab) {
      bins[k][tid] += 1.f;
      bins[NBINS + k][tid] += conf;
      bins[2 * NBINS + k][tid] += aerr;
    }
    if (nig_out) {
      // plane bases live in the constant bank: one IMAD.WIDE per store address
      __stcs(planes.p[0] + e, p.gamma);
      __stcs(planes.p[1] + e, p.nu);
      __stcs(planes.p[2] + e, p.alpha);
      __stcs(planes.p[3] + e, p.beta);
      __stcs(planes.p[4] + e, alea);
      __stcs(planes.p[5] + e, epis);
      __stcs(planes.p[6] + e, alea + epis);
    }
  };
  auto pair = [&](const RawNig& r0, const RawNig& r1, int e0, int e1) {
    const NigT<P2> p = derive_nig<from_evidence>(P2(r0.v.x, r1.v.x), P2(r0.v.y, r1.v.y), P2(r0.v.z, r1.v.z),
                                                 P2(r0.v.w, r1.v.w));
    const StatsOut<P2> o = stats_math(p, P2(r0.y, r1.y), eps, inv_two_pi_eps, log1eps, eps_is_1e8, nig_out);
    const M2 m{r0.lab, r1.lab};
    a_nll = a_nll + keep(o.nll, m);
    a_reg = a_reg + keep(o.reg, m);
    a_kla = a_kla + keep(o.kla, m);
    a_klb = a_klb + keep(o.klb, m);
    a_u = a_u + keep(o.u, m);
    if constexpr (kMask) a_n += (r0.lab ? 1.f : 0.f) + (r1.lab ? 1.f : 0.f);
    NigT<float> q0, q1;
    q0.gamma = p.gamma.x; q0.nu = p.nu.x; q0.alpha = p.alpha.x; q0.beta = p.beta.x;
    q1.gamma = p.gamma.y; q1.nu = p.nu.y; q1.alpha = p.alpha.y; q1.beta = p.beta.y;
    tail(o.conf.x, o.aerr.x, q0, o.alea.x, o.epis.x, e0, r0.lab);
    tail(o.conf.y, o.aerr.y, q1, o.alea.y, o.epis.y, e1, r1.lab);
  };
  auto single = [&](const RawNig& r, int e) {
    const NigT<float> p = derive_nig<from_evidence>(r.v.x, r.v.y, r.v.z, r.v.w);
    const StatsOut<float> o = stats_math(p, r.y, eps, inv_two_pi_eps, log1eps, eps_is_1e8, nig_out);
    a_nll.x += keep(o.nll, r.lab);
    a_reg.x += keep(o.reg, r.lab);
    a_kla.x += keep(o.kla, r.lab);
    a_klb.x += keep(o.klb, r.lab);
    a_u.x += keep(o.u, r.lab);
    if constexpr (kMask) a_n += r.lab ? 1.f : 0.f;
    tail(o.conf, o.aerr, p, o.alea, o.epis, e, r.lab);
  };
  int eb = (int)blockIdx.x * LOSS_THREADS + tid;
  if constexpr (PIPE) {
    // software pipeline: the loads of trip i+1 are issued before trip i is computed, so every warp keeps 80 bytes per
    // thread in flight WHILE it computes (with load -> compute -> load the memory system idles during the math)
    bool have = eb + (LOSS_UNROLL - 1) * stride < total;
    RawNig rr[LOSS_UNROLL];
    if (have) {
#pragma unroll
      for (int q = 0; q < LOSS_UNROLL; q++)
        rr[q] = fetch_nig<KEEP, from_evidence, kMask>(evidence, gamma, nu, alpha, beta, targets, mask,
                                                      eb + q * stride, pol);
    }
    while (have) {
      const int en = eb + LOSS_UNROLL * stride;
      const bool more = en + (LOSS_UNROLL - 1) * stride < total;
      RawNig nx[LOSS_UNROLL];
      if (more) {
#pragma unroll
        for (int q = 0; q < LOSS_UNROLL; q++)
          nx[q] = fetch_nig<KEEP, from_evidence, kMask>(evidence, gamma, nu, alpha, beta, targets, mask,
                                                        en + q * stride, pol);
      }
#pragma unroll
      for (int q = 0; q < LOSS_UNROLL; q += 2) pair(rr[q], rr[q + 1], eb + q * stride, eb + (q + 1) * stride);
      if (more) {
#pragma unroll
        for (int q = 0; q < LOSS_UNROLL; q++) rr[q] = nx[q];
      }
      eb = en;
      have = more;
    }
  } else {
    for (; eb + (LOSS_UNROLL - 1) * stride < total; eb += LOSS_UNROLL * stride) {
      RawNig rr[LOSS_UNROLL];
#pragma unroll
      for (int q = 0; q < LOSS_UNROLL; q++)
        rr[q] = fetch_nig<KEEP, from_evidence, kMask>(evidence, gamma, nu, alpha, beta, targets, mask,
                                                      eb + q * stride, pol);
#pragma unroll
      for (int q = 0; q < LOSS_UNROLL; q += 2) pair(rr[q], rr[q + 1], eb + q * stride, eb + (q + 1) * stride);
    }
  }
  for (; eb < total; eb += stride)
    single(fetch_nig<KEEP, from_evidence, kMask>(evidence, gamma, nu, alpha, beta, targets, mask, eb, pol), eb);
  red[0][tid] = hsum(a_nll);
  red[1][tid] = hsum(a_reg);
  red[2][tid] = hsum(a_kla);
  red[3][tid] = hsum(a_klb);
  red[4][tid] = hsum(a_u);
  if constexpr (kMask) red[NRED - 1][tid] = a_n;
  __syncthreads();
  // thread (d, s) for s < NRS sums the columns of threads whose dimension is d (tid % D == d)
  const int first_e_dim = ((int)blockIdx.x * LOSS_THREADS) % D;
  for (int w = tid; w < D * NRS; w += LOSS_THREADS) {
    const int d = w / NRS, s = w % NRS;
    // threads t with (first_e_dim + t) % D == d
    int t0 = (d - first_e_dim) % D;
    if (t0 < 0) t0 += D;
    float acc = 0.f;
    const float* src = s < 5 ? red[s] : (kMask && s == 35 ? red[NRED - 1] : bins[s - 5]);
    for (int t = t0; t < LOSS_THREADS; t += D) acc += src[t];
    if (acc != 0.f) atomicAdd(stats + d * NSTAT + s, acc);
  }
}

struct DimCoef {
  float sign[NBINS];  // ECE bin signs
  float cross;        // d cross_dim / d ubar_d
  float w;            // task weight
};

// ---- phase 2, per-value math: d total / d (gamma, nu, alpha, beta) up to the ECE term (which needs the element's bin)
template <class V>
struct GradOut {
  V dg, dn, da, db;
  V conf, u, rden, err;   // for the ECE / cross-dimension terms
};
template <class V>
__device__ __forceinline__ GradOut<V> grad_math(const NigT<V>& p, V y, float eps, float log1eps, float reg_w, float kl_w) {
  GradOut<V> o;
  const V err = y - p.gamma, e2 = err * err;
  const V S = vfma(p.nu * V(0.5f), e2, p.beta + V(eps));
  const V ah = p.alpha + V(0.5f);
  const V be = p.beta + V(eps);
  // reciprocals in pairs: 1/a = b * rcp(ab), 1/b = a * rcp(ab) (the MUFU pipe is the busiest one in this kernel)
  const V rSb = vrcp(S * be);
  const V rS = be * rSb, rbe = S * rSb, lbe = vlog(be);
  const V am1 = p.alpha - V(1.f);
  const V den = am1 + V(eps);
  const V rnd = vrcp(p.nu * den);
  const V rnu = den * rnd, rden = p.nu * rnd;
  const V ahrS = ah * rS;
  // nll + reg + kl
  //   dg = -ah nu err / S            - reg_w (4 beta err + 4 nu e2 err)
  //   dn = -1/(2 nu) + ah e2 / (2 S) + reg_w e2^2
  //   da = -log(be) + psi(alpha+eps) + log S + kl_w 2 (alpha - 1)
  //   db = -alpha / be + ah / S      + reg_w 2 e2 + kl_w 0.2 (log be - log(1+eps)) / be
  const V nue2 = p.nu * e2;
  o.dg = V(0.f) - err * vfma(V(4.f * reg_w), p.beta + nue2, ahrS * p.nu);
  o.dn = vfma(e2, vfma(V(reg_w), e2, ahrS * V(0.5f)), rnu * V(-0.5f));
  o.da = vfma(V(2.f * kl_w), am1, digamma_ge1_fast(p.alpha + V(eps)) + (vlog(S) - lbe));
  o.db = vfma(V(2.f * reg_w), e2, ahrS) + rbe * vfma(V(0.2f * kl_w), lbe - V(log1eps), V(0.f) - p.alpha);
  o.u = p.beta * rden;
  o.conf = vrcp(V(1.f) + o.u);
  o.rden = rden;
  o.err = err;
  return o;
}

// kMask: the means of dimension d are over its N_d labelled elements (statistic 35; B_global is not used), the
// cross-dimension term covers the dimensions with N_d > 0, and unlabelled elements get a zero gradient
template <bool from_evidence, bool PIPE, bool kMask>
__global__ void __launch_bounds__(LOSS_THREADS, PIPE ? LOSS_MIN_BLOCKS_PIPE : LOSS_MIN_BLOCKS) nig_loss_finish_kernel(
    const float* __restrict__ evidence, const float* __restrict__ gamma, const float* __restrict__ nu,
    const float* __restrict__ alpha, const float* __restrict__ beta, const float* __restrict__ targets,
    const float* __restrict__ bin_edges, const float* __restrict__ stats, const float* __restrict__ task_weights,
    float reg_w, float kl_w, float ece_w, float cross_w, float eps, int total_local, long long B_global, int D,
    float grad_scale, float* __restrict__ losses, float* __restrict__ d_out, const unsigned char* __restrict__ mask,
    float* __restrict__ counts) {
  DEER_PDL_ENTRY();
  __shared__ DimCoef coef[8];
  __shared__ float sedges[NBINS + 1];
  __shared__ float ubar[8];
  __shared__ float sinvn[kMask ? 8 : 1];   // kMask: 1 / N_d, 0 for a dimension without labels
  const int tid = threadIdx.x;
  const float invN = 1.f / (float)B_global;
  if (tid <= NBINS) sedges[tid] = bin_edges[tid];
  if (tid < D) {
    if constexpr (kMask) {
      const float n = stats[tid * NSTAT + 35];
      sinvn[tid] = n > 0.f ? 1.f / n : 0.f;
      ubar[tid] = stats[tid * NSTAT + 4] * sinvn[tid];
    } else {
      ubar[tid] = stats[tid * NSTAT + 4] * invN;
    }
  }
  __syncthreads();
  auto inv_n = [&](int d) -> float {
    if constexpr (kMask) return sinvn[d];
    else return invN;
  };
  auto present = [&](int d) -> bool {   // dimension d takes part in the cross-dimension term
    if constexpr (kMask) return sinvn[d] > 0.f;
    else return true;
  };
  auto num_pairs = [&]() -> int {   // pairs of dimensions in the cross-dimension term
    int n = D;
    if constexpr (kMask) {
      n = 0;
      for (int j = 0; j < D; j++) n += present(j) ? 1 : 0;
    }
    return n * (n - 1) / 2;
  };
  __shared__ float ece_part[8][NBINS];
  if (tid < D * NBINS) {  // one thread per (dimension, bin): no serial chain of dependent global loads and divisions
    const int dd = tid / NBINS, k = tid % NBINS;
    const float* st = stats + dd * NSTAT;
    const float cnt = st[5 + k], sc = st[15 + k], se = st[25 + k];
    float sg = 0.f, part = 0.f;
    if (cnt > 0.f) {
      const float diff = sc / cnt - (1.f - se / cnt);
      part = (cnt * inv_n(dd)) * fabsf(diff);
      sg = diff > 0.f ? 1.f : (diff < 0.f ? -1.f : 0.f);
    }
    coef[dd].sign[k] = sg;
    ece_part[dd][k] = part;
  }
  if (tid < D) {
    float cs = 0.f;
    for (int j = 0; j < D; j++)
      if (j != tid && present(j)) cs += ubar[tid] - ubar[j];
    const int npairs = num_pairs();
    coef[tid].cross = (npairs > 0 && present(tid)) ? 2.f * cs / (float)npairs : 0.f;
    coef[tid].w = task_weights ? task_weights[tid] : 1.f;
  }
  __syncthreads();
  if (blockIdx.x == 0 && losses) {
    if (tid < D) {
      const float* st = stats + tid * NSTAT;
      float ece = 0.f;
      for (int k = 0; k < NBINS; k++) ece += ece_part[tid][k];
      const float in = inv_n(tid);   // a dimension without labels: every sum is 0, and so is every entry
      const float nll = st[0] * in, reg = st[1] * in;
      const float kl = st[2] * in + 0.1f * st[3] * in;
      float* L = losses + tid * 5;
      L[0] = nll + reg_w * reg + kl_w * kl + ece_w * ece;
      L[1] = nll;
      L[2] = reg;
      L[3] = kl;
      L[4] = ece;
      if (kMask && counts) counts[tid] = st[35];
    }
    __syncthreads();
    if (tid == 0) {
      float cd = 0.f;
      for (int i = 0; i < D; i++)
        for (int j = i + 1; j < D; j++)
          if (present(i) && present(j)) cd += (ubar[i] - ubar[j]) * (ubar[i] - ubar[j]);
      const int npairs = num_pairs();
      if (npairs > 0) cd /= (float)npairs;
      float tot = 0.f;
      for (int i = 0; i < D; i++) tot += coef[i].w * losses[i * 5];
      if (cross_w > 0.f && D > 1) tot += cross_w * cd;
      losses[D * 5] = cd;
      losses[D * 5 + 1] = tot / (float)D;
    }
  }
  if (d_out == nullptr) return;
  const float invD = 1.f / (float)D;
  const float log1eps = logf(1.f + eps);
  const int stride = (int)gridDim.x * LOSS_THREADS;  // multiple of D: the dimension is fixed per thread
  const int d = ((int)blockIdx.x * LOSS_THREADS + tid) % D;
  const float w = coef[d].w;
  const float base_w = grad_scale * invD * inv_n(d) * w;   // task weight folded into the output scale
  const bool eps_is_1e8 = eps == 1e-8f;
  // cross-dimension term enters UNWEIGHTED by the task weight: pre-divide by w where w != 0 (w == 0: term dropped,
  // handled by the separate scale below)
  const float cross_c = (cross_w > 0.f && D > 1) ? cross_w * coef[d].cross : 0.f;
  const float base = grad_scale * invD * inv_n(d);
  const float ece_on = ece_w > 0.f ? ece_w : 0.f;
  const float* __restrict__ sgn = coef[d].sign;
  // ECE bin sign of one element (scalar: a bin search and a shared-memory lookup), pre-multiplied by the ECE weight
  auto bin_sign = [&](float conf) -> float {
    const int k = ece_bin(conf, sedges);
    return k >= 0 ? sgn[max(k, 0)] * ece_on : 0.f;
  };
  // ECE and cross-dimension corrections, task weight, chain rule back to the evidence: value-typed like the rest
  auto finish = [&](auto g, const auto& p, auto sg, auto m) {
    using V = decltype(g.dg);
    if (ece_on > 0.f) {  // uniform
      const V t = V(0.f) - sg * (g.conf * g.conf) * g.rden;  // sg * dconf/du * 1/den
      g.db = g.db + t;
      g.da = g.da - t * g.u;
      g.dg = g.dg - vsignmul(g.err, sg);
    }
    V ox = g.dg * V(base_w), oy = g.dn * V(base_w), oz = g.da * V(base_w), ow = g.db * V(base_w);
    // cross-dimension consistency: d/d ubar_d * (1/N) * du/d(alpha,beta), u = beta/(alpha-1+1e-8); not task-weighted
    if (cross_c != 0.f) {  // uniform
      const V r8 = eps_is_1e8 ? g.rden : vrcp((p.alpha - V(1.f)) + V(1e-8f));  // same denominator under the default epsilon
      const V cb = r8 * V(base * cross_c);
      ow = ow + cb;
      oz = oz - cb * (p.beta * r8);
    }
    if (from_evidence) {
      oy = oy * p.sn;
      oz = oz * p.sa;
      ow = ow * p.sb;
    }
    if constexpr (kMask) {   // exactly 0 at an unlabelled element
      ox = vsel(m, ox, V(0.f));
      oy = vsel(m, oy, V(0.f));
      oz = vsel(m, oz, V(0.f));
      ow = vsel(m, ow, V(0.f));
    }
    g.dg = ox; g.dn = oy; g.da = oz; g.db = ow;
    return g;
  };
  auto pair = [&](const RawNig& r0, const RawNig& r1, int e0, int e1) {
    const NigT<P2> p = derive_nig<from_evidence>(P2(r0.v.x, r1.v.x), P2(r0.v.y, r1.v.y), P2(r0.v.z, r1.v.z),
                                                 P2(r0.v.w, r1.v.w));
    GradOut<P2> g = grad_math(p, P2(r0.y, r1.y), eps, log1eps, reg_w, kl_w);
    const P2 sg = ece_on > 0.f ? P2(bin_sign(g.conf.x), bin_sign(g.conf.y)) : P2(0.f);
    g = finish(g, p, sg, M2{r0.lab, r1.lab});
    __stcs(reinterpret_cast<float4*>(d_out) + e0, make_float4(g.dg.x, g.dn.x, g.da.x, g.db.x));
    __stcs(reinterpret_cast<float4*>(d_out) + e1, make_float4(g.dg.y, g.dn.y, g.da.y, g.db.y));
  };
  auto single = [&](const RawNig& r, int e) {
    const NigT<float> p = derive_nig<from_evidence>(r.v.x, r.v.y, r.v.z, r.v.w);
    GradOut<float> g = grad_math(p, r.y, eps, log1eps, reg_w, kl_w);
    const float sg = ece_on > 0.f ? bin_sign(g.conf) : 0.f;
    g = finish(g, p, sg, r.lab);
    __stcs(reinterpret_cast<float4*>(d_out) + e, make_float4(g.dg, g.dn, g.da, g.db));
  };
  int eb = (int)blockIdx.x * LOSS_THREADS + tid;
  if constexpr (PIPE) {   // software-pipelined like phase 1
    bool have = eb + (LOSS_UNROLL - 1) * stride < total_local;
    RawNig rr[LOSS_UNROLL];
    if (have) {
#pragma unroll
      for (int q = 0; q < LOSS_UNROLL; q++)
        rr[q] = fetch_nig<false, from_evidence, kMask>(evidence, gamma, nu, alpha, beta, targets, mask,
                                                       eb + q * stride, 0ull);
    }
    while (have) {
      const int en = eb + LOSS_UNROLL * stride;
      const bool more = en + (LOSS_UNROLL - 1) * stride < total_local;
      RawNig nx[LOSS_UNROLL];
      if (more) {
#pragma unroll
        for (int q = 0; q < LOSS_UNROLL; q++)
          nx[q] = fetch_nig<false, from_evidence, kMask>(evidence, gamma, nu, alpha, beta, targets, mask,
                                                         en + q * stride, 0ull);
      }
#pragma unroll
      for (int q = 0; q < LOSS_UNROLL; q += 2) pair(rr[q], rr[q + 1], eb + q * stride, eb + (q + 1) * stride);
      if (more) {
#pragma unroll
        for (int q = 0; q < LOSS_UNROLL; q++) rr[q] = nx[q];
      }
      eb = en;
      have = more;
    }
  } else {
    for (; eb + (LOSS_UNROLL - 1) * stride < total_local; eb += LOSS_UNROLL * stride) {
      RawNig rr[LOSS_UNROLL];
#pragma unroll
      for (int q = 0; q < LOSS_UNROLL; q++)
        rr[q] = fetch_nig<false, from_evidence, kMask>(evidence, gamma, nu, alpha, beta, targets, mask,
                                                       eb + q * stride, 0ull);
#pragma unroll
      for (int q = 0; q < LOSS_UNROLL; q += 2) pair(rr[q], rr[q + 1], eb + q * stride, eb + (q + 1) * stride);
    }
  }
  for (; eb < total_local; eb += stride)
    single(fetch_nig<false, from_evidence, kMask>(evidence, gamma, nu, alpha, beta, targets, mask, eb, 0ull), eb);
}

// ------------------------------------------------------------------ stand-alone head
__global__ void __launch_bounds__(256) nig_head_fwd_kernel(const float* __restrict__ evidence, float* __restrict__ mu,
                                                           float* __restrict__ nu, float* __restrict__ alpha,
                                                           float* __restrict__ beta, float* __restrict__ alea,
                                                           float* __restrict__ epis, float* __restrict__ tot,
                                                           long long N) {
  DEER_PDL_ENTRY();
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < N; e += (long long)gridDim.x * blockDim.x) {
    const float4 r = reinterpret_cast<const float4*>(evidence)[e];
    const float n = softplus_f(r.y) + 1e-6f, a = softplus_f(r.z) + 1.0f, b = softplus_f(r.w) + 1e-6f;
    const float al = b / (a - 1.f), ep = b / (n * (a - 1.f));
    mu[e] = r.x;
    nu[e] = n;
    alpha[e] = a;
    beta[e] = b;
    alea[e] = al;
    epis[e] = ep;
    tot[e] = al + ep;
  }
}

__global__ void __launch_bounds__(256) nig_head_bwd_kernel(const float* __restrict__ evidence,
                                                           const float* __restrict__ dmu, const float* __restrict__ dnu,
                                                           const float* __restrict__ dalpha,
                                                           const float* __restrict__ dbeta,
                                                           const float* __restrict__ dalea,
                                                           const float* __restrict__ depis,
                                                           const float* __restrict__ dtot, float* __restrict__ dev,
                                                           long long N) {
  DEER_PDL_ENTRY();
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < N; e += (long long)gridDim.x * blockDim.x) {
    const float4 r = reinterpret_cast<const float4*>(evidence)[e];
    const float n = softplus_f(r.y) + 1e-6f, a = softplus_f(r.z) + 1.0f, b = softplus_f(r.w) + 1e-6f;
    const float am1 = a - 1.f;
    const float gal = (dalea ? dalea[e] : 0.f) + (dtot ? dtot[e] : 0.f);  // grad wrt aleatoric
    const float gep = (depis ? depis[e] : 0.f) + (dtot ? dtot[e] : 0.f);  // grad wrt epistemic
    // aleatoric = b/am1 ; epistemic = b/(n*am1)
    float gn = (dnu ? dnu[e] : 0.f) + gep * (-b / (n * n * am1));
    float ga = (dalpha ? dalpha[e] : 0.f) + gal * (-b / (am1 * am1)) + gep * (-b / (n * am1 * am1));
    float gb = (dbeta ? dbeta[e] : 0.f) + gal / am1 + gep / (n * am1);
    float4 o;
    o.x = dmu ? dmu[e] : 0.f;
    o.y = gn * softplus_grad_f(r.y);
    o.z = ga * softplus_grad_f(r.z);
    o.w = gb * softplus_grad_f(r.w);
    reinterpret_cast<float4*>(dev)[e] = o;
  }
}

// ------------------------------------------------------------------ Amini-style loss (deer.py:111-195)
__global__ void __launch_bounds__(256) amini_loss_kernel(const float* __restrict__ mu, const float* __restrict__ nu,
                                                         const float* __restrict__ alpha,
                                                         const float* __restrict__ beta,
                                                         const float* __restrict__ targets, float ew, float kw,
                                                         long long N, float* __restrict__ dparams,
                                                         float* __restrict__ scratch) {
  DEER_PDL_ENTRY();
  __shared__ float red[32];
  float s_nll = 0.f, s_reg = 0.f, s_kl = 0.f, s_mse = 0.f;
  const float invN = 1.f / (float)N;
  const float PI = 3.14159265358979f;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < N; e += (long long)gridDim.x * blockDim.x) {
    const float m = mu[e], n = nu[e], a = alpha[e], b = beta[e];
    const float err = targets[e] - m, se = err * err;
    const float S = b + n * se * 0.5f, ah = a + 0.5f;
    const float lga = lgammaf(a), lgah = lgammaf(ah);
    s_nll += 0.5f * logf(PI / n) - a * logf(2.f * b) + lga - lgah + ah * logf(S);
    const float num = n * se + 2.f * b * (1.f + n), den = 2.f * n * (1.f + n);
    s_reg += num / den;
    const float kl = 0.5f * (n - 1.f) + a * logf(b) - lga + lgah - 0.5f * logf(2.f * PI * b);
    s_kl += fmaxf(kl, 0.f);
    s_mse += se;
    if (dparams) {
      const float psa = digamma_f(a), psah = digamma_f(ah);
      float dm = ah * (-n * err) / S;
      float dn = -0.5f / n + ah * se * 0.5f / S;
      float da = -logf(2.f * b) + psa - psah + logf(S);
      float db = -a / b + ah / S;
      dm += ew * (-2.f * n * err / den);
      dn += ew * ((se + 2.f * b) / den - num * (2.f + 4.f * n) / (den * den));
      db += ew * (1.f / n);
      if (kl > 0.f) {
        dn += kw * 0.5f;
        da += kw * (logf(b) - psa + psah);
        db += kw * (a / b - 0.5f / b);
      }
      dparams[e] = dm * invN;
      dparams[N + e] = dn * invN;
      dparams[2 * N + e] = da * invN;
      dparams[3 * N + e] = db * invN;
    }
  }
  s_nll = block_sum(s_nll, red);
  s_reg = block_sum(s_reg, red);
  s_kl = block_sum(s_kl, red);
  s_mse = block_sum(s_mse, red);
  if (threadIdx.x == 0) {
    atomicAdd(scratch + 0, s_nll);
    atomicAdd(scratch + 1, s_reg);
    atomicAdd(scratch + 2, s_kl);
    atomicAdd(scratch + 3, s_mse);
  }
}
__global__ void amini_finish_kernel(const float* scratch, float ew, float kw, long long N, float* losses) {
  DEER_PDL_ENTRY();
  const float invN = 1.f / (float)N;
  const float nll = scratch[0] * invN, reg = scratch[1] * invN, kl = scratch[2] * invN, mse = scratch[3] * invN;
  losses[0] = nll + ew * reg + kw * kl;
  losses[1] = nll;
  losses[2] = reg;
  losses[3] = kl;
  losses[4] = mse;
}

// grid of the two loss passes: exactly the number of co-resident blocks (one wave; the grid-stride loops cover the
// rest), never 8 blocks per SM when only 6 fit - the partial second wave ran at a third of the occupancy
template <typename K>
static int resident_grid(K kernel, long long n, int threads) {
  static int per_sm = 0;  // per template instantiation (one kernel each)
  if (per_sm == 0) {
    int b = 0;
    if (cudaOccupancyMaxActiveBlocksPerMultiprocessor(&b, kernel, threads, 0) != cudaSuccess || b < 1) b = 4;
    per_sm = b;
  }
  long long g = cdiv(n, (long long)threads * LOSS_UNROLL);  // every thread gets a full unrolled trip when it can
  const long long cap = (long long)kNumSMs * per_sm;
  if (g > cap) g = cap;
  return (int)(g < 1 ? 1 : g);
}

static int stream_grid(long long n, int threads) {
  long long g = cdiv(n, threads);
  const long long cap = (long long)kNumSMs * 8;
  if (g > cap) g = cap;
  return (int)(g < 1 ? 1 : g);
}

int g_nig_pipe = 1;   // DEER_OPT_NIG_PIPELINE

// launchers shared by the plain and the mask entries (kMask: target_mask [B,D] bytes, nonzero = labelled)
template <bool kMask>
static int nig_loss_stats_launch(const float* evidence, const float* gamma, const float* nu, const float* alpha,
                                 const float* beta, const float* targets, const unsigned char* mask,
                                 const float* bin_edges, float* stats, float* nig_out, long long B, int D,
                                 int from_evidence, float eps, void* stream) {
  DEER_CHECK_ARG(targets && bin_edges && stats && B > 0, "nig_loss_stats: bad args");
  DEER_CHECK_ARG(from_evidence ? evidence != nullptr : (gamma && nu && alpha && beta), "nig_loss_stats: inputs");
  if (D < 1 || D > 8 || LOSS_THREADS % D != 0) {
    set_error("nig_loss_stats: D=%d unsupported (need a divisor of %d, <=8)", D, LOSS_THREADS);
    return DEER_ERR_UNSUPPORTED;
  }
  const long long total = B * D;
  if (total > DEER_NIG_MAX_ELEMENTS) {
    set_error("nig_loss_stats: B*D=%lld exceeds %lld", total, (long long)DEER_NIG_MAX_ELEMENTS);
    return DEER_ERR_UNSUPPORTED;
  }
  NigPlanes planes;
  for (int i = 0; i < 7; i++) planes.p[i] = nig_out ? nig_out + (long long)i * total : nullptr;
  const int has_out = nig_out != nullptr;
  // operands (20 B per element) small enough to stay in the 126 MB L2 between the two passes?
  const bool keep = total * 20 <= (long long)DEER_NIG_L2_KEEP_BYTES;
#define DEER_NIG_STATS_GO(K, FE, PP)                                                                                  \
  DEER_LAUNCH((nig_loss_stats_kernel<K, FE, PP, kMask>),                                                               \
              resident_grid(nig_loss_stats_kernel<K, FE, PP, kMask>, total, LOSS_THREADS), LOSS_THREADS, 0, stream,   \
              evidence, gamma, nu, alpha, beta, targets, bin_edges, stats, planes, has_out, (int)total, D, eps, mask)
#define DEER_NIG_STATS_GO2(K, FE)            \
  do {                                       \
    if (g_nig_pipe) DEER_NIG_STATS_GO(K, FE, true); \
    else DEER_NIG_STATS_GO(K, FE, false);    \
  } while (0)
  if (keep) {
    if (from_evidence) DEER_NIG_STATS_GO2(true, true);
    else DEER_NIG_STATS_GO2(true, false);
  } else {
    if (from_evidence) DEER_NIG_STATS_GO2(false, true);
    else DEER_NIG_STATS_GO2(false, false);
  }
#undef DEER_NIG_STATS_GO2
#undef DEER_NIG_STATS_GO
  return DEER_OK;
}

template <bool kMask>
static int nig_loss_finish_launch(const float* evidence, const float* gamma, const float* nu, const float* alpha,
                                  const float* beta, const float* targets, const unsigned char* mask,
                                  const float* bin_edges, const float* stats, const float* task_weights, float reg_w,
                                  float kl_w, float ece_w, float cross_w, float eps, long long B_local,
                                  long long B_global, int D, int from_evidence, float grad_scale, float* losses,
                                  float* d_out, float* counts, void* stream) {
  DEER_CHECK_ARG(targets && bin_edges && stats && B_local > 0, "nig_loss_finish: bad args");
  DEER_CHECK_ARG(from_evidence ? evidence != nullptr : (gamma && nu && alpha && beta), "nig_loss_finish: inputs");
  DEER_CHECK_ARG(losses || d_out, "nig_loss_finish: nothing to do");
  if (D < 1 || D > 8) {
    set_error("nig_loss_finish: D=%d unsupported", D);
    return DEER_ERR_UNSUPPORTED;
  }
  const long long total = B_local * D;
  if (total > DEER_NIG_MAX_ELEMENTS) {
    set_error("nig_loss_finish: B*D=%lld exceeds %lld", total, (long long)DEER_NIG_MAX_ELEMENTS);
    return DEER_ERR_UNSUPPORTED;
  }
#define DEER_NIG_FINISH_GO(FE, PP)                                                                                    \
  DEER_LAUNCH((nig_loss_finish_kernel<FE, PP, kMask>),                                                                 \
              resident_grid(nig_loss_finish_kernel<FE, PP, kMask>, total, LOSS_THREADS), LOSS_THREADS, 0, stream,     \
              evidence, gamma, nu, alpha, beta, targets, bin_edges, stats, task_weights, reg_w, kl_w, ece_w, cross_w, \
              eps, (int)total, B_global, D, grad_scale, losses, d_out, mask, counts)
  if (from_evidence) {
    if (g_nig_pipe) DEER_NIG_FINISH_GO(true, true);
    else DEER_NIG_FINISH_GO(true, false);
  } else {
    if (g_nig_pipe) DEER_NIG_FINISH_GO(false, true);
    else DEER_NIG_FINISH_GO(false, false);
  }
#undef DEER_NIG_FINISH_GO
  return DEER_OK;
}


}  // namespace deer

using namespace deer;

extern "C" {

int deer_nig_head_fwd(const float* evidence, float* mu, float* nu, float* alpha, float* beta, float* aleatoric,
                      float* epistemic, float* total, long long N, void* stream) {
  DEER_CHECK_ARG(evidence && mu && nu && alpha && beta && aleatoric && epistemic && total && N > 0,
                 "nig_head_fwd: bad args");
  DEER_LAUNCH(nig_head_fwd_kernel, stream_grid(N, 256), 256, 0, stream, evidence, mu, nu, alpha, beta, aleatoric,
              epistemic, total, N);
  return DEER_OK;
}

int deer_nig_head_bwd(const float* evidence, const float* dmu, const float* dnu, const float* dalpha,
                      const float* dbeta, const float* daleatoric, const float* depistemic, const float* dtotal,
                      float* devidence, long long N, void* stream) {
  DEER_CHECK_ARG(evidence && devidence && N > 0, "nig_head_bwd: bad args");
  DEER_LAUNCH(nig_head_bwd_kernel, stream_grid(N, 256), 256, 0, stream, evidence, dmu, dnu, dalpha, dbeta, daleatoric,
              depistemic, dtotal, devidence, N);
  return DEER_OK;
}

int deer_nig_loss_stats(const float* evidence, const float* gamma, const float* nu, const float* alpha,
                        const float* beta, const float* targets, const float* bin_edges, float* stats, float* nig_out,
                        long long B, int D, int from_evidence, float eps, void* stream) {
  return nig_loss_stats_launch<false>(evidence, gamma, nu, alpha, beta, targets, nullptr, bin_edges, stats, nig_out, B,
                                      D, from_evidence, eps, stream);
}

int deer_nig_loss_stats_mask(const float* evidence, const float* gamma, const float* nu, const float* alpha,
                             const float* beta, const float* targets, const void* target_mask, const float* bin_edges,
                             float* stats, float* nig_out, long long B, int D, int from_evidence, float eps,
                             void* stream) {
  DEER_CHECK_ARG(target_mask, "nig_loss_stats_mask: target_mask");
  return nig_loss_stats_launch<true>(evidence, gamma, nu, alpha, beta, targets,
                                     static_cast<const unsigned char*>(target_mask), bin_edges, stats, nig_out, B, D,
                                     from_evidence, eps, stream);
}

int deer_nig_loss_finish(const float* evidence, const float* gamma, const float* nu, const float* alpha,
                         const float* beta, const float* targets, const float* bin_edges, const float* stats,
                         const float* task_weights, float reg_w, float kl_w, float ece_w, float cross_w, float eps,
                         long long B_local, long long B_global, int D, int from_evidence, float grad_scale,
                         float* losses, float* d_out, void* stream) {
  DEER_CHECK_ARG(B_global >= B_local, "nig_loss_finish: bad args");
  return nig_loss_finish_launch<false>(evidence, gamma, nu, alpha, beta, targets, nullptr, bin_edges, stats,
                                       task_weights, reg_w, kl_w, ece_w, cross_w, eps, B_local, B_global, D,
                                       from_evidence, grad_scale, losses, d_out, nullptr, stream);
}

int deer_nig_loss_finish_mask(const float* evidence, const float* gamma, const float* nu, const float* alpha,
                              const float* beta, const float* targets, const void* target_mask,
                              const float* bin_edges, const float* stats, const float* task_weights, float reg_w,
                              float kl_w, float ece_w, float cross_w, float eps, long long B_local, int D,
                              int from_evidence, float grad_scale, float* losses, float* d_out, float* counts,
                              void* stream) {
  DEER_CHECK_ARG(target_mask, "nig_loss_finish_mask: target_mask");
  DEER_CHECK_ARG(losses || !counts, "nig_loss_finish_mask: counts are written with the losses");
  return nig_loss_finish_launch<true>(evidence, gamma, nu, alpha, beta, targets,
                                      static_cast<const unsigned char*>(target_mask), bin_edges, stats, task_weights,
                                      reg_w, kl_w, ece_w, cross_w, eps, B_local, B_local, D, from_evidence, grad_scale,
                                      losses, d_out, counts, stream);
}

int deer_amini_loss(const float* mu, const float* nu, const float* alpha, const float* beta, const float* targets,
                    float evidence_w, float kl_w, long long N, float* losses, float* dparams, float* scratch,
                    void* stream) {
  DEER_CHECK_ARG(mu && nu && alpha && beta && targets && losses && scratch && N > 0, "amini_loss: bad args");
  cudaError_t e = cudaMemsetAsync(scratch, 0, 8 * sizeof(float), (cudaStream_t)stream);
  if (e != cudaSuccess) return cuda_status(e, "amini memset");
  DEER_LAUNCH(amini_loss_kernel, stream_grid(N, 256), 256, 0, stream, mu, nu, alpha, beta, targets, evidence_w, kl_w, N,
              dparams, scratch);
  DEER_LAUNCH(amini_finish_kernel, 1, 1, 0, stream, scratch, evidence_w, kl_w, N, losses);
  return DEER_OK;
}

}  // extern "C"
