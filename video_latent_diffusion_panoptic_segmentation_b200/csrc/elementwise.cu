// Small HBM-/latency-bound kernels of the sampler loop: DDIM, DPM-Solver++ and UniPC updates, timestep sinusoid +
// GEMV chain, the few-channel 3x3 convs at the ends of the UNet / seg-AE (fused with concat+cast), nearest upsample,
// stride-2 im2col.
#include "common.cuh"
#include "host_util.h"

namespace {
using namespace ldm;

// ---------------------------------------------------------------- DDIM update (ddim_scheduler.py:234-267)
// Explicit round-to-nearest mul/sub/div/add intrinsics keep the reference's op order (no FMA contraction) so the
// fp32 result is bit-identical to torch eager on the CPU.
// `prev` / `x0out` may alias `sample` (in-place update by the sampler loop): no __restrict__ on those.
// With `eps_text` the noise prediction is first combined as classifier-free guidance does (trainers_ldm_cond.py:1147-1149):
// eps = eps_uncond + g * (eps_text - eps_uncond), three roundings in the reference's order.
// kRows: t_index holds one row per image, element i reads row t_index[i / epi] (epi % 4 == 0, so a float4 lies in one
// image); the row's scalars are reloaded only when a thread's element moves to another image.
template <bool kRows>
__global__ void ddim_step_kernel(const float* __restrict__ eps, const float* __restrict__ eps_text, float guidance,
                                 const float* sample, const float* __restrict__ coef,
                                 const int32_t* __restrict__ t_index, float* prev, float* x0out, long long n,
                                 float clip, int reclip_eps, long long epi) {
  // clip > 0: pred_original_sample is clamped to [-clip, clip] (clip_sample, :253-257); reclip_eps: the noise is then
  // re-derived from the clamped x0 (use_clipped_model_output, :259-261), both in the reference's op order
  const int ti = kRows ? 0 : (t_index ? *t_index : 0);
  float s1m_at = coef[ti * 4 + 0];   // sqrt(1 - alpha_t)
  float s_at = coef[ti * 4 + 1];     // sqrt(alpha_t)
  float s_ap = coef[ti * 4 + 2];     // sqrt(alpha_prev)
  float s1m_ap = coef[ti * 4 + 3];   // sqrt(1 - alpha_prev)
  long long img = 0;
  auto select = [&](long long elem) {
    if constexpr (kRows) {
      if (elem / epi != img) {
        img = elem / epi;
        const int r = __ldg(t_index + img);
        s1m_at = __ldg(coef + r * 4 + 0); s_at = __ldg(coef + r * 4 + 1);
        s_ap = __ldg(coef + r * 4 + 2); s1m_ap = __ldg(coef + r * 4 + 3);
      }
    }
  };
  if constexpr (kRows) img = -1;
  const long long nv = n / 4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long long)gridDim.x * blockDim.x) {
    select(i * 4);
    const float4 e = __ldg(reinterpret_cast<const float4*>(eps) + i);
    const float4 x = reinterpret_cast<const float4*>(sample)[i];
    float ev[4] = {e.x, e.y, e.z, e.w};
    if (eps_text) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(eps_text) + i);
      const float tv[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) ev[j] = __fadd_rn(ev[j], __fmul_rn(guidance, __fsub_rn(tv[j], ev[j])));
    }
    const float xv[4] = {x.x, x.y, x.z, x.w};
    float p0[4], pv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      p0[j] = __fdiv_rn(__fsub_rn(xv[j], __fmul_rn(s1m_at, ev[j])), s_at);
      if (clip > 0.f) p0[j] = fminf(fmaxf(p0[j], -clip), clip);
      if (reclip_eps) ev[j] = __fdiv_rn(__fsub_rn(xv[j], __fmul_rn(s_at, p0[j])), s1m_at);
      pv[j] = __fadd_rn(__fmul_rn(s_ap, p0[j]), __fmul_rn(s1m_ap, ev[j]));
    }
    if (prev) reinterpret_cast<float4*>(prev)[i] = make_float4(pv[0], pv[1], pv[2], pv[3]);
    if (x0out) reinterpret_cast<float4*>(x0out)[i] = make_float4(p0[0], p0[1], p0[2], p0[3]);
  }
  // tail
  for (long long i = nv * 4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    select(i);
    float e = eps[i];
    if (eps_text) e = __fadd_rn(e, __fmul_rn(guidance, __fsub_rn(eps_text[i], e)));
    float p0 = __fdiv_rn(__fsub_rn(sample[i], __fmul_rn(s1m_at, e)), s_at);
    if (clip > 0.f) p0 = fminf(fmaxf(p0, -clip), clip);
    if (reclip_eps) e = __fdiv_rn(__fsub_rn(sample[i], __fmul_rn(s_at, p0)), s1m_at);
    if (prev) prev[i] = __fadd_rn(__fmul_rn(s_ap, p0), __fmul_rn(s1m_ap, e));
    if (x0out) x0out[i] = p0;
  }
}

// ---------------------------------------------------------------- DPM-Solver++ (2M, midpoint) update
// Row *step_index of `coef` (ldmseg/schedulers/dpm_solver.py) holds {sig_i, alpha_i, A, Bc, c, hb, order, 0}:
//   x0 = (x - sig_i * eps) / alpha_i;  prev = A * x - Bc * x0  [ - hb * (c * (x0 - x0_prev)) when order == 2 ]
// in that op order with round-to-nearest intrinsics, as ddim_step_kernel. x0 replaces x0_prev in place (the same thread
// reads and writes each element); `prev` may alias `sample`. kRows: row step_index[i / epi] per image, as
// ddim_step_kernel<true>.
constexpr int kDpmCoefCols = 8;
template <bool kRows>
__global__ void dpmpp_step_kernel(const float* __restrict__ eps, const float* __restrict__ eps_text, float guidance,
                                  const float* sample, const float* __restrict__ coef,
                                  const int32_t* __restrict__ step_index, float* prev, float* x0_prev, long long n,
                                  long long epi) {
  float sig, alpha, A, Bc, c, hb;
  bool second;
  auto load = [&](const int32_t* idx) {
    const float* row = coef + (long long)__ldg(idx) * kDpmCoefCols;
    sig = __ldg(row + 0); alpha = __ldg(row + 1); A = __ldg(row + 2); Bc = __ldg(row + 3);
    c = __ldg(row + 4); hb = __ldg(row + 5);
    second = __ldg(row + 6) > 1.5f;
  };
  long long img = -1;
  auto select = [&](long long elem) {
    if constexpr (kRows) {
      if (elem / epi != img) {
        img = elem / epi;
        load(step_index + img);
      }
    }
  };
  if constexpr (!kRows) load(step_index);
  const long long nv = n / 4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long long)gridDim.x * blockDim.x) {
    select(i * 4);
    const float4 e = __ldg(reinterpret_cast<const float4*>(eps) + i);
    const float4 x = reinterpret_cast<const float4*>(sample)[i];
    float ev[4] = {e.x, e.y, e.z, e.w};
    if (eps_text) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(eps_text) + i);
      const float tv[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) ev[j] = __fadd_rn(ev[j], __fmul_rn(guidance, __fsub_rn(tv[j], ev[j])));
    }
    const float xv[4] = {x.x, x.y, x.z, x.w};
    float qv[4] = {0.f, 0.f, 0.f, 0.f};
    if (second) {
      const float4 q = reinterpret_cast<const float4*>(x0_prev)[i];
      qv[0] = q.x; qv[1] = q.y; qv[2] = q.z; qv[3] = q.w;
    }
    float p0[4], pv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      p0[j] = __fdiv_rn(__fsub_rn(xv[j], __fmul_rn(sig, ev[j])), alpha);
      pv[j] = __fsub_rn(__fmul_rn(A, xv[j]), __fmul_rn(Bc, p0[j]));
      if (second) pv[j] = __fsub_rn(pv[j], __fmul_rn(hb, __fmul_rn(c, __fsub_rn(p0[j], qv[j]))));
    }
    reinterpret_cast<float4*>(prev)[i] = make_float4(pv[0], pv[1], pv[2], pv[3]);
    reinterpret_cast<float4*>(x0_prev)[i] = make_float4(p0[0], p0[1], p0[2], p0[3]);
  }
  // tail
  for (long long i = nv * 4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    select(i);
    float e = eps[i];
    if (eps_text) e = __fadd_rn(e, __fmul_rn(guidance, __fsub_rn(eps_text[i], e)));
    const float x = sample[i];
    const float p0 = __fdiv_rn(__fsub_rn(x, __fmul_rn(sig, e)), alpha);
    float p = __fsub_rn(__fmul_rn(A, x), __fmul_rn(Bc, p0));
    if (second) p = __fsub_rn(p, __fmul_rn(hb, __fmul_rn(c, __fsub_rn(p0, x0_prev[i]))));
    prev[i] = p;
    x0_prev[i] = p0;
  }
}

// ---------------------------------------------------------------- UniPC (bh2, data prediction) update
// Row *step_index of `coef` (ldmseg/schedulers/unipc.py, include/ldmseg_b200.h) holds the scalars of the corrector of
// the previous step's result and of the predictor to the next sigma; the op order is that of oracle/unipc_oracle.py,
// with round-to-nearest intrinsics as ddim_step_kernel. Each thread owns its elements: it reads sample, last and the
// history m1..mQ of an element before it writes prev (which may alias sample), last and the shifted history.
constexpr int kUniPCCoefCols = 20;
struct UniPCRow {
  float sig, alpha;
  int p, q;                                  // predictor order 1..3, corrector order 0 (off) .. 3
  float Ap, Pp, Bp, rp1, rp2, rhop1, rhop2;  // predictor: a = i -> t = i + 1
  float Ac, Pc, Bc, rc1, rc2, rhoc1, rhoc2, rhocm;  // corrector: a = i - 1 -> t = i
};

__device__ __forceinline__ UniPCRow unipc_row(const float* __restrict__ coef, const int32_t* __restrict__ step_index) {
  const float* r = coef + (long long)__ldg(step_index) * kUniPCCoefCols;
  UniPCRow c;
  c.sig = __ldg(r + 0); c.alpha = __ldg(r + 1);
  c.p = __float2int_rn(__ldg(r + 2)); c.q = __float2int_rn(__ldg(r + 3));
  c.Ap = __ldg(r + 4); c.Pp = __ldg(r + 5); c.Bp = __ldg(r + 6); c.rp1 = __ldg(r + 7); c.rp2 = __ldg(r + 8);
  c.rhop1 = __ldg(r + 9); c.rhop2 = __ldg(r + 10);
  c.Ac = __ldg(r + 11); c.Pc = __ldg(r + 12); c.Bc = __ldg(r + 13); c.rc1 = __ldg(r + 14); c.rc2 = __ldg(r + 15);
  c.rhoc1 = __ldg(r + 16); c.rhoc2 = __ldg(r + 17); c.rhocm = __ldg(r + 18);
  return c;
}

// One element: e is the (guided) noise prediction, x the sample, last the corrected sample of the previous step and
// h[0..2] = m1..m3. Returns prev; last and h are updated in place (h[k] for k >= the history length is scratch).
__device__ __forceinline__ float unipc_elem(const UniPCRow& c, float e, float x, float& last, float (&h)[3]) {
  const float m = __fdiv_rn(__fsub_rn(x, __fmul_rn(c.sig, e)), c.alpha);
  float xc = x;
  if (c.q > 0) {
    float s = __fmul_rn(c.rhocm, __fsub_rn(m, h[0]));
    if (c.q > 1) {
      float d = __fmul_rn(c.rhoc1, __fdiv_rn(__fsub_rn(h[1], h[0]), c.rc1));
      if (c.q > 2) d = __fadd_rn(d, __fmul_rn(c.rhoc2, __fdiv_rn(__fsub_rn(h[2], h[0]), c.rc2)));
      s = __fadd_rn(d, s);
    }
    xc = __fsub_rn(__fsub_rn(__fmul_rn(c.Ac, last), __fmul_rn(c.Pc, h[0])), __fmul_rn(c.Bc, s));
  }
  float prev = __fsub_rn(__fmul_rn(c.Ap, xc), __fmul_rn(c.Pp, m));
  if (c.p > 1) {
    float s = __fmul_rn(c.rhop1, __fdiv_rn(__fsub_rn(h[0], m), c.rp1));
    if (c.p > 2) s = __fadd_rn(s, __fmul_rn(c.rhop2, __fdiv_rn(__fsub_rn(h[1], m), c.rp2)));
    prev = __fsub_rn(prev, __fmul_rn(c.Bp, s));
  }
  last = xc;
  h[2] = h[1];
  h[1] = h[0];
  h[0] = m;
  return prev;
}

// Q = solver_order: the number of history buffers read and shifted. kRows: row step_index[i / epi] per image, as
// ddim_step_kernel<true>.
template <int Q, bool kRows>
__global__ void unipc_step_kernel(const float* __restrict__ eps, const float* __restrict__ eps_text, float guidance,
                                  const float* sample, const float* __restrict__ coef,
                                  const int32_t* __restrict__ step_index, float* prev, float* __restrict__ last,
                                  float* __restrict__ m1, float* __restrict__ m2, float* __restrict__ m3, long long n,
                                  long long epi) {
  UniPCRow c;
  if constexpr (!kRows) c = unipc_row(coef, step_index);
  long long img = -1;
  auto select = [&](long long elem) {
    if constexpr (kRows) {
      if (elem / epi != img) {
        img = elem / epi;
        c = unipc_row(coef, step_index + img);
      }
    }
  };
  float* const hist[3] = {m1, m2, m3};
  const long long nv = n / 4;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < nv; i += (long long)gridDim.x * blockDim.x) {
    select(i * 4);
    const float4 e4 = __ldg(reinterpret_cast<const float4*>(eps) + i);
    const float4 x4 = reinterpret_cast<const float4*>(sample)[i];
    float ev[4] = {e4.x, e4.y, e4.z, e4.w};
    if (eps_text) {
      const float4 t = __ldg(reinterpret_cast<const float4*>(eps_text) + i);
      const float tv[4] = {t.x, t.y, t.z, t.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) ev[j] = __fadd_rn(ev[j], __fmul_rn(guidance, __fsub_rn(tv[j], ev[j])));
    }
    const float xv[4] = {x4.x, x4.y, x4.z, x4.w};
    float lv[4] = {0.f, 0.f, 0.f, 0.f};
    if (c.q > 0) {
      const float4 l = reinterpret_cast<const float4*>(last)[i];
      lv[0] = l.x; lv[1] = l.y; lv[2] = l.z; lv[3] = l.w;
    }
    float hv[4][3] = {};
#pragma unroll
    for (int k = 0; k < Q; ++k) {
      const float4 m = reinterpret_cast<const float4*>(hist[k])[i];
      hv[0][k] = m.x; hv[1][k] = m.y; hv[2][k] = m.z; hv[3][k] = m.w;
    }
    float pv[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) pv[j] = unipc_elem(c, ev[j], xv[j], lv[j], hv[j]);
    reinterpret_cast<float4*>(prev)[i] = make_float4(pv[0], pv[1], pv[2], pv[3]);
    reinterpret_cast<float4*>(last)[i] = make_float4(lv[0], lv[1], lv[2], lv[3]);
#pragma unroll
    for (int k = 0; k < Q; ++k)
      reinterpret_cast<float4*>(hist[k])[i] = make_float4(hv[0][k], hv[1][k], hv[2][k], hv[3][k]);
  }
  // tail
  for (long long i = nv * 4 + (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n;
       i += (long long)gridDim.x * blockDim.x) {
    select(i);
    float e = eps[i];
    if (eps_text) e = __fadd_rn(e, __fmul_rn(guidance, __fsub_rn(eps_text[i], e)));
    float l = c.q > 0 ? last[i] : 0.f;
    float hv[3] = {};
#pragma unroll
    for (int k = 0; k < Q; ++k) hv[k] = hist[k][i];
    prev[i] = unipc_elem(c, e, sample[i], l, hv);
    last[i] = l;
#pragma unroll
    for (int k = 0; k < Q; ++k) hist[k][i] = hv[k];
  }
}

// ---------------------------------------------------------------- timestep sinusoid (diffusers Timesteps)
// out[0:half] = cos(t * f_i), out[half:2*half] = sin(t * f_i)   (flip_sin_to_cos=True, freq_shift=0)
// kRows: one CTA per image b, t = timesteps[b], out row b of [B, 2*half].
template <bool kRows>
__global__ void timestep_sinusoid_kernel(const long long* __restrict__ timesteps, const int32_t* __restrict__ t_index,
                                         const float* __restrict__ freqs, float* __restrict__ out, int half) {
  const float t = (float)timesteps[kRows ? (int)blockIdx.x : (t_index ? *t_index : 0)];
  if constexpr (kRows) out += (long long)blockIdx.x * 2 * half;
  for (int i = threadIdx.x; i < half; i += blockDim.x) {
    const float a = __fmul_rn(t, freqs[i]);
    out[i] = cosf(a);
    out[half + i] = sinf(a);
  }
}

// ---------------------------------------------------------------- GEMV: out[n] = act(bias[n] + bias2[n] + w[n,:] . x)
// one warp per output row; x (fp32) staged in shared memory; w bf16 row-major [N,K], K % 8 == 0.
// kRows: x is [B, K] with image b = blockIdx.y; out is [B, N], or with seg_offs (nseg + 1 ascending column offsets
// from 0 to N) segment-major: column n of segment s lands at seg_offs[s] * B + b * width_s + (n - seg_offs[s]).
// Every output element takes the arithmetic of the single-vector kernel, so row b equals it bit for bit.
template <bool kRows>
__global__ void gemv_bf16_kernel(const __nv_bfloat16* __restrict__ w, const float* __restrict__ bias,
                                 const float* __restrict__ bias2, const float* __restrict__ x, float* __restrict__ out,
                                 int N, int K, int silu_out, const int32_t* __restrict__ seg_offs, int nseg) {
  extern __shared__ float xs[];
  if constexpr (kRows) x += (long long)blockIdx.y * K;
  for (int i = threadIdx.x; i < K; i += blockDim.x) xs[i] = x[i];
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  for (int n = blockIdx.x * wpb + (threadIdx.x >> 5); n < N; n += gridDim.x * wpb) {
    const __nv_bfloat16* row = w + (long long)n * K;
    float acc = 0.f;
    for (int k = lane * 8; k < K; k += 256) {
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(row + k));
      const float2 a = unpack_bf16(u.x), b = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
      acc += a.x * xs[k] + a.y * xs[k + 1] + b.x * xs[k + 2] + b.y * xs[k + 3] + c.x * xs[k + 4] + c.y * xs[k + 5] +
             d.x * xs[k + 6] + d.y * xs[k + 7];
    }
    acc = warp_sum(acc);
    if (lane == 0) {
      float v = acc + (bias ? bias[n] : 0.f) + (bias2 ? bias2[n] : 0.f);
      long long o = n;
      if constexpr (kRows) {
        const long long b = blockIdx.y, B = gridDim.y;
        if (seg_offs) {
          int s = 0;
          while (s + 1 < nseg && n >= seg_offs[s + 1]) ++s;
          const int lo = seg_offs[s];
          o = lo * B + b * (seg_offs[s + 1] - lo) + (n - lo);
        } else {
          o = b * N + n;
        }
      }
      out[o] = silu_out ? silu_f(v) : v;
    }
  }
}

// ---------------------------------------------------------------- few-input-channel conv3x3 (conv_in / AE conv_in)
// Input: up to 3 NCHW fp32 sources of `cps` channels each (the latent concat, trainers_ldm_cond.py:1134-1141),
// scaled by `scale`; weights fp32 [cin, 3, 3, cout] (output channel innermost); output bf16 NHWC. One thread per output channel, a CTA per
// strip of pixels in one image row; the input patch is staged in shared memory (broadcast reads).
constexpr int kStrip = 32;
__global__ void conv3x3_small_cin_kernel(const float* __restrict__ s0, const float* __restrict__ s1,
                                         const float* __restrict__ s2, int nsrc, int cps, float scale, float shift,
                                         const float* __restrict__ w, const float* __restrict__ bias,
                                         __nv_bfloat16* __restrict__ out, int B, int h, int wd, int cout, int silu) {
  extern __shared__ float patch[];  // [cin][3][kStrip+2]
  const int cin = nsrc * cps;
  const int strips = (wd + kStrip - 1) / kStrip;
  const int bid = blockIdx.x;
  const int sx = bid % strips;
  const int y = (bid / strips) % h;
  const int b = bid / (strips * h);
  const int x0 = sx * kStrip;
  const int pw = kStrip + 2;
  for (int i = threadIdx.x; i < cin * 3 * pw; i += blockDim.x) {
    const int c = i / (3 * pw);
    const int r = (i / pw) % 3;
    const int px = i % pw;
    const int yy = y + r - 1, xx = x0 + px - 1;
    float v = 0.f;
    if (yy >= 0 && yy < h && xx >= 0 && xx < wd) {
      const int si = c / cps, cc = c % cps;
      const float* src = si == 0 ? s0 : (si == 1 ? s1 : s2);
      // (two roundings, as `2. * images - 1.` of encode_inputs; the conv's zero padding stays zero)
      v = __fadd_rn(__fmul_rn(src[(((long long)b * cps + cc) * h + yy) * wd + xx], scale), shift);
    }
    patch[i] = v;
  }
  __syncthreads();
  const int co = threadIdx.x;
  if (co >= cout) return;
  float acc[kStrip];
  const float bv = bias ? bias[co] : 0.f;
#pragma unroll
  for (int i = 0; i < kStrip; ++i) acc[i] = bv;
  for (int c = 0; c < cin; ++c) {
    float wk[9];
#pragma unroll
    for (int t = 0; t < 9; ++t) wk[t] = __ldg(&w[((long long)c * 9 + t) * cout + co]);  // [cin,3,3,cout]: coalesced over co
#pragma unroll
    for (int r = 0; r < 3; ++r) {
      const float* prow = patch + (c * 3 + r) * pw;
#pragma unroll
      for (int i = 0; i < kStrip; ++i)
        acc[i] += wk[r * 3] * prow[i] + wk[r * 3 + 1] * prow[i + 1] + wk[r * 3 + 2] * prow[i + 2];
    }
  }
  for (int i = 0; i < kStrip; ++i) {
    const int x = x0 + i;
    if (x < wd) out[(((long long)b * h + y) * wd + x) * cout + co] = __float2bfloat16_rn(silu ? silu_f(acc[i]) : acc[i]);
  }
}

// ---------------------------------------------------------------- conv_out: bf16 NHWC [B,h,w,cin] -> fp32 NCHW [B,cout,h,w]
// one warp per output pixel; lanes split the channels; weights staged in smem as [tap][cin][cout] fp32.
constexpr int kMaxCoutSmall = 8;
__global__ void conv_out_kernel(const __nv_bfloat16* __restrict__ x, const float* __restrict__ w,
                                const float* __restrict__ bias, float* __restrict__ out, int B, int h, int wd,
                                int cin, int cout) {
  extern __shared__ float ws[];  // [9][cin][cout]
  for (int i = threadIdx.x; i < 9 * cin * cout; i += blockDim.x) {
    const int co = i % cout;
    const int c = (i / cout) % cin;
    const int t = i / (cout * cin);
    ws[i] = w[((long long)co * cin + c) * 9 + t];
  }
  __syncthreads();
  const int lane = threadIdx.x & 31;
  const int wpb = blockDim.x >> 5;
  const long long npix = (long long)B * h * wd;
  const int nvec = cin / 8;
  for (long long pix = (long long)blockIdx.x * wpb + (threadIdx.x >> 5); pix < npix;
       pix += (long long)gridDim.x * wpb) {
    const int xx = (int)(pix % wd);
    const int yy = (int)((pix / wd) % h);
    const int b = (int)(pix / ((long long)wd * h));
    float acc[kMaxCoutSmall];
#pragma unroll
    for (int o = 0; o < kMaxCoutSmall; ++o) acc[o] = 0.f;
    for (int t = 0; t < 9; ++t) {
      const int sy = yy + t / 3 - 1, sx = xx + t % 3 - 1;
      if (sy < 0 || sy >= h || sx < 0 || sx >= wd) continue;
      const __nv_bfloat16* src = x + (((long long)b * h + sy) * wd + sx) * cin;
      for (int v = lane; v < nvec; v += 32) {
        const uint4 u = __ldg(reinterpret_cast<const uint4*>(src + v * 8));
        const float2 a = unpack_bf16(u.x), b2 = unpack_bf16(u.y), c = unpack_bf16(u.z), d = unpack_bf16(u.w);
        const float f[8] = {a.x, a.y, b2.x, b2.y, c.x, c.y, d.x, d.y};
        const float* wp = ws + ((long long)t * cin + v * 8) * cout;
#pragma unroll
        for (int j = 0; j < 8; ++j) {
#pragma unroll
          for (int o = 0; o < kMaxCoutSmall; ++o)
            if (o < cout) acc[o] += f[j] * wp[j * cout + o];
        }
      }
    }
#pragma unroll
    for (int o = 0; o < kMaxCoutSmall; ++o) {
      if (o < cout) {
        const float s = warp_sum(acc[o]);
        if (lane == 0) out[(((long long)b * cout + o) * h + yy) * wd + xx] = s + (bias ? bias[o] : 0.f);
      }
    }
  }
}

// ---------------------------------------------------------------- nearest upsample (F.interpolate mode="nearest")
__global__ void upsample_nearest_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ out, int B,
                                        int h, int w, int C, int oh, int ow, float sh_, float sw_) {
  const int vpp = C / 8;
  const long long total = (long long)B * oh * ow * vpp;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % vpp);
    long long p = i / vpp;
    const int ox = (int)(p % ow);
    p /= ow;
    const int oy = (int)(p % oh);
    const int b = (int)(p / oh);
    int sy = (int)floorf(__fmul_rn((float)oy, sh_));
    int sx = (int)floorf(__fmul_rn((float)ox, sw_));
    sy = sy < h - 1 ? sy : h - 1;
    sx = sx < w - 1 ? sx : w - 1;
    const uint4 u = __ldg(reinterpret_cast<const uint4*>(x + (((long long)b * h + sy) * w + sx) * C) + v);
    reinterpret_cast<uint4*>(out + (((long long)b * oh + oy) * ow + ox) * C)[v] = u;
  }
}

// ---------------------------------------------------------------- im2col for the stride-2 Downsample2D conv
__global__ void im2col3x3_s2_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ out, int B, int h,
                                    int w, int C, int oh, int ow, int pad) {
  const int vpp = C / 8;
  const long long total = (long long)B * oh * ow * 9 * vpp;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total;
       i += (long long)gridDim.x * blockDim.x) {
    const int v = (int)(i % vpp);
    long long p = i / vpp;
    const int t = (int)(p % 9);
    p /= 9;
    const int ox = (int)(p % ow);
    p /= ow;
    const int oy = (int)(p % oh);
    const int b = (int)(p / oh);
    const int sy = 2 * oy + t / 3 - pad, sx = 2 * ox + t % 3 - pad;
    uint4 u = make_uint4(0, 0, 0, 0);
    if (sy >= 0 && sy < h && sx >= 0 && sx < w)
      u = __ldg(reinterpret_cast<const uint4*>(x + (((long long)b * h + sy) * w + sx) * C) + v);
    reinterpret_cast<uint4*>(out)[i] = u;
  }
}

int grid_for(long long work_items, int threads) {
  long long g = (work_items + threads - 1) / threads;
  const long long cap = (long long)ldm_host::num_sms() * 16;
  if (g > cap) g = cap;
  if (g < 1) g = 1;
  return (int)g;
}

}  // namespace

extern "C" int ldm_ddim_step(const float* eps, const float* sample, const float* coef, const int32_t* t_index,
                             float* prev_sample, float* pred_x0, int64_t n, ldm_stream_t stream) {
  return ldm_ddim_step_clip(eps, nullptr, 0.f, sample, coef, t_index, prev_sample, pred_x0, n, 0.f, 0, stream);
}

extern "C" int ldm_ddim_step_cfg(const float* eps_uncond, const float* eps_text, float guidance_scale,
                                 const float* sample, const float* coef, const int32_t* t_index, float* prev_sample,
                                 float* pred_x0, int64_t n, ldm_stream_t stream) {
  return ldm_ddim_step_clip(eps_uncond, eps_text, guidance_scale, sample, coef, t_index, prev_sample, pred_x0, n, 0.f, 0,
                            stream);
}

extern "C" int ldm_ddim_step_clip(const float* eps_uncond, const float* eps_text, float guidance_scale,
                                  const float* sample, const float* coef, const int32_t* t_index, float* prev_sample,
                                  float* pred_x0, int64_t n, float clip_sample_range, int32_t use_clipped_model_output,
                                  ldm_stream_t stream) {
  using namespace ldm_host;
  LDM_REQUIRE(clip_sample_range >= 0.f, LDM_ERR_BAD_ARG, "ldm_ddim_step: clip_sample_range=%g (0 = no clipping)",
              (double)clip_sample_range);
  LDM_REQUIRE(eps_uncond && sample && coef, LDM_ERR_BAD_ARG, "ldm_ddim_step: null arg");
  LDM_REQUIRE(n > 0, LDM_ERR_BAD_SHAPE, "ldm_ddim_step: n=%lld", (long long)n);
  LDM_REQUIRE(((uintptr_t)eps_uncond | (uintptr_t)eps_text | (uintptr_t)sample | (uintptr_t)prev_sample |
               (uintptr_t)pred_x0) % 16 == 0,
              LDM_ERR_ALIGNMENT, "ldm_ddim_step: pointers must be 16-byte aligned");
  ddim_step_kernel<false><<<grid_for(n / 4 + 1, 256), 256, 0, as_stream(stream)>>>(
      eps_uncond, eps_text, guidance_scale, sample, coef, t_index, prev_sample, pred_x0, n, clip_sample_range,
      use_clipped_model_output != 0, n);
  count_launch();
  return check_launch("ddim_step_kernel");
}

extern "C" int ldm_dpmpp_step(const float* eps_uncond, const float* eps_text, float guidance_scale, const float* sample,
                              const float* coef, const int32_t* step_index, float* prev_sample, float* x0_prev, int64_t n,
                              ldm_stream_t stream) {
  using namespace ldm_host;
  LDM_REQUIRE(eps_uncond && sample && coef && step_index && prev_sample && x0_prev, LDM_ERR_BAD_ARG,
              "ldm_dpmpp_step: null arg");
  LDM_REQUIRE(n > 0, LDM_ERR_BAD_SHAPE, "ldm_dpmpp_step: n=%lld", (long long)n);
  LDM_REQUIRE(((uintptr_t)eps_uncond | (uintptr_t)eps_text | (uintptr_t)sample | (uintptr_t)prev_sample |
               (uintptr_t)x0_prev) % 16 == 0,
              LDM_ERR_ALIGNMENT, "ldm_dpmpp_step: pointers must be 16-byte aligned");
  dpmpp_step_kernel<false><<<grid_for(n / 4 + 1, 256), 256, 0, as_stream(stream)>>>(
      eps_uncond, eps_text, guidance_scale, sample, coef, step_index, prev_sample, x0_prev, n, n);
  count_launch();
  return check_launch("dpmpp_step_kernel");
}

extern "C" int ldm_unipc_step(const float* eps_uncond, const float* eps_text, float guidance_scale, const float* sample,
                              const float* coef, const int32_t* step_index, float* prev_sample, float* last, float* m1,
                              float* m2, float* m3, int32_t solver_order, int64_t n, ldm_stream_t stream) {
  using namespace ldm_host;
  LDM_REQUIRE(solver_order >= 1 && solver_order <= 3, LDM_ERR_BAD_ARG, "ldm_unipc_step: solver_order=%d",
              (int)solver_order);
  LDM_REQUIRE(eps_uncond && sample && coef && step_index && prev_sample && last && m1 && (solver_order < 2 || m2) &&
                  (solver_order < 3 || m3),
              LDM_ERR_BAD_ARG, "ldm_unipc_step: null arg");
  LDM_REQUIRE(n > 0, LDM_ERR_BAD_SHAPE, "ldm_unipc_step: n=%lld", (long long)n);
  LDM_REQUIRE(((uintptr_t)eps_uncond | (uintptr_t)eps_text | (uintptr_t)sample | (uintptr_t)prev_sample |
               (uintptr_t)last | (uintptr_t)m1 | (uintptr_t)m2 | (uintptr_t)m3) % 16 == 0,
              LDM_ERR_ALIGNMENT, "ldm_unipc_step: pointers must be 16-byte aligned");
  const dim3 grid = grid_for(n / 4 + 1, 256);
  auto s = as_stream(stream);
  if (solver_order == 1)
    unipc_step_kernel<1, false><<<grid, 256, 0, s>>>(eps_uncond, eps_text, guidance_scale, sample, coef, step_index,
                                                     prev_sample, last, m1, m2, m3, n, n);
  else if (solver_order == 2)
    unipc_step_kernel<2, false><<<grid, 256, 0, s>>>(eps_uncond, eps_text, guidance_scale, sample, coef, step_index,
                                                     prev_sample, last, m1, m2, m3, n, n);
  else
    unipc_step_kernel<3, false><<<grid, 256, 0, s>>>(eps_uncond, eps_text, guidance_scale, sample, coef, step_index,
                                                     prev_sample, last, m1, m2, m3, n, n);
  count_launch();
  return check_launch("unipc_step_kernel");
}

extern "C" int ldm_timestep_sinusoid(const int64_t* timesteps, const int32_t* t_index, const float* freqs, float* out,
                                     int32_t half, ldm_stream_t stream) {
  using namespace ldm_host;
  LDM_REQUIRE(timesteps && freqs && out && half > 0, LDM_ERR_BAD_ARG, "ldm_timestep_sinusoid: bad arg");
  timestep_sinusoid_kernel<false><<<1, 256, 0, as_stream(stream)>>>(reinterpret_cast<const long long*>(timesteps),
                                                                    t_index, freqs, out, half);
  count_launch();
  return check_launch("timestep_sinusoid_kernel");
}

extern "C" int ldm_gemv_bf16(const void* w, const float* bias, const float* bias2, const float* x, float* out,
                             int32_t N, int32_t K, int32_t silu_out, ldm_stream_t stream) {
  using namespace ldm_host;
  LDM_REQUIRE(w && x && out, LDM_ERR_BAD_ARG, "ldm_gemv_bf16: null arg");
  LDM_REQUIRE(N > 0 && K > 0 && K % 8 == 0 && K <= 8192, LDM_ERR_BAD_SHAPE, "ldm_gemv_bf16: N=%d K=%d", N, K);
  const int wpb = 8;
  int grid = (N + wpb - 1) / wpb;
  const int cap = num_sms() * 8;
  if (grid > cap) grid = cap;
  gemv_bf16_kernel<false><<<grid, wpb * 32, sizeof(float) * K, as_stream(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(w), bias, bias2, x, out, N, K, silu_out, nullptr, 0);
  count_launch();
  return check_launch("gemv_bf16_kernel");
}

// ---------------------------------------------------------------- per-image rows (streaming sampler)
extern "C" int ldm_timestep_sinusoid_rows(const int64_t* timesteps, const float* freqs, float* out, int32_t half,
                                          int32_t B, ldm_stream_t stream) {
  using namespace ldm_host;
  LDM_REQUIRE(timesteps && freqs && out && half > 0 && B > 0 && B <= 65535, LDM_ERR_BAD_ARG,
              "ldm_timestep_sinusoid_rows: bad arg (half=%d, B=%d)", (int)half, (int)B);
  timestep_sinusoid_kernel<true><<<B, 256, 0, as_stream(stream)>>>(reinterpret_cast<const long long*>(timesteps),
                                                                   nullptr, freqs, out, half);
  count_launch();
  return check_launch("timestep_sinusoid_kernel");
}

extern "C" int ldm_gemv_bf16_rows(const void* w, const float* bias, const float* bias2, const float* x, float* out,
                                  int32_t N, int32_t K, int32_t B, const int32_t* seg_offs, int32_t nseg,
                                  int32_t silu_out, ldm_stream_t stream) {
  using namespace ldm_host;
  LDM_REQUIRE(w && x && out, LDM_ERR_BAD_ARG, "ldm_gemv_bf16_rows: null arg");
  LDM_REQUIRE(N > 0 && K > 0 && K % 8 == 0 && K <= 8192 && B > 0 && B <= 65535, LDM_ERR_BAD_SHAPE,
              "ldm_gemv_bf16_rows: N=%d K=%d B=%d", N, K, B);
  LDM_REQUIRE(!seg_offs || nseg > 0, LDM_ERR_BAD_ARG, "ldm_gemv_bf16_rows: nseg=%d", nseg);
  const int wpb = 8;
  int grid = (N + wpb - 1) / wpb;
  const int cap = num_sms() * 8;
  if (grid > cap) grid = cap;
  gemv_bf16_kernel<true><<<dim3(grid, B), wpb * 32, sizeof(float) * K, as_stream(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(w), bias, bias2, x, out, N, K, silu_out, seg_offs, nseg);
  count_launch();
  return check_launch("gemv_bf16_kernel");
}

static int check_rows_args(const char* what, const float* const* ptrs, int nptrs, const int32_t* rows, int64_t n,
                           int64_t elems_per_image) {
  using namespace ldm_host;
  LDM_REQUIRE(rows != nullptr, LDM_ERR_BAD_ARG, "%s: null rows", what);
  LDM_REQUIRE(n > 0 && elems_per_image > 0 && elems_per_image % 4 == 0, LDM_ERR_BAD_SHAPE,
              "%s: n=%lld elems_per_image=%lld (a positive multiple of 4)", what, (long long)n,
              (long long)elems_per_image);
  uintptr_t a = 0;
  for (int i = 0; i < nptrs; ++i) a |= (uintptr_t)ptrs[i];
  LDM_REQUIRE(a % 16 == 0, LDM_ERR_ALIGNMENT, "%s: pointers must be 16-byte aligned", what);
  return LDM_OK;
}

extern "C" int ldm_ddim_step_rows(const float* eps, const float* sample, const float* coef, const int32_t* rows,
                                  float* prev_sample, float* pred_x0, int64_t n, int64_t elems_per_image,
                                  ldm_stream_t stream) {
  using namespace ldm_host;
  LDM_REQUIRE(eps && sample && coef, LDM_ERR_BAD_ARG, "ldm_ddim_step_rows: null arg");
  const float* ptrs[] = {eps, sample, prev_sample, pred_x0};
  if (int rc = check_rows_args("ldm_ddim_step_rows", ptrs, 4, rows, n, elems_per_image)) return rc;
  ddim_step_kernel<true><<<grid_for(n / 4 + 1, 256), 256, 0, as_stream(stream)>>>(
      eps, nullptr, 0.f, sample, coef, rows, prev_sample, pred_x0, n, 0.f, 0, elems_per_image);
  count_launch();
  return check_launch("ddim_step_kernel");
}

extern "C" int ldm_dpmpp_step_rows(const float* eps, const float* sample, const float* coef, const int32_t* rows,
                                   float* prev_sample, float* x0_prev, int64_t n, int64_t elems_per_image,
                                   ldm_stream_t stream) {
  using namespace ldm_host;
  LDM_REQUIRE(eps && sample && coef && prev_sample && x0_prev, LDM_ERR_BAD_ARG, "ldm_dpmpp_step_rows: null arg");
  const float* ptrs[] = {eps, sample, prev_sample, x0_prev};
  if (int rc = check_rows_args("ldm_dpmpp_step_rows", ptrs, 4, rows, n, elems_per_image)) return rc;
  dpmpp_step_kernel<true><<<grid_for(n / 4 + 1, 256), 256, 0, as_stream(stream)>>>(
      eps, nullptr, 0.f, sample, coef, rows, prev_sample, x0_prev, n, elems_per_image);
  count_launch();
  return check_launch("dpmpp_step_kernel");
}

extern "C" int ldm_unipc_step_rows(const float* eps, const float* sample, const float* coef, const int32_t* rows,
                                   float* prev_sample, float* last, float* m1, float* m2, float* m3,
                                   int32_t solver_order, int64_t n, int64_t elems_per_image, ldm_stream_t stream) {
  using namespace ldm_host;
  LDM_REQUIRE(solver_order >= 1 && solver_order <= 3, LDM_ERR_BAD_ARG, "ldm_unipc_step_rows: solver_order=%d",
              (int)solver_order);
  LDM_REQUIRE(eps && sample && coef && prev_sample && last && m1 && (solver_order < 2 || m2) && (solver_order < 3 || m3),
              LDM_ERR_BAD_ARG, "ldm_unipc_step_rows: null arg");
  const float* ptrs[] = {eps, sample, prev_sample, last, m1, m2, m3};
  if (int rc = check_rows_args("ldm_unipc_step_rows", ptrs, 7, rows, n, elems_per_image)) return rc;
  const dim3 grid = grid_for(n / 4 + 1, 256);
  auto s = as_stream(stream);
  if (solver_order == 1)
    unipc_step_kernel<1, true><<<grid, 256, 0, s>>>(eps, nullptr, 0.f, sample, coef, rows, prev_sample, last, m1, m2,
                                                    m3, n, elems_per_image);
  else if (solver_order == 2)
    unipc_step_kernel<2, true><<<grid, 256, 0, s>>>(eps, nullptr, 0.f, sample, coef, rows, prev_sample, last, m1, m2,
                                                    m3, n, elems_per_image);
  else
    unipc_step_kernel<3, true><<<grid, 256, 0, s>>>(eps, nullptr, 0.f, sample, coef, rows, prev_sample, last, m1, m2,
                                                    m3, n, elems_per_image);
  count_launch();
  return check_launch("unipc_step_kernel");
}

extern "C" int ldm_conv3x3_small_cin(const float* s0, const float* s1, const float* s2, int32_t nsrc, int32_t cps,
                                     float scale, const float* w, const float* bias, void* out, int32_t B, int32_t h,
                                     int32_t wd, int32_t cout, ldm_stream_t stream) {
  return ldm_conv3x3_small_cin_act(s0, s1, s2, nsrc, cps, scale, w, bias, out, B, h, wd, cout, 0, stream);
}

extern "C" int ldm_conv3x3_small_cin_act(const float* s0, const float* s1, const float* s2, int32_t nsrc, int32_t cps,
                                         float scale, const float* w, const float* bias, void* out, int32_t B, int32_t h,
                                         int32_t wd, int32_t cout, int32_t silu, ldm_stream_t stream) {
  return ldm_conv3x3_small_cin_affine(s0, s1, s2, nsrc, cps, scale, 0.f, w, bias, out, B, h, wd, cout, silu, stream);
}

extern "C" int ldm_conv3x3_small_cin_affine(const float* s0, const float* s1, const float* s2, int32_t nsrc,
                                            int32_t cps, float scale, float shift, const float* w, const float* bias,
                                            void* out, int32_t B, int32_t h, int32_t wd, int32_t cout, int32_t silu,
                                            ldm_stream_t stream) {
  using namespace ldm_host;
  LDM_REQUIRE(s0 && w && out && nsrc >= 1 && nsrc <= 3 && (nsrc < 2 || s1) && (nsrc < 3 || s2), LDM_ERR_BAD_ARG,
              "ldm_conv3x3_small_cin: bad sources");
  LDM_REQUIRE(B > 0 && h > 0 && wd > 0 && cps > 0 && cout > 0 && cout <= 1024 && nsrc * cps <= 64, LDM_ERR_BAD_SHAPE,
              "ldm_conv3x3_small_cin: bad shape");
  const int threads = ((cout + 31) / 32) * 32;
  const int strips = (wd + kStrip - 1) / kStrip;
  const size_t shb = sizeof(float) * nsrc * cps * 3 * (kStrip + 2);
  conv3x3_small_cin_kernel<<<B * h * strips, threads, shb, as_stream(stream)>>>(
      s0, s1, s2, nsrc, cps, scale, shift, w, bias, reinterpret_cast<__nv_bfloat16*>(out), B, h, wd, cout, silu);
  count_launch();
  return check_launch("conv3x3_small_cin_kernel");
}

extern "C" int ldm_conv_out(const void* x, const float* w, const float* bias, float* out, int32_t B, int32_t h,
                            int32_t wd, int32_t cin, int32_t cout, ldm_stream_t stream) {
  using namespace ldm_host;
  LDM_REQUIRE(x && w && out, LDM_ERR_BAD_ARG, "ldm_conv_out: null arg");
  LDM_REQUIRE(cout > 0 && cout <= kMaxCoutSmall && cin % 8 == 0 && 9 * cin * cout * 4 <= 200 * 1024, LDM_ERR_BAD_SHAPE,
              "ldm_conv_out: cin=%d cout=%d unsupported", cin, cout);
  const size_t shb = sizeof(float) * 9 * cin * cout;
  cudaFuncSetAttribute(conv_out_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 200 * 1024);  // (per device)
  const int grid = num_sms() * 2;
  conv_out_kernel<<<grid, 256, shb, as_stream(stream)>>>(reinterpret_cast<const __nv_bfloat16*>(x), w, bias, out, B, h,
                                                         wd, cin, cout);
  count_launch();
  return check_launch("conv_out_kernel");
}

extern "C" int ldm_upsample_nearest(const void* x, void* out, int32_t B, int32_t h, int32_t w, int32_t C, int32_t oh,
                                    int32_t ow, ldm_stream_t stream) {
  using namespace ldm_host;
  LDM_REQUIRE(x && out && C % 8 == 0 && B > 0 && h > 0 && w > 0 && oh > 0 && ow > 0, LDM_ERR_BAD_ARG,
              "ldm_upsample_nearest: bad arg");
  // torch: scale = in/out in float unless an explicit scale_factor was given; for exact 2x both give 0.5
  const float sh_ = (oh == 2 * h) ? 0.5f : (float)h / (float)oh;
  const float sw_ = (ow == 2 * w) ? 0.5f : (float)w / (float)ow;
  const long long total = (long long)B * oh * ow * (C / 8);
  upsample_nearest_kernel<<<grid_for(total, 256), 256, 0, as_stream(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(x), reinterpret_cast<__nv_bfloat16*>(out), B, h, w, C, oh, ow, sh_, sw_);
  count_launch();
  return check_launch("upsample_nearest_kernel");
}

extern "C" int ldm_im2col3x3_s2(const void* x, void* out, int32_t B, int32_t h, int32_t w, int32_t C, int32_t oh,
                                int32_t ow, ldm_stream_t stream) {
  return ldm_im2col3x3_s2_pad(x, out, B, h, w, C, oh, ow, 1, stream);
}

extern "C" int ldm_im2col3x3_s2_pad(const void* x, void* out, int32_t B, int32_t h, int32_t w, int32_t C, int32_t oh,
                                    int32_t ow, int32_t pad_lo, ldm_stream_t stream) {
  using namespace ldm_host;
  LDM_REQUIRE(x && out && C % 8 == 0 && B > 0 && (pad_lo == 0 || pad_lo == 1), LDM_ERR_BAD_ARG,
              "ldm_im2col3x3_s2: bad arg");
  // rows / columns before the image: pad_lo; after it: 1 (conv pad 1, or F.pad(x, (0, 1, 0, 1)) in front of a pad-0 conv)
  LDM_REQUIRE(oh == (h + pad_lo - 2) / 2 + 1 && ow == (w + pad_lo - 2) / 2 + 1, LDM_ERR_BAD_SHAPE,
              "ldm_im2col3x3_s2: output %dx%d does not match the stride-2 conv of %dx%d (pad %d before, 1 after)", oh, ow,
              h, w, pad_lo);
  const long long total = (long long)B * oh * ow * 9 * (C / 8);
  im2col3x3_s2_kernel<<<grid_for(total, 256), 256, 0, as_stream(stream)>>>(
      reinterpret_cast<const __nv_bfloat16*>(x), reinterpret_cast<__nv_bfloat16*>(out), B, h, w, C, oh, ow, pad_lo);
  count_launch();
  return check_launch("im2col3x3_s2_kernel");
}
