// Fused flash-style self-attention for the 40-wide heads (320 channels / 8 heads: the 48x156 level, 7 488 tokens, 85 % of
// the attention time of one UNet forward; and the 96x312 level of the 768x2496 frames).
//
// What bounds this shape (measured, tools/microbench/): every score costs one exponential (MUFU: 7.8 cycles per warp
// instruction per scheduler) plus about four cycles of FMA / ALU issue, against 160 tensor FLOP -- the softmax is the
// kernel, the MMAs ride along. The generic kernel (attn_tc.cu: one thread per query row, two query groups) keeps only two
// softmax warps per scheduler; its per-block barrier round trips and the MUFU-free stretches of its exponential pass
// leave the MUFU pipe 40 % idle (tools/microbench/attn_trace.cu). This kernel runs FOUR softmax warps per scheduler:
//
//   grid = (ceil(seq / 256), B*heads); one CTA = two groups of 128 queries; 640 threads
//     warp 0            TMA producer : Q tiles once, then a ring of (K block | two V^T atoms) stages, 96 keys per block
//     warp 1            MMA issuer   : S = Q K^T (N = 96) and, per half, O_h += P_h V_h with P read straight from TMEM
//     warps 4..19       softmax      : TWO threads per query row. Thread h of a row owns keys [48h, 48h+48) of every
//                                      block and runs its own online softmax over them: own reference maximum, own row
//                                      sum, own accumulator O_h in TMEM. The halves never have to agree on anything while
//                                      the keys stream by (no per-block exchange, every guard stays exact per thread);
//                                      they are merged once at the end: O = (a0 O_0 + a1 O_1) / (a0 l_0 + a1 l_1) with
//                                      a_h = 2^(m_h - max(m_0, m_1)).
//   TMEM columns of one group (stride 256): a ring of 144 columns shared by S and P, then O_0 and O_1 (48 each).
//     S of an even block at [0, 96), its P (bf16 pairs, 48 columns) at [0, 48); S of an odd block at [48, 144), its P at
//     [96, 144). P of half 1 lands on score columns of half 0, so a thread's first P store of a block waits until all
//     256 threads of the group have their scores in registers (the s_free barrier, complete long before). S of block
//     j+1 never overlaps P of block j, and S of block j+2 is issued after PV of block j on the in-order tensor pipe --
//     so the softmax threads never wait for a PV MMA (only the rare rescale of O_h does).
//   V^T tile of a block: two 64-key SWIZZLE_128B atoms, keys [0, 64) and [32, 96) of the block; half 0 uses k-steps 0..2
//     of the first, half 1 k-steps 1..3 of the second (a 96-key block is 1.5 atoms wide).
//   Layouts as in attn_tc.cu: q, k [B*heads, seq, 64] (zero padded), vt [B*heads, 48, seq_pad] with row 40 = 1.0 (the PV
//   MMA then also produces the softmax row sums in column 40 of O_h), out [B*seq, heads*40]; all bf16.
#include <stdlib.h>

#include "attn_common.cuh"
#include "host_util.h"

namespace {
using namespace ldm;
using namespace ldm_attn;

constexpr int kD = 40;
constexpr int kDN = 48;            // UMMA N of the PV MMAs (40 channels + the ones row, padded to 16)
constexpr int kBKV = 96;           // keys per block
constexpr int kHalf = kBKV / 2;    // keys per thread and block
constexpr int kStages = 5;
constexpr int kQBytes = 128 * 128;                 // one group's Q tile (128 rows x 64 bf16)
constexpr int kKBytes = kBKV * 128;
constexpr int kVAtomBytes = kDN * 128;             // 48 rows x 64 keys
constexpr int kStageBytes = kKBytes + 2 * kVAtomBytes;  // 24 KB
constexpr int kMergeStride = 43;   // floats per row in the merge buffer (m, l, 40 x O; odd stride: no bank conflicts)
constexpr int kMergeBytes = 2 * 128 * kMergeStride * 4;
constexpr int kSmem = 2 * kQBytes + kStages * kStageBytes + kMergeBytes + 1024 + 512;
constexpr int kThreads = 128 + 2 * 256;
constexpr int kGroupStride = 256;  // TMEM columns
constexpr int kRing = kBKV + kBKV / 2;
static_assert(kRing + 2 * kDN <= kGroupStride, "TMEM budget");
static_assert(kStageBytes % 1024 == 0, "stage alignment");
static_assert(kSmem <= 227 * 1024, "smem budget");

template <int kPoly>
__global__ void __launch_bounds__(kThreads, 1)
flash_attn40_kernel(const __grid_constant__ CUtensorMap tmQ, const __grid_constant__ CUtensorMap tmK,
                    const __grid_constant__ CUtensorMap tmV, const AttnParams p) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t* smem = smem_raw + ((1024u - (smem_u32(smem_raw) & 1023u)) & 1023u);  // an offset, not an integer round trip: the compiler keeps the shared address space (LDS / STS instead of generic LD / ST)
  uint8_t* sQ = smem;                   // 2 * kQBytes
  uint8_t* sKV = sQ + 2 * kQBytes;      // kStages * kStageBytes
  float* sMerge = reinterpret_cast<float*>(sKV + kStages * kStageBytes);  // kMergeBytes
  uint64_t* bars = reinterpret_cast<uint64_t*>(sKV + kStages * kStageBytes + kMergeBytes);
  uint64_t* q_full = bars;              // [2]
  uint64_t* kv_full = q_full + 2;       // [kStages]
  uint64_t* kv_empty = kv_full + 8;     // [kStages]
  uint64_t* s_full = kv_empty + 8;      // [2]
  uint64_t* p_full = s_full + 2;        // [2][2]: one barrier per (group, block parity), see the MMA warp's wait
  uint64_t* o_full = p_full + 4;        // [2]
  uint64_t* s_free = o_full + 2;        // [2]
  uint64_t* o_done = s_free + 2;        // [2] completes ONCE, when the last block's PV MMAs have landed (see the final wait)
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(o_done + 2);

  const int warp = __shfl_sync(0xffffffffu, (int)(threadIdx.x >> 5), 0);
  const int lane = threadIdx.x & 31;
  const int bh = blockIdx.y;
  const int q_base = blockIdx.x * 256;
  const int nblk = (p.kv_seq + kBKV - 1) / kBKV;

  if (warp == 0 && lane == 0) {
    tma_prefetch_desc(&tmQ);
    tma_prefetch_desc(&tmK);
    tma_prefetch_desc(&tmV);
    for (int g = 0; g < 2; ++g) {
      mbar_init(&q_full[g], 1);
      mbar_init(&s_full[g], 1);
      mbar_init(&p_full[2 * g], 256);
      mbar_init(&p_full[2 * g + 1], 256);
      mbar_init(&o_full[g], 1);
      mbar_init(&o_done[g], 1);
      mbar_init(&s_free[g], 256);
    }
    for (int s = 0; s < kStages; ++s) {
      mbar_init(&kv_full[s], 1);
      mbar_init(&kv_empty[s], 1);
    }
    mbar_fence_init();
  }
  if (warp == 1) {
    tmem_alloc(tmem_slot, 512);
    tmem_relinquish();
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  pdl_launch_dependents();
  pdl_wait();

  // 640 threads start at 96 registers (61 440 for the CTA, the pool setmaxnreg works in): 128 x 56 + 512 x 104 fits
  if (warp < 4) {
    asm volatile("setmaxnreg.dec.sync.aligned.u32 56;");
    if (warp == 0) {
      // ------------------------------------------------------------------ TMA producer
      if (elect_one()) {
        for (int g = 0; g < 2; ++g) {
          mbar_arrive_expect_tx(&q_full[g], kQBytes);
          tma_load_3d(sQ + g * kQBytes, &tmQ, &q_full[g], 0, q_base + g * 128, bh);
        }
      }
      int stage = 0;
      uint32_t phase = 0;
      for (int j = 0; j < nblk; ++j) {
        mbar_wait(&kv_empty[stage], phase ^ 1);
        uint8_t* sk = sKV + stage * kStageBytes;
        uint8_t* sv = sk + kKBytes;
        if (elect_one()) {
          mbar_arrive_expect_tx(&kv_full[stage], kStageBytes);
          tma_load_3d(sk, &tmK, &kv_full[stage], 0, j * kBKV, bh);
          tma_load_3d(sv, &tmV, &kv_full[stage], j * kBKV, 0, bh);
          tma_load_3d(sv + kVAtomBytes, &tmV, &kv_full[stage], j * kBKV + 32, 0, bh);
        }
        __syncwarp();
        if (++stage == kStages) {
          stage = 0;
          phase ^= 1;
        }
      }
      __syncwarp();
    } else if (warp == 1) {
      // ------------------------------------------------------------------ MMA issuer (all lanes wait, one lane issues)
      const uint32_t idesc_s = umma_idesc_bf16(128, kBKV);
      const uint32_t idesc_o = umma_idesc_bf16(128, kDN);
      auto issue_s = [&](int g, int stage, int blk) {
        const uint32_t qa = smem_u32(sQ + g * kQBytes);
        const uint32_t ka = smem_u32(sKV + stage * kStageBytes);
        const uint32_t d_tmem = tmem_base + g * kGroupStride + (blk & 1) * (kBKV / 2);
        if (elect_one()) {
#pragma unroll
          for (int kk = 0; kk < 3; ++kk)
            umma_bf16(d_tmem, umma_desc_k_sw128(qa + kk * 32), umma_desc_k_sw128(ka + kk * 32), idesc_s, kk != 0);
          umma_commit(&s_full[g]);
        }
        __syncwarp();
      };
      auto issue_o = [&](int g, int stage, int blk) {
        const uint32_t pa = tmem_base + g * kGroupStride + (blk & 1) * kBKV;  // 8 columns per k-step, 24 per half
        const uint32_t va = smem_u32(sKV + stage * kStageBytes + kKBytes);
        const uint32_t d_tmem = tmem_base + g * kGroupStride + kRing;
        if (elect_one()) {
#pragma unroll
          for (int h = 0; h < 2; ++h)
#pragma unroll
            for (int kk = 0; kk < 3; ++kk)
              umma_bf16_ts(d_tmem + h * kDN, pa + h * 24 + kk * 8,
                           umma_desc_k_sw128(va + h * kVAtomBytes + (kk + h) * 32), idesc_o, blk > 0 || kk != 0);
          umma_commit(&o_full[g]);
          if (blk == nblk - 1) umma_commit(&o_done[g]);
        }
        __syncwarp();
      };
      for (int g = 0; g < 2; ++g) mbar_wait(&q_full[g], 0);
      mbar_wait(&kv_full[0], 0);
      tc_fence_after();
      for (int g = 0; g < 2; ++g) {
        TRACE(2 + g, 0);
        issue_s(g, 0, 0);
      }
      for (int j = 0; j < nblk; ++j) {
        const int stage = j % kStages, nstage = (j + 1) % kStages;
        if (j + 1 < nblk) {
          // S of the next block as soon as the softmax threads have pulled this block's scores out of TMEM
          mbar_wait(&kv_full[nstage], ((j + 1) / kStages) & 1);
          for (int g = 0; g < 2; ++g) {
            mbar_wait(&s_free[g], j & 1);
            tc_fence_after();
            TRACE(2 + g, j + 1);
            issue_s(g, nstage, j + 1);
          }
        }
        for (int g = 0; g < 2; ++g) {
          // Two barriers per group, alternating with the block parity. With one, a group whose softmax threads finish
          // blocks j AND j + 1 (S of j + 1 is issued above, before this wait) while this warp is still held up by the
          // other group's s_free would complete two phases before the wait looks: a parity wait then never returns.
          // Arrivals for block j + 2 need S of j + 2, which is only issued after this wait has returned.
          mbar_wait(&p_full[2 * g + (j & 1)], (j >> 1) & 1);
          tc_fence_after();
          TRACE(4 + g, j);
          issue_o(g, stage, j);
        }
        if (elect_one()) umma_commit(&kv_empty[stage]);
        __syncwarp();
      }
      __syncwarp();
    }
  } else {
    // ------------------------------------------------------------------ softmax: two threads per query row
    asm volatile("setmaxnreg.inc.sync.aligned.u32 104;");
    const int sw = warp - 4;            // 0..15
    const int g = sw >> 3;              // query group
    const int h = (sw >> 2) & 1;        // which half of every key block
    const int quad = warp & 3;          // TMEM lane quadrant this warp may touch
    const int r = quad * 32 + lane;     // query row inside the group
    const int qrow = q_base + g * 128 + r;
    const uint32_t t_g = tmem_base + ((uint32_t)(quad * 32) << 16) + g * kGroupStride;
    const uint32_t t_o = t_g + kRing + h * kDN;
    float m = -INFINITY;                // reference maximum P / O_h are relative to (log2 domain)
    float m_seen = -INFINITY;           // running maximum of this half including the previous block
    constexpr float kLazy = 8.0f;       // rescale O_h only when the maximum grew by more than 2^8 ...
    constexpr float kRedo = 64.0f;      // ... and redo a block's exponentials if it alone jumps by more than 2^64

    for (int j = 0; j < nblk; ++j) {
      const int nvalid = p.kv_seq - j * kBKV - h * kHalf;  // keys of this half inside the sequence (may be <= 0)
      const uint32_t t_s = t_g + (j & 1) * (kBKV / 2) + h * kHalf;  // this half's scores ...
      const uint32_t t_p = t_g + (j & 1) * kBKV + h * (kHalf / 2);  // ... and where its P goes
      TRACE(0, j);
      mbar_wait(&s_full[g], j & 1);
      tc_fence_after();
      TRACE(1, j);
      uint32_t sv[kHalf];
      tmem_ld32(t_s, sv);
      tmem_ld16(t_s + 32, sv + 32);
      tmem_ld_wait();
      TRACE(2, j);
      tc_fence_before();
      mbar_arrive(&s_free[g]);  // the S columns may be overwritten by the next block's QK^T now
      if (nvalid < kHalf) {     // only the last block of a ragged sequence
#pragma unroll
        for (int i = 0; i < kHalf; ++i)
          if (i >= nvalid) sv[i] = 0xff800000u;  // -inf
      }

      // O_h (TMEM) moves to the new reference max(m, target) for the rows that need it
      auto rescale = [&](bool need, float target) {
        if (j > 0) mbar_wait(&o_full[g], (j - 1) & 1);  // PV of the previous block has landed in O_h
        tc_fence_after();
        const float m_new = need ? target : m;
        const float alpha = ex2(m - m_new);  // 1 for the rows that keep their reference
        m = m_new;
#pragma unroll
        for (int c = 0; c < kDN; c += 16) {
          uint32_t v[16];
          tmem_ld16(t_o + c, v);
          tmem_ld_wait();
#pragma unroll
          for (int i = 0; i < 16; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) * alpha);
          tmem_st16(t_o + c, v);
        }
        tmem_st_wait();
      };
      // P = exp2(s*scale - m) as bf16 pairs into TMEM; the block maximum is tracked in the same pass
      auto exp_pass = [&](float& bmax) {
        float mx0 = -INFINITY, mx1 = -INFINITY;
        const uint64_t scale2 = pack2(p.scale_log2, p.scale_log2), negm2 = pack2(-m, -m);
#pragma unroll
        for (int c = 0; c < kHalf; c += 16) {
          uint32_t u[8];
#pragma unroll
          for (int q = 0; q < 8; ++q) {  // pairs of keys; kPoly of every 8 pairs take the FMA-pipe exp2
            const float s0 = __uint_as_float(sv[c + 2 * q]), s1 = __uint_as_float(sv[c + 2 * q + 1]);
            if (q & 1) mx1 = fmax3(mx1, s0, s1); else mx0 = fmax3(mx0, s0, s1);
            const uint64_t x = ffma2(pack2(s0, s1), scale2, negm2);
            float e0, e1;
            if (q < 8 - kPoly) {
              float x0, x1;
              unpack2(x, x0, x1);
              e0 = ex2(x0);
              e1 = ex2(x1);
            } else {
              ex2_poly2(x, e0, e1);
            }
            u[q] = pack_bf16(e0, e1);
          }
          if (c == 0) mbar_wait(&s_free[g], j & 1);  // every thread of the group has read its scores (see the ring)
          tmem_st8(t_p + (c >> 1), u);  // keys c .. c+15 of this half = 8 columns of bf16 pairs
        }
        bmax = fmaxf(mx0, mx1) * p.scale_log2;  // scale > 0
      };

      if (j == 0) {
        // the first block needs its true maximum up front (nothing to be relative to yet)
        float mx0 = -INFINITY, mx1 = -INFINITY;
#pragma unroll
        for (int i = 0; i < kHalf; i += 4) {
          mx0 = fmax3(mx0, __uint_as_float(sv[i]), __uint_as_float(sv[i + 1]));
          mx1 = fmax3(mx1, __uint_as_float(sv[i + 2]), __uint_as_float(sv[i + 3]));
        }
        m = fmaxf(mx0, mx1) * p.scale_log2;
        if (m == -INFINITY) m = 0.f;  // this half has no key at all (kv_seq <= 48): P = 0, l = 0 (see the merge)
        m_seen = m;
      } else {
        const bool need = m_seen - m > kLazy;
        if (__any_sync(0xffffffffu, need)) rescale(need, m_seen);
      }
      float bmax;
      exp_pass(bmax);
      if (j > 0) {
        const bool redo = bmax - m > kRedo;  // would leave the comfortable fp32 / bf16 range: never on sane inputs
        if (__any_sync(0xffffffffu, redo)) {
          rescale(redo, bmax);
          exp_pass(bmax);
        }
      }
      m_seen = fmaxf(m_seen, bmax);
      TRACE(3, j);
      tmem_st_wait();
      tc_fence_before();
      mbar_arrive(&p_full[2 * g + (j & 1)]);
      TRACE(4, j);
    }
    // NOT o_full with the parity of the last block: a softmax thread never waits for a PV MMA inside the loop, so here
    // it can be TWO commits ahead of the tensor pipe (s_full of block j only implies PV of block j-2), and a parity wait
    // cannot tell "phase nblk-3 complete" from "phase nblk-1 complete" -- a fast warp then read O without the last two
    // blocks (seen as a run-to-run difference of one warp's rows). o_done has a single phase.
    mbar_wait(&o_done[g], 0);
    tc_fence_after();
    float o_acc[kDN];
    {
      uint32_t v[kDN];
#pragma unroll
      for (int c = 0; c < kDN; c += 16) tmem_ld16(t_o + c, v + c);
      tmem_ld_wait();
#pragma unroll
      for (int i = 0; i < kDN; ++i) o_acc[i] = __uint_as_float(v[i]);
    }
    // merge the two halves of a row: half 1 publishes (m, l, O) through shared memory, half 0 combines. Half 0 always
    // has a key; half 1 has none when kv_seq <= 48 and then enters with m = -inf, i.e. weight a1 = 0, a0 = 1. (Its
    // placeholder m = 0 would give a0 = 2^(m0 - 0) = 0 and 1 / 0 for a row whose scores all lie below -126 log2 units.)
    float* mg = sMerge + (g * 128 + r) * kMergeStride;
    if (h == 1) {
      mg[0] = p.kv_seq > kHalf ? m : -INFINITY;
      mg[1] = o_acc[kD];
#pragma unroll
      for (int c = 0; c < kD; ++c) mg[2 + c] = o_acc[c];
    }
    named_bar_sync(1 + g, 256);
    if (h == 0 && qrow < p.seq) {
      const float m1 = mg[0], l1 = mg[1];
      const float mm = fmaxf(m, m1);
      const float a0 = ex2(m - mm), a1 = ex2(m1 - mm);
      const float inv = 1.0f / (a0 * o_acc[kD] + a1 * l1);
      const float w0 = a0 * inv, w1 = a1 * inv;
      const int b = bh / p.heads, head = bh - b * p.heads;
      __nv_bfloat16* dst = p.out + ((long long)b * p.seq + qrow) * (p.heads * kD) + head * kD;
#pragma unroll
      for (int c = 0; c < kD; c += 8) {
        float o[8];
#pragma unroll
        for (int i = 0; i < 8; ++i) o[i] = w0 * o_acc[c + i] + w1 * mg[2 + c + i];
        uint4 u;
        u.x = pack_bf16(o[0], o[1]);
        u.y = pack_bf16(o[2], o[3]);
        u.z = pack_bf16(o[4], o[5]);
        u.w = pack_bf16(o[6], o[7]);
        *reinterpret_cast<uint4*>(dst + c) = u;
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, 512);
  }
}

template <int kPoly>
int launch(const ldm_attn_desc* d, cudaStream_t s) {
  using namespace ldm_host;
  const int BH = d->B * d->heads;
  const int kv_seq = d->kv_seq > 0 ? d->kv_seq : d->seq;
  CUtensorMap tmQ, tmK, tmV;
  {
    const uint64_t dims[3] = {(uint64_t)d->dpad, (uint64_t)d->seq, (uint64_t)BH};
    const uint64_t str[2] = {(uint64_t)d->dpad * 2, (uint64_t)d->dpad * 2 * d->seq};
    const uint64_t dimsk[3] = {(uint64_t)d->dpad, (uint64_t)kv_seq, (uint64_t)BH};
    const uint64_t strk[2] = {(uint64_t)d->dpad * 2, (uint64_t)d->dpad * 2 * kv_seq};
    const uint32_t boxq[3] = {64, 128, 1};
    const uint32_t boxk[3] = {64, (uint32_t)kBKV, 1};
    int rc = make_tmap(&tmQ, d->q, 3, dims, str, boxq, 2, true);
    if (rc) return rc;
    rc = make_tmap(&tmK, d->k, 3, dimsk, strk, boxk, 2, true);
    if (rc) return rc;
  }
  {
    const uint64_t dims[3] = {(uint64_t)kv_seq, (uint64_t)d->vt_rows, (uint64_t)BH};
    const uint64_t str[2] = {(uint64_t)d->seq_pad * 2, (uint64_t)d->seq_pad * 2 * d->vt_rows};
    const uint32_t box[3] = {64, (uint32_t)kDN, 1};
    int rc = make_tmap(&tmV, d->vt, 3, dims, str, box, 2, true);
    if (rc) return rc;
  }
  AttnParams p;
  p.seq = d->seq;
  p.kv_seq = kv_seq;
  p.heads = d->heads;
  p.head_dim = d->head_dim;
  p.scale_log2 = d->scale * 1.4426950408889634f;
  p.out = reinterpret_cast<__nv_bfloat16*>(d->out);
  auto kern = flash_attn40_kernel<kPoly>;
  {  // per launch (the attribute is per device; see gemm_tc_inst.cuh)
    cudaError_t e = cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, kSmem);
    if (e != cudaSuccess) return set_error(LDM_ERR_CUDA, "cudaFuncSetAttribute(attn40): %s", cudaGetErrorString(e));
  }
  dim3 grid((d->seq + 255) / 256, BH);
  cudaError_t le = launch_pdl(kern, grid, dim3(kThreads), (size_t)kSmem, s, 1, tmQ, tmK, tmV, p);
  if (le != cudaSuccess) return set_error(LDM_ERR_CUDA, "flash_attn40_kernel launch: %s", cudaGetErrorString(le));
  count_launch();
  return check_launch("flash_attn40_kernel");
}

}  // namespace

int ldm_launch_attn40(const ldm_attn_desc* d, cudaStream_t s) {
  // LDM_ATTN_POLY=0..4 (diagnostic builds): A/B timing of the FMA-pipe exp2 share (n of 8 pairs)
  switch (ldm_host::diag_env("LDM_ATTN_POLY", 2)) {
    case 0: return launch<0>(d, s);
    case 1: return launch<1>(d, s);
    case 3: return launch<3>(d, s);
    case 4: return launch<4>(d, s);
    default: return launch<2>(d, s);
  }
}
