// Single-head attention over all T = H * W positions of the VQ-GAN bottleneck as ONE streaming tcgen05 kernel:
//
//     O = softmax(Q K^T * C^-1/2) V + b_v                   (per image, every query against every key)
//
// reference: AttnBlock.forward between the q / k / v convolutions and proj_out (ldm/modules/diffusionmodules/model.py:
// 180-203); the reference runs large latents through xformers' MemoryEfficientAttnBlock (:205-270).  Neither S nor P
// leaves the SM, so the workspace has no T^2 term (the three-GEMM path of vq.inc writes S of every image to memory).
//
//   * inputs: Q, K the NHWC fp16 outputs of the .q / .k 1x1 convs ([N][T][C]), V^T [N][C][T] fp16 WITHOUT the value bias
//     (the per-image GEMM of vq.inc produces it; it is the K-major B operand of PV), b_v fp32 [C]; output [N][T][C] fp16;
//   * a CTA owns one 128-query block of one image and one channel part of O: C <= 256 in one part (DV = C), larger C in
//     two (DV = C / 2, each part recomputes Q K^T: 1.5x the algorithmic FLOPs at C = 512).  Grid = (T / 128, C / DV, N);
//   * key blocks of 128: S_j = Q K_j^T (M = 128, N = 128, K = C in 64-channel k-blocks) into one of two TMEM S buffers,
//     so S_{j+1} runs on the tensor core while the softmax warps work on S_j; O += P_j V_j (N = DV / n_vc per MMA);
//   * online softmax in fp32, one thread per query row (TMEM lane): running max m and sum l in registers.  The max is
//     kept STALE until a block raises it by more than 8 (log2 units): P then stays <= 2^8, exact in fp16's range, and the
//     O accumulator is rescaled in TMEM only on those rare blocks (O and l always share the same m, so the result is the
//     same).  P is rounded to fp16 for PV (the three-GEMM path rounds S and P to fp16 too); O is normalised by 1 / l at the
//     end and b_v is added there (rows of P sum to 1: vq.inc's header);
//   * keys beyond T (a last block of 64) are masked to -inf and their V^T half-block is neither loaded nor multiplied;
//     query rows beyond T are computed on zero-filled Q and not stored.  No atomics: runs are bit-reproducible.
//
// TMEM (512 columns, the whole of it: one CTA per SM, which the shared memory forces anyway):
//     [0, 128) S buffer 0, [128, 256) S buffer 1, [256, 256 + DV) O  (DV <= 256).
// Shared memory (dynamic, C = 512):  Q block 128 x C fp16 resident (C / 64 k-blocks x 16 KB = 128 KB) | P 128 x 128 fp16
// (32 KB, two 64-key k-blocks) | a four-slot ring of 16 KB TMA tiles (K k-blocks [128 keys x 64 ch], V^T tiles
// [<= 128 ch x 64 keys]) = 64 KB | barriers: 225.25 KB + 1 KB alignment slack.
//
// Warp roles (192 threads): warps 0-3 softmax / O correction / epilogue (warp w <-> TMEM lanes [32 w, +32)), warp 4 TMA
// producer, warp 5 TMEM allocation + MMA issue.  The producer and the issuer walk the same sequence of ring tiles:
//     K_0, then for every key block j: K_{j+1} (if any), V_j.
#pragma once

#include "common.cuh"

namespace rs {

constexpr int kVqaThreads = 192;
constexpr int kVqaTmaWarp = 4, kVqaMmaWarp = 5;
constexpr int kVqaSlots = 4;
constexpr int kVqaSlotBytes = 16384;
constexpr int kVqaSlack = 1024;

struct VqAttnParams {
  CUtensorMap tmQ;         // {C, T, N} fp16, box {64, 128, 1}
  CUtensorMap tmK;         // {C, T, N} fp16, box {64, 128, 1}
  CUtensorMap tmVt;        // {T, C, N} fp16, box {64, VC, 1}
  const float* bias;       // b_v [C]
  __half* out;             // [N][T][ld_out]
  int ld_out;
  int T, C;
  int DV;                  // O channels per CTA (C or C / 2)
  int n_vc;                // V^T tiles (MMAs) per 64-key half-block: DV / VC
  int VC;                  // channels per V^T tile (<= 128)
  float scale_log2;        // C^-1/2 * log2(e)
};

// host and device agree on the layout
__host__ __device__ inline int vqa_off_p(int C) { return (C / 64) * 16384; }
__host__ __device__ inline int vqa_off_ring(int C) { return vqa_off_p(C) + 32768; }
__host__ __device__ inline int vqa_off_bars(int C) { return vqa_off_ring(C) + kVqaSlots * kVqaSlotBytes; }
__host__ __device__ inline int vqa_smem_bytes(int C) { return vqa_off_bars(C) + 256 + kVqaSlack; }

#ifdef __CUDACC__

__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* m, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.tile.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(m)), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// registers -> TMEM: 32 lanes x 32-bit, 16 consecutive columns per thread (the inverse of tmem_ld16)
__device__ __forceinline__ void tmem_st16(uint32_t taddr, const uint32_t (&v)[16]) {
  asm volatile(
      "tcgen05.st.sync.aligned.32x32b.x16.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, %16};"
      ::"r"(taddr), "r"(v[0]), "r"(v[1]), "r"(v[2]), "r"(v[3]), "r"(v[4]), "r"(v[5]), "r"(v[6]), "r"(v[7]), "r"(v[8]),
      "r"(v[9]), "r"(v[10]), "r"(v[11]), "r"(v[12]), "r"(v[13]), "r"(v[14]), "r"(v[15])
      : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ float vqa_ex2(float x) {
  float y;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(y) : "f"(x));
  return y;
}
__device__ __forceinline__ uint32_t vqa_pack_h2(float a, float b) {
  __half2 h = __floats2half2_rn(a, b);
  return *reinterpret_cast<uint32_t*>(&h);
}

__global__ void __launch_bounds__(kVqaThreads, 1) vq_attn_tc_kernel(const __grid_constant__ VqAttnParams p) {
  extern __shared__ __align__(1024) uint8_t vqa_smem_raw[];
  const uint32_t base_pad = (1024u - (smem_u32(vqa_smem_raw) & 1023u)) & 1023u;
  if (base_pad > (uint32_t)kVqaSlack) __trap();
  uint8_t* smem = vqa_smem_raw + base_pad;
  const int C = p.C, T = p.T, DV = p.DV, VC = p.VC, n_vc = p.n_vc;
  const int nkb = C / 64;                       // 64-channel k-blocks of Q K^T
  const int nk = (T + 127) / 128;               // key blocks
  const int q0 = blockIdx.x * 128, part = blockIdx.y, img = blockIdx.z;
  const uint32_t sQ = smem_u32(smem), sP = sQ + (uint32_t)vqa_off_p(C), sRing = sQ + (uint32_t)vqa_off_ring(C);
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + vqa_off_bars(C));
  uint64_t* full = bars;                        // [4] TMA -> MMA
  uint64_t* empty = bars + 4;                   // [4] MMA commit -> TMA
  uint64_t* q_full = bars + 8;
  uint64_t* s_full = bars + 9;                  // [2] commit of S_j (buffer j & 1)
  uint64_t* p_full = bars + 11;                 // 4 softmax warps: P_j in shared memory, O corrected, S_j read
  uint64_t* o_full = bars + 12;                 // commit of PV_j
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 13);
  // 64-key halves of key block j that hold keys < T
  auto halves = [&](int j) { return min(2, (T - j * 128) / 64); };

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  if (warp == kVqaTmaWarp && lane == 0) {
    tma_prefetch_desc(&p.tmQ); tma_prefetch_desc(&p.tmK); tma_prefetch_desc(&p.tmVt);
    for (int s = 0; s < kVqaSlots; ++s) { mbar_init(&full[s], 1); mbar_init(&empty[s], 1); }
    mbar_init(q_full, 1);
    mbar_init(&s_full[0], 1); mbar_init(&s_full[1], 1);
    mbar_init(p_full, 4); mbar_init(o_full, 1);
    mbar_fence_init();
  }
  if (warp == kVqaMmaWarp) { tmem_alloc_dyn(tmem_slot, 512u); tmem_relinquish(); }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;
  const uint32_t tmO = tmem_base + 256;
  pdl_trigger();
  pdl_wait();                                   // Q / K / V^T come from the previous kernels; the output may alias their inputs

  if (warp == kVqaTmaWarp) {
    // ===================== TMA producer =====================
    const bool el = elect_one();
    if (el) {
      mbar_arrive_expect_tx(q_full, (uint32_t)nkb * 16384u);
      for (int kb = 0; kb < nkb; ++kb) tma_load_3d(smem + kb * 16384, &p.tmQ, q_full, kb * 64, q0, img);
    }
    int slot = 0; uint32_t ph = 0;
    auto next = [&]() { if (++slot == kVqaSlots) { slot = 0; ph ^= 1; } };
    auto load_k = [&](int j) {
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(&empty[slot], ph ^ 1);
        if (el) {
          mbar_arrive_expect_tx(&full[slot], 16384u);
          tma_load_3d(smem + vqa_off_ring(C) + slot * kVqaSlotBytes, &p.tmK, &full[slot], kb * 64, j * 128, img);
        }
        next();
      }
    };
    auto load_v = [&](int j) {
      for (int kh = 0; kh < halves(j); ++kh)
        for (int vc = 0; vc < n_vc; ++vc) {
          mbar_wait(&empty[slot], ph ^ 1);
          if (el) {
            mbar_arrive_expect_tx(&full[slot], (uint32_t)VC * 128u);
            tma_load_3d(smem + vqa_off_ring(C) + slot * kVqaSlotBytes, &p.tmVt, &full[slot], j * 128 + kh * 64,
                        part * DV + vc * VC, img);
          }
          next();
        }
    };
    load_k(0);
    for (int j = 0; j < nk; ++j) {
      if (j + 1 < nk) load_k(j + 1);
      load_v(j);
    }
  } else if (warp == kVqaMmaWarp) {
    // ===================== MMA issuer =====================
    const bool el = elect_one();
    const uint32_t idesc_s = umma_idesc_f16(128, 128), idesc_pv = umma_idesc_f16(128, VC);
    int slot = 0; uint32_t ph = 0;
    auto next = [&]() { if (++slot == kVqaSlots) { slot = 0; ph ^= 1; } };
    mbar_wait(q_full, 0);
    tc_fence_after();
    // S_j = Q K_j^T into S buffer j & 1 (its previous contents, S_{j-2}, were read before p_full of j - 2, which the
    // issuer waited for before PV_{j-2}: earlier in the sequence)
    auto issue_s = [&](int j) {
      const uint32_t d = tmem_base + (uint32_t)(j & 1) * 128u;
      for (int kb = 0; kb < nkb; ++kb) {
        mbar_wait(&full[slot], ph);
        tc_fence_after();
        if (el) {
          const uint64_t ad = umma_desc_sw128(sQ + (uint32_t)kb * 16384u);
          const uint64_t bd = umma_desc_sw128(sRing + (uint32_t)slot * kVqaSlotBytes);
#pragma unroll
          for (int k = 0; k < 4; ++k) umma_f16(d, ad + 2 * k, bd + 2 * k, idesc_s, (kb | k) != 0 ? 1u : 0u);
          umma_commit(&empty[slot]);
        }
        __syncwarp();
        next();
      }
      if (el) umma_commit(&s_full[j & 1]);
      __syncwarp();
    };
    // O (+)= P_j V_j: per 64-key half, n_vc MMAs of N = VC into consecutive O columns
    auto issue_pv = [&](int j) {
      mbar_wait(p_full, (uint32_t)j & 1u);
      tc_fence_after();
      for (int kh = 0; kh < halves(j); ++kh)
        for (int vc = 0; vc < n_vc; ++vc) {
          mbar_wait(&full[slot], ph);
          tc_fence_after();
          if (el) {
            const uint64_t ad = umma_desc_sw128(sP + (uint32_t)kh * 16384u);
            const uint64_t bd = umma_desc_sw128(sRing + (uint32_t)slot * kVqaSlotBytes);
            const uint32_t d = tmO + (uint32_t)(vc * VC);
#pragma unroll
            for (int k = 0; k < 4; ++k) umma_f16(d, ad + 2 * k, bd + 2 * k, idesc_pv, (j | kh | k) != 0 ? 1u : 0u);
            umma_commit(&empty[slot]);
          }
          __syncwarp();
          next();
        }
      if (el) umma_commit(o_full);
      __syncwarp();
    };
    issue_s(0);
    for (int j = 0; j < nk; ++j) {
      if (j + 1 < nk) issue_s(j + 1);
      issue_pv(j);
    }
  } else {
    // ===================== softmax warps: thread r owns query row q0 + r (TMEM lane r) =====================
    const int r = tid;
    const uint32_t lane_base = (uint32_t)(warp * 32) << 16;
    uint8_t* const pP = smem + vqa_off_p(C);
    const int rsw = r & 7;
    float m_run = -INFINITY, l_run = 0.f;
    for (int j = 0; j < nk; ++j) {
      mbar_wait(&s_full[j & 1], (uint32_t)(j >> 1) & 1u);
      tc_fence_after();
      float s[128];
      {
        const uint32_t ts = tmem_base + lane_base + (uint32_t)(j & 1) * 128u;
#pragma unroll
        for (int c = 0; c < 8; ++c) {
          uint32_t v[16];
          tmem_ld16(ts + (uint32_t)(16 * c), v);
          tmem_ld_wait16(v);
#pragma unroll
          for (int i = 0; i < 16; ++i) s[16 * c + i] = __uint_as_float(v[i]);
        }
      }
      const int valid = T - j * 128;              // keys of this block below T (64 or >= 128)
      float mx4[4] = {-INFINITY, -INFINITY, -INFINITY, -INFINITY};
#pragma unroll
      for (int c = 0; c < 128; ++c) {
        s[c] = c < valid ? s[c] * p.scale_log2 : -INFINITY;
        mx4[c & 3] = fmaxf(mx4[c & 3], s[c]);
      }
      const float mx = fmaxf(fmaxf(mx4[0], mx4[1]), fmaxf(mx4[2], mx4[3]));
      float alpha = 1.f;
      bool rescale = false;
      if (j == 0) {
        m_run = mx;
      } else if (mx > m_run + 8.0f) {
        alpha = vqa_ex2(m_run - mx);
        m_run = mx;
        rescale = true;
      }
      uint32_t pk[64];
      float sum4[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int c = 0; c < 64; ++c) {
        const float e0 = vqa_ex2(s[2 * c] - m_run), e1 = vqa_ex2(s[2 * c + 1] - m_run);
        sum4[c & 3] += e0 + e1;
        pk[c] = vqa_pack_h2(e0, e1);
      }
      l_run = fmaf(l_run, alpha, (sum4[0] + sum4[1]) + (sum4[2] + sum4[3]));
      if (j > 0) {
        // PV_{j-1} has completed: O is up to date and P may be overwritten
        mbar_wait(o_full, (uint32_t)(j - 1) & 1u);
        tc_fence_after();
        if (__any_sync(0xffffffffu, rescale)) {
          for (int c = 0; c < DV; c += 16) {
            uint32_t v[16];
            tmem_ld16(tmO + lane_base + (uint32_t)c, v);
            tmem_ld_wait16(v);
#pragma unroll
            for (int i = 0; i < 16; ++i) v[i] = __float_as_uint(__uint_as_float(v[i]) * alpha);
            tmem_st16(tmO + lane_base + (uint32_t)c, v);
          }
          tmem_st_wait();
        }
      }
      // P_j: row r of two K-major 128B-swizzled [128 rows][64 keys] tiles
#pragma unroll
      for (int u = 0; u < 16; ++u) {
        uint8_t* dst = pP + (u >> 3) * 16384 + r * 128 + (((u & 7) ^ rsw) << 4);
        *reinterpret_cast<uint4*>(dst) = make_uint4(pk[4 * u], pk[4 * u + 1], pk[4 * u + 2], pk[4 * u + 3]);
      }
      fence_proxy_async_smem();
      tc_fence_before();
      __syncwarp();
      if (lane == 0) mbar_arrive(p_full);
    }
    // ---- epilogue: O / l + b_v -> fp16, row q0 + r, channels [part * DV, +DV) ----
    mbar_wait(o_full, (uint32_t)(nk - 1) & 1u);
    tc_fence_after();
    const float inv = 1.0f / l_run;
    const int row = q0 + r;
    const int c0 = part * DV;
    __half* orow = p.out + ((size_t)img * T + (size_t)min(row, T - 1)) * p.ld_out + c0;
    for (int c = 0; c < DV; c += 16) {
      uint32_t v[16];
      tmem_ld16(tmO + lane_base + (uint32_t)c, v);
      tmem_ld_wait16(v);
      uint32_t h[8];
#pragma unroll
      for (int i = 0; i < 8; ++i)
        h[i] = vqa_pack_h2(fmaf(__uint_as_float(v[2 * i]), inv, __ldg(p.bias + c0 + c + 2 * i)),
                           fmaf(__uint_as_float(v[2 * i + 1]), inv, __ldg(p.bias + c0 + c + 2 * i + 1)));
      if (row < T) {
        reinterpret_cast<uint4*>(orow + c)[0] = make_uint4(h[0], h[1], h[2], h[3]);
        reinterpret_cast<uint4*>(orow + c)[1] = make_uint4(h[4], h[5], h[6], h[7]);
      }
    }
  }

  tc_fence_before();
  __syncthreads();
  if (warp == kVqaMmaWarp) { tc_fence_after(); tmem_dealloc_dyn(tmem_base, 512u); }
}

#endif  // __CUDACC__
}  // namespace rs
