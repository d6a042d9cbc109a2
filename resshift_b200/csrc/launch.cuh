// Host-side launch helpers: TMA descriptor encoding and one launcher per kernel family.
#pragma once

#include <algorithm>
#include <cstdlib>
#include <cmath>
#include <cstring>
#include <utility>
#include <vector>

#include "common.cuh"
#include "conv_gemm.cuh"
#include "conv_persist.cuh"
#include "elementwise.cuh"
#include "mlp_fused.cuh"
#include "norm_act.cuh"
#include "window_attn.cuh"
#include "swin_attn_fused.cuh"
#include "swin_attn_tc.cuh"
#include "vq_attn_tc.cuh"

namespace rs {

// ---- driver entry point for cuTensorMapEncodeTiled (the .so does not link libcuda) --------------
typedef CUresult (*PFN_encodeTiled)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                    const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                    CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

inline PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  if (!fn) {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult q;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &q) == cudaSuccess &&
        q == cudaDriverEntryPointSuccess)
      fn = reinterpret_cast<PFN_encodeTiled>(p);
  }
  return fn;
}

// NHWC fp16 view descriptor used by the host code.
struct View {
  __half* ptr = nullptr;   // resolved at bind time
  int tens = -1;           // owning workspace tensor
  long long off = 0;       // element offset inside the tensor (channel slice + batch slice)
  int c0 = 0, n0 = 0;      // bookkeeping of the same slice: first channel / first image inside the owning tensor
  int N = 0, H = 0, W = 0, C = 0, ld = 0;
  long long sW() const { return ld; }
  long long sH() const { return (long long)W * ld; }
  long long sN() const { return (long long)H * W * ld; }
};

// 4-D activation map {C, W, H, N} with explicit element strides; box {64, bw, bh, bn}, 128B swizzle.
inline int encode_act_map(CUtensorMap* m, const __half* base, int C, int W, int H, int N, long long sW,
                          long long sH, long long sN, int bw, int bh, int bn, int box_c = kConvBK) {
  PFN_encodeTiled enc = get_encode_tiled();
  RS_CHECK(enc != nullptr, "cuTensorMapEncodeTiled entry point not available (no CUDA driver?)");
  cuuint64_t dims[4] = {(cuuint64_t)C, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)N};
  cuuint64_t strides[3] = {(cuuint64_t)sW * 2, (cuuint64_t)sH * 2, (cuuint64_t)sN * 2};
  cuuint32_t box[4] = {(cuuint32_t)box_c, (cuuint32_t)bw, (cuuint32_t)bh, (cuuint32_t)bn};
  const CUtensorMapSwizzle swz = box_c == 64 ? CU_TENSOR_MAP_SWIZZLE_128B
                                 : (box_c == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  RS_CHECK(box_c == 64 || box_c == 32 || box_c == 16, "activation box width");
  cuuint32_t estr[4] = {1, 1, 1, 1};
  RS_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0, "activation base must be 16-byte aligned");
  RS_CHECK(sW % 8 == 0 && sH % 8 == 0 && sN % 8 == 0, "activation strides must be multiples of 16 bytes");
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 4, const_cast<__half*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  RS_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(activation) failed with CUresult " + std::to_string((int)r));
  return 0;
}
// 2-D weight map {Ktot, Cout}, box {64, BN}.
inline int encode_weight_map(CUtensorMap* m, const __half* base, int Ktot, int Cout, int BN) {
  PFN_encodeTiled enc = get_encode_tiled();
  RS_CHECK(enc != nullptr, "cuTensorMapEncodeTiled entry point not available (no CUDA driver?)");
  cuuint64_t dims[2] = {(cuuint64_t)Ktot, (cuuint64_t)Cout};
  cuuint64_t strides[1] = {(cuuint64_t)Ktot * 2};
  cuuint32_t box[2] = {(cuuint32_t)kConvBK, (cuuint32_t)BN};
  cuuint32_t estr[2] = {1, 1};
  RS_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0 && Ktot % 8 == 0, "weight matrix must be 16-byte aligned");
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 2, const_cast<__half*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  RS_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(weights) failed with CUresult " + std::to_string((int)r));
  return 0;
}

inline int env_int(const char* name, int dflt) {
  const char* v = std::getenv(name);
  return v ? std::atoi(v) : dflt;
}
inline bool env_is(const char* name, const char* val) {
  const char* v = std::getenv(name);
  return v && std::strcmp(v, val) == 0;
}

// All kernels go through this launcher: cudaLaunchKernelEx with the programmatic-stream-serialization
// attribute (PDL), so kernel N+1's prologue overlaps kernel N's tail, also inside captured graphs.
// RS_PDL=0 turns the attribute off.
template <typename... KArgs, typename... Args>
inline cudaError_t launch_kc(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                             int cluster_x, Args&&... args) {
  static const int use_pdl = env_int("RS_PDL", 1);
  cudaLaunchConfig_t cfg{};
  cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = st;
  cudaLaunchAttribute attr[2];
  int n = 0;
  if (use_pdl) {
    attr[n].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[n].val.programmaticStreamSerializationAllowed = 1;
    ++n;
  }
  if (cluster_x > 1) {
    attr[n].id = cudaLaunchAttributeClusterDimension;
    attr[n].val.clusterDim.x = cluster_x; attr[n].val.clusterDim.y = 1; attr[n].val.clusterDim.z = 1;
    ++n;
  }
  cfg.attrs = attr; cfg.numAttrs = n;
  return cudaLaunchKernelEx(&cfg, kernel, std::forward<Args>(args)...);
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_k(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t st,
                            Args&&... args) {
  return launch_kc(kernel, grid, block, smem, st, 1, std::forward<Args>(args)...);
}

inline int pow2_floor_div(int x, int cap) {   // largest power of two dividing x, capped
  int p = 1;
  while (p * 2 <= cap && x % (p * 2) == 0) p *= 2;
  return p;
}

// Host description of one conv / linear layer instance.
struct ConvDesc {
  View in;                 // input view (for stride 2: the full-resolution input)
  int ksize = 1, stride = 1;
  int pad_lo = 1;          // stride-2 convs: 1 = symmetric padding 1 (UNet Downsample, reference models/unet.py:99-108);
                           // 0 = pad (0,1,0,1) then a padding-free conv (VQ-GAN Downsample, ldm/.../model.py:78-87)
  const __half* wt = nullptr;   // [Cout][taps][ipad]
  int ipad = 0;
  const float* bias = nullptr;
  int Cout = 0;
  View out;                // NHWC fp16 output view (ptr may be null when out_f32 is used)
  bool has_out = true;
  View res; bool has_res = false;
  float* out_f32 = nullptr;
  int act = ACT_NONE;
  int bn_override = 0;
  unsigned long long* dbg = nullptr;
  float* partial = nullptr;       // split-K scratch [S][pixels][Cout] fp32 (caller-provided when the plan chose S > 1)
  bool allow_split = false;
  SplitKReduceParams red;         // filled by finalize() when S > 1
  int red_grid_x = 0, red_grid_z = 1; size_t red_smem = 0;
  // fused GroupNorm statistics of the output (up to two consumers; gn_stats.cuh).  `expected` is filled by finalize()
  // (slots * cstride) unless the caller set it (a statistics buffer only partly covered by this producer: unit tests)
  GnSink sink[2] = {};
  // filled by finalize()
  ConvParams prm;
  ConvSimtSrc simt;
  int grid = 0; size_t smem = 0;
};

struct TileConfig { int BN = 0, msub = 1, stages = 2, occ = 1, cg = 1, splitk = 1, persist = 0, cluster_split = 0; double est_cycles = 1e30; };

// Cost model calibrated on B200 timelines (profiles/r1_s5_*, r1_s6_*).  Per 64-channel k-block and 128-pixel tile the
// tensor pipe needs 2*BN cycles; every operand byte crosses shared memory twice (TMA write + UMMA read, 128 B/clk
// per SM), which is what actually bounds a single-CTA tile (A 16 KB + B BN*128 B);  a CTA pair (cg = 2,
// tcgen05 cta_group::2) stages only half of B per SM.  Shallow rings are additionally latency-bound (~3000 cycles
// per load).  The epilogue (~18 cycles per column + set-up) hides under a co-resident CTA; whole waves are counted.
inline TileConfig pick_tile_config(int m_tiles, int cout16, int num_kb, int f_bn, bool allow_split = false, bool allow_persist = false,
                                   bool allow_cluster_split = false) {
  const int f_msub = env_int("RS_CONV_MSUB", 0), f_occ = env_int("RS_CONV_OCC", 0), f_stages = env_int("RS_CONV_STAGES", 0);
  const int f_cg = env_int("RS_CONV_CG", 0);
  TileConfig best, bestp;      // best one-tile-per-CTA configuration (ranking model below), best persistent one
  double best_real = 1e30;     // realistic estimate of `best` (see the end of the function)
  for (int cand = std::min(cout16, 256); cand >= 16; cand -= 16) {
    if (f_bn ? (cand != std::min(f_bn, std::min(cout16, 256))) : (cout16 % cand != 0)) continue;
    const int n_tiles = (cout16 + cand - 1) / cand;
    for (int cg = 1; cg <= 2; ++cg) {
      if (f_cg && cg != f_cg && !(f_cg == 2 && m_tiles < 2)) continue;   // a single tile cannot form a pair
      if (cg == 2 && (cand % 16 != 0 || m_tiles < 2)) continue;
      // persistent kernel (conv_persist.cuh): one CTA (pair) per SM walks ceil(units / workers) tiles; the epilogue
      // (~5000 + 3 cycles per column with double-buffered staging, profiles/r1_s38_persist_sweep.log) hides under the next tile's main loop, so
      // a tile costs max(main loop, epilogue) and set-up / first round trip / last epilogue are paid once
      if (allow_persist && 2 * cand <= 512) {
        const long long units_p = (long long)((m_tiles + cg - 1) / cg) * n_tiles;
        const int workers = cg == 2 ? 74 : 148;
        const int sbytes_p = kConvBM * kConvBK * 2 + (cand / cg) * kConvBK * 2;
        const size_t extra = (size_t)2 * cand * kConvBM * 2 + (size_t)cand * 40 + 1280 + sizeof(GnArriveList);   // two staging buffers, wsum, two bias slots, arrival list
        const int st_p = (int)std::min<size_t>(8, ((size_t)227 * 1024 - extra) / (size_t)sbytes_p);
        // (only layers with at least two PIXEL tiles per worker: that is where the model below was calibrated; getting
        // there through many narrow channel tiles would re-read the A operand once per channel tile)
        if ((m_tiles + cg - 1) / cg >= 2 * workers && st_p >= 2) {
          const double kb_p = std::max(std::max(2.0 * cand, 2.0 * sbytes_p / 128.0), 2600.0 / st_p);
          const double epi_p = 5000.0 + 3.0 * cand;
          const double rounds = std::ceil((double)units_p / workers);
          const double total = rounds * std::max(num_kb * kb_p, epi_p) + epi_p + 3000.0;
          if (total < bestp.est_cycles) {
            bestp.est_cycles = total; bestp.BN = cand; bestp.msub = 1; bestp.stages = std::min(st_p, std::max(2, num_kb));
            bestp.occ = 1; bestp.cg = cg; bestp.splitk = 1; bestp.persist = 1;
          }
        }
      }
      for (int ms = 1; ms <= 2; ++ms) {
        if (ms == 2 && (f_msub != 2 || cg == 2 || m_tiles % 2 || 2 * cand > 512)) continue;   // msub = 2 only on request
        const int sbytes = ms * kConvBM * kConvBK * 2 + (cand / cg) * kConvBK * 2;
        for (int occ = 1; occ <= 2; ++occ) {
          if (f_occ && occ != f_occ) continue;
          if (occ == 2 && ms * cand > 256) continue;                       // TMEM: 512 columns per SM
          const int budget = (occ == 2 ? 111 : 222) * 1024 - 2048;
          int st = std::min(std::min(8, std::max(2, num_kb)), budget / sbytes);
          // the staged epilogue (output tile + statistics scratch) reuses the ring: it must be at least that large
          // (short-K layers with wide channel tiles in pair mode: 2 stages x (16 KB + BN/2 x 128 B) < BN x 288 B)
          {
            const int st_need = (int)(((size_t)ms * ((size_t)cand * kConvBM * 2 + (size_t)4 * cand * 2 * sizeof(float)) + 16 + sbytes - 1) / sbytes);
            if (st_need > budget / sbytes) continue;
            st = std::max(st, st_need);
          }
          if (f_stages) st = f_stages;
          if (st < 2 || (size_t)st * sbytes + 2304 > (size_t)(occ == 2 ? 113 : 227) * 1024) continue;
          const double smem_cycles = (sbytes + ms * (kConvBM * kConvBK * 2.0 + (cand / cg) * kConvBK * 2.0)) / 128.0;
          // SM time for every resident CTA to advance one k-block: tensor / smem work of each, or the load latency
          // amortised over the ring depth
          // load latency: ~3000 cycles when many tiles share each weight tile (L2 hits), ~7500 when the layer has so few
          // pixel tiles that every weight tile is a fresh HBM read for a handful of CTAs (profiles/r1_s12_smallm_sweep.log)
          const double load_lat = m_tiles >= 64 ? 3000.0 : 7500.0;
          const double kb_cycles = std::max(occ * std::max(ms * 2.0 * cand, smem_cycles), load_lat / st);
          const double epi = 18.0 * cand * ms + 3000.0 + (cg == 2 ? 2500.0 : 0.0);  // + pipeline fill / set-up (+ cluster syncs)
          const long long units = (long long)((m_tiles + cg * ms - 1) / (cg * ms)) * n_tiles;   // CTAs or CTA pairs
          const double slots = (cg == 2 ? 74.0 : 148.0) * occ;
          // split-K: S CTAs (pairs) share one output tile's K loop; costs an fp32 round trip + a small reduce kernel
          const int f_split = env_int("RS_CONV_SPLITK", 0);
          const int kSplits[6] = {1, 2, 3, 4, 6, 8};
          // split-K flavours: 0 = none / global (fp32 partials in HBM scratch + splitk_reduce_kernel), 1 = cluster (the S
          // pairs of a tile are one cluster of 2S CTAs and reduce through distributed shared memory: pair mode)
          const char* f_mode = std::getenv("RS_CONV_SPLITK_MODE");
          for (int mode = 0; mode < 2; ++mode)
          for (int si = 0; si < 6; ++si) {
            const int S = kSplits[si];
            // (S = 2 only: clusters of 8 CTAs with ~200 KB of shared memory each schedule poorly — 30 us vs 21 us for the
            //  8x8 640->640 layer, profiles/r1_s35_cluster_split_sweep.log)
            if (mode == 1 && (S != 2 || !allow_cluster_split || cg != 2 || occ != 1 || (cand / S) % 8 != 0)) continue;
            if (mode == 1 && f_mode && std::strcmp(f_mode, "global") == 0) continue;
            if (mode == 0 && S > 1 && f_mode && std::strcmp(f_mode, "cluster") == 0) continue;
            if (mode == 1 && (size_t)kConvBM * (cand * 4 + 16) + (size_t)kConvBM * (cand / S) * 2 + (size_t)4 * (cand / S) * 4 + 16 > (size_t)st * sbytes) continue;
            if (S > 1 && ((mode == 0 && !allow_split) || ms != 1 || num_kb / S < 6)) continue;
            if (f_split && (allow_split || allow_cluster_split) && ms == 1 && num_kb / f_split >= 6 && S != f_split) continue;
            const double waves = std::ceil((double)units * S / slots);
            const double kbs = std::ceil((double)num_kb / S);
            const double round = kbs * kb_cycles + (occ == 2 ? 0.5 * epi : epi);
            // global: fp32 partials written once by the conv epilogue and read once by the reduce kernel (~2 KB/clk
            // chip-wide each way in practice), plus a second kernel launch / drain (~10 us of fixed cost for the pair);
            // cluster: a cluster barrier and one pass over the tile through distributed shared memory
            const double part_bytes = 4.0 * m_tiles * 128.0 * cout16 * S;
            const double total = waves * round + (S == 1 ? 0.0 : mode == 1 ? 6000.0 : 19000.0 + 2.0 * part_bytes / 2048.0);
            if (total < best.est_cycles) {
              best.est_cycles = total; best.BN = cand; best.msub = ms;
              best.stages = std::max(std::min(st, (int)std::max(2.0, kbs)), std::min(st, (int)(((size_t)ms * ((size_t)cand * kConvBM * 2 + (size_t)4 * cand * 2 * sizeof(float)) + 16 + sbytes - 1) / sbytes)));
              best.occ = occ; best.cg = cg; best.splitk = S; best.persist = 0; best.cluster_split = (S > 1 && mode == 1) ? 1 : 0;
              // what a wave really costs (timelines r1_s25): co-resident CTAs run in lockstep, so set-up, the first
              // operand round trip and the whole epilogue are exposed once per wave
              best_real = waves * (kbs * kb_cycles + epi + 5000.0) + (S == 1 ? 0.0 : mode == 1 ? 6000.0 : 19000.0 + 2.0 * part_bytes / 2048.0);
            }
          }
        }
      }
    }
  }
  // the ranking model above orders one-tile-per-CTA configurations well (scripts/conv_sweep.py) but is optimistic in
  // absolute terms; the persistent estimate is calibrated in absolute cycles, so compare it with the realistic figure
  // (ties go to the persistent kernel: it measured faster on every >= 2-tiles-per-SM layer of the model)
  if (bestp.BN && 0.85 * bestp.est_cycles < best_real) return bestp;
  return best;
}

// geometry-only preview of the configuration conv_finalize() will choose (used at plan time to size split-K scratch)
inline TileConfig conv_preview_config(int N, int Hin, int Win, int Cin, int Cout, int ksize, int stride, bool allow_split) {
  const int Hout = Hin / stride, Wout = Win / stride;
  const int bw = pow2_floor_div(Wout, kConvBM);
  const int bh = pow2_floor_div(Hout, kConvBM / bw);
  const int bn = kConvBM / (bw * bh);
  const int m_tiles = (Wout / bw) * (Hout / bh) * ((N + bn - 1) / bn);
  const bool contiguous = (bw == Wout) || (bh == 1);
  const int num_kb = ksize * ksize * ((Cin + kConvBK - 1) / kConvBK);
  const bool sp = allow_split && contiguous && bn <= 2;
  return pick_tile_config(m_tiles, (Cout + 15) / 16 * 16, num_kb, env_int("RS_CONV_BN", 0), sp, false, sp && Cout % 8 == 0);
}

inline int conv_finalize(ConvDesc& d) {
  ConvParams& p = d.prm;
  std::memset(&p, 0, sizeof(p));
  const int Hin = d.in.H, Win = d.in.W;
  RS_CHECK(d.ksize == 1 || d.ksize == 3, "kernel size must be 1 or 3");
  RS_CHECK(d.stride == 1 || (d.stride == 2 && d.ksize == 3 && Hin % 2 == 0 && Win % 2 == 0), "unsupported stride");
  const int Hout = Hin / d.stride, Wout = Win / d.stride, N = d.in.N;
  p.Hout = Hout; p.Wout = Wout; p.Nimg = N; p.Cout = d.Cout;
  p.num_taps = d.ksize * d.ksize;
  p.kchunks = (d.in.C + kConvBK - 1) / kConvBK;
  {
    const int tail = d.in.C - (p.kchunks - 1) * kConvBK;                 // real channels of the last 64-channel chunk
    p.tail_k16 = env_int("RS_CONV_TAILSKIP", 1) ? (tail + 15) / 16 : kConvBK / 16;
  }
  p.w_tap_stride = d.ipad;
  RS_CHECK(d.ipad % 8 == 0 && d.ipad >= d.in.C, "weight channel padding");
  // pixel box
  p.bw = pow2_floor_div(Wout, kConvBM);
  p.bh = pow2_floor_div(Hout, kConvBM / p.bw);
  p.bn = kConvBM / (p.bw * p.bh);
  p.tiles_w = Wout / p.bw; p.tiles_h = Hout / p.bh; p.tiles_n = (N + p.bn - 1) / p.bn;
  const int m_tiles = p.tiles_w * p.tiles_h * p.tiles_n;
  // ---- tile configuration: channel tile BN, sub-tiles per CTA (msub), CTAs per SM (occ), ring depth (stages) ----
  // Chosen by a small cost model calibrated on B200 timelines (profiles/r1_s5_*): the main loop is bound by the bytes
  // of TMA loads in flight per SM (ring capacity / ~3000-cycle load latency, at most ~75 B/clk) unless the tensor
  // pipe is slower (2*BN cycles per 64-channel k-block per 128-pixel sub-tile); the epilogue (~18 cycles per output
  // column per sub-tile) hides under the other resident CTA when two fit; whole waves of CTAs are counted.
  const int cout16 = (d.Cout + 15) / 16 * 16;
  const int num_kb = p.num_taps * p.kchunks;
  const bool contiguous_tiles = (p.bw == Wout) || (p.bh == 1);
  const bool can_split = d.allow_split && d.partial != nullptr && contiguous_tiles && p.bn <= 2 && d.has_out && !d.out_f32;
  const int want_persist = env_int("RS_CONV_PERSIST", -1);           // 0 / 1 disables / forces the persistent kernel
  // (the persistent kernel batches its GroupNorm arrivals in a shared list of kGnListCap (sink, image) entries)
  const bool persist_ok = d.has_out && !d.out_f32 && want_persist != 0 && !env_is("RS_CONV_EPI", "direct") &&
                          !env_is("RS_CONV_IMPL", "simt") && env_int("RS_CONV_MSUB", 0) != 2 &&
                          (!(d.sink[0].part || d.sink[1].part) || 2 * N <= kGnListCap);
  const bool can_cluster_split = d.allow_split && contiguous_tiles && p.bn <= 2 && d.has_out && !d.out_f32 && d.Cout % 8 == 0;
  const TileConfig tc = pick_tile_config(m_tiles, cout16, num_kb, d.bn_override ? d.bn_override : env_int("RS_CONV_BN", 0), can_split,
                                         persist_ok && want_persist != 1, can_cluster_split);
  const int BN = tc.BN, msub = tc.msub, stages = tc.stages, cg = tc.cg;
  p.cg = cg;
  p.splitk = tc.splitk; p.partial = d.partial; p.splitk_cluster = tc.cluster_split;
  RS_CHECK(BN >= 16 && BN <= 256 && BN % 16 == 0, "no valid tile configuration");
  p.BN = BN; p.n_tiles = (cout16 + BN - 1) / BN;
  p.msub = msub;
  int cols = 32; while (cols < msub * BN) cols *= 2;
  p.tmem_cols = cols;
  const int stage_bytes = msub * kConvBM * kConvBK * 2 + (BN / cg) * kConvBK * 2;
  p.stages = stages;
  d.smem = (size_t)stages * stage_bytes + 1024 + 256 + 1024;   // ring + alignment slack + barriers + bias tile
  RS_CHECK(d.smem <= 227 * 1024, "shared memory budget exceeded");
  d.grid = (cg == 2 ? ((m_tiles + 1) / 2) * p.n_tiles * 2 : (m_tiles / msub) * p.n_tiles) * p.splitk;
  // taps
  if (d.stride == 1) {
    int t = 0;
    for (int ky = 0; ky < d.ksize; ++ky)
      for (int kx = 0; kx < d.ksize; ++kx, ++t) {
        p.tap_src[t] = 0; p.tap_dh[t] = ky - d.ksize / 2; p.tap_dw[t] = kx - d.ksize / 2;
      }
  } else {
    int t = 0;
    for (int ky = 0; ky < 3; ++ky)
      for (int kx = 0; kx < 3; ++kx, ++t) {
        if (d.pad_lo == 1) {        // input row 2i + ky - 1: parity (ky != 1), one step back for ky = 0
          const int hp = (ky == 1) ? 0 : 1, wp = (kx == 1) ? 0 : 1;
          p.tap_src[t] = hp * 2 + wp; p.tap_dh[t] = (ky == 0) ? -1 : 0; p.tap_dw[t] = (kx == 0) ? -1 : 0;
        } else {                    // input row 2i + ky: parity (ky == 1), one step forward for ky = 2 (TMA zero fill = the pad)
          const int hp = (ky == 1) ? 1 : 0, wp = (kx == 1) ? 1 : 0;
          p.tap_src[t] = hp * 2 + wp; p.tap_dh[t] = (ky == 2) ? 1 : 0; p.tap_dw[t] = (kx == 2) ? 1 : 0;
        }
      }
  }
  // epilogue
  p.bias = d.bias; p.act = d.act;
  if (d.has_res) {
    RS_CHECK(d.res.H == Hout && d.res.W == Wout && d.res.N == N && d.res.C >= d.Cout, "residual geometry");
    p.residual = d.res.ptr; p.res_sN = d.res.sN(); p.res_sH = d.res.sH(); p.res_sW = d.res.sW();
  }
  if (d.has_out) {
    RS_CHECK(d.out.H == Hout && d.out.W == Wout && d.out.N == N, "output geometry");
    p.out = d.out.ptr; p.out_sN = d.out.sN(); p.out_sH = d.out.sH(); p.out_sW = d.out.sW();
    RS_CHECK(d.out.ld % 8 == 0 && (reinterpret_cast<uintptr_t>(d.out.ptr) & 15) == 0, "output alignment");
  }
  p.out_f32_nchw = d.out_f32;
  p.dbg = d.dbg;
  // staged epilogue (TMA store / TMA residual load) for fp16 NHWC outputs
  p.tma_out = (d.has_out && !d.out_f32 && p.splitk == 1 && !env_is("RS_CONV_EPI", "direct") && !env_is("RS_CONV_IMPL", "simt")) ? 1 : 0;
  p.tma_res = (p.tma_out && d.has_res) ? 1 : 0;
  p.epi_bc = (BN % 64 == 0) ? 64 : (BN % 32 == 0 ? 32 : 16);
  if (p.tma_out) {
    int rc = encode_act_map(&p.tmOut, d.out.ptr, d.Cout, Wout, Hout, N, d.out.sW(), d.out.sH(), d.out.sN(), p.bw, p.bh, p.bn, p.epi_bc);
    if (rc) return rc;
    if (p.tma_res) {
      rc = encode_act_map(&p.tmRes, d.res.ptr, d.Cout, Wout, Hout, N, d.res.sW(), d.res.sH(), d.res.sN(), p.bw, p.bh, p.bn, p.epi_bc);
      if (rc) return rc;
    }
    // the staging area (column blocks + per-warp GN partials) must fit in the operand ring
    // (the persistent kernel stages in buffers of its own, sized below)
    const size_t need = (size_t)msub * ((size_t)BN * kConvBM * 2 + (size_t)4 * BN * 2 * sizeof(float)) + 16;
    RS_CHECK(tc.persist || need <= (size_t)stages * stage_bytes, "epilogue staging does not fit in the pipeline shared memory");
  }
  // persistent variant (conv_persist.cuh) when the cost model chose it (every SM / pair gets at least two tiles), or
  // when RS_CONV_PERSIST = 1 forces it for any eligible layer
  {
    const int units = (cg == 2 ? (m_tiles + 1) / 2 : m_tiles) * p.n_tiles;
    const int workers = cg == 2 ? 74 : 148;
    const bool eligible = persist_ok && p.tma_out && p.splitk == 1 && msub == 1 && 2 * BN <= 512;
    p.persist = (eligible && (tc.persist || want_persist == 1)) ? 1 : 0;
    RS_CHECK(!tc.persist || p.persist, "persistent configuration chosen for an ineligible layer");
    p.num_units = units;
    if (p.persist) {
      const size_t extra = (size_t)2 * BN * kConvBM * 2 + (size_t)4 * BN * 2 * sizeof(float) + (size_t)2 * BN * sizeof(float) + 256 + 1024 + sizeof(GnArriveList);
      const int st = (int)std::min<size_t>(8, ((size_t)227 * 1024 - extra) / (size_t)stage_bytes);
      RS_CHECK(st >= 2, "persistent conv: shared memory budget");
      p.stages = std::min(st, std::max(2, num_kb));
      d.smem = (size_t)p.stages * stage_bytes + extra;
      int cols2 = 32; while (cols2 < 2 * BN) cols2 *= 2;
      p.tmem_cols = cols2;
      d.grid = cg * std::min(units, workers);
    }
  }
  p.gn_slots = p.tiles_w * p.tiles_h;
  RS_CHECK(!(d.sink[0].part || d.sink[1].part) || p.bn <= 2, "fused GroupNorm statistics need tiles of at most two images");
  auto fill_sinks = [&](GnSink* dst) {
    int k = 0;
    for (int i = 0; i < 2; ++i) {
      dst[i] = GnSink{};
      if (!d.sink[i].part) continue;
      dst[k] = d.sink[i];
      if (dst[k].expected == 0) dst[k].expected = (unsigned)(p.gn_slots * dst[k].cstride);
      if (dst[k].eps == 0.f) dst[k].eps = 1e-5f;
      ++k;
    }
  };
  {
    GnSink none[2] = {};
    if (p.tma_out) fill_sinks(p.sink); else { p.sink[0] = none[0]; p.sink[1] = none[1]; }
  }
  if (p.splitk > 1 && p.splitk_cluster) {
    // cluster split-K: the conv kernel finishes the layer itself (DSMEM reduce + direct epilogue), statistics included
    fill_sinks(p.sink);
    RS_CHECK(cg == 2 && d.Cout % 8 == 0 && (BN / p.splitk) % 8 == 0, "cluster split-K configuration");
  } else if (p.splitk > 1) {
    // the conv kernel only produces fp32 partial sums; bias / activation / residual / fp16 store / GroupNorm statistics
    // happen in the reduce kernel, one CTA per (128-pixel slot, image)
    SplitKReduceParams& r = d.red;
    std::memset(&r, 0, sizeof(r));
    r.partial = d.partial; r.S = p.splitk; r.N = N; r.HW = Hout * Wout; r.C = d.Cout;
    r.bias = d.bias; r.act = d.act;
    if (d.has_res) { r.residual = d.res.ptr; r.res_sN = d.res.sN(); r.res_ld = d.res.ld; }
    r.out = d.out.ptr; r.out_sN = d.out.sN(); r.out_ld = d.out.ld;
    r.rows_per_slot = p.bw * p.bh; r.slots = p.tiles_w * p.tiles_h;
    fill_sinks(r.sink);
    RS_CHECK(d.Cout % 8 == 0 && d.Cout <= 2048, "split-K reduce needs Cout % 8 == 0");
    p.bias = nullptr; p.residual = nullptr; p.act = ACT_NONE; p.sink[0] = GnSink{}; p.sink[1] = GnSink{};
    d.red_grid_x = r.slots;
    // column blocks so that the reduce kernel fills the machine even with one slot per image
    int cpc = d.Cout;
    while (cpc > 64 && cpc % 16 == 0 && (long long)r.slots * N * (d.Cout / cpc) < 2 * 148) cpc /= 2;
    r.cols_per_cta = cpc;
    d.red_grid_z = (d.Cout + cpc - 1) / cpc;
    const int lanes = 256 / std::max(1, cpc / 8);
    d.red_smem = (size_t)std::max(1, lanes) * cpc * 3 * sizeof(float) + 16;
  }
  // tensor maps + SIMT mirrors
  ConvSimtSrc& s = d.simt;
  std::memset(&s, 0, sizeof(s));
  s.C = d.in.C; s.wt = d.wt;
  const int nsrc = d.stride == 1 ? 1 : 4;
  for (int i = 0; i < kMaxSrc; ++i) {
    const int j = i < nsrc ? i : 0;
    const int hp = d.stride == 2 ? (j >> 1) : 0, wp = d.stride == 2 ? (j & 1) : 0;
    const __half* base = d.in.ptr + (long long)hp * d.in.sH() + (long long)wp * d.in.sW();
    const long long sW = d.in.sW() * d.stride, sH = d.in.sH() * d.stride, sN = d.in.sN();
    s.ptr[i] = base; s.sN[i] = sN; s.sH[i] = sH; s.sW[i] = sW; s.H[i] = Hout; s.W[i] = Wout;
    if (!env_is("RS_CONV_IMPL", "simt")) {
      int rc = encode_act_map(&p.tmA[i], base, d.in.C, Wout, Hout, N, sW, sH, sN, p.bw, p.bh, p.bn);
      if (rc) return rc;
    }
  }
  if (!env_is("RS_CONV_IMPL", "simt")) {
    int rc = encode_weight_map(&p.tmB, d.wt, p.num_taps * d.ipad, d.Cout, BN / cg);
    if (rc) return rc;
  }
  return 0;
}

inline int conv_init() {   // once per process, outside any stream capture
  static bool attr_set = false;
  if (!attr_set) {
    RS_CUDA_OK(cudaFuncSetAttribute(conv_gemm_sm100_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    RS_CUDA_OK(cudaFuncSetAttribute(conv_gemm_sm100_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    RS_CUDA_OK(cudaFuncSetAttribute(conv_gemm_persist_sm100_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    RS_CUDA_OK(cudaFuncSetAttribute(conv_gemm_persist_sm100_kernel<2>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    RS_CUDA_OK(cudaFuncSetAttribute(window_attn_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 160 * 1024));
    RS_CUDA_OK(cudaFuncSetAttribute(mlp_fused_sm100_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    RS_CUDA_OK(cudaFuncSetAttribute(swin_attn_fused_kernel<192>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SwinSmem<192>::total));
    RS_CUDA_OK(cudaFuncSetAttribute(swin_attn_fused_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SwinSmem<64>::total));
    RS_CUDA_OK(cudaFuncSetAttribute(swin_attn_tc_kernel<192>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SwinTcSmem<192>::total));
    RS_CUDA_OK(cudaFuncSetAttribute(swin_attn_tc_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)SwinTcSmem<64>::total));
    RS_CUDA_OK(cudaFuncSetAttribute(vq_attn_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, vqa_smem_bytes(512)));
    attr_set = true;
  }
  return 0;
}

inline int conv_launch(const ConvDesc& d, cudaStream_t st) {
  if (env_is("RS_CONV_IMPL", "simt")) {
    const long long npix = (long long)d.prm.Nimg * d.prm.Hout * d.prm.Wout;
    const int warps = 8;
    (void)launch_k(conv_simt_kernel, dim3((unsigned)((npix + warps - 1) / warps)), dim3(warps * 32), (size_t)(0), st, d.prm, d.simt);
  } else {
    if (d.prm.persist && d.prm.cg == 2)
      (void)launch_kc(conv_gemm_persist_sm100_kernel<2>, dim3(d.grid), dim3(kConvThreads), (size_t)(d.smem), st, 2, d.prm);
    else if (d.prm.persist)
      (void)launch_kc(conv_gemm_persist_sm100_kernel<1>, dim3(d.grid), dim3(kConvThreads), (size_t)(d.smem), st, 1, d.prm);
    else if (d.prm.cg == 2)
      (void)launch_kc(conv_gemm_sm100_kernel<2>, dim3(d.grid), dim3(kConvThreads), (size_t)(d.smem), st,
                      d.prm.splitk_cluster ? 2 * d.prm.splitk : 2, d.prm);
    else
      (void)launch_kc(conv_gemm_sm100_kernel<1>, dim3(d.grid), dim3(kConvThreads), (size_t)(d.smem), st, 1, d.prm);
    if (d.prm.splitk > 1 && !d.prm.splitk_cluster)
      (void)launch_k(splitk_reduce_kernel, dim3(d.red_grid_x, d.prm.Nimg, d.red_grid_z), dim3(256), d.red_smem, st, d.red);
  }
  RS_CUDA_OK(cudaGetLastError());
  return 0;
}

// ---- GroupNorm -------------------------------------------------------------------------------
// number of 128-pixel tile slots per image the conv kernel uses for an H x W output (and whether its epilogue can
// produce per-image statistics: tiles must not span more than two images)
inline int conv_tile_slots(int H, int W, bool* fusable = nullptr) {
  const int bw = pow2_floor_div(W, kConvBM);
  const int bh = pow2_floor_div(H, kConvBM / bw);
  if (fusable) *fusable = (kConvBM / (bw * bh)) <= 2;
  return (W / bw) * (H / bh);
}

struct GnDesc {
  View in, out;
  const float* gamma = nullptr; const float* beta = nullptr;
  const float* film = nullptr; long long film_sN = 0;   // resolved per launch for FiLM layers
  int film_off = -1;      // offset of this layer's [2C] slice inside an embedding row, or -1
  int film_n0 = 0;        // first image of this (batch-sliced) op inside the plan's batch: row offset into per-image FiLM
  int silu = 0;
  float* part = nullptr;  // [N][slots][C][2] (mean, M2) pairs
  float* gstat = nullptr; // [N][32][2] (mean, rstd), finalised by the last producer CTA of each image
  unsigned int* counter = nullptr;   // [N]
  float eps = 1e-5f;
  int slots = 0;
  bool fused = false;     // statistics already delivered by the producing kernels' epilogues
  bool win_slots = false; // the producer is the fused Swin attention kernel: one slot per 8x8 window (64 values each)
  bool finalize_kernel = false;   // fused statistics with many slots: reduce part -> gstat with gn_finalize_kernel first
};

inline void gn_chunks(int HW, int N, int* chunks, int* rows) {
  // enough CTAs to fill the machine, at least 32 rows each, and every chunk with the SAME number of rows (the
  // statistics combine assumes equal counts per slot): the largest divisor of HW not above the target
  int c = std::max(1, std::min((HW + 31) / 32, (148 * 4 + N - 1) / N));
  while (c > 1 && HW % c != 0) --c;
  *chunks = c; *rows = HW / c;
}

inline int gn_launch(const GnDesc& g, cudaStream_t st) {
  const int C = g.in.C, HW = g.in.H * g.in.W, N = g.in.N;
  RS_CHECK(C % 32 == 0 && C % 8 == 0 && C <= 2048, "GroupNorm channel count");
  RS_CHECK(g.in.ld % 8 == 0 && g.out.ld % 8 == 0, "GroupNorm view alignment");
  int chunks, rows;
  gn_chunks(HW, N, &chunks, &rows);
  int slots = g.slots;
  RS_CHECK(g.gstat != nullptr || g.part != nullptr, "GroupNorm needs a statistics buffer");
  if (!g.fused) {
    slots = chunks;
    const int lanes = 256 / (C / 8);
    RS_CHECK(g.part != nullptr && (g.gstat == nullptr || g.counter != nullptr), "GroupNorm statistics buffers");
    GnStatsParams sp{};
    sp.x = g.in.ptr; sp.sN = g.in.sN(); sp.ld = g.in.ld; sp.C = C; sp.HW = HW; sp.N = N;
    sp.sink.part = g.part; sp.sink.gstat = g.gstat; sp.sink.counter = g.counter; sp.sink.cstride = C; sp.sink.coff = 0;
    sp.sink.expected = (unsigned)(slots * C); sp.sink.eps = g.eps;
    sp.slots = slots; sp.rows_per_slot = rows;
    (void)launch_k(gn_stats_kernel, dim3(chunks, N), dim3(256), (size_t)lanes * C * 3 * sizeof(float) + 16, st, sp);
    RS_CUDA_OK(cudaGetLastError());
  }
  if (g.fused && g.finalize_kernel) {
    RS_CHECK(g.part != nullptr && g.gstat != nullptr && slots > 0 && HW % slots == 0, "GroupNorm finalisation buffers");
    GnFinalizeParams fp{g.part, g.gstat, slots, C, (float)(HW / slots), g.eps};
    (void)launch_k(gn_finalize_kernel, dim3(32, N), dim3(256), (size_t)0, st, fp);
    RS_CUDA_OK(cudaGetLastError());
  }
  // apply: ~4 CTAs per SM in total, all resident at once (each CTA re-derives the per-channel affine from the
  // partials — a latency, not a bandwidth cost), at least 16 rows each
  int actas = std::max(1, std::min((HW + 15) / 16, (148 * 4 + N - 1) / N));
  const int arows = (HW + actas - 1) / actas;
  actas = (HW + arows - 1) / arows;
  // small tensors: split the channels too (slices aligned to GroupNorm groups and to 8-channel vectors) until there
  // are ~1.5 CTAs per SM — a 8x8 C=640 layer would otherwise run on 64 CTAs
  int csplit = 1;
  {
    const int cpg = C / 32;
    int unit = cpg; while (unit % 8) unit += cpg;                   // lcm(8, channels per group)
    for (int cs = 2; actas * N * csplit < 222 && cs <= C / unit; ++cs)
      if (C % cs == 0 && (C / cs) % unit == 0) csplit = cs;
  }
  GnApplyParams ap{g.in.ptr, g.in.sN(), g.in.ld, g.out.ptr, g.out.sN(), g.out.ld, C, HW, N, g.gstat, g.part, slots, g.eps,
                   g.gamma, g.beta, g.film, g.film_sN, g.silu, arows, C / csplit};
  (void)launch_k(gn_apply_kernel, dim3(actas, N, csplit), dim3(256), (size_t)(4 * (C / csplit) + 64) * sizeof(float), st, ap);
  RS_CUDA_OK(cudaGetLastError());
  return 0;
}

// ---- fused Swin MLP ---------------------------------------------------------------------------
struct MlpDesc {
  View in, out, res;
  bool has_res = true;
  const __half* w1 = nullptr; const float* b1 = nullptr;    // fc1: [Hd][E] fp16
  const __half* w2 = nullptr; const float* b2 = nullptr;    // fc2: [E][Hd] fp16
  int E = 0, Hd = 0;
  GnSink sink[2] = {};
  long long* dbg = nullptr;
  // optional fused input GroupNorm (plain affine): `in` is then the un-normalised tensor
  const float* gn_in_gstat = nullptr;      // finalised group statistics, or
  const float* gn_in_part = nullptr; int gn_in_slots = 0;   // the producers' (mean, M2) pairs to combine in the kernel
  const float* gn_in_gamma = nullptr; const float* gn_in_beta = nullptr;
  MlpParams prm;
  int grid = 0; size_t smem = 0;
};

inline bool mlp_supported(int E, int Hd, int H, int W, int N) {
  bool fus = false;
  const int slots = conv_tile_slots(H, W, &fus);
  const int bw = pow2_floor_div(W, kConvBM), bh = pow2_floor_div(H, kConvBM / bw), bn = kConvBM / (bw * bh);
  const int tiles = slots * ((N + bn - 1) / bn);
  return E % 64 == 0 && E <= 256 && Hd % kMlpHc == 0 && fus && tiles % 2 == 0;   // the kernel runs as CTA pairs
}

inline int mlp_finalize(MlpDesc& d) {
  MlpParams& p = d.prm;
  std::memset(&p, 0, sizeof(p));
  const int H = d.in.H, W = d.in.W, N = d.in.N;
  RS_CHECK(mlp_supported(d.E, d.Hd, H, W, N), "fused MLP: unsupported shape (E % 64, E <= 256, hidden % 128, even tile count)");
  RS_CHECK(d.in.C == d.E && d.out.C == d.E, "fused MLP: channel mismatch");
  p.E = d.E; p.Hd = d.Hd; p.bias1 = d.b1; p.bias2 = d.b2;
  p.bw = pow2_floor_div(W, kConvBM);
  p.bh = pow2_floor_div(H, kConvBM / p.bw);
  p.bn = kConvBM / (p.bw * p.bh);
  p.tiles_w = W / p.bw; p.tiles_h = H / p.bh;
  const int tiles_n = (N + p.bn - 1) / p.bn;
  p.Wout = W; p.Hout = H; p.Nimg = N;
  // shared memory per CTA: X (E/64 tiles) + two H buffers + barriers + both bias vectors; the rest is ring slots for
  // this CTA's HALF of the weight tiles: two hidden chunks of the fc2 stream, everything else to the fc1 stream
  const size_t kW1 = (size_t)(kMlpHc / 2) * 128;
  const size_t slot2 = (size_t)(d.E / 2) * 128;
  const int kHT = kMlpHc / 64, kx = d.E / 64;
  const size_t fixed = (size_t)kx * 16384 + (size_t)2 * kHT * 16384 + 1024 + 512 + (size_t)(d.Hd + d.E) * sizeof(float) +
                       (size_t)(2 * d.E * 2 + 2 * 32 * 2) * sizeof(float);   // + input-GN affine / group statistics
  RS_CHECK(fixed + kHT * slot2 + (size_t)kx * kW1 <= 227 * 1024, "fused MLP: not enough shared memory for the weight rings");
  const size_t budget = 227 * 1024 - fixed;
  p.ring2 = (int)std::min<size_t>(2 * kHT, (budget - (size_t)kx * kW1) / slot2);
  p.ring1 = (int)std::min<size_t>(12, (budget - (size_t)p.ring2 * slot2) / kW1);
  p.has_res = d.has_res ? 1 : 0;
  const int tiles = p.tiles_w * p.tiles_h * tiles_n;      // even (mlp_supported): CTA pairs
  // few-tile layers (8x8 / 16x16 levels): split the hidden dimension over two pairs of one cluster; partial outputs
  // meet in distributed shared memory (RS_MLP_HSPLIT = 1 disables, = 2 forces)
  {
    const int want = env_int("RS_MLP_HSPLIT", 0);
    const bool can = (d.Hd / kMlpHc) >= 2 && (d.E / 2) % 8 == 0 &&
                     (size_t)kConvBM * (d.E * 4 + 16) + (size_t)kConvBM * (d.E / 2) * 2 + (size_t)2 * d.E * 4 <= (size_t)200 * 1024;
    p.hsplit = (can && want != 1 && (want == 2 || tiles <= 64)) ? 2 : 1;
  }
  d.grid = tiles * p.hsplit;
  p.out_ptr = d.out.ptr; p.out_sN = d.out.sN(); p.out_sH = d.out.sH(); p.out_sW = d.out.sW();
  p.res_ptr = d.has_res ? d.res.ptr : nullptr;
  if (d.has_res) { p.res_sN = d.res.sN(); p.res_sH = d.res.sH(); p.res_sW = d.res.sW(); }
  d.smem = fixed + (size_t)p.ring1 * kW1 + (size_t)p.ring2 * slot2;
  RS_CHECK(d.smem <= 227 * 1024, "fused MLP: shared memory budget exceeded");
  int rc = encode_act_map(&p.tmX, d.in.ptr, d.E, W, H, N, d.in.sW(), d.in.sH(), d.in.sN(), p.bw, p.bh, p.bn, 64);
  if (rc) return rc;
  rc = encode_weight_map(&p.tmW1, d.w1, d.E, d.Hd, kMlpHc / 2); if (rc) return rc;   // each CTA of a pair fetches half a tile
  rc = encode_weight_map(&p.tmW2, d.w2, d.Hd, d.E, d.E / 2); if (rc) return rc;
  rc = encode_act_map(&p.tmOut, d.out.ptr, d.E, W, H, N, d.out.sW(), d.out.sH(), d.out.sN(), p.bw, p.bh, p.bn, 64);
  if (rc) return rc;
  if (d.has_res) {
    rc = encode_act_map(&p.tmRes, d.res.ptr, d.E, W, H, N, d.res.sW(), d.res.sH(), d.res.sN(), p.bw, p.bh, p.bn, 64);
    if (rc) return rc;
  }
  p.dbg = d.dbg;
  p.gn_in_gstat = d.gn_in_gstat; p.gn_in_part = d.gn_in_part; p.gn_in_slots = d.gn_in_slots;
  p.gn_in_gamma = d.gn_in_gamma; p.gn_in_beta = d.gn_in_beta; p.gn_in_eps = 1e-5f;
  RS_CHECK(!(d.gn_in_gstat || d.gn_in_part) || (d.gn_in_gamma && d.gn_in_beta && d.Hd >= 4 * d.E && d.E % 32 == 0),
           "fused MLP: input GroupNorm arguments");
  p.gn_slots = p.tiles_w * p.tiles_h;
  {
    int k = 0;
    p.sink[0] = GnSink{}; p.sink[1] = GnSink{};
    for (int i = 0; i < 2; ++i) {
      if (!d.sink[i].part) continue;
      p.sink[k] = d.sink[i];
      if (p.sink[k].expected == 0) p.sink[k].expected = (unsigned)(p.gn_slots * p.sink[k].cstride);
      if (p.sink[k].eps == 0.f) p.sink[k].eps = 1e-5f;
      ++k;
    }
  }
  return 0;
}

inline int mlp_launch(const MlpDesc& d, cudaStream_t st) {
  (void)launch_kc(mlp_fused_sm100_kernel, dim3(d.grid), dim3(kMlpThreads), d.smem, st, 2 * d.prm.hsplit, d.prm);
  RS_CUDA_OK(cudaGetLastError());
  return 0;
}

// ---- fused attention half of a Swin block (swin_attn_fused.cuh, swin_attn_tc.cuh) -----------------
static long long* g_swin_timeline = nullptr;   // rs_debug_swin_timeline
struct SwinAttnDesc {
  View x, y;                               // input / output token tensors [N, H, W, E] (y may alias x)
  int heads = 0, shift = 0;
  const float* gn_part = nullptr; int gn_slots = 0; const float* gn_gstat = nullptr;
  const float* gamma = nullptr; const float* beta = nullptr;
  const __half* wqkv = nullptr; int wqkv_ld = 0; const float* bqkv = nullptr;
  const float* relbias = nullptr;
  const __half* wproj = nullptr; int wproj_ld = 0; const float* bproj = nullptr;
  GnSink sink[2] = {};
  SwinAttnParams prm;
  SwinTcParams tc;                         // tcgen05 version (swin_attn_tc.cuh): tensor maps of the two weight matrices
  bool use_tc = false;
  long long* dbg = nullptr;
  int grid = 0;
};
inline bool swin_attn_uses_tc() { return !env_is("RS_SWIN_IMPL", "mma"); }
inline bool swin_attn_supported(int E, int heads, int H, int W) {
  return (E == 192 || E == 64) && heads * 32 == E && H % 8 == 0 && W % 8 == 0;
}
inline int swin_attn_finalize(SwinAttnDesc& d) {
  SwinAttnParams& p = d.prm;
  std::memset(&p, 0, sizeof(p));
  const int E = d.x.C;
  RS_CHECK(swin_attn_supported(E, d.heads, d.x.H, d.x.W), "fused Swin attention: E in {64, 192}, head_dim 32, H and W multiples of 8");
  RS_CHECK(d.y.C == E && d.y.H == d.x.H && d.y.W == d.x.W && d.y.N == d.x.N, "fused Swin attention: output geometry");
  RS_CHECK(d.x.ld % 8 == 0 && d.y.ld % 8 == 0 && d.wqkv_ld % 8 == 0 && d.wproj_ld % 8 == 0, "fused Swin attention: 16-byte rows");
  RS_CHECK((d.gn_part && d.gn_slots > 0) || d.gn_gstat, "fused Swin attention: norm1 statistics");
  p.x = d.x.ptr; p.x_ld = d.x.ld; p.y = d.y.ptr; p.y_ld = d.y.ld;
  p.N = d.x.N; p.H = d.x.H; p.W = d.x.W; p.heads = d.heads; p.shift = d.shift; p.scale = 0.17677669529663687f;
  p.gn_part = d.gn_part; p.gn_slots = d.gn_slots; p.gn_gstat = d.gn_gstat; p.gamma = d.gamma; p.beta = d.beta; p.eps = 1e-5f;
  p.wqkv = d.wqkv; p.wqkv_ld = d.wqkv_ld; p.bqkv = d.bqkv; p.relbias = d.relbias;
  p.wproj = d.wproj; p.wproj_ld = d.wproj_ld; p.bproj = d.bproj;
  p.total_windows = d.x.N * (d.x.H / 8) * (d.x.W / 8);
  {
    int k = 0;
    for (int i = 0; i < 2; ++i) {
      if (!d.sink[i].part) continue;
      p.sink[k] = d.sink[i];
      if (p.sink[k].expected == 0) p.sink[k].expected = (unsigned)((d.x.H / 8) * (d.x.W / 8) * p.sink[k].cstride);
      if (p.sink[k].eps == 0.f) p.sink[k].eps = 1e-5f;
      ++k;
    }
  }
  const int pairs = (p.total_windows + 1) / 2;
  d.grid = std::min(pairs, 148);
  // tcgen05 version unless RS_SWIN_IMPL=mma (the mma.sync kernel stays as the tested restatement of the same arithmetic)
  d.use_tc = swin_attn_uses_tc() && d.wqkv_ld == E && d.wproj_ld == E;
  if (!d.use_tc)                                            // the mma.sync kernel delivers pairs only: consumers combine them
    for (int k = 0; k < 2; ++k) { p.sink[k].gstat = nullptr; p.sink[k].counter = nullptr; }
  if (d.use_tc) {
    std::memset(&d.tc, 0, sizeof(d.tc));
    d.tc.a = p; d.tc.dbg = d.dbg;
    int rc = encode_weight_map(&d.tc.tmWqkv, d.wqkv, E, 3 * E, 64); if (rc) return rc;
    rc = encode_weight_map(&d.tc.tmWproj, d.wproj, E, E, E); if (rc) return rc;
  }
  return 0;
}
inline int swin_attn_launch(const SwinAttnDesc& d, cudaStream_t st) {
  if (d.use_tc) {
    if (d.x.C == 192) (void)launch_k(swin_attn_tc_kernel<192>, dim3(d.grid), dim3(kTcThreads), (size_t)SwinTcSmem<192>::total, st, d.tc);
    else (void)launch_k(swin_attn_tc_kernel<64>, dim3(d.grid), dim3(kTcThreads), (size_t)SwinTcSmem<64>::total, st, d.tc);
    RS_CUDA_OK(cudaGetLastError());
    return 0;
  }
  if (d.x.C == 192) (void)launch_k(swin_attn_fused_kernel<192>, dim3(d.grid), dim3(kSwinThreads), SwinSmem<192>::total, st, d.prm);
  else (void)launch_k(swin_attn_fused_kernel<64>, dim3(d.grid), dim3(kSwinThreads), SwinSmem<64>::total, st, d.prm);
  RS_CUDA_OK(cudaGetLastError());
  return 0;
}

// Fused single-head attention of the VQ-GAN bottleneck (vq_attn_tc.cuh): q, k [N][T][C], vt [N][C][T] fp16, out
// [N][T][ld_out] fp16.
struct VqAttnDesc {
  const __half* q = nullptr; const __half* k = nullptr; const __half* vt = nullptr;
  const float* bias = nullptr;
  __half* out = nullptr; int ld_out = 0;
  int N = 0, T = 0, C = 0;
  VqAttnParams prm;
  dim3 grid;
};
inline bool vq_attn_supported(int T, int C) { return C % 64 == 0 && C >= 64 && C <= 512 && T % 64 == 0 && T >= 64; }
// 3-D fp16 map {d0, d1, d2} (d0 contiguous), 128B swizzle, box {64, box1, 1}
inline int encode_3d_map(CUtensorMap* m, const __half* base, long long d0, long long d1, long long d2, long long s1,
                         long long s2, int box1) {
  PFN_encodeTiled enc = get_encode_tiled();
  RS_CHECK(enc != nullptr, "cuTensorMapEncodeTiled entry point not available (no CUDA driver?)");
  RS_CHECK((reinterpret_cast<uintptr_t>(base) & 15) == 0 && s1 % 8 == 0 && s2 % 8 == 0, "attention operands: 16-byte rows");
  cuuint64_t dims[3] = {(cuuint64_t)d0, (cuuint64_t)d1, (cuuint64_t)d2};
  cuuint64_t strides[2] = {(cuuint64_t)s1 * 2, (cuuint64_t)s2 * 2};
  cuuint32_t box[3] = {64, (cuuint32_t)box1, 1};
  cuuint32_t estr[3] = {1, 1, 1};
  CUresult r = enc(m, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, const_cast<__half*>(base), dims, strides, box, estr,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  RS_CHECK(r == CUDA_SUCCESS, "cuTensorMapEncodeTiled(attention operand) failed with CUresult " + std::to_string((int)r));
  return 0;
}
inline int vq_attn_finalize(VqAttnDesc& d) {
  RS_CHECK(d.q && d.k && d.vt && d.bias && d.out && d.N > 0, "fused VQ attention: null operand");
  RS_CHECK(vq_attn_supported(d.T, d.C), "fused VQ attention: C a multiple of 64 in [64, 512], T a multiple of 64");
  RS_CHECK(d.ld_out >= d.C && d.ld_out % 8 == 0, "fused VQ attention: output row stride");
  VqAttnParams& p = d.prm;
  std::memset(&p, 0, sizeof(p));
  p.T = d.T; p.C = d.C;
  p.DV = d.C <= 256 ? d.C : d.C / 2;
  p.n_vc = p.DV > 128 ? 2 : 1;
  p.VC = p.DV / p.n_vc;
  p.scale_log2 = 1.4426950408889634f / std::sqrt((float)d.C);
  p.bias = d.bias; p.out = d.out; p.ld_out = d.ld_out;
  int rc = encode_3d_map(&p.tmQ, d.q, d.C, d.T, d.N, d.C, (long long)d.T * d.C, 128); if (rc) return rc;
  rc = encode_3d_map(&p.tmK, d.k, d.C, d.T, d.N, d.C, (long long)d.T * d.C, 128); if (rc) return rc;
  rc = encode_3d_map(&p.tmVt, d.vt, d.T, d.C, d.N, d.T, (long long)d.T * d.C, p.VC); if (rc) return rc;
  d.grid = dim3((unsigned)((d.T + 127) / 128), (unsigned)(d.C / p.DV), (unsigned)d.N);
  return 0;
}
inline int vq_attn_launch(const VqAttnDesc& d, cudaStream_t st) {
  (void)launch_k(vq_attn_tc_kernel, d.grid, dim3(kVqaThreads), (size_t)vqa_smem_bytes(d.C), st, d.prm);
  RS_CUDA_OK(cudaGetLastError());
  return 0;
}

inline size_t attn_smem_bytes(int E) {
  return (size_t)2 * 3 * 64 * kAttnPad * 2 + (size_t)64 * (E + 8) * 2 + 64 * sizeof(int);
}

inline int attn_launch(const View& qkv, const View& out, const float* bias, int heads, int E, int shift,
                       cudaStream_t st) {
  RS_CHECK(qkv.H % 8 == 0 && qkv.W % 8 == 0, "window attention needs H, W multiples of 8");
  RS_CHECK(E == heads * 32 && E % 8 == 0, "window attention kernel is specialised for head_dim 32");
  const int windows = qkv.N * (qkv.H / 8) * (qkv.W / 8);
  // heads per CTA: all of them when there are plenty of windows, fewer (more CTAs) otherwise
  int hpc = heads;
  while (hpc > 1 && (long long)windows * (heads / hpc) < 4 * 148 && hpc % 2 == 0) hpc /= 2;
  if (hpc > 1 && (long long)windows * (heads / hpc) < 4 * 148 && heads % hpc == 0) hpc = 1;
  WinAttnParams p{qkv.ptr, qkv.ld, out.ptr, out.ld, bias, qkv.N, qkv.H, qkv.W, heads, E, shift, 0.17677669529663687f, hpc};
  if (env_is("RS_ATTN_IMPL", "simt")) {
    (void)launch_k(window_attn_simt_kernel, dim3(windows, heads), dim3(64), (size_t)0, st, p);
  } else {
    const size_t smem = attn_smem_bytes(E);
    RS_CHECK(smem <= 160 * 1024, "attention tile does not fit in shared memory");   // limit raised in conv_init()
    (void)launch_k(window_attn_kernel, dim3(windows, heads / hpc), dim3(128), smem, st, p);
  }
  RS_CUDA_OK(cudaGetLastError());
  return 0;
}

}  // namespace rs
