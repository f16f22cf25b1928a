// mlp_bwd.cu -- backward of one SharedMLP layer of a set-abstraction block on tcgen05 (sm_100a).
//
// Replaces, for one [1x1 conv -> BatchNorm2d -> ReLU] layer l inside PointnetSAModuleVotes
// (reference pointnet2_modules.py:245-267 / pytorch_utils.py:11-36,67-120), what autograd runs as
//   max_pool2d backward (top layer) -> threshold_backward (ReLU) -> cudnn bn_bw -> cuDNN dgrad conv
//   -> cuDNN wgrad conv (+ for layer 0: cat / div / sub backward and two group_points_grad
//   scatters, _ext_src/src/group_points_gpu.cu:48-69)
// i.e. ~8 full passes over (B, C, npoint, nsample) tensors, by ONE persistent, warp-specialised
// kernel per layer.  Per tile of NT positions:
//
//   X[pos, k]    the layer's input, RECOMPUTED like the forward prologue (gathered rows, or
//                relu(bn(z_prev)))                                            -> smem, BF16
//   DZ[pos, co]  = a[co]*g + b[co]*z[pos,co] + c[co]   (BatchNorm backward; a,b,c from
//                b2r_bn_bwd_finalize).  Dense layers: g = gr and z are read from HBM.  Pooled top
//                layer: z is RECOMPUTED on the tensor cores (D1 = W X^T, never stored by the
//                forward) and g is the max-pool-routed output gradient, non-zero at ONE sample
//                per (centre, channel)                                          -> smem, BF16
//   dgrad        D2[k, pos]  = sum_co W[co,k] DZ[pos,co]                 TMEM, fresh per tile
//   wgrad        D3[co, k]  += sum_pos DZ[pos,co] X[pos,k]               TMEM, accumulated over
//                                                                        ALL tiles of the CTA
//   epilogue     dense: gr_prev = D2 * [relu(bn(z_prev)) > 0] + the next BatchNorm-backward sums;
//                gather layer: D2 scatter-added (red.global.add.f32) into the POINT-major feature
//                / xyz / centre gradients.  End of kernel: D3 -> atomicAdd into dW (Cout, Cin).
//
// Operands are BF16 (FP32 accumulate).  Every tile lives in shared memory ONCE, in the K-major
// 128B-swizzled layout; wgrad, which contracts over positions, reads the SAME bytes through
// MN-major descriptors, and dgrad reads the forward-oriented weight image MN-major as W^T.
// (For 32-bit TF32 data the MN-major view needs a different byte layout -- SWIZZLE_128B_BASE32B --
// hence a second copy of every tile; both facts measured with scripts/probe/umma_probe*.cu, logs
// under profiles/r01/.  The first version of this kernel was TF32 with doubled tiles: it could
// not double-buffer the 128->256 layers in 227 KB.)  BF16 operand rounding (2^-9) adds ~3e-3 to a
// gradient whose TF32-forward noise floor is 3-4e-2 (profiles/r01/tf32_gradient_noise*.log).
//
// Warp roles (12 warps): EW = 4 (or 8, top layer) epilogue warps (one TMEM lane quadrant each),
// then 1 MMA-issue warp (one thread), then the producers (global loads -> transform -> smem).  Two smem stages and two TMEM
// stages for D1/D2, mbarrier hand-offs (full / empty / z_done / dz_ready / mma_done / d2_free):
// producers run up to two tiles ahead of the tensor core, stores and scatters trail behind.
// Layers beyond one launch's TMEM / shared memory run as channel-slice launches
// (b2r_sa_layer_bwd_slices): an output slice adds its rows of dW and, dense layers, accumulates
// its share of gr_prev after the first slice; a feature slice of a gather layer owns its dgrad
// rows and dW columns.
#include <cuda_bf16.h>

#include "mlp_common.cuh"

namespace b2r {
using namespace mlp;
namespace {

// 12 warps = 3 per SM sub-partition -> 168 registers/thread.  EW epilogue warps (4, or 8 for the
// pooled top layer whose epilogue warps also turn the recomputed z into DZ and are the critical
// role there), 1 MMA warp, 11 - EW producer warps.
constexpr int kBwdWarps = 12;
constexpr int kBwdThreads = kBwdWarps * 32;   // 384

struct BwdArgs {
  int B, N, NP, NS, Cin, Cout, mode, top;
  const float *xyz, *new_xyz, *feat_t;
  const int *idx;
  float radius;
  int normalize_xyz;
  const float *z_prev, *scale_prev, *shift_prev;
  const void *w_image;                          // BF16 image from b2r_mlp_pack_weight_bf16
  const float *dz;                              // direct dz (M,Cout), or NULL and:
  const float *gr, *z;                          //   dense: (M,Cout) each
  const float *dysel;                           //   top:   (B*NP,Cout)
  const int *asel;                              //   top:   (B*NP,Cout)
  const float *coef_a, *coef_b, *coef_c;        // (Cout)
  float *dW;
  float *gr_prev;
  double *stats_prev;
  float *g_feat_t, *g_xyz, *g_new_xyz;
  int do_dgrad;
  int Kp, KA, WA, Cout_pad, num_tiles;   // KA: 64-wide atoms of packed K; WA: atoms in the image
  int ch8_shift;                         // log2(feature 16-byte chunks per row) or -1
  int ns_shift;                          // log2(NS) or -1
  const int *cidx, *ccen, *cmeta;        // compacted position space (csrc/compact.cu) or NULL
  // channel slice (Cin / Cout above are the slice's): row pitch of dz / gr / z / dysel / asel (the
  // whole layer's Cout), row pitch of feat_t / g_feat_t (the whole layer's features) and of dW
  // (its Cin), first feature column of the slice in dW, whether the slice owns the xyz columns,
  // and gr_prev += instead of gr_prev =
  int ldo, ldf, ldw, kofs, xyz_cols, accumulate;
};

// packed K extent of a layer in THIS kernel's operand order: gather layers put the C feature
// channels first (padded to a multiple of 8 = one 16-byte BF16 chunk), then dx,dy,dz and 5 zeros
__host__ __device__ inline int packed_k16(int Cin, int gather) {
  if (!gather) return (Cin + 7) & ~7;
  return ((Cin - 3 + 7) & ~7) + 8;
}

struct BwdSmem {
  uint32_t w_off, w_bytes, x_off[2], dz_off[2], x_bytes, dz_bytes, coef_off, scale_off, idx_off,
      cen_off, meta_off, route_off, flush_off, bar_off, total;
};
// cmp: compacted position space -- a second 4-deep ring for the rows' centre ids, the plan's meta
// words, and routed-gradient stages for NT/8 (instead of NT/16) centres per tile
__host__ __device__ inline BwdSmem bwd_smem_layout(int Kp, int KA, int WA, int Cout, int Cout_pad,
                                                   int NT, int top, int cmp = 0) {
  BwdSmem s;
  s.w_off = 0;
  s.w_bytes = (uint32_t)Cout_pad * WA * 128u;
  s.x_bytes = (uint32_t)NT * KA * 128u;
  s.dz_bytes = (uint32_t)NT * (Cout_pad >> 6) * 128u;
  uint32_t o = s.w_bytes;
  for (int st = 0; st < 2; ++st) {
    s.x_off[st] = o;
    o += s.x_bytes;
    s.dz_off[st] = o;
    o += s.dz_bytes;
  }
  s.coef_off = o;
  s.scale_off = s.coef_off + 3u * Cout * 4u;
  s.idx_off = s.scale_off + 2u * Kp * 4u;
  s.cen_off = s.idx_off + 4u * (uint32_t)NT * 4u;                    // idx: 4 buffers (below)
  s.meta_off = s.cen_off + (cmp ? 4u * (uint32_t)NT * 4u : 0u);
  s.route_off = (s.meta_off + (cmp ? 32u : 0u) + 15u) & ~15u;
  s.flush_off = s.route_off +
                (top ? 4u * (uint32_t)(NT / (cmp ? 8 : 16)) * Cout_pad * 4u : 0u);   // 2 stages
  // wgrad flush staging: a padded 32x32 tile per warp.  With a plan it reuses the operand stages
  // when they are large enough (the flush runs after the CTA's last MMA has completed, when no
  // producer or tensor-core access to them is outstanding): the wider routed-gradient stages
  // would otherwise push the 128->256 top layer down to 32-position tiles.
  const uint32_t flush_bytes = 8u * 32u * 33u * 4u;
  if (cmp && 2u * (s.x_bytes + s.dz_bytes) >= flush_bytes) {
    s.bar_off = s.flush_off;
    s.flush_off = s.x_off[0];
  } else {
    s.bar_off = s.flush_off + flush_bytes;
  }
  s.total = s.bar_off + 13 * 8 + 16 + 1024;                        // + alignment slack
  return s;
}

// byte offset of 16-byte chunk `chunk` (8 consecutive BF16 channels) of row `row` in a K-major
// SW128 BF16 operand with `rows` rows: 64-channel atoms, then 8-row groups of 1024 B
__device__ __forceinline__ uint32_t bf_off(int row, int chunk, int rows) {
  const int a = chunk >> 3, c = chunk & 7, g = row >> 3, r8 = row & 7;
  return (uint32_t)(((a * (rows >> 3) + g) << 10) + (r8 << 7) + ((c ^ r8) << 4));
}
// kind::f16 instruction descriptor: BF16 x BF16 -> F32, M = 128, N = n
__host__ __device__ constexpr uint32_t idesc_bf16(int n, int a_mn, int b_mn) {
  return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)a_mn << 15) | ((uint32_t)b_mn << 16) |
         ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24);
}
__device__ __forceinline__ void umma_bf16(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
  const __nv_bfloat162 v = __floats2bfloat162_rn(lo, hi);
  return *reinterpret_cast<const uint32_t *>(&v);
}
template <int N>
__device__ __forceinline__ void bar_named(int id) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "n"(N));
}

// W (Cout, Cin) fp32 -> BF16 K-major SW128 image, rows = Cout (padded to 128), contraction
// dimension = packed K (this kernel's order), WA 64-wide atoms (zero padded)
__global__ void pack_weight_bf16_kernel(const float *__restrict__ w, int Cout, int Cin, int gather,
                                        int Kp, int Cout_pad, int WA,
                                        __nv_bfloat16 *__restrict__ image) {
  const long long total = (long long)Cout_pad * WA * 64;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    const int co = (int)(e / (WA * 64)), kp = (int)(e % (WA * 64));
    float v = 0.f;
    if (co < Cout && kp < Kp) {
      int k = -1;
      if (gather) {
        const int C = Cin - 3, Cf8 = (C + 7) & ~7;
        if (kp < C) k = 3 + kp;
        else if (kp >= Cf8 && kp < Cf8 + 3) k = kp - Cf8;
      } else if (kp < Cin) {
        k = kp;
      }
      if (k >= 0) v = w[(size_t)co * Cin + k];
    }
    image[(bf_off(co, kp >> 3, Cout_pad) >> 1) + (kp & 7)] = __float2bfloat16_rn(v);
  }
}

// MODE (0 gather layer, 1 dense layer) and TOP (pooled top layer: z recomputed, DZ built by the
// epilogue warps) are compile-time: every instantiation carries only its own producer /
// epilogue code.  One runtime-branched kernel was 52,872 SASS instructions (846 KB) and spent
// 25 % of its warp-stall samples waiting for instruction fetch (ncu, stall_no_inst).
// CMP: positions are those of a b2r_compact_plan (csrc/compact.cu).  Incoming gradients (gr,
// dysel) and everything derived from them carry the positions' multiplicities implicitly: only
// the DENSE BatchNorm-backward term b*z + c, which every padded position receives once, is
// scaled by the multiplicity (1 + NS - class size for a centre's first sample, 0 for dead rows).
// SL: a channel-slice launch (ldo / ldf / ldw / kofs / xyz_cols / accumulate); the whole-layer
// instantiations keep the addressing they had before slices existed
template <int NT, int EW, int MODE, int TOP, bool CMP, bool SL>
__global__ void __launch_bounds__(kBwdThreads, 1) sa_layer_bwd_kernel(const BwdArgs a) {
  constexpr int kMode = MODE;
  constexpr bool kTop = TOP != 0;
  constexpr int kRC = CMP ? NT / 8 : NT / 16;   // centres per tile a routed-gradient stage holds
  constexpr int kEpiThreads = EW * 32, kProdThreads = (kBwdWarps - 1 - EW) * 32;
  auto bar_epi = [] { bar_named<kEpiThreads>(1); };
  auto bar_prod = [] { bar_named<kProdThreads>(2); };
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t *base = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                              ~(uintptr_t)1023);
  const BwdSmem L = bwd_smem_layout(a.Kp, a.KA, a.WA, a.Cout, a.Cout_pad, NT, kTop, CMP ? 1 : 0);
  uint8_t *s_w = base + L.w_off;
  float *s_ca = reinterpret_cast<float *>(base + L.coef_off);
  float *s_cb = s_ca + a.Cout;
  float *s_cc = s_cb + a.Cout;
  float *s_scale = reinterpret_cast<float *>(base + L.scale_off);
  float *s_shift = s_scale + a.Kp;
  // ball-query indices per tile, 4-deep ring: the producers may write tile k while the scatter
  // epilogue still reads tile k-3 (MMA(k-2) only waits for the epilogue of tile k-4)
  int *s_idx4 = reinterpret_cast<int *>(base + L.idx_off);
  int *s_cen4 = reinterpret_cast<int *>(base + L.cen_off);     // CMP: centre of every row, same ring
  int *s_meta = reinterpret_cast<int *>(base + L.meta_off);    // CMP: plan meta words 0..7
  float *s_dy = reinterpret_cast<float *>(base + L.route_off);
  int *s_as = reinterpret_cast<int *>(s_dy + 2 * kRC * a.Cout_pad);
  uint64_t *s_bar = reinterpret_cast<uint64_t *>(base + L.bar_off);
  uint32_t *s_tmem = reinterpret_cast<uint32_t *>(s_bar + 13);
  // mbarriers: [0,1] full  [2,3] empty  [4,5] z_done  [6,7] dz_ready  [8,9] mma_done
  //            [10,11] d2_free  [12] weights
  auto bar = [&](int i) { return smem_u32(&s_bar[i]); };

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int KA = a.KA;
  const int MTp = (KA + 1) >> 1;          // 128-row M tiles of the dgrad output (packed K rows)
  const int MTl = a.Cout_pad >> 7;        // 128-row M tiles over Cout (recompute, wgrad)
  constexpr int NCH = NT / 32;
  const bool has_coef = a.dz == nullptr;
  const int w12 = ((kTop && MTl > (a.do_dgrad ? MTp : 0)) ? MTl : (a.do_dgrad ? MTp : 0)) * NT;
  const uint32_t d3_col0 = 2u * (uint32_t)w12;
  constexpr uint32_t kTmemCols = 512;
  const long long per_scene = (long long)a.NP * a.NS;
  const int C = a.Cin - 3, Cf8 = (C + 7) & ~7;   // gather layers: feature channels
  const int ldo = SL ? a.ldo : a.Cout;             // row pitch of dz / gr / z / dysel / asel
  const int ldf = SL ? a.ldf : C;                  // row pitch of feat_t / g_feat_t
  int num_tiles = a.num_tiles;
  if constexpr (CMP) {
    num_tiles = __ldg(a.cmeta + 8) / NT;
    if (tid < 8) s_meta[tid] = __ldg(a.cmeta + tid);
  }

  if (tid == 0) {
    // full (0,1) and d2_free (10,11) are completed by ONE arrival per warp of the role -- a named
    // barrier + single arrival made every warp of the role wait for its slowest sibling once per
    // tile (stall_barrier 13-22 % of the samples, profiles/r02/ncu_stalls_sa1_bwd.txt)
    for (int i = 0; i < 13; ++i)
      mbar_init(bar(i), (i == 0 || i == 1) ? (uint32_t)(kProdThreads / 32)
                        : (i == 10 || i == 11) ? (uint32_t)EW : 1u);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == EW) tmem_alloc(smem_u32(s_tmem), kTmemCols);
  {  // zero both stages of both tiles once: padding chunks are never written again
    const uint32_t zb = 2u * (L.x_bytes + L.dz_bytes);
    for (uint32_t i = tid * 16; i < zb; i += kBwdThreads * 16)
      *reinterpret_cast<uint4 *>(base + L.x_off[0] + i) = make_uint4(0, 0, 0, 0);
  }
  if (kMode == 1)
    for (int i = tid; i < a.Cin; i += kBwdThreads) {
      s_scale[i] = a.scale_prev[i];
      s_shift[i] = a.shift_prev[i];
    }
  if (has_coef)
    for (int i = tid; i < a.Cout; i += kBwdThreads) {
      s_ca[i] = a.coef_a[i];
      s_cb[i] = a.coef_b[i];
      s_cc[i] = a.coef_c[i];
    }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;
  const bool need_w = kTop || a.do_dgrad;
  if (tid == 0 && need_w) {
    mbar_expect_tx(bar(12), L.w_bytes);
    bulk_g2s(smem_u32(s_w), a.w_image, L.w_bytes, bar(12));
  }
  const int grid = (int)gridDim.x;

  if (warp > EW) {
    // =============================== PRODUCERS (7 warps) ========================================
    const int ptid = tid - (kEpiThreads + 32);
    const int CH8 = a.Cout >> 3;     // 16-byte BF16 chunks per DZ row
    const int ch8s = (CH8 & (CH8 - 1)) == 0 ? 31 - __clz(CH8) : -1;   // log2 or -1: no division
    const int CHx = a.Cin >> 3;      // dense layers: 16-byte BF16 chunks per X row
    const int chxs = (CHx > 0 && (CHx & (CHx - 1)) == 0) ? 31 - __clz(CHx) : -1;
    int nidx = 0, ncen = 0;   // prefetched ball-query index (centre) of the next tile
    for (int k = 0, tile = blockIdx.x; tile < num_tiles; tile += grid, ++k) {
      const int s = k & 1, n = k >> 1;
      mbar_wait(bar(2 + s), (uint32_t)((n & 1) ^ 1));   // MMAs of tile k-2 are done with stage s
      const long long pos0 = (long long)tile * NT;
      uint8_t *sx = base + L.x_off[s], *sdz = base + L.dz_off[s];
      int *s_idx = s_idx4 + (k & 3) * NT;
      int *s_cen = s_cen4 + (k & 3) * NT;
      TileClass tc{};
      int p64 = 0;
      if constexpr (CMP) {
        tc = tile_class(s_meta, pos0, a.NS);
        p64 = (int)(pos0 & 63);
      }
      if (ptid == 0 && tile + 2 * grid < num_tiles) {   // pull tile k+2 into L2 meanwhile
        const size_t pn = (size_t)(pos0 + 2ll * grid * NT);
        if (!kTop) {
          if (!has_coef) prefetch_l2(a.dz + pn * ldo, (uint32_t)NT * ldo * 4u);
          else {
            prefetch_l2(a.gr + pn * ldo, (uint32_t)NT * ldo * 4u);
            prefetch_l2(a.z + pn * ldo, (uint32_t)NT * ldo * 4u);
          }
        }
        if (kMode == 1) prefetch_l2(a.z_prev + pn * a.Cin, (uint32_t)NT * a.Cin * 4u);
      }
      // ---- DZ tile from HBM (dense layers / direct dz); the top layer's DZ comes from D1 ------
      if (!kTop) {
        const int total = NT * CH8;
        const size_t o0 = (size_t)pos0 * ldo;
        for (int i0 = ptid; i0 < total; i0 += kProdThreads * 4) {
          float4 g[4][2], zz[4][2];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * kProdThreads;
            if (i < total) {
              // chunk i sits at float4 2 i of the tile for a whole layer, at row * ldo + ch * 8
              // floats for a slice
              size_t e = 0;
              int e4 = 2 * i;
              if constexpr (SL) {
                const int row = ch8s >= 0 ? (i >> ch8s) : (i / CH8);
                e = (size_t)row * ldo + (size_t)(i - row * CH8) * 8;
                e4 = 0;
              }
              if (!has_coef) {
                const float4 *p = reinterpret_cast<const float4 *>(a.dz + o0 + e) + e4;
                g[u][0] = __ldg(p); g[u][1] = __ldg(p + 1);
              } else {
                const float4 *p = reinterpret_cast<const float4 *>(a.gr + o0 + e) + e4;
                const float4 *qz = reinterpret_cast<const float4 *>(a.z + o0 + e) + e4;
                g[u][0] = __ldg(p); g[u][1] = __ldg(p + 1);
                zz[u][0] = __ldg(qz); zz[u][1] = __ldg(qz + 1);
              }
            }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * kProdThreads;
            if (i < total) {
              const int row = ch8s >= 0 ? (i >> ch8s) : (i / CH8), ch = i - row * CH8;
              float v[8] = {g[u][0].x, g[u][0].y, g[u][0].z, g[u][0].w,
                            g[u][1].x, g[u][1].y, g[u][1].z, g[u][1].w};
              if (has_coef) {
                const float zv[8] = {zz[u][0].x, zz[u][0].y, zz[u][0].z, zz[u][0].w,
                                     zz[u][1].x, zz[u][1].y, zz[u][1].z, zz[u][1].w};
                float ca8[8], cb8[8], cc8[8];
                *reinterpret_cast<float4 *>(ca8) = *reinterpret_cast<const float4 *>(s_ca + ch * 8);
                *reinterpret_cast<float4 *>(ca8 + 4) = *reinterpret_cast<const float4 *>(s_ca + ch * 8 + 4);
                *reinterpret_cast<float4 *>(cb8) = *reinterpret_cast<const float4 *>(s_cb + ch * 8);
                *reinterpret_cast<float4 *>(cb8 + 4) = *reinterpret_cast<const float4 *>(s_cb + ch * 8 + 4);
                *reinterpret_cast<float4 *>(cc8) = *reinterpret_cast<const float4 *>(s_cc + ch * 8);
                *reinterpret_cast<float4 *>(cc8 + 4) = *reinterpret_cast<const float4 *>(s_cc + ch * 8 + 4);
                if constexpr (CMP) {
                  const float wgt = row < tc.live
                                        ? ((((p64 + row) & (tc.ns - 1)) == 0) ? 1.f + tc.wx : 1.f)
                                        : 0.f;
#pragma unroll
                  for (int e = 0; e < 8; ++e)
                    v[e] = fmaf(ca8[e], v[e], wgt * fmaf(cb8[e], zv[e], cc8[e]));
                } else {
#pragma unroll
                  for (int e = 0; e < 8; ++e) v[e] = fmaf(ca8[e], v[e], fmaf(cb8[e], zv[e], cc8[e]));
                }
              }
              *reinterpret_cast<uint4 *>(sdz + bf_off(row, ch, NT)) =
                  make_uint4(pack_bf16(v[0], v[1]), pack_bf16(v[2], v[3]), pack_bf16(v[4], v[5]),
                             pack_bf16(v[6], v[7]));
            }
          }
        }
      }
      // ---- X tile ---------------------------------------------------------------------------
      if (kMode == 0) {
        // indices of this tile were requested one tile ago (nidx): no dependent global wait here
        if constexpr (kProdThreads < NT) {
          // fewer producer threads than rows (8 epilogue warps leave 3 producer warps: a one-layer
          // block, gather AND pooled top, on 128-position tiles): plain loop, no register prefetch
          for (int r = ptid; r < NT; r += kProdThreads) {
            if constexpr (CMP) {
              s_idx[r] = __ldg(a.cidx + pos0 + r);
              s_cen[r] = __ldg(a.ccen + pos0 + r);
            } else {
              s_idx[r] = __ldg(a.idx + pos0 + r);
            }
          }
        } else if (ptid < NT) {
          if constexpr (CMP) {
            s_idx[ptid] = (k == 0) ? a.cidx[pos0 + ptid] : nidx;
            s_cen[ptid] = (k == 0) ? a.ccen[pos0 + ptid] : ncen;
            if (tile + grid < num_tiles) {
              nidx = __ldg(a.cidx + pos0 + (long long)grid * NT + ptid);
              ncen = __ldg(a.ccen + pos0 + (long long)grid * NT + ptid);
            }
          } else {
            s_idx[ptid] = (k == 0) ? a.idx[pos0 + ptid] : nidx;
            if (tile + grid < num_tiles) nidx = __ldg(a.idx + pos0 + (long long)grid * NT + ptid);
          }
        }
        bar_prod();
        // CMP: s_idx holds global source rows and s_cen global centres: scene 0's base pointers
        const int b = CMP ? 0 : (int)(pos0 / per_scene);
        const int in_scene0 = CMP ? 0 : (int)(pos0 - (long long)b * per_scene);
        const int CH8f = Cf8 >> 3;
        for (int row = ptid; row < NT; row += kProdThreads) {   // relative xyz chunk
          const int p = s_idx[row];
          const int j = CMP ? max(s_cen[row], 0) : (in_scene0 + row) / a.NS;
          const float *pp = a.xyz + ((size_t)b * a.N + p) * 3;
          const float *qq = a.new_xyz + ((size_t)b * a.NP + j) * 3;
          const float px = __ldg(pp), py = __ldg(pp + 1), pz = __ldg(pp + 2);
          const float qx = __ldg(qq), qy = __ldg(qq + 1), qz = __ldg(qq + 2);
          float d0 = __fsub_rn(px, qx), d1 = __fsub_rn(py, qy), d2 = __fsub_rn(pz, qz);
          if (a.normalize_xyz) {
            d0 = __fdiv_rn(d0, a.radius);
            d1 = __fdiv_rn(d1, a.radius);
            d2 = __fdiv_rn(d2, a.radius);
          }
          *reinterpret_cast<uint4 *>(sx + bf_off(row, CH8f, NT)) =
              make_uint4(pack_bf16(d0, d1), pack_bf16(d2, 0.f), 0u, 0u);
        }
        if (CH8f > 0) {
          const float *fb = a.feat_t + (size_t)b * a.N * ldf;
          const int total = NT * CH8f;
          if ((C & 7) == 0) {
            for (int i0 = ptid; i0 < total; i0 += kProdThreads * 4) {
              float4 t[4][2];
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * kProdThreads;
                if (i < total) {
                  const int row = a.ch8_shift >= 0 ? (i >> a.ch8_shift) : (i / CH8f);
                  const int ch = i - row * CH8f;
                  const float4 *p =
                      reinterpret_cast<const float4 *>(fb + (size_t)s_idx[row] * ldf) + 2 * ch;
                  t[u][0] = __ldg(p); t[u][1] = __ldg(p + 1);
                }
              }
#pragma unroll
              for (int u = 0; u < 4; ++u) {
                const int i = i0 + u * kProdThreads;
                if (i < total) {
                  const int row = a.ch8_shift >= 0 ? (i >> a.ch8_shift) : (i / CH8f);
                  const int ch = i - row * CH8f;
                  *reinterpret_cast<uint4 *>(sx + bf_off(row, ch, NT)) =
                      make_uint4(pack_bf16(t[u][0].x, t[u][0].y), pack_bf16(t[u][0].z, t[u][0].w),
                                 pack_bf16(t[u][1].x, t[u][1].y), pack_bf16(t[u][1].z, t[u][1].w));
                }
              }
            }
          } else {
            for (int i = ptid; i < total; i += kProdThreads) {
              const int row = i / CH8f, ch = i - row * CH8f;
              const float *src = fb + (size_t)s_idx[row] * ldf + ch * 8;
              float f[8];
#pragma unroll
              for (int e = 0; e < 8; ++e) f[e] = (ch * 8 + e < C) ? __ldg(src + e) : 0.f;
              *reinterpret_cast<uint4 *>(sx + bf_off(row, ch, NT)) =
                  make_uint4(pack_bf16(f[0], f[1]), pack_bf16(f[2], f[3]), pack_bf16(f[4], f[5]),
                             pack_bf16(f[6], f[7]));
            }
          }
        }
      } else {
        const int CH = a.Cin >> 3;
        const int total = NT * CH;
        const float4 *src = reinterpret_cast<const float4 *>(a.z_prev + (size_t)pos0 * a.Cin);
        for (int i0 = ptid; i0 < total; i0 += kProdThreads * 4) {
          float4 t[4][2];
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * kProdThreads;
            if (i < total) { t[u][0] = __ldg(src + 2 * i); t[u][1] = __ldg(src + 2 * i + 1); }
          }
#pragma unroll
          for (int u = 0; u < 4; ++u) {
            const int i = i0 + u * kProdThreads;
            if (i < total) {
              const int row = chxs >= 0 ? (i >> chxs) : (i / CH), ch = i - row * CH;
              const float *sc = s_scale + ch * 8, *sh = s_shift + ch * 8;
              const float x0 = fmaxf(fmaf(t[u][0].x, sc[0], sh[0]), 0.f);
              const float x1 = fmaxf(fmaf(t[u][0].y, sc[1], sh[1]), 0.f);
              const float x2 = fmaxf(fmaf(t[u][0].z, sc[2], sh[2]), 0.f);
              const float x3 = fmaxf(fmaf(t[u][0].w, sc[3], sh[3]), 0.f);
              const float x4 = fmaxf(fmaf(t[u][1].x, sc[4], sh[4]), 0.f);
              const float x5 = fmaxf(fmaf(t[u][1].y, sc[5], sh[5]), 0.f);
              const float x6 = fmaxf(fmaf(t[u][1].z, sc[6], sh[6]), 0.f);
              const float x7 = fmaxf(fmaf(t[u][1].w, sc[7], sh[7]), 0.f);
              *reinterpret_cast<uint4 *>(sx + bf_off(row, ch, NT)) =
                  make_uint4(pack_bf16(x0, x1), pack_bf16(x2, x3), pack_bf16(x4, x5),
                             pack_bf16(x6, x7));
            }
          }
        }
      }
      fence_async_smem();   // generic-proxy writes -> visible to the tensor core (async proxy)
      __syncwarp();
      if (lane == 0) mbar_arrive(bar(0 + s));
    }
  } else if (warp == EW) {
    // =============================== MMA ISSUE (one thread) =====================================
    if (lane == 0) {
      if (need_w) mbar_wait(bar(12), 0);
      const uint32_t wa = smem_u32(s_w);
      const uint32_t lbo_w = (uint32_t)(a.Cout_pad >> 3) * 1024u;   // 64-wide K atoms of the image
      const uint32_t lbo_t = (uint32_t)(NT >> 3) * 1024u;           // 64-wide atoms of the tiles
      const int KS16 = (a.Kp + 15) >> 4, KSl16 = (a.Cout + 15) >> 4;
      for (int k = 0, tile = blockIdx.x; tile < num_tiles; tile += grid, ++k) {
        const int s = k & 1, n = k >> 1;
        const uint32_t xa = smem_u32(base + L.x_off[s]), dza = smem_u32(base + L.dz_off[s]);
        const uint32_t d12 = tmem_base + (uint32_t)(s * w12);
        mbar_wait(bar(0 + s), (uint32_t)(n & 1));           // X (and DZ) of tile k are in smem
        mbar_wait(bar(10 + s), (uint32_t)((n & 1) ^ 1));    // epilogue of tile k-2 left D1/D2[s]
        tc_fence_after();
        if (kTop) {
          // D1[co, pos] = W (K-major) * X (K-major): the top layer's z, never stored by the forward
          for (int ml = 0; ml < MTl; ++ml)
            for (int ks = 0; ks < KS16; ++ks) {
              const uint64_t ad = smem_desc_sw128(wa + (uint32_t)(ks >> 2) * lbo_w +
                                                  (uint32_t)ml * 16u * 1024u + (uint32_t)(ks & 3) * 32u);
              const uint64_t bd =
                  smem_desc_sw128(xa + (uint32_t)(ks >> 2) * lbo_t + (uint32_t)(ks & 3) * 32u);
              umma_bf16(d12 + (uint32_t)ml * NT, ad, bd, idesc_bf16(NT, 0, 0), ks > 0 ? 1u : 0u);
            }
          umma_commit(bar(4 + s));
          mbar_wait(bar(6 + s), (uint32_t)(n & 1));         // epilogue warps wrote DZ from D1
          tc_fence_after();
        }
        if (a.do_dgrad) {
          // D2[k rows, pos] = W^T (the image viewed MN-major) * DZ (K-major)
          for (int m = 0; m < MTp; ++m)
            for (int ks = 0; ks < KSl16; ++ks) {
              const uint64_t ad = smem_desc_sw128_mn(
                  wa + (uint32_t)(2 * m) * lbo_w + (uint32_t)ks * 2048u, lbo_w, 1024u);
              const uint64_t bd =
                  smem_desc_sw128(dza + (uint32_t)(ks >> 2) * lbo_t + (uint32_t)(ks & 3) * 32u);
              umma_bf16(d12 + (uint32_t)m * NT, ad, bd, idesc_bf16(NT, 1, 0), ks > 0 ? 1u : 0u);
            }
        }
        // D3[co rows, k cols] += DZ^T * X: both tiles viewed MN-major, contraction over positions
        for (int ml = 0; ml < MTl; ++ml)
          for (int a0 = 0; a0 < KA; a0 += 4) {
            const int na = (KA - a0) < 4 ? (KA - a0) : 4;
            const uint32_t idw = idesc_bf16(na * 64, 1, 1);
            for (int k16 = 0; k16 < NT / 16; ++k16) {
              const uint64_t ad = smem_desc_sw128_mn(
                  dza + (uint32_t)(2 * ml) * lbo_t + (uint32_t)k16 * 2048u, lbo_t, 1024u);
              const uint64_t bd = smem_desc_sw128_mn(
                  xa + (uint32_t)a0 * lbo_t + (uint32_t)k16 * 2048u, lbo_t, 1024u);
              umma_bf16(tmem_base + d3_col0 + (uint32_t)(ml * KA + a0) * 64u, ad, bd, idw,
                        (k > 0 || k16 > 0) ? 1u : 0u);
            }
          }
        umma_commit(bar(8 + s));   // -> epilogue
        umma_commit(bar(2 + s));   // -> producers: stage s may be overwritten
      }
    }
    __syncwarp();
  } else {
    // =============================== EPILOGUE (4 warps, one TMEM lane quadrant each) ============
    // warp w: TMEM lane quadrant q = w & 3; with 8 epilogue warps the two warps of a quadrant
    // split the 32-column chunks by parity h = w >> 2
    const int q = warp & 3, h = warp >> 2;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    float s1[3] = {0.f, 0.f, 0.f}, s2[3] = {0.f, 0.f, 0.f};
    double d1[3] = {0.0, 0.0, 0.0}, d2[3] = {0.0, 0.0, 0.0};
    int ntiles = 0;
    // Top layer: D1 (recomputed z) -> dz = a*dy_routed + b*z + c -> DZ tile (BF16) of tile k.
    // Called one tile AHEAD of the D2 epilogue (software pipelining): while these warps turn
    // D1(k+1) into DZ(k+1), the tensor core runs dgrad/wgrad(k), so neither waits for the other.
    // Routed gradient (dysel, asel) of every centre touching tile k (<= NT/16 centres), parked in
    // smem stage k & 1.  Fetched with cp.async TWO tiles ahead (issued at the end of
    // produce_dz(k-2)): a plain load here was an exposed HBM round trip per tile (13 % of this
    // kernel's stall samples, ncu).  Every thread reads back only entries it copied itself (the
    // two warps of a quadrant copy the same entries), so cp.async.wait_group is all the
    // synchronisation needed.  One (possibly empty) group is committed per call.
    auto fetch_route = [&](int k, int tile) {
      if (tile < num_tiles) {
        const int s = k & 1;
        const long long pos0 = (long long)tile * NT;
        int ns_t = a.NS, shift_t = a.ns_shift;
        if constexpr (CMP) {
          ns_t = tile_class(s_meta, pos0, a.NS).ns;
          shift_t = 31 - __clz(ns_t);
        }
        const long long centre0 = pos0 >> shift_t;
        const int base_s = (int)(pos0 & (ns_t - 1));
        const int ncen = ((base_s + NT - 1) >> shift_t) + 1;
        float *my_dy = s_dy + (size_t)s * kRC * a.Cout_pad;
        int *my_as = s_as + (size_t)s * kRC * a.Cout_pad;
        // global centre of the tile's c-th centre (its first in-tile position), dead padding = -1:
        // lane c fetches it ONCE for the warp (ncen <= NT/8 + 1 <= 17) and the loop below takes it
        // by shuffle -- a dependent global load per centre and thread in front of every cp.async
        // pair was 15 % of this kernel's stall samples (profiles/r02/ncu_stalls_sa1_bwd.txt)
        int cg_lane = -1;
        if constexpr (CMP) {
          if (lane < ncen) cg_lane = __ldg(a.ccen + pos0 + (lane == 0 ? 0 : lane * ns_t - base_s));
        }
        for (int c = 0; c < ncen; ++c) {
          long long cg = centre0 + c;
          if constexpr (CMP) cg = __shfl_sync(0xffffffffu, cg_lane, c);
          for (int ml = 0; ml < MTl; ++ml) {
            const int co = ml * 128 + q * 32 + lane;
            if (co < a.Cout) {
              if constexpr (CMP) {
                if (cg < 0) {
                  my_dy[c * a.Cout_pad + co] = 0.f;
                  my_as[c * a.Cout_pad + co] = -1;
                  continue;
                }
              }
              const size_t o = (size_t)cg * ldo + co;
              asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(
                               smem_u32(my_dy + c * a.Cout_pad + co)),
                           "l"(a.dysel + o)
                           : "memory");
              asm volatile("cp.async.ca.shared.global [%0], [%1], 4;" ::"r"(
                               smem_u32(my_as + c * a.Cout_pad + co)),
                           "l"(a.asel + o)
                           : "memory");
            }
          }
        }
      }
      asm volatile("cp.async.commit_group;" ::: "memory");
    };
    auto produce_dz = [&](int k, int tile) {
      const int s = k & 1, n = k >> 1;
      const long long pos0 = (long long)tile * NT;
      const uint32_t d12 = tmem_base + (uint32_t)(s * w12);
      uint8_t *sdz = base + L.dz_off[s];
      TileClass tc{};
      int ns_t = a.NS, shift_t = a.ns_shift;
      if constexpr (CMP) {
        tc = tile_class(s_meta, pos0, a.NS);
        ns_t = tc.ns;
        shift_t = 31 - __clz(ns_t);
      }
      const int ns_mask = ns_t - 1;                         // NS is a power of two >= 16 (host)
      const int base_s = (int)(pos0 & ns_mask);
      const float *my_dy = s_dy + (size_t)s * kRC * a.Cout_pad;
      const int *my_as = s_as + (size_t)s * kRC * a.Cout_pad;
      asm volatile("cp.async.wait_group 1;" ::: "memory");   // tile k's routes have landed
      mbar_wait(bar(4 + s), (uint32_t)(n & 1));
      tc_fence_after();
#pragma unroll
      for (int ml = 0; ml < 2; ++ml) {
        if (ml >= MTl) continue;
        const int co = ml * 128 + q * 32 + lane;
        const bool ok = co < a.Cout;
        const float ca = ok ? s_ca[co] : 0.f, cb = ok ? s_cb[co] : 0.f, cc = ok ? s_cc[co] : 0.f;
#pragma unroll
        for (int c0 = 0; c0 < NCH; c0 += (EW == 8 ? 2 : 1)) {
          const int ch = c0 + (EW == 8 ? h : 0);   // 8 warps: the quadrant's two warps alternate
          uint32_t r[32];
          cuda::ptx::tcgen05_ld_32x32b(r, d12 + lane_addr + (uint32_t)(ml * NT + ch * 32));
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (ok && CMP) {
#pragma unroll
            for (int sg = 0; sg < 4; ++sg) {   // 8 columns lie inside one centre, live or dead
              const int colb = ch * 32 + sg * 8;
              const int t0 = base_s + colb;
              const int c = t0 >> shift_t;
              const int s0 = t0 & ns_mask;
              const float dyv = my_dy[c * a.Cout_pad + co];
              const int as = my_as[c * a.Cout_pad + co] - s0;   // routed sample, relative
              const float w0 = colb < tc.live ? 1.f : 0.f;
#pragma unroll
              for (int i = 0; i < 8; ++i) {
                const float dy = (i == as) ? dyv : 0.f;
                const float wgt = (s0 + i == 0) ? w0 * (1.f + tc.wx) : w0;
                const float v =
                    fmaf(ca, dy, wgt * fmaf(cb, __uint_as_float(r[sg * 8 + i]), cc));
                *reinterpret_cast<__nv_bfloat16 *>(
                    sdz + bf_off(colb + i, co >> 3, NT) + (co & 7) * 2) = __float2bfloat16_rn(v);
              }
            }
          } else if (ok) {
#pragma unroll
            for (int hf = 0; hf < 2; ++hf) {   // 16 columns = one centre (NS >= 16, aligned)
              const int t0 = base_s + ch * 32 + hf * 16;
              const int c = t0 >> a.ns_shift;
              const int s0 = t0 & ns_mask;
              const float dyv = my_dy[c * a.Cout_pad + co];
              const int as = my_as[c * a.Cout_pad + co] - s0;   // routed sample, relative
#pragma unroll
              for (int i = 0; i < 16; ++i) {
                const float dy = (i == as) ? dyv : 0.f;
                const float v = fmaf(ca, dy, fmaf(cb, __uint_as_float(r[hf * 16 + i]), cc));
                *reinterpret_cast<__nv_bfloat16 *>(
                    sdz + bf_off(ch * 32 + hf * 16 + i, co >> 3, NT) + (co & 7) * 2) =
                    __float2bfloat16_rn(v);
              }
            }
          }
        }
      }
      tc_fence_before();
      fence_async_smem();
      // A full role barrier here, not per-warp arrivals: the two warps of a quadrant refill the SAME
      // route entries of stage s right below (fetch_route), so neither may start before both have
      // read them (compute-sanitizer racecheck flags exactly that when this is a per-warp arrival)
      bar_epi();
      if (tid == 0) mbar_arrive(bar(6 + s));
      fetch_route(k + 2, tile + 2 * grid);   // stage s is free again: this thread's reads are done
    };
    if (kTop) {
      fetch_route(0, blockIdx.x);
      fetch_route(1, blockIdx.x + grid);
      if ((int)blockIdx.x < num_tiles) produce_dz(0, blockIdx.x);
    }
    for (int k = 0, tile = blockIdx.x; tile < num_tiles; tile += grid, ++k, ++ntiles) {
      const int s = k & 1, n = k >> 1;
      const long long pos0 = (long long)tile * NT;
      const uint32_t d12 = tmem_base + (uint32_t)(s * w12);
      const int *s_idx = s_idx4 + (k & 3) * NT;
      const int *s_cen = s_cen4 + (k & 3) * NT;
      if (kTop && tile + grid < num_tiles) produce_dz(k + 1, tile + grid);
      mbar_wait(bar(8 + s), (uint32_t)(n & 1));
      tc_fence_after();
      if (a.do_dgrad) {
        int tile_b = 0, in_scene0 = 0;
        if (kMode == 0 && !CMP) {
          tile_b = (int)(pos0 / per_scene);
          in_scene0 = (int)(pos0 - (long long)tile_b * per_scene);
        }
        int ns_t = a.NS;   // CMP: class size of this tile's centres (s_idx / s_cen are global)
        if constexpr (CMP) {
          if (kMode == 0) {
            ns_t = tile_class(s_meta, pos0, a.NS).ns;
            in_scene0 = (int)(pos0 & 63);
          }
        }
#pragma unroll
        for (int m = 0; m < 3; ++m) {
          if (m >= MTp) continue;
#pragma unroll
          for (int c0 = 0; c0 < NCH; c0 += (EW == 8 ? 2 : 1)) {
            const int cc = c0 + (EW == 8 ? h : 0);
            uint32_t r[32];
            cuda::ptx::tcgen05_ld_32x32b(r, d12 + lane_addr + (uint32_t)(m * NT + cc * 32));
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            const int kp = m * 128 + q * 32 + lane;   // packed K row owned by this thread
            const long long p0 = pos0 + cc * 32;
            if (kMode == 1) {
              if (kp < a.Cin) {
                const float sc = s_scale[kp], sh = s_shift[kp];
                const float *zp = a.z_prev + (size_t)p0 * a.Cin + kp;
                float *gp = a.gr_prev + (size_t)p0 * a.Cin + kp;
                float t1 = 0.f, t2 = 0.f;
                float zv[32];   // all 32 (L2-resident) loads in flight before the first store
#pragma unroll
                for (int i = 0; i < 32; ++i) zv[i] = __ldg(zp + (size_t)i * a.Cin);
                if (SL && a.accumulate) {
                  // a later output slice: add its share of dz W to the earlier slices' (the mask
                  // and the sums below are linear in it, so partial sums add up)
#pragma unroll
                  for (int i = 0; i < 32; ++i) {
                    const float g = fmaf(zv[i], sc, sh) > 0.f ? __uint_as_float(r[i]) : 0.f;
                    gp[(size_t)i * a.Cin] += g;
                    t1 += g;
                    t2 = fmaf(g, zv[i], t2);
                  }
                } else {
#pragma unroll
                  for (int i = 0; i < 32; ++i) {
                    const float g = fmaf(zv[i], sc, sh) > 0.f ? __uint_as_float(r[i]) : 0.f;
                    gp[(size_t)i * a.Cin] = g;
                    t1 += g;
                    t2 = fmaf(g, zv[i], t2);
                  }
                }
                s1[m] += t1;
                s2[m] += t2;
              }
            } else {
              // gather layer: scatter-add into the point-major feature / xyz / centre gradients
              const bool is_feat = kp < C;
              const int e = kp - Cf8;                 // 0..2 for the dx,dy,dz rows
              const bool is_xyz = (e >= 0 && e < 3);
              if (is_feat && a.g_feat_t != nullptr) {
                float *gb = a.g_feat_t + (size_t)tile_b * a.N * ldf + kp;
#pragma unroll
                for (int i = 0; i < 32; ++i)
                  atomicAdd(gb + (size_t)s_idx[cc * 32 + i] * ldf, __uint_as_float(r[i]));
              } else if (is_xyz && (a.g_xyz != nullptr || a.g_new_xyz != nullptr)) {
                float run = 0.f;
                float *gx = a.g_xyz != nullptr ? a.g_xyz + (size_t)tile_b * a.N * 3 + e : nullptr;
#pragma unroll
                for (int i = 0; i < 32; ++i) {
                  const int ins = in_scene0 + cc * 32 + i;   // position inside the scene
                  float v = __uint_as_float(r[i]);
                  if (a.normalize_xyz) v = __fdiv_rn(v, a.radius);
                  if (gx != nullptr) atomicAdd(gx + (size_t)s_idx[cc * 32 + i] * 3, v);
                  run += v;
                  if constexpr (CMP) {
                    if (((ins + 1) & (ns_t - 1)) == 0 || i == 31) {   // end of this centre's run
                      const int cg = s_cen[cc * 32 + i];
                      if (a.g_new_xyz != nullptr && cg >= 0)
                        atomicAdd(a.g_new_xyz + (size_t)cg * 3 + e, -run);
                      run = 0.f;
                    }
                  } else if (((ins + 1) % a.NS) == 0 || i == 31) {   // end of this centre's run
                    if (a.g_new_xyz != nullptr)
                      atomicAdd(a.g_new_xyz + ((size_t)tile_b * a.NP + ins / a.NS) * 3 + e, -run);
                    run = 0.f;
                  }
                }
              }
            }
          }
        }
        if (kMode == 1) {
#pragma unroll
          for (int m = 0; m < 3; ++m) {
            d1[m] += (double)s1[m];
            d2[m] += (double)s2[m];
            s1[m] = 0.f;
            s2[m] = 0.f;
          }
        }
      }
      tc_fence_before();
      __syncwarp();   // every thread of this warp is done with D1/D2[s] (and, gather layers, s_idx)
      if (lane == 0) mbar_arrive(bar(10 + s));
    }

    if (a.do_dgrad && kMode == 1 && a.stats_prev != nullptr) {
#pragma unroll
      for (int m = 0; m < 3; ++m) {
        const int kp = m * 128 + q * 32 + lane;
        if (m < MTp && kp < a.Cin) {
          atomicAdd(a.stats_prev + kp, d1[m]);
          atomicAdd(a.stats_prev + a.Cin + kp, d2[m]);
        }
      }
    }
    // ---- wgrad accumulator -> dW (Cout, Cin): the last mma_done wait covered every MMA ----------
    // TMEM hands each thread one ROW (output channel) of a 32x32 chunk; adding it to dW as it is
    // would make every warp-wide red.global touch 32 rows = 32 cache lines.  Each warp transposes
    // its chunk through a private padded smem tile so that one instruction adds 32 CONSECUTIVE
    // input channels of one row: one 128-byte line per instruction (32x fewer L2 transactions --
    // this flush is a fixed cost per CTA and dominated the small SA3/SA4/vote layers).
    if (ntiles > 0) {
      tc_fence_after();
      float *stg = reinterpret_cast<float *>(base + L.flush_off) + warp * (32 * 33);
      for (int ml = 0; ml < MTl; ++ml) {
        const int co0 = ml * 128 + q * 32;
        for (int at = (EW == 8 ? h : 0); at < KA * 2; at += (EW == 8 ? 2 : 1)) {
          uint32_t r[32];
          cuda::ptx::tcgen05_ld_32x32b(
              r, tmem_base + lane_addr + d3_col0 + (uint32_t)(ml * KA * 64 + at * 32));
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
          for (int i = 0; i < 32; ++i) stg[lane * 33 + i] = __uint_as_float(r[i]);
          __syncwarp();
          const int kp = at * 32 + lane;   // this lane's packed input channel
          int kk = -1;
          if (kMode == 0) {
            if (kp < C) kk = 3 + (SL ? a.kofs : 0) + kp;
            else if ((!SL || a.xyz_cols) && kp >= Cf8 && kp < Cf8 + 3) kk = kp - Cf8;
          } else if (kp < a.Cin) {
            kk = kp;
          }
          if (kk >= 0) {
            const int rows = min(32, a.Cout - co0);
            for (int rr = 0; rr < rows; ++rr)
              atomicAdd(a.dW + (size_t)(co0 + rr) * (SL ? a.ldw : a.Cin) + kk, stg[rr * 33 + lane]);
          }
          __syncwarp();
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == EW) tmem_dealloc(tmem_base, kTmemCols);
}

// ---- max-pool / ReLU / BatchNorm backward of the pooled top layer: the sparse part ------------
// Forward kept, per (centre, channel): zmax, zmin and their sample indices.  The pooled output
// was y = relu(scale*zsel + shift) with zsel = (scale >= 0 ? zmax : zmin).  Its gradient reaches
// exactly ONE sample per (centre, channel):
//   dysel = dout * [y > 0],  asel = arg of zsel
// and the BatchNorm-backward sums over all positions reduce to sums over centres:
//   sum(gr) = sum(dysel),   sum(gr * z) = sum(dysel * zsel).
// One 32 x 32 (centre, channel) tile per CTA: the channel-major output gradient is read with
// coalesced rows along the centres, transposed through shared memory, and everything else
// (zmax / zmin / arg reads, dysel / asel writes) runs coalesced along the channels; the tile's
// contribution to the two per-channel sums is reduced in shared memory: one double atomic pair
// per channel per CTA.
__global__ void pool_bwd_prep_kernel(const float *__restrict__ dout_cm,
                                     const float *__restrict__ dout_pm,
                                     const float *__restrict__ zmax, const float *__restrict__ zmin,
                                     const int *__restrict__ amax, const int *__restrict__ amin,
                                     const float *__restrict__ scale,
                                     const float *__restrict__ shift, int NP, int Cch,
                                     float *__restrict__ dysel, int *__restrict__ asel,
                                     double *__restrict__ stats) {
  __shared__ float t[32][33];
  __shared__ double r1[8][32], r2[8][32];
  const int b = blockIdx.z;
  const int j0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  if (dout_cm != nullptr) {
    for (int i = threadIdx.y; i < 32; i += blockDim.y) {   // rows = channels, lanes = centres
      const int cc = c0 + i, j = j0 + threadIdx.x;
      t[i][threadIdx.x] = (cc < Cch && j < NP) ? dout_cm[((size_t)b * Cch + cc) * NP + j] : 0.f;
    }
    __syncthreads();
  }
  const int ch = c0 + threadIdx.x;
  const float s = ch < Cch ? scale[ch] : 0.f, sh = ch < Cch ? shift[ch] : 0.f;
  const bool pos = s >= 0.f;
  double a1 = 0.0, a2 = 0.0;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {     // rows = centres, lanes = channels
    const int j = j0 + i;
    if (j < NP && ch < Cch) {
      const size_t o = ((size_t)b * NP + j) * Cch + ch;
      const float zs = pos ? zmax[o] : zmin[o];
      const int as = pos ? amax[o] : amin[o];
      float g = dout_cm != nullptr ? t[threadIdx.x][i] : 0.f;
      if (dout_pm != nullptr) g += dout_pm[o];
      g = fmaf(zs, s, sh) > 0.f ? g : 0.f;
      dysel[o] = g;
      asel[o] = as;
      a1 += (double)g;
      a2 += (double)g * (double)zs;
    }
  }
  r1[threadIdx.y][threadIdx.x] = a1;
  r2[threadIdx.y][threadIdx.x] = a2;
  __syncthreads();
  if (threadIdx.y == 0 && ch < Cch) {
    for (int k = 1; k < 8; ++k) {
      a1 += r1[k][threadIdx.x];
      a2 += r2[k][threadIdx.x];
    }
    atomicAdd(stats + ch, a1);
    atomicAdd(stats + Cch + ch, a2);
  }
}

// BatchNorm backward bookkeeping of one layer from  S1 = sum(gr), S2 = sum(gr*z)  (one thread per
// channel).  training: dz = a*gr + b*z + c with
//    gs = gamma*invstd, k1 = S1/M, k2 = (S2 - mean*S1)*invstd/M, a = gs, b = -gs*k2*invstd,
//    c = -gs*k1 - b*mean;       eval (running statistics): dz = gs*gr.
// dgamma = (S2 - mean*S1)*invstd, dbeta = S1.  Also emits the epilogue-2 form (k1,k2,gs).
__global__ void bn_bwd_finalize_kernel(const double *__restrict__ stats, int Cch, double count,
                                       double inv_count,
                                       const float *__restrict__ gamma,
                                       const float *__restrict__ mean,
                                       const float *__restrict__ invstd, int training,
                                       float *__restrict__ coef_a, float *__restrict__ coef_b,
                                       float *__restrict__ coef_c, float *__restrict__ k1_out,
                                       float *__restrict__ k2_out, float *__restrict__ gs_out,
                                       float *__restrict__ dgamma, float *__restrict__ dbeta,
                                       float *__restrict__ dbias_conv) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch >= Cch) return;
  const double S1 = stats[ch], S2 = stats[Cch + ch];
  const double mu = (double)mean[ch], is = (double)invstd[ch];
  const double g = gamma ? (double)gamma[ch] : 1.0;
  const double sx = (S2 - mu * S1) * is;   // sum(gr * xhat)
  const double gs = g * is;
  double k1 = 0.0, k2 = 0.0;
  if (training) {
    k1 = S1 * inv_count;
    k2 = sx * inv_count;
  }
  const double b = -gs * k2 * is;
  if (coef_a) coef_a[ch] = (float)gs;
  if (coef_b) coef_b[ch] = (float)b;
  if (coef_c) coef_c[ch] = (float)(-gs * k1 - b * mu);
  if (k1_out) k1_out[ch] = (float)k1;
  if (k2_out) k2_out[ch] = (float)k2;
  if (gs_out) gs_out[ch] = (float)gs;
  if (dgamma) dgamma[ch] = (float)sx;
  if (dbeta) dbeta[ch] = (float)S1;
  // gradient of a bias added by the convolution BEFORE this BatchNorm: sum over positions of
  // dz = a*gr + b*z + c, i.e. a*S1 + count*(b*mean + c) -- zero with batch statistics, gs*S1 with
  // running statistics (nn.Conv1d(bias=True) -> BatchNorm1d in the voting / proposal heads)
  if (dbias_conv) dbias_conv[ch] = (float)(gs * S1 + count * (b * mu + (-gs * k1 - b * mu)));
}

}  // namespace

}  // namespace b2r

using namespace b2r;

namespace {
struct Geometry {
  int Kp, KA, WA, Cout_pad;
};
Geometry bwd_geometry(int Cout, int Cin, int gather) {
  Geometry g;
  g.Kp = packed_k16(Cin, gather);
  g.KA = (g.Kp + 63) >> 6;
  const int MTp = (g.KA + 1) >> 1;
  g.WA = g.KA > 2 * MTp ? g.KA : 2 * MTp;   // dgrad reads the image in whole 128-wide M tiles
  g.Cout_pad = (Cout + 127) & ~127;
  return g;
}
}  // namespace

namespace {
// positions per tile for one backward launch: the widest tile whose two smem stages and two TMEM
// stages fit; 0 = the layer does not fit at all
int bwd_pick_nt(const Geometry &g, int Cout, int mode, int top, int do_dgrad, int NS, long long M,
                long long per_scene, int cmp = 0) {
  const int MTp = (g.KA + 1) >> 1, MTl = g.Cout_pad >> 7;
  if (MTp > 3) return 0;
  for (int nt : {128, 64, 32}) {
    if (M % nt) continue;
    if (!cmp && mode == 0 && per_scene % nt) continue;   // a tile must lie inside one scene
    if (top && (nt % NS) != 0 && (NS % nt) != 0) continue;
    const BwdSmem L = bwd_smem_layout(g.Kp, g.KA, g.WA, Cout, g.Cout_pad, nt, top, cmp);
    const int w12 = ((top && MTl > (do_dgrad ? MTp : 0)) ? MTl : (do_dgrad ? MTp : 0)) * nt;
    const int cols = 2 * w12 + MTl * g.KA * 64;
    if (L.total <= 227u * 1024u && cols <= 512) return nt;
  }
  return 0;
}

// whether ONE launch can hold a layer of these channel counts at all (dgrad on, the narrowest
// tile, which also satisfies every nsample rule); compact: with a plan's extra shared memory
bool bwd_fits(int Cin, int Cout, int gather, int top, int cmp) {
  if (Cout > 256) return false;
  const Geometry g = bwd_geometry(Cout, Cin, gather);
  if (((g.KA + 1) >> 1) > 3) return false;
  const int MTp = (g.KA + 1) >> 1, MTl = g.Cout_pad >> 7;
  const BwdSmem L = bwd_smem_layout(g.Kp, g.KA, g.WA, Cout, g.Cout_pad, 32, top, cmp);
  const int w12 = ((top && MTl > MTp) ? MTl : MTp) * 32;
  return L.total <= 227u * 1024u && 2 * w12 + MTl * g.KA * 64 <= 512;
}
}  // namespace

// Slice grid (include/b2r.h): the same search as b2r_sa_layer_fwd_slices over the backward's
// limits (shared memory, TMEM columns, at most three 128-row dgrad tiles)
extern "C" int b2r_sa_layer_bwd_slices(int Cin, int Cout, int gather, int top, int *co_step,
                                       int *ci_step) {
  int best = 0, best_kn = 0, bco = 0, bci = 0;
  if (Cin > 0 && Cout > 0 && (Cout % 8) == 0 && (gather ? Cin >= 3 : (Cin % 8) == 0)) {
    if (bwd_fits(Cin, Cout, gather, top, 0)) {
      best = 1; bco = Cout; bci = 0;
    } else {
      const int C = Cin - 3;
      for (int cs : {256, 128}) {
        const int co = cs < Cout ? cs : Cout;
        for (int kn = 1; kn <= 16; kn *= 2) {
          int ci = 0;
          if (kn > 1) {
            if (!gather || top || C % 8 != 0) break;
            ci = ((C + kn - 1) / kn + 7) & ~7;
            if (ci * (kn - 1) >= C) continue;
          }
          if (!bwd_fits(kn > 1 ? 3 + ci : Cin, co, gather, top, 1)) continue;
          const int n = ((Cout + co - 1) / co) * (kn > 1 ? (C + ci - 1) / ci : 1);
          if (best == 0 || n < best || (n == best && kn < best_kn)) {
            best = n; best_kn = kn; bco = co; bci = ci;
          }
          break;
        }
      }
    }
  }
  if (co_step) *co_step = bco;
  if (ci_step) *ci_step = bci;
  return best;
}

extern "C" int b2r_sa_layer_bwd_supported(int B, int NP, int NS, int Cin, int Cout, int gather,
                                          int top) {
  if (B <= 0 || NP <= 0 || NS <= 0 || Cin <= 0 || Cout <= 0) return 0;
  if ((Cout % 8) != 0 || (!gather && (Cin % 8) != 0) || (gather && Cin < 3)) return 0;
  if (top && pow2_shift(NS) < 0) return 0;
  int co = 0, ci = 0;
  if (b2r_sa_layer_bwd_slices(Cin, Cout, gather, top, &co, &ci) == 0) return 0;
  const int Cin_s = ci > 0 ? 3 + ci : Cin;   // the widest slice decides the tile
  const Geometry g = bwd_geometry(co, Cin_s, gather);
  const long long per_scene = (long long)NP * NS, M = (long long)B * per_scene;
  // worst case for the tile choice: every gradient requested (dgrad on)
  return bwd_pick_nt(g, co, gather ? 0 : 1, top, 1, NS, M, per_scene) > 0 ? 1 : 0;
}

extern "C" int b2r_sa_layer_bwd_tile(int B, int NP, int NS, int Cin, int Cout, int gather, int top,
                                     int dgrad, int compact) {
  if (B <= 0 || NP <= 0 || NS <= 0 || Cin <= 0 || Cout <= 0) return 0;
  const Geometry g = bwd_geometry(Cout, Cin, gather);
  const long long per_scene = (long long)NP * NS;
  const long long M = compact ? b2r_compact_capacity(B, NP, NS) : (long long)B * per_scene;
  return bwd_pick_nt(g, Cout, gather ? 0 : 1, top, dgrad, NS, M, per_scene, compact ? 1 : 0);
}

extern "C" long long b2r_mlp_weight_bf16_image_bytes(int Cout, int Cin, int gather) {
  if (Cout <= 0 || Cin <= 0) return 0;
  const Geometry g = bwd_geometry(Cout, Cin, gather);
  return (long long)g.Cout_pad * g.WA * 128;
}

extern "C" int b2r_mlp_pack_weight_bf16(const float *w, int Cout, int Cin, int gather, void *image,
                                        void *stream) {
  B2R_REQUIRE(w && image && Cout > 0 && Cin > 0, "b2r_mlp_pack_weight_bf16: bad argument");
  B2R_REQUIRE(!gather || Cin >= 3, "b2r_mlp_pack_weight_bf16: gather layers need Cin >= 3");
  const Geometry g = bwd_geometry(Cout, Cin, gather);
  const long long total = (long long)g.Cout_pad * g.WA * 64;
  pack_weight_bf16_kernel<<<ceil_div(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      w, Cout, Cin, gather, g.Kp, g.Cout_pad, g.WA, static_cast<__nv_bfloat16 *>(image));
  B2R_CHECK_LAUNCH();
  return B2R_OK;
}

extern "C" int b2r_sa_layer_bwd(const b2r_sa_layer_bwd_desc *d, void *stream) {
  B2R_REQUIRE(d != nullptr, "b2r_sa_layer_bwd: null descriptor");
  B2R_REQUIRE(d->B > 0 && d->NP > 0 && d->NS > 0 && d->Cin > 0 && d->Cout > 0,
              "b2r_sa_layer_bwd: non-positive size");
  B2R_REQUIRE(d->mode == 0 || d->mode == 1, "b2r_sa_layer_bwd: mode must be 0 or 1");
  B2R_REQUIRE(d->dW != nullptr, "b2r_sa_layer_bwd: null dW");
  const bool co_sliced = d->co_n != 0, ci_sliced = d->ci_n != 0;
  B2R_REQUIRE(co_sliced ? (d->co0 >= 0 && d->co_n > 0 && d->co0 <= d->Cout - d->co_n &&
                           d->co0 % 8 == 0)
                        : d->co0 == 0,
              "b2r_sa_layer_bwd: output slice [%d, +%d) outside Cout=%d or not 8-aligned", d->co0,
              d->co_n, d->Cout);
  B2R_REQUIRE(!ci_sliced || d->mode == 0, "b2r_sa_layer_bwd: feature slices are for gather layers");
  B2R_REQUIRE(ci_sliced ? (d->ci0 >= 0 && d->ci_n > 0 && d->ci0 <= d->Cin - 3 - d->ci_n &&
                           d->ci0 % 8 == 0 && d->ci_n % 8 == 0)
                        : d->ci0 == 0,
              "b2r_sa_layer_bwd: feature slice [%d, +%d) outside the %d features or not a "
              "multiple of 8", d->ci0, d->ci_n, d->Cin - 3);
  B2R_REQUIRE(!d->accumulate || (d->accumulate == 1 && d->mode == 1),
              "b2r_sa_layer_bwd: accumulate is 0, or 1 for a dense layer (gather layers always "
              "scatter-add)");
  const int Cout_s = co_sliced ? d->co_n : d->Cout;
  const int Cin_s = ci_sliced ? 3 + d->ci_n : d->Cin;
  const int co0 = d->co0;
  const bool top = d->dysel != nullptr;
  B2R_REQUIRE(d->dz != nullptr || (d->coef_a && d->coef_b && d->coef_c &&
                                   ((d->gr && d->z) || (top && d->asel))),
              "b2r_sa_layer_bwd: needs dz, or gr + z + coef_a/b/c, or dysel + asel + coef_a/b/c");
  // a slice launch: the kernel sees a layer of Cin_s -> Cout_s channels; the pointers below are
  // moved to the slice's first output channel / feature column, the pitches stay the layer's
  auto off = [](const float *p, long long o) { return p != nullptr ? p + o : nullptr; };
  BwdArgs a;
  a.B = d->B; a.N = d->N; a.NP = d->NP; a.NS = d->NS; a.Cin = Cin_s; a.Cout = Cout_s;
  a.mode = d->mode;
  a.top = (d->dz == nullptr && top) ? 1 : 0;
  a.xyz = d->xyz; a.new_xyz = d->new_xyz; a.feat_t = off(d->feat_t, d->ci0); a.idx = d->idx;
  a.radius = d->radius; a.normalize_xyz = d->normalize_xyz;
  a.z_prev = d->z_prev; a.scale_prev = d->scale_prev; a.shift_prev = d->shift_prev;
  a.w_image = d->w_image_bf16;
  a.dz = off(d->dz, co0); a.gr = off(d->gr, co0); a.z = off(d->z, co0);
  a.dysel = off(d->dysel, co0); a.asel = d->asel != nullptr ? d->asel + co0 : nullptr;
  a.coef_a = off(d->coef_a, co0); a.coef_b = off(d->coef_b, co0); a.coef_c = off(d->coef_c, co0);
  a.dW = d->dW + (size_t)co0 * d->Cin; a.gr_prev = d->gr_prev; a.stats_prev = d->stats_prev;
  a.g_feat_t = d->g_feat_t != nullptr ? d->g_feat_t + d->ci0 : nullptr;
  // the xyz rows of a gather layer belong to the feature slice that starts at 0
  a.g_xyz = d->ci0 == 0 ? d->g_xyz : nullptr;
  a.g_new_xyz = d->ci0 == 0 ? d->g_new_xyz : nullptr;
  a.ldo = d->Cout; a.ldf = d->Cin - 3; a.ldw = d->Cin; a.kofs = d->ci0;
  a.xyz_cols = d->ci0 == 0 ? 1 : 0; a.accumulate = d->accumulate;
  const Geometry g = bwd_geometry(Cout_s, Cin_s, d->mode == 0);
  a.Kp = g.Kp; a.KA = g.KA; a.WA = g.WA; a.Cout_pad = g.Cout_pad;
  a.ch8_shift = pow2_shift((((Cin_s - 3 + 7) & ~7) >> 3));
  a.ns_shift = pow2_shift(d->NS);
  a.cidx = d->cidx; a.ccen = d->ccen; a.cmeta = d->cmeta;
  const int cmp = d->cmeta != nullptr ? 1 : 0;
  B2R_REQUIRE(!cmp || (d->cidx && d->ccen), "b2r_sa_layer_bwd: a plan needs cidx, ccen and cmeta");
  if (cmp && !(d->NS == 16 || d->NS == 32 || d->NS == 64)) {
    set_error("b2r_sa_layer_bwd: a compacted plan needs nsample 16/32/64 (got %d)", d->NS);
    return B2R_ERR_UNSUPPORTED;
  }
  if (a.top && a.ns_shift < 0) {
    set_error("b2r_sa_layer_bwd: the pooled top layer needs a power-of-two nsample (got %d)", d->NS);
    return B2R_ERR_UNSUPPORTED;
  }
  a.num_tiles = 0;
  if (d->mode == 0) {
    B2R_REQUIRE(d->Cin >= 3 && d->xyz && d->new_xyz && (d->idx || cmp) && (d->feat_t || d->Cin == 3),
                "b2r_sa_layer_bwd: gather mode needs xyz, new_xyz, idx (and feat_t when Cin > 3)");
    a.do_dgrad = (a.g_feat_t != nullptr && Cin_s > 3) || a.g_xyz != nullptr ||
                 a.g_new_xyz != nullptr;
  } else {
    B2R_REQUIRE(d->z_prev && d->scale_prev && d->shift_prev,
                "b2r_sa_layer_bwd: dense mode needs z_prev/scale/shift");
    B2R_REQUIRE(d->gr_prev != nullptr, "b2r_sa_layer_bwd: dense mode needs gr_prev");
    a.do_dgrad = 1;
  }
  B2R_REQUIRE(!(a.do_dgrad || a.top) || d->w_image_bf16 != nullptr,
              "b2r_sa_layer_bwd: null weight image");
  // thin first layer without an input gradient (SA1: xyz / height are leaves): streaming kernel
  if (!co_sliced && !ci_sliced && thin::bwd_applicable(d)) return thin::bwd_launch(d, stream);
  // with a plan the launch is sized for the plan's CAPACITY; the live tile count is on the device
  const long long M = cmp ? b2r_compact_capacity(d->B, d->NP, d->NS)
                          : (long long)d->B * d->NP * d->NS;
  const long long per_scene = (long long)d->NP * d->NS;
  if (a.Cout_pad > 256 || (Cout_s % 8) != 0 || (d->mode == 1 && (d->Cin % 8) != 0)) {
    set_error("b2r_sa_layer_bwd: needs Cout %% 8 == 0, Cout <= 256 per launch (see "
              "b2r_sa_layer_bwd_slices), dense Cin %% 8 == 0 (Cin=%d Cout=%d)", Cin_s, Cout_s);
    return B2R_ERR_UNSUPPORTED;
  }
  const int NT = bwd_pick_nt(g, Cout_s, d->mode, a.top, a.do_dgrad, d->NS, M, per_scene, cmp);
  if (NT == 0) {
    set_error("b2r_sa_layer_bwd: layer Cin=%d Cout=%d M=%lld does not fit shared memory / TMEM",
              Cin_s, Cout_s, M);
    return B2R_ERR_UNSUPPORTED;
  }
  const BwdSmem L = bwd_smem_layout(a.Kp, a.KA, a.WA, a.Cout, a.Cout_pad, NT, a.top, cmp);
  a.num_tiles = (int)(M / NT);
  int sms = kNumSMs;
  if (d->sm_limit > 0 && d->sm_limit < kNumSMs) sms = d->sm_limit;
  const int grid = a.num_tiles < sms ? a.num_tiles : sms;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool sliced = co_sliced || ci_sliced || d->accumulate;
#define B2R_LAUNCH_BWD3(NTV, EWV, MV, TV, CV, SLV)                                              \
  do {                                                                                          \
    B2R_CUDA(cudaFuncSetAttribute(sa_layer_bwd_kernel<NTV, EWV, MV, TV, CV, SLV>,               \
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));  \
    sa_layer_bwd_kernel<NTV, EWV, MV, TV, CV, SLV><<<grid, kBwdThreads, L.total, st>>>(a);      \
  } while (0)
#define B2R_LAUNCH_BWD2(NTV, EWV, MV, TV, CV)                                                   \
  do {                                                                                          \
    if (sliced) B2R_LAUNCH_BWD3(NTV, EWV, MV, TV, CV, true);                                    \
    else B2R_LAUNCH_BWD3(NTV, EWV, MV, TV, CV, false);                                          \
  } while (0)
#define B2R_LAUNCH_BWD1(NTV, EWV, MV, TV)                                                       \
  do {                                                                                          \
    if (cmp) B2R_LAUNCH_BWD2(NTV, EWV, MV, TV, true); else B2R_LAUNCH_BWD2(NTV, EWV, MV, TV, false); \
  } while (0)
  // the pooled top layer runs 8 epilogue warps (they also build DZ from the recomputed z) on
  // tiles of >= 64 positions
#define B2R_LAUNCH_BWD(NTV, EWTOP)                                                              \
  do {                                                                                          \
    if (a.top) {                                                                                \
      if (a.mode == 0) B2R_LAUNCH_BWD1(NTV, EWTOP, 0, 1); else B2R_LAUNCH_BWD1(NTV, EWTOP, 1, 1); \
    } else {                                                                                    \
      if (a.mode == 0) B2R_LAUNCH_BWD1(NTV, 4, 0, 0); else B2R_LAUNCH_BWD1(NTV, 4, 1, 0);       \
    }                                                                                           \
  } while (0)
  if (NT == 128) B2R_LAUNCH_BWD(128, 8);
  else if (NT == 64) B2R_LAUNCH_BWD(64, 8);
  else B2R_LAUNCH_BWD(32, 4);
#undef B2R_LAUNCH_BWD
#undef B2R_LAUNCH_BWD1
#undef B2R_LAUNCH_BWD2
#undef B2R_LAUNCH_BWD3
  B2R_CHECK_LAUNCH();
  return B2R_OK;
}

extern "C" int b2r_pool_bwd_prep(const float *dout_cm, const float *dout_pm, const float *zmax,
                                 const float *zmin, const int *amax, const int *amin,
                                 const float *scale, const float *shift, int B, int NP, int C,
                                 float *dysel, int *asel, double *stats, void *stream) {
  B2R_REQUIRE((dout_cm || dout_pm) && zmax && zmin && amax && amin && scale && shift && dysel &&
                  asel && stats && B > 0 && NP > 0 && C > 0 && C <= 1024,
              "b2r_pool_bwd_prep: bad argument");
  B2R_REQUIRE(B <= 65535, "b2r_pool_bwd_prep: B=%d exceeds gridDim.z", B);
  dim3 grid(ceil_div(NP, 32), ceil_div(C, 32), B), block(32, 8);
  pool_bwd_prep_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(
      dout_cm, dout_pm, zmax, zmin, amax, amin, scale, shift, NP, C, dysel, asel, stats);
  B2R_CHECK_LAUNCH();
  return B2R_OK;
}

extern "C" int b2r_bn_bwd_finalize_ex(const double *stats, int C, double count, const float *gamma,
                                      const float *mean, const float *invstd, int training,
                                      float *coef_a, float *coef_b, float *coef_c, float *k1,
                                      float *k2, float *gs, float *dgamma, float *dbeta,
                                      float *dbias_conv, void *stream) {
  B2R_REQUIRE(stats && mean && invstd && C > 0 && count > 0, "b2r_bn_bwd_finalize: bad argument");
  bn_bwd_finalize_kernel<<<ceil_div(C, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      stats, C, count, 1.0 / count, gamma, mean, invstd, training, coef_a, coef_b, coef_c, k1, k2, gs, dgamma,
      dbeta, dbias_conv);
  B2R_CHECK_LAUNCH();
  return B2R_OK;
}

extern "C" int b2r_bn_bwd_finalize(const double *stats, int C, double count, const float *gamma,
                                   const float *mean, const float *invstd, int training,
                                   float *coef_a, float *coef_b, float *coef_c, float *k1,
                                   float *k2, float *gs, float *dgamma, float *dbeta,
                                   void *stream) {
  return b2r_bn_bwd_finalize_ex(stats, C, count, gamma, mean, invstd, training, coef_a, coef_b,
                                coef_c, k1, k2, gs, dgamma, dbeta, nullptr, stream);
}
