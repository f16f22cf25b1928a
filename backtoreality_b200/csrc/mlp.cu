// mlp.cu -- the SharedMLP block of a set-abstraction layer on tcgen05 tensor cores (sm_100a).
//
// Replaces, for PointnetSAModuleVotes (reference pointnet2_modules.py:245-267), the chain
//   QueryAndGroup (group xyz, -= centre, /= radius, group features, cat)      5 HBM passes
//   3 x [cuDNN 1x1 conv -> BatchNorm2d -> ReLU]                                 ~9 HBM passes
//   F.max_pool2d over nsample                                                   1 HBM pass
// which materialises every (B, C, npoint, nsample) intermediate.
//
// One kernel, `sa_layer_fwd_kernel`, runs ONE conv layer as a fused GEMM
//        D[Cout x positions] = W[Cout x K] * X[positions x K]^T          (TF32 in, FP32 accumulate)
// with the neighbouring memory-bound work folded into its prologue / epilogue:
//   prologue  mode 0: X rows are GATHERED on the fly (ball-query idx -> point-major features +
//                     relative, radius-normalised xyz): the grouped tensor never exists in HBM.
//             mode 1: X rows are the previous layer's raw conv output with that layer's
//                     BatchNorm scale/shift + ReLU applied while loading.
//   epilogue  0: per-channel sum / sum-of-squares (BatchNorm batch statistics) + store raw z.
//             1: statistics + max AND min over the `nsample` positions of every centre (+ arg
//                indices).  BN+ReLU are monotone per channel, so max-pool(relu(bn(z))) is
//                relu(bn(max z)) for a non-negative BN scale and relu(bn(min z)) otherwise:
//                the (B,C,npoint,nsample) activation of the last layer is never stored.
// Orientation "channels on TMEM lanes": the accumulator row (TMEM lane) is an output channel and
// the column a position, so BN statistics, BN scale/shift and the max-pool over `nsample` are all
// per-THREAD register work in the epilogue (one thread owns one channel), no shuffles.
//
// Warp-specialised and double-buffered (see the role table above the kernel).
// Blackwell specifics: tcgen05.mma (kind::tf32, cta_group::1, M=128, N=64/128, K=8) issued by one
// elected thread, operands in 128B-swizzled K-major shared memory, accumulators in TMEM read back
// with tcgen05.ld.32x32b.x32, MMA completion signalled through tcgen05.commit -> mbarrier.
// The weight operand is staged by the TMA unit: one cp.async.bulk (UBLKCP) of a pre-swizzled
// weight image built by `pack_weight_kernel`.
// A layer whose image does not fit (or with Cout > 256) runs as a grid of channel-slice launches
// of the same kernel (b2r_sa_layer_fwd_slices, DESIGN.md section 4): output slices write their own
// columns of the whole layer's z / statistics / pool outputs; feature slices of a gather layer add
// their partial z in the storing epilogue (ldz, ldf, accumulate in LayerArgs).
#include "mlp_common.cuh"

namespace b2r {
using namespace mlp;
namespace {

// W (Cout, Cin) row-major fp32 (a 1x1 conv weight) -> TF32-rounded shared-memory image of the A
// operand: Cout padded to 128 rows per M tile, K padded to 32-element atoms, SW128 K-major.
__global__ void pack_weight_kernel(const float *__restrict__ w, int Cout, int Cin, int gather,
                                   int Kp, int Cout_pad, float *__restrict__ image) {
  const int KA = (Kp + 31) >> 5;
  const long long total = (long long)Cout_pad * KA * 32;
  for (long long e = (long long)blockIdx.x * blockDim.x + threadIdx.x; e < total;
       e += (long long)gridDim.x * blockDim.x) {
    const int m = (int)(e / (KA * 32)), kp = (int)(e % (KA * 32));
    float v = 0.f;
    if (m < Cout && kp < Kp) {
      int k = -1;  // source column in the reference order [dx,dy,dz, f0..fC-1]
      if (gather) {
        const int C = Cin - 3, Cf4 = (C + 3) & ~3;
        if (kp < C) k = 3 + kp;
        else if (kp >= Cf4 && kp < Cf4 + 3) k = kp - Cf4;
      } else if (kp < Cin) {
        k = kp;
      }
      if (k >= 0) v = __uint_as_float(to_tf32(w[(size_t)m * Cin + k]));
    }
    const uint32_t off = sw128_off(m, kp >> 2, Cout_pad) + (kp & 3) * 4;
    image[off >> 2] = v;
  }
}

struct LayerArgs {
  int B, N, NP, NS, Cin, Cout, mode, epilogue;
  const float *xyz, *new_xyz, *feat_t;
  const int *idx;
  float radius;
  int normalize_xyz;
  const float *z_prev, *scale_prev, *shift_prev;
  const float *w_image;
  float *z;
  double *stats;
  float *zmax, *zmin;
  int *amax, *amin;
  int Kp, Cout_pad, num_tiles, chf_shift, ns_shift, raw_stage;
  const int *cidx, *ccen, *cmeta;   // compacted position space (csrc/compact.cu) or NULL
  // channel slice: row pitch of z / zmax / zmin / amax / amin and offset of the sum-of-squares
  // half of stats (the whole layer's Cout; Cout above is the slice's), row pitch of feat_t, and
  // z += product instead of z = product (a feature slice after the first)
  int ldz, ldf, accumulate;
};

// Warp roles (16 warps = 4 per SM sub-partition -> 128 registers/thread):
//   0-7  epilogue   two warps per TMEM lane quadrant (warp & 3), each takes one half of the tile's
//                   columns: TMEM -> registers (8 columns at a time, software-pipelined) ->
//                   statistics, store / pool.  A rolled loop over 8-column sample groups: the
//                   fully unrolled 128-column epilogue of round 1 was 1,500 straight-line
//                   instructions per tile and spent 35 % of its issue slots waiting for
//                   instruction fetch (ncu, profiles/r02/ncu_sa1_fwd_pooled_epilogue.txt)
//   8    MMA issue  one elected thread
//   9-15 producers  global loads (batched) -> BN+ReLU / gather -> TF32 -> swizzled smem tile
// Two smem stages for the X tile and two TMEM stages for the accumulator, mbarrier hand-offs
// (full / empty / mma_done / d_free): producers run up to two tiles ahead of the tensor core and
// the epilogue's stores trail behind, so HBM reads, MMAs and HBM writes of different tiles overlap.
constexpr int kFwdEpiThreads = 256, kFwdProdThreads = 224, kFwdMmaWarp = 8;
constexpr int kFwdThreads = kFwdEpiThreads + 32 + kFwdProdThreads;   // 512

struct FwdSmem {
  uint32_t w_off, w_bytes, x_off[2], x_bytes, raw_off[2], raw_bytes, scale_off, idx_off, cen_off,
      bar_off, total;
};
// raw_cin > 0 (dense layers): two raw staging buffers of NT x raw_cin fp32, filled by TMA bulk
// copies two tiles ahead, so the producers never wait on a global load
// cmp: compacted position space -- per-row centre ids for the producers (NT ints), a two-stage
// ring of them for the pooling epilogue (2 NT ints) and a copy of the plan's meta words (8 ints)
__host__ __device__ inline FwdSmem fwd_smem_layout(int Kp, int Cout_pad, int NT, int raw_cin,
                                                   int cmp = 0) {
  FwdSmem s;
  const uint32_t KA = (uint32_t)(Kp + 31) >> 5;
  s.w_off = 0;
  s.w_bytes = (uint32_t)Cout_pad * KA * 128u;
  s.x_bytes = (uint32_t)NT * KA * 128u;
  s.x_off[0] = s.w_bytes;
  s.x_off[1] = s.w_bytes + s.x_bytes;
  s.raw_bytes = (uint32_t)NT * raw_cin * 4u;
  s.raw_off[0] = s.x_off[1] + s.x_bytes;
  s.raw_off[1] = s.raw_off[0] + s.raw_bytes;
  s.scale_off = s.raw_off[1] + s.raw_bytes;
  s.idx_off = s.scale_off + 2u * Kp * 4u;
  s.cen_off = s.idx_off + (uint32_t)NT * 4u;
  s.bar_off = (s.cen_off + (cmp ? 3u * (uint32_t)NT * 4u + 32u : 0u) + 15u) & ~15u;
  s.total = s.bar_off + 11 * 8 + 16 + 1024;   // + alignment slack
  return s;
}
__device__ __forceinline__ void fwd_bar_epi() {
  asm volatile("bar.sync 1, %0;" ::"n"(kFwdEpiThreads));
}
__device__ __forceinline__ void fwd_bar_prod() {
  asm volatile("bar.sync 2, %0;" ::"n"(kFwdProdThreads));
}
__device__ __forceinline__ void mbar_arrive1(uint32_t bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(bar) : "memory");
}

// NT = positions per tile (MMA N); MT = Cout_pad / 128 accumulator M tiles (1 or 2).
// CMP: positions are those of a b2r_compact_plan (csrc/compact.cu): the tile count comes from
// the plan's meta words on the device, gather rows from cidx / ccen, and the epilogue works on
// 8-column sample groups whose class (8/16/32/64 samples per centre), liveness and first-sample
// weight are per-TILE constants.
// SL: a channel-slice launch (ldz / ldf / accumulate); the whole-layer instantiations keep the
// arithmetic and addressing they had before slices existed
template <int NT, bool CMP, bool SL>
__global__ void __launch_bounds__(kFwdThreads, 1) sa_layer_fwd_kernel(const LayerArgs a) {
  extern __shared__ __align__(1024) uint8_t smem_raw[];
  uint8_t *base = reinterpret_cast<uint8_t *>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) &
                                              ~(uintptr_t)1023);
  const FwdSmem L = fwd_smem_layout(a.Kp, a.Cout_pad, NT, a.raw_stage ? a.Cin : 0, CMP ? 1 : 0);
  uint8_t *s_w = base + L.w_off;
  float *s_scale = reinterpret_cast<float *>(base + L.scale_off);
  float *s_shift = s_scale + a.Kp;
  int *s_idx = reinterpret_cast<int *>(base + L.idx_off);
  int *s_cenp = reinterpret_cast<int *>(base + L.cen_off);   // CMP: producers' centre per row
  int *s_cene = s_cenp + NT;                                 // CMP: pooling epilogue's, 2 stages
  int *s_meta = s_cene + 2 * NT;                             // CMP: plan meta words 0..7
  uint64_t *s_bar = reinterpret_cast<uint64_t *>(base + L.bar_off);
  uint32_t *s_tmem = reinterpret_cast<uint32_t *>(s_bar + 11);
  // mbarriers: [0,1] full  [2,3] empty  [4,5] mma_done  [6,7] d_free  [8] weights  [9,10] raw
  auto bar = [&](int i) { return smem_u32(&s_bar[i]); };

  const int tid = threadIdx.x, warp = tid >> 5, lane = tid & 31;
  const int MT = a.Cout_pad >> 7;
  const int ldz = SL ? a.ldz : a.Cout;
  constexpr int NCH = NT / 32;
  constexpr uint32_t kTmemCols = 512;
  const int grid = (int)gridDim.x;
  int num_tiles = a.num_tiles;
  if constexpr (CMP) {
    num_tiles = __ldg(a.cmeta + 8) / NT;
    if (tid < 8) s_meta[tid] = __ldg(a.cmeta + tid);
  }

  if (tid == 0) {
    for (int i = 0; i < 11; ++i) mbar_init(bar(i), 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == kFwdMmaWarp) tmem_alloc(smem_u32(s_tmem), kTmemCols);
  for (uint32_t i = tid * 16; i < 2u * L.x_bytes; i += kFwdThreads * 16)   // padding stays zero
    *reinterpret_cast<uint4 *>(base + L.x_off[0] + i) = make_uint4(0, 0, 0, 0);
  if (a.mode == 1)
    for (int i = tid; i < a.Cin; i += kFwdThreads) {
      s_scale[i] = a.scale_prev[i];
      s_shift[i] = a.shift_prev[i];
    }
  fence_async_smem();
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *s_tmem;
  if (tid == 0) {  // TMA unit stages the whole pre-swizzled weight image
    mbar_expect_tx(bar(8), L.w_bytes);
    bulk_g2s(smem_u32(s_w), a.w_image, L.w_bytes, bar(8));
  }

  if (warp > kFwdMmaWarp) {
    // =============================== PRODUCERS ==================================================
    const int ptid = tid - (kFwdEpiThreads + 32);
    const long long per_scene = (long long)a.NP * a.NS;
    GatherSrc gsrc;
    gsrc.xyz = a.xyz; gsrc.new_xyz = a.new_xyz; gsrc.feat_t = a.feat_t;
    gsrc.N = a.N; gsrc.NP = a.NP; gsrc.NS = a.NS; gsrc.C = a.Cin - 3;
    gsrc.Cf4 = (a.Cin - 3 + 3) & ~3;
    gsrc.ldf = SL ? a.ldf : gsrc.C; gsrc.chf_shift = a.chf_shift; gsrc.radius = a.radius; gsrc.normalize_xyz = a.normalize_xyz;
    if (a.raw_stage && ptid == 0) {   // prime the raw ring with this CTA's first two tiles
      for (int k = 0; k < 2; ++k) {
        const long long tile = (long long)blockIdx.x + (long long)k * grid;
        if (tile < num_tiles) {
          mbar_expect_tx(bar(9 + k), L.raw_bytes);
          bulk_g2s(smem_u32(base + L.raw_off[k]), a.z_prev + (size_t)(tile * NT) * a.Cin,
                   L.raw_bytes, bar(9 + k));
        }
      }
    }
    int nidx = 0, ncen = 0;   // prefetched ball-query index (centre) of the next tile
    for (int k = 0, tile = blockIdx.x; tile < num_tiles; tile += grid, ++k) {
      const int s = k & 1, n = k >> 1;
      mbar_wait(bar(2 + s), (uint32_t)((n & 1) ^ 1));   // MMAs of tile k-2 are done with stage s
      const long long pos0 = (long long)tile * NT;
      uint8_t *sx = base + L.x_off[s];
      if (CMP && a.mode == 0) {
        if (ptid < NT) {
          s_idx[ptid] = (k == 0) ? a.cidx[pos0 + ptid] : nidx;
          s_cenp[ptid] = (k == 0) ? a.ccen[pos0 + ptid] : ncen;
          if (tile + grid < num_tiles) {
            nidx = __ldg(a.cidx + pos0 + (long long)grid * NT + ptid);
            ncen = __ldg(a.ccen + pos0 + (long long)grid * NT + ptid);
          }
        }
        fwd_bar_prod();
        build_x_gather<NT, kFwdProdThreads>(gsrc, 0, 0, s_idx, sx, ptid,
                                            [](int row, int ch) { return sw128_off(row, ch, NT); },
                                            s_cenp);
      } else if (a.mode == 0) {
        // ball-query indices of this tile were requested one tile ago (nidx): the gathers below
        // start without waiting on a dependent global load
        if (ptid < NT) {
          s_idx[ptid] = (k == 0) ? a.idx[pos0 + ptid] : nidx;
          if (tile + grid < num_tiles) nidx = __ldg(a.idx + pos0 + (long long)grid * NT + ptid);
        }
        fwd_bar_prod();
        const int b = (int)(pos0 / per_scene);
        const int in_scene0 = (int)(pos0 - (long long)b * per_scene);
        build_x_gather<NT, kFwdProdThreads>(gsrc, b, in_scene0, s_idx, sx, ptid,
                                            [](int row, int ch) { return sw128_off(row, ch, NT); });
      } else if (a.raw_stage) {
        // dense layer, TMA-staged: the tile (one contiguous block of z_prev) was bulk-copied into
        // raw[s] two tiles ago; producers only transform smem -> smem (BN + ReLU + TF32 + swizzle)
        const int CH = a.Cin >> 2;
        const int total = NT * CH;
        const int chs = (CH & (CH - 1)) == 0 ? 31 - __clz(CH) : -1;   // log2(CH) or -1
        mbar_wait(bar(9 + s), (uint32_t)(n & 1));
        const float4 *src = reinterpret_cast<const float4 *>(base + L.raw_off[s]);
        for (int i = ptid; i < total; i += kFwdProdThreads) {
          const float4 t = src[i];
          const int row = chs >= 0 ? (i >> chs) : (i / CH), ch = i - row * CH;
          const float4 sc = *reinterpret_cast<const float4 *>(s_scale + ch * 4);
          const float4 sh = *reinterpret_cast<const float4 *>(s_shift + ch * 4);
          uint4 out;
          out.x = to_tf32(fmaxf(fmaf(t.x, sc.x, sh.x), 0.f));
          out.y = to_tf32(fmaxf(fmaf(t.y, sc.y, sh.y), 0.f));
          out.z = to_tf32(fmaxf(fmaf(t.z, sc.z, sh.z), 0.f));
          out.w = to_tf32(fmaxf(fmaf(t.w, sc.w, sh.w), 0.f));
          *reinterpret_cast<uint4 *>(sx + sw128_off(row, ch, NT)) = out;
        }
      } else {
        // dense layer, register-staged fallback (operands too large for the raw buffers):
        // 8 independent 16-byte loads per thread in flight, tile k+2 prefetched into L2
        const int CH = a.Cin >> 2;
        const int total = NT * CH;
        const int chs = (CH & (CH - 1)) == 0 ? 31 - __clz(CH) : -1;
        if (ptid == 0 && tile + 2 * grid < num_tiles)
          prefetch_l2(a.z_prev + (size_t)(pos0 + 2ll * grid * NT) * a.Cin, (uint32_t)total * 16u);
        const float4 *src = reinterpret_cast<const float4 *>(a.z_prev + (size_t)pos0 * a.Cin);
        for (int i0 = ptid; i0 < total; i0 += kFwdProdThreads * 8) {
          float4 t[8];
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int i = i0 + u * kFwdProdThreads;
            if (i < total) t[u] = __ldg(src + i);
          }
#pragma unroll
          for (int u = 0; u < 8; ++u) {
            const int i = i0 + u * kFwdProdThreads;
            if (i < total) {
              const int row = chs >= 0 ? (i >> chs) : (i / CH), ch = i - row * CH;
              const float4 sc = *reinterpret_cast<const float4 *>(s_scale + ch * 4);
              const float4 sh = *reinterpret_cast<const float4 *>(s_shift + ch * 4);
              uint4 out;
              out.x = to_tf32(fmaxf(fmaf(t[u].x, sc.x, sh.x), 0.f));
              out.y = to_tf32(fmaxf(fmaf(t[u].y, sc.y, sh.y), 0.f));
              out.z = to_tf32(fmaxf(fmaf(t[u].z, sc.z, sh.z), 0.f));
              out.w = to_tf32(fmaxf(fmaf(t[u].w, sc.w, sh.w), 0.f));
              *reinterpret_cast<uint4 *>(sx + sw128_off(row, ch, NT)) = out;
            }
          }
        }
      }
      fence_async_smem();   // generic-proxy accesses ordered before the async proxy (MMA, TMA)
      fwd_bar_prod();
      if (ptid == 0) {
        mbar_arrive1(bar(0 + s));
        if (a.raw_stage && tile + 2 * grid < num_tiles) {   // refill raw[s] with tile k+2
          mbar_expect_tx(bar(9 + s), L.raw_bytes);
          bulk_g2s(smem_u32(base + L.raw_off[s]),
                   a.z_prev + (size_t)(pos0 + 2ll * grid * NT) * a.Cin, L.raw_bytes, bar(9 + s));
        }
      }
    }
  } else if (warp == kFwdMmaWarp) {
    // =============================== MMA ISSUE (one thread) =====================================
    if (lane == 0) {
      mbar_wait(bar(8), 0);
      const uint32_t wa = smem_u32(s_w);
      const int KS = (a.Kp + 7) >> 3;  // K = 8 slices actually issued
      const uint32_t idesc = idesc_tf32(NT);
      for (int k = 0, tile = blockIdx.x; tile < num_tiles; tile += grid, ++k) {
        const int s = k & 1, n = k >> 1;
        const uint32_t xa = smem_u32(base + L.x_off[s]);
        mbar_wait(bar(0 + s), (uint32_t)(n & 1));          // X tile of tile k is in smem
        mbar_wait(bar(6 + s), (uint32_t)((n & 1) ^ 1));    // epilogue of tile k-2 left D[s]
        tc_fence_after();
        for (int m = 0; m < MT; ++m)
          for (int ks = 0; ks < KS; ++ks) {
            const uint32_t koff = (uint32_t)(ks >> 2) * 1024u;
            const uint64_t da = smem_desc_sw128(wa + koff * (uint32_t)(a.Cout_pad >> 3) +
                                                (uint32_t)m * 16u * 1024u + (uint32_t)(ks & 3) * 32u);
            const uint64_t db =
                smem_desc_sw128(xa + koff * (uint32_t)(NT >> 3) + (uint32_t)(ks & 3) * 32u);
            umma_tf32(tmem_base + (uint32_t)((s * MT + m) * NT), da, db, idesc, ks > 0 ? 1u : 0u);
          }
        umma_commit(bar(4 + s));   // -> epilogue
        umma_commit(bar(2 + s));   // -> producers: stage s may be overwritten
      }
    }
    __syncwarp();
  } else {
    // =============================== EPILOGUE (8 warps) =========================================
    const int q = warp & 3, h = warp >> 2;
    const uint32_t lane_addr = (uint32_t)(q * 32) << 16;
    double acc_s[2] = {0.0, 0.0}, acc_ss[2] = {0.0, 0.0};
    // the quadrant's two warps take one half of the tile's columns each -- whole centres when
    // NT/2 >= nsample (a centre's running max must stay in one thread); otherwise warp h = 0 pools
    // the whole tile alone.  Storing layers (epilogue 0) always split.
    constexpr int kGroups = NT / 8;   // 8-column sample groups per tile
    const bool split = a.epilogue == 0 || NT / 2 >= a.NS;
    const int sg_begin = split ? h * (kGroups / 2) : 0;
    const int sg_end = split ? sg_begin + kGroups / 2 : (h == 0 ? kGroups : 0);
    int ncen_e = -1;   // CMP pooling: centre of this thread's column in the NEXT tile
    if constexpr (CMP) {
      if (a.epilogue == 1) {
        if (tid < NT)
          s_cene[tid] = ((int)blockIdx.x < num_tiles) ? a.ccen[(long long)blockIdx.x * NT + tid] : -1;
        fwd_bar_epi();
      }
    }
    for (int k = 0, tile = blockIdx.x; tile < num_tiles; tile += grid, ++k) {
      const int s = k & 1, n = k >> 1;
      const long long pos0 = (long long)tile * NT;
      // per-tile class: samples per centre, live rows, extra weight of a centre's first sample
      // (padded position space: the block's nsample, every row live, no extra weight)
      TileClass tc;
      tc.ns = a.NS; tc.live = NT; tc.wx = 0.f;
      if constexpr (CMP) {
        tc = tile_class(s_meta, pos0, a.NS);
        if (a.epilogue == 1 && tid < NT && tile + grid < num_tiles)
          ncen_e = __ldg(a.ccen + pos0 + (long long)grid * NT + tid);
      }
      const int nsm = tc.ns - 1;
      const int p64 = (int)(pos0 & 63);
      mbar_wait(bar(4 + s), (uint32_t)(n & 1));
      tc_fence_after();
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        if (m >= MT) continue;
        const int c = m * 128 + q * 32 + lane;   // output channel owned by this thread
        const bool c_ok = c < a.Cout;
        float ts = 0.f, tss = 0.f;
        // running max / min (+ sample index) of the current centre, as TWO independent chains
        // (even / odd columns) merged at the centre's end: the epilogue is bound by the latency
        // of these dependent compare-select chains, not by issue slots
        float mx = 0.f, mn = 0.f, mx1 = 0.f, mn1 = 0.f;
        int ax = 0, an = 0, ax1 = 0, an1 = 0;
        const uint32_t t0 = tmem_base + lane_addr + (uint32_t)((s * MT + m) * NT);
        // one 8-column sample group: wholly live or wholly dead, inside one centre; the centre's
        // first sample stands for its NS - ns pad copies as well (weight 1 + wx)
        auto process = [&](uint32_t (&r)[8], int sg) {
          if (!c_ok) return;
          const int col0 = sg * 8;
          if (a.epilogue == 0) {   // dead rows are stored too: later layers must read finite z
            float *zp = a.z + (size_t)(pos0 + col0) * ldz + c;
            if constexpr (SL) {
              if (a.accumulate) {   // earlier feature slices' partial z first, then this product
#pragma unroll
                for (int i = 0; i < 8; ++i)
                  r[i] = __float_as_uint(zp[(size_t)i * ldz] + __uint_as_float(r[i]));
              }
            }
#pragma unroll
            for (int i = 0; i < 8; ++i) zp[(size_t)i * ldz] = __uint_as_float(r[i]);
          }
          if (col0 >= tc.live) return;
          const int s0 = (p64 + col0) & nsm;
          float t = 0.f, tt = 0.f, tb = 0.f, ttb = 0.f;
#pragma unroll
          for (int i = 0; i < 8; i += 2) {
            const float x = __uint_as_float(r[i]), y = __uint_as_float(r[i + 1]);
            t += x;
            tt = fmaf(x, x, tt);
            tb += y;
            ttb = fmaf(y, y, ttb);
          }
          t += tb;
          tt += ttb;
          if (CMP && s0 == 0) {
            const float x0 = __uint_as_float(r[0]);
            t = fmaf(tc.wx, x0, t);
            tt = fmaf(tc.wx * x0, x0, tt);
          }
          ts += t;
          tss += tt;
          if (a.epilogue == 1) {
            // max AND min over the centre's samples with strict compares: the first extremum
            // wins, like max_pool2d
            if (s0 == 0) {
              mx = mx1 = -INFINITY; mn = mn1 = INFINITY; ax = an = ax1 = an1 = 0;
            }
#pragma unroll
            for (int i = 0; i < 8; i += 2) {
              const float x = __uint_as_float(r[i]), y = __uint_as_float(r[i + 1]);
              if (x > mx) { mx = x; ax = s0 + i; }
              if (x < mn) { mn = x; an = s0 + i; }
              if (y > mx1) { mx1 = y; ax1 = s0 + i + 1; }
              if (y < mn1) { mn1 = y; an1 = s0 + i + 1; }
            }
            if (s0 + 8 == tc.ns) {
              // merge the two chains: larger value wins, equal values -> the earlier sample
              if (mx1 > mx || (mx1 == mx && ax1 < ax)) { mx = mx1; ax = ax1; }
              if (mn1 < mn || (mn1 == mn && an1 < an)) { mn = mn1; an = an1; }
              long long centre;
              if constexpr (CMP) centre = s_cene[(k & 1) * NT + col0];
              else centre = (pos0 + col0) >> a.ns_shift;
              if (centre >= 0) {
                const size_t o = (size_t)centre * ldz + c;
                a.zmax[o] = mx; a.zmin[o] = mn; a.amax[o] = ax; a.amin[o] = an;
              }
            }
          }
        };
        // software-pipelined TMEM loads: group sg+1 is in flight while group sg is processed
        uint32_t ra[8], rb[8];
        if (sg_begin < sg_end) cuda::ptx::tcgen05_ld_32x32b(ra, t0 + (uint32_t)(sg_begin * 8));
#pragma unroll 1
        for (int sg = sg_begin; sg < sg_end; sg += 2) {
          asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
          if (sg + 1 < sg_end) cuda::ptx::tcgen05_ld_32x32b(rb, t0 + (uint32_t)((sg + 1) * 8));
          process(ra, sg);
          if (sg + 1 < sg_end) {
            asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
            if (sg + 2 < sg_end) cuda::ptx::tcgen05_ld_32x32b(ra, t0 + (uint32_t)((sg + 2) * 8));
            process(rb, sg + 1);
          }
        }
        acc_s[m] += (double)ts;
        acc_ss[m] += (double)tss;
      }
      if constexpr (CMP) {
        if (a.epilogue == 1 && tid < NT) s_cene[((k + 1) & 1) * NT + tid] = ncen_e;
      }
      tc_fence_before();
      fwd_bar_epi();   // every epilogue thread has read D[s]
      if (tid == 0) mbar_arrive1(bar(6 + s));
    }
    if (a.stats != nullptr) {
#pragma unroll
      for (int m = 0; m < 2; ++m) {
        const int c = m * 128 + q * 32 + lane;
        if (m < MT && c < a.Cout) {
          atomicAdd(a.stats + c, acc_s[m]);
          atomicAdd(a.stats + ldz + c, acc_ss[m]);
        }
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == kFwdMmaWarp) tmem_dealloc(tmem_base, kTmemCols);
}

// BatchNorm bookkeeping from the accumulated statistics (one thread per channel):
//   scale = gamma / sqrt(var_biased + eps), shift = beta - mean * scale        (training)
//   running_mean/var updated with `momentum` (unbiased variance), like nn.BatchNorm2d
// kDevMomentum: the momentum is read from device memory (*momentum_dev) when the kernel runs, so a
// replayed CUDA graph follows a momentum schedule; otherwise it is the by-value `momentum`.
template <bool kDevMomentum>
__global__ void bn_finalize_kernel(const double *__restrict__ stats, int Cch, double inv_count,
                                   float unbias,
                                   const float *__restrict__ gamma, const float *__restrict__ beta,
                                   float eps, float momentum_val,
                                   const float *__restrict__ momentum_dev,
                                   float *__restrict__ running_mean,
                                   float *__restrict__ running_var, float *__restrict__ scale,
                                   float *__restrict__ shift, float *__restrict__ mean_out,
                                   float *__restrict__ invstd_out,
                                   long long *__restrict__ num_batches_tracked) {
  const int ch = blockIdx.x * blockDim.x + threadIdx.x;
  if (ch == 0 && num_batches_tracked != nullptr) *num_batches_tracked += 1;
  if (ch >= Cch) return;
  // FP64 only where cancellation needs it (mean, E[z^2] - mean^2): two multiplies and one FMA.
  // Divisions and the square root in double cost ~2 us of this single-CTA kernel on B200's few
  // FP64 lanes, and it sits between two dependent layer kernels 23 times per step.
  // (1/count and count/(count-1) come from the host.)
  const double mean = stats[ch] * inv_count;
  double var = fma(stats[Cch + ch], inv_count, -mean * mean);
  if (var < 0.0) var = 0.0;
  const float invstd = 1.0f / sqrtf((float)var + eps);
  const float g = gamma ? gamma[ch] : 1.f, bta = beta ? beta[ch] : 0.f;
  scale[ch] = g * invstd;
  shift[ch] = bta - (float)mean * g * invstd;
  if (mean_out) mean_out[ch] = (float)mean;
  if (invstd_out) invstd_out[ch] = invstd;
  if (running_mean) {
    const float momentum = kDevMomentum ? *momentum_dev : momentum_val;
    const float unbiased = (float)var * unbias;
    running_mean[ch] = (1.f - momentum) * running_mean[ch] + momentum * (float)mean;
    running_var[ch] = (1.f - momentum) * running_var[ch] + momentum * unbiased;
  }
}

// out = relu(scale * (scale >= 0 ? zmax : zmin) + shift), written channel-major (B,C,NP) for the
// reference API and point-major (B,NP,C) for the next layer's gather.  One 32 x 32 (centre,
// channel) tile per CTA, transposed through shared memory so that BOTH layouts are read and
// written with 128-byte coalesced rows.
__global__ void pool_finalize_kernel(const float *__restrict__ zmax, const float *__restrict__ zmin,
                                     const float *__restrict__ scale,
                                     const float *__restrict__ shift, int NP, int Cch,
                                     float *__restrict__ out_cm, float *__restrict__ out_pm) {
  __shared__ float t[32][33];
  const int b = blockIdx.z;
  const int j0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int ch = c0 + threadIdx.x;
  const float s = ch < Cch ? scale[ch] : 0.f, sh = ch < Cch ? shift[ch] : 0.f;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int j = j0 + i;
    float y = 0.f;
    if (j < NP && ch < Cch) {
      const size_t e = ((size_t)b * NP + j) * Cch + ch;
      const float z = s >= 0.f ? zmax[e] : zmin[e];
      y = fmaxf(fmaf(z, s, sh), 0.f);
      if (out_pm) out_pm[e] = y;
    }
    t[i][threadIdx.x] = y;
  }
  if (out_cm == nullptr) return;
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int cc = c0 + i, j = j0 + threadIdx.x;
    if (cc < Cch && j < NP) out_cm[((size_t)b * Cch + cc) * NP + j] = t[threadIdx.x][i];
  }
}

// (B,C,N) channel-major -> (B,N,C) point-major (tile transpose through shared memory)
__global__ void to_point_major_kernel(const float *__restrict__ in, int Cch, int N,
                                      float *__restrict__ out) {
  __shared__ float t[32][33];
  const int b = blockIdx.z;
  const int n0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  in += (size_t)b * Cch * N;
  out += (size_t)b * Cch * N;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int cc = c0 + i, n = n0 + threadIdx.x;
    t[i][threadIdx.x] = (cc < Cch && n < N) ? in[(size_t)cc * N + n] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int n = n0 + i, cc = c0 + threadIdx.x;
    if (n < N && cc < Cch) out[(size_t)n * Cch + cc] = t[threadIdx.x][i];
  }
}

}  // namespace
}  // namespace b2r

using namespace b2r;

extern "C" long long b2r_mlp_weight_image_bytes(int Cout, int Cin, int gather) {
  if (Cout <= 0 || Cin <= 0) return 0;
  const int Kp = packed_k(Cin, gather);
  const int KA = (Kp + 31) >> 5;
  const int Cout_pad = (Cout + 127) & ~127;
  return (long long)Cout_pad * KA * 128;
}

extern "C" int b2r_mlp_pack_weight(const float *w, int Cout, int Cin, int gather, float *image,
                                   void *stream) {
  B2R_REQUIRE(w && image && Cout > 0 && Cin > 0, "b2r_mlp_pack_weight: bad argument");
  B2R_REQUIRE(!gather || Cin >= 3, "b2r_mlp_pack_weight: gather layers need Cin >= 3");
  const int Kp = packed_k(Cin, gather);
  const int KA = (Kp + 31) >> 5;
  const int Cout_pad = (Cout + 127) & ~127;
  const long long total = (long long)Cout_pad * KA * 32;
  pack_weight_kernel<<<ceil_div(total, 256), 256, 0, static_cast<cudaStream_t>(stream)>>>(
      w, Cout, Cin, gather, Kp, Cout_pad, image);
  B2R_CHECK_LAUNCH();
  return B2R_OK;
}

namespace {
// positions per tile for one forward launch (0 = does not fit) and whether dense tiles are
// TMA-staged: the widest tile whose two smem stages + two TMEM stages fit; a gather tile must lie
// inside one scene and a pooling tile must hold whole centres
int fwd_pick_nt(int Kp, int Cout_pad, int Cin, int mode, int epilogue, int NS, long long M,
                long long per_scene, int *raw_stage, int cmp = 0) {
  const int MT = Cout_pad >> 7;
  for (int raw = (mode == 1 ? 1 : 0); raw >= 0; --raw)
    for (int nt : {128, 64, 32}) {
      if (M % nt) continue;
      if (!cmp && mode == 0 && per_scene % nt) continue;   // (a plan's tiles hold global rows)
      if (epilogue == 1 && (nt % NS) != 0) continue;
      if (raw && nt < 64) continue;   // prefer wider register-staged tiles over tiny TMA ones
      const FwdSmem L = fwd_smem_layout(Kp, Cout_pad, nt, raw ? Cin : 0, cmp);
      if (L.total <= 227u * 1024u && 2 * MT * nt <= 512) {
        *raw_stage = raw;
        return nt;
      }
    }
  *raw_stage = 0;
  return 0;
}

// whether ONE launch can hold a layer of these channel counts at all: the narrowest tile (32
// positions, register-staged) within shared memory and TMEM; compact: with a plan's extra words
bool fwd_fits(int Cin, int Cout, int gather, int cmp) {
  if (Cout > 256) return false;
  const int Cout_pad = (Cout + 127) & ~127;
  const FwdSmem L = fwd_smem_layout(packed_k(Cin, gather), Cout_pad, 32, 0, cmp);
  return L.total <= 227u * 1024u && 2 * (Cout_pad >> 7) * 32 <= 512;
}
}  // namespace

// Slice grid (include/b2r.h).  A layer that fits one launch keeps it.  Otherwise output slices of
// 256 or 128 channels, and for gather layers (not pooled) feature slices of C/2, C/4, ... channels
// (multiples of 8), checked with the plan's extra shared memory: the grid with the fewest launches,
// then the fewest feature slices (each one after the first re-reads z).
extern "C" int b2r_sa_layer_fwd_slices(int Cin, int Cout, int gather, int pooled, int *co_step,
                                       int *ci_step) {
  if (Cin <= 0 || Cout <= 0 || (gather && Cin < 3) || (!gather && (Cin % 4) != 0)) return 0;
  int best = 0, best_kn = 0, bco = 0, bci = 0;
  if (fwd_fits(Cin, Cout, gather, 0)) {
    best = 1; bco = Cout; bci = 0;
  } else if (Cout % 8 == 0) {
    const int C = Cin - 3;
    for (int cs : {256, 128}) {
      const int co = cs < Cout ? cs : Cout;
      for (int kn = 1; kn <= 16; kn *= 2) {
        int ci = 0;
        if (kn > 1) {
          if (!gather || pooled || C % 8 != 0) break;
          ci = ((C + kn - 1) / kn + 7) & ~7;
          if (ci * (kn - 1) >= C) continue;
        }
        if (!fwd_fits(kn > 1 ? 3 + ci : Cin, co, gather, 1)) continue;
        const int n = ((Cout + co - 1) / co) * (kn > 1 ? (C + ci - 1) / ci : 1);
        if (best == 0 || n < best || (n == best && kn < best_kn)) {
          best = n; best_kn = kn; bco = co; bci = ci;
        }
        break;   // more feature slices only add launches at this output width
      }
    }
  }
  if (co_step) *co_step = bco;
  if (ci_step) *ci_step = bci;
  return best;
}

extern "C" int b2r_sa_layer_fwd_supported(int B, int NP, int NS, int Cin, int Cout, int gather,
                                          int pooled) {
  if (B <= 0 || NP <= 0 || NS <= 0 || Cin <= 0 || Cout <= 0) return 0;
  if (gather ? Cin < 3 : (Cin % 4) != 0) return 0;
  if (pooled && !(NS == 16 || NS == 32 || NS == 64)) return 0;
  int co = 0, ci = 0;
  if (b2r_sa_layer_fwd_slices(Cin, Cout, gather, pooled, &co, &ci) == 0) return 0;
  const int Cin_s = ci > 0 ? 3 + ci : Cin;   // the widest slice decides the tile
  const long long per_scene = (long long)NP * NS, M = (long long)B * per_scene;
  int raw = 0;
  return fwd_pick_nt(packed_k(Cin_s, gather), (co + 127) & ~127, Cin_s, gather ? 0 : 1,
                     pooled ? 1 : 0, NS, M, per_scene, &raw) > 0 ? 1 : 0;
}

extern "C" int b2r_sa_layer_fwd_tile(int B, int NP, int NS, int Cin, int Cout, int gather,
                                     int pooled, int compact) {
  if (B <= 0 || NP <= 0 || NS <= 0 || Cin <= 0 || Cout <= 0 || Cout > 256) return 0;
  const long long per_scene = (long long)NP * NS;
  const long long M = compact ? b2r_compact_capacity(B, NP, NS) : (long long)B * per_scene;
  int raw = 0;
  return fwd_pick_nt(packed_k(Cin, gather), (Cout + 127) & ~127, Cin, gather ? 0 : 1,
                     pooled ? 1 : 0, NS, M, per_scene, &raw, compact ? 1 : 0);
}

extern "C" int b2r_sa_layer_fwd(const b2r_sa_layer *d, void *stream) {
  B2R_REQUIRE(d != nullptr, "b2r_sa_layer_fwd: null descriptor");
  B2R_REQUIRE(d->B > 0 && d->NP > 0 && d->NS > 0 && d->Cin > 0 && d->Cout > 0,
              "b2r_sa_layer_fwd: non-positive size");
  B2R_REQUIRE(d->mode == 0 || d->mode == 1, "b2r_sa_layer_fwd: mode must be 0 or 1");
  B2R_REQUIRE(d->epilogue == 0 || d->epilogue == 1, "b2r_sa_layer_fwd: epilogue must be 0 or 1");
  B2R_REQUIRE(d->w_image != nullptr, "b2r_sa_layer_fwd: null weight image");
  const bool co_sliced = d->co_n != 0, ci_sliced = d->ci_n != 0;
  B2R_REQUIRE(co_sliced ? (d->co0 >= 0 && d->co_n > 0 && d->co0 <= d->Cout - d->co_n)
                        : d->co0 == 0,
              "b2r_sa_layer_fwd: output slice [%d, +%d) outside Cout=%d", d->co0, d->co_n, d->Cout);
  B2R_REQUIRE(!ci_sliced || (d->mode == 0 && d->epilogue == 0),
              "b2r_sa_layer_fwd: feature slices are for gather layers that store z");
  B2R_REQUIRE(ci_sliced ? (d->ci0 >= 0 && d->ci_n > 0 && d->ci0 <= d->Cin - 3 - d->ci_n &&
                           d->ci0 % 8 == 0 && d->ci_n % 8 == 0)
                        : d->ci0 == 0,
              "b2r_sa_layer_fwd: feature slice [%d, +%d) outside the %d features or not a "
              "multiple of 8", d->ci0, d->ci_n, d->Cin - 3);
  B2R_REQUIRE(!d->accumulate || (d->accumulate == 1 && d->epilogue == 0),
              "b2r_sa_layer_fwd: accumulate is 0, or 1 for a layer that stores z");
  const int Cout_s = co_sliced ? d->co_n : d->Cout;
  const int Cin_s = ci_sliced ? 3 + d->ci_n : d->Cin;
  LayerArgs a;
  // a slice launch: the kernel sees a layer of Cin_s -> Cout_s channels whose outputs sit at
  // column co0 of the whole layer's rows and whose features start at column ci0 of feat_t's rows
  const int co0 = d->co0;
  a.B = d->B; a.N = d->N; a.NP = d->NP; a.NS = d->NS; a.Cin = Cin_s; a.Cout = Cout_s;
  a.mode = d->mode; a.epilogue = d->epilogue;
  a.xyz = d->xyz; a.new_xyz = d->new_xyz; a.idx = d->idx;
  a.feat_t = d->feat_t != nullptr ? d->feat_t + d->ci0 : nullptr;
  a.radius = d->radius; a.normalize_xyz = d->normalize_xyz;
  a.z_prev = d->z_prev; a.scale_prev = d->scale_prev; a.shift_prev = d->shift_prev;
  a.w_image = d->w_image;
  a.z = d->z != nullptr ? d->z + co0 : nullptr;
  a.stats = d->stats != nullptr ? d->stats + co0 : nullptr;
  a.zmax = d->zmax != nullptr ? d->zmax + co0 : nullptr;
  a.zmin = d->zmin != nullptr ? d->zmin + co0 : nullptr;
  a.amax = d->amax != nullptr ? d->amax + co0 : nullptr;
  a.amin = d->amin != nullptr ? d->amin + co0 : nullptr;
  a.ldz = d->Cout; a.ldf = d->Cin - 3; a.accumulate = d->accumulate;
  a.Kp = packed_k(Cin_s, d->mode == 0);
  a.Cout_pad = (Cout_s + 127) & ~127;
  a.chf_shift = pow2_shift(((Cin_s - 3 + 3) & ~3) >> 2);
  a.ns_shift = pow2_shift(d->NS);
  a.cidx = d->cidx; a.ccen = d->ccen; a.cmeta = d->cmeta;
  const int cmp = d->cmeta != nullptr ? 1 : 0;
  B2R_REQUIRE(!cmp || (d->cidx && d->ccen), "b2r_sa_layer_fwd: a plan needs cidx, ccen and cmeta");
  if (cmp && !(d->NS == 16 || d->NS == 32 || d->NS == 64)) {
    set_error("b2r_sa_layer_fwd: a compacted plan needs nsample 16/32/64 (got %d)", d->NS);
    return B2R_ERR_UNSUPPORTED;
  }
  // with a plan the launch is sized for the plan's CAPACITY; the live tile count is on the device
  const long long M = cmp ? b2r_compact_capacity(d->B, d->NP, d->NS)
                          : (long long)d->B * d->NP * d->NS;
  const long long per_scene = (long long)d->NP * d->NS;
  if (d->mode == 0) {
    B2R_REQUIRE(d->Cin >= 3 && d->xyz && d->new_xyz && (d->idx || cmp) && (d->feat_t || d->Cin == 3),
                "b2r_sa_layer_fwd: gather mode needs xyz, new_xyz, idx (and feat_t when Cin > 3)");
    B2R_REQUIRE(d->Cin == 3 || ((reinterpret_cast<uintptr_t>(d->feat_t) & 15u) == 0),
                "b2r_sa_layer_fwd: feat_t must be 16-byte aligned");
  } else {
    B2R_REQUIRE(d->z_prev && d->scale_prev && d->shift_prev && (d->Cin % 4) == 0,
                "b2r_sa_layer_fwd: dense mode needs z_prev/scale/shift and Cin %% 4 == 0");
  }
  if (d->epilogue == 0) {
    B2R_REQUIRE(d->z != nullptr, "b2r_sa_layer_fwd: epilogue 0 needs z");
  } else {
    B2R_REQUIRE(d->zmax && d->zmin && d->amax && d->amin,
                "b2r_sa_layer_fwd: epilogue 1 needs pool outputs");
    if (!(d->NS == 16 || d->NS == 32 || d->NS == 64)) {
      set_error("b2r_sa_layer_fwd: pooling supports nsample 16/32/64 (got %d)", d->NS);
      return B2R_ERR_UNSUPPORTED;
    }
  }
  if (a.Cout_pad > 256) {
    set_error("b2r_sa_layer_fwd: needs Cout <= 256 per launch (got %d; see "
              "b2r_sa_layer_fwd_slices)", Cout_s);
    return B2R_ERR_UNSUPPORTED;
  }
  // thin first layer (Cin <= 8): a streaming CUDA-core kernel, not a tensor-core tile pipeline
  if (!co_sliced && !ci_sliced && !d->accumulate && thin::fwd_applicable(d))
    return thin::fwd_launch(d, stream);
  const int NT = fwd_pick_nt(a.Kp, a.Cout_pad, Cin_s, d->mode, d->epilogue, d->NS, M, per_scene,
                             &a.raw_stage, cmp);
  if (NT == 0) {
    set_error("b2r_sa_layer_fwd: layer Cin=%d Cout=%d M=%lld NP*NS=%lld does not fit (needs "
              "B*NP*NS %% 32 == 0, gather layers NP*NS %% 32 == 0, operands within 227 KB)",
              Cin_s, Cout_s, M, per_scene);
    return B2R_ERR_UNSUPPORTED;
  }
  const FwdSmem L = fwd_smem_layout(a.Kp, a.Cout_pad, NT, a.raw_stage ? Cin_s : 0, cmp);
  a.num_tiles = (int)(M / NT);
  // persistent grid: one CTA per SM, or fewer when the caller keeps SMs free for kernels running
  // concurrently on another stream (the geometry pre-pass: FPS needs whole SMs to itself)
  int sms = kNumSMs;
  if (d->sm_limit > 0 && d->sm_limit < kNumSMs) sms = d->sm_limit;
  const int grid = a.num_tiles < sms ? a.num_tiles : sms;
  cudaStream_t st = static_cast<cudaStream_t>(stream);
  const bool sliced = co_sliced || ci_sliced || d->accumulate;
#define B2R_LAUNCH_FWD2(NTV, CMPV, SLV)                                                         \
  do {                                                                                          \
    B2R_CUDA(cudaFuncSetAttribute(sa_layer_fwd_kernel<NTV, CMPV, SLV>,                          \
                                  cudaFuncAttributeMaxDynamicSharedMemorySize, (int)L.total));  \
    sa_layer_fwd_kernel<NTV, CMPV, SLV><<<grid, kFwdThreads, L.total, st>>>(a);                 \
  } while (0)
#define B2R_LAUNCH_FWD(NTV, CMPV)                                                               \
  do {                                                                                          \
    if (sliced) B2R_LAUNCH_FWD2(NTV, CMPV, true); else B2R_LAUNCH_FWD2(NTV, CMPV, false);       \
  } while (0)
  if (cmp) {
    if (NT == 128) B2R_LAUNCH_FWD(128, true);
    else if (NT == 64) B2R_LAUNCH_FWD(64, true);
    else B2R_LAUNCH_FWD(32, true);
  } else {
    if (NT == 128) B2R_LAUNCH_FWD(128, false);
    else if (NT == 64) B2R_LAUNCH_FWD(64, false);
    else B2R_LAUNCH_FWD(32, false);
  }
#undef B2R_LAUNCH_FWD
#undef B2R_LAUNCH_FWD2
  B2R_CHECK_LAUNCH();
  return B2R_OK;
}

// the two entries below: same validation, same kernel template, momentum by value or on the device
template <bool kDevMomentum>
static int bn_finalize_launch(const char *name, const double *stats, int C, double count,
                              const float *gamma, const float *beta, float eps, float momentum,
                              const float *momentum_dev, float *running_mean, float *running_var,
                              float *scale, float *shift, float *mean_out, float *invstd_out,
                              long long *num_batches_tracked, void *stream) {
  B2R_REQUIRE(stats && scale && shift && C > 0 && count > 0, "%s: bad argument", name);
  B2R_REQUIRE((running_mean == nullptr) == (running_var == nullptr),
              "%s: running_mean and running_var must both be given or both be NULL", name);
  B2R_REQUIRE(!kDevMomentum || running_mean == nullptr || momentum_dev != nullptr,
              "%s: running statistics given without a momentum pointer", name);
  bn_finalize_kernel<kDevMomentum><<<ceil_div(C, 128), 128, 0, static_cast<cudaStream_t>(stream)>>>(
      stats, C, 1.0 / count, count > 1.0 ? (float)(count / (count - 1.0)) : 1.0f, gamma, beta, eps,
      momentum, momentum_dev, running_mean, running_var, scale, shift,
      mean_out, invstd_out, num_batches_tracked);
  B2R_CHECK_LAUNCH();
  return B2R_OK;
}

extern "C" int b2r_bn_finalize(const double *stats, int C, double count, const float *gamma,
                               const float *beta, float eps, float momentum, float *running_mean,
                               float *running_var, float *scale, float *shift, float *mean_out,
                               float *invstd_out, long long *num_batches_tracked, void *stream) {
  return bn_finalize_launch<false>("b2r_bn_finalize", stats, C, count, gamma, beta, eps, momentum,
                                   nullptr, running_mean, running_var, scale, shift, mean_out,
                                   invstd_out, num_batches_tracked, stream);
}

extern "C" int b2r_bn_finalize_dev(const double *stats, int C, double count, const float *gamma,
                                   const float *beta, float eps, const float *momentum,
                                   float *running_mean, float *running_var, float *scale,
                                   float *shift, float *mean_out, float *invstd_out,
                                   long long *num_batches_tracked, void *stream) {
  return bn_finalize_launch<true>("b2r_bn_finalize_dev", stats, C, count, gamma, beta, eps, 0.f,
                                  momentum, running_mean, running_var, scale, shift, mean_out,
                                  invstd_out, num_batches_tracked, stream);
}

extern "C" int b2r_pool_finalize(const float *zmax, const float *zmin, const float *scale,
                                 const float *shift, int B, int NP, int C, float *out_cm,
                                 float *out_pm, void *stream) {
  B2R_REQUIRE(zmax && zmin && scale && shift && B > 0 && NP > 0 && C > 0,
              "b2r_pool_finalize: bad argument");
  B2R_REQUIRE(B <= 65535, "b2r_pool_finalize: B=%d exceeds gridDim.z", B);
  dim3 grid(ceil_div(NP, 32), ceil_div(C, 32), B), block(32, 8);
  pool_finalize_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(
      zmax, zmin, scale, shift, NP, C, out_cm, out_pm);
  B2R_CHECK_LAUNCH();
  return B2R_OK;
}

extern "C" int b2r_to_point_major(const float *in, int B, int C, int N, float *out, void *stream) {
  B2R_REQUIRE(B >= 0 && C >= 0 && N >= 0, "b2r_to_point_major: negative size");
  if (B == 0 || C == 0 || N == 0) return B2R_OK;
  B2R_REQUIRE(in && out, "b2r_to_point_major: null pointer");
  dim3 grid(ceil_div(N, 32), ceil_div(C, 32), B), block(32, 8);
  to_point_major_kernel<<<grid, block, 0, static_cast<cudaStream_t>(stream)>>>(in, C, N, out);
  B2R_CHECK_LAUNCH();
  return B2R_OK;
}
