// mlp_common.cuh -- device helpers shared by the tcgen05 SharedMLP kernels (mlp.cu, mlp_bwd.cu):
// inline PTX for mbarrier / TMA bulk copy / tcgen05 alloc-mma-commit-fence, shared-memory matrix
// descriptors for the 128-byte-swizzled canonical layouts (K-major and MN-major views of the SAME
// bytes), and the address function of that layout.
#pragma once
#include <cuda/ptx>

#include "common.cuh"

namespace b2r {
namespace mlp {


// ----------------------------------------------------------------------------- PTX helpers --
__device__ __forceinline__ uint32_t to_tf32(float x) {
  uint32_t r;
  asm("cvt.rna.tf32.f32 %0, %1;" : "=r"(r) : "f"(x));
  return r;
}
__device__ __forceinline__ void mbar_init(uint32_t bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(bar), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint32_t bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes)
               : "memory");
}
__device__ __forceinline__ void mbar_wait(uint32_t bar, uint32_t parity) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "MLP_WAIT_%=:\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n\t"
      "@p bra MLP_DONE_%=;\n\t"
      "bra MLP_WAIT_%=;\n\t"
      "MLP_DONE_%=:\n\t"
      "}" ::"r"(bar),
      "r"(parity)
      : "memory");
}
__device__ __forceinline__ void bulk_g2s(uint32_t dst, const void *src, uint32_t bytes,
                                         uint32_t bar) {
  asm volatile(
      "cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::
          "r"(dst),
      "l"(src), "r"(bytes), "r"(bar)
      : "memory");
}
// Ask the L2 to fetch a contiguous block ahead of use (one instruction, no registers, no smem):
// issued by one thread for the NEXT tile while the current one is being processed.
__device__ __forceinline__ void prefetch_l2(const void *p, uint32_t bytes) {
  asm volatile("cp.async.bulk.prefetch.L2.global [%0], %1;" ::"l"(p), "r"(bytes) : "memory");
}
__device__ __forceinline__ void fence_async_smem() {
  asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_before() {
  asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tc_fence_after() {
  asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
}
__device__ __forceinline__ void tmem_alloc(uint32_t smem_dst, uint32_t ncols) {
  asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_dst),
               "r"(ncols)
               : "memory");
  asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
}
__device__ __forceinline__ void tmem_dealloc(uint32_t taddr, uint32_t ncols) {
  asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(taddr), "r"(ncols)
               : "memory");
}
// D[tmem] (+)= A[smem] * B[smem]^T, TF32 operands, FP32 accumulate
__device__ __forceinline__ void umma_tf32(uint32_t d_tmem, uint64_t a_desc, uint64_t b_desc,
                                          uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t"
      ".reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n\t"
      "}" ::"r"(d_tmem),
      "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma_commit(uint32_t bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(
                   bar)
               : "memory");
}

// Shared-memory matrix descriptor, K-major, 128-byte swizzle (canonical layout: 8-row x 128-byte
// atoms, 16-byte chunk index XOR (row & 7); consecutive 8-row groups 1024 B apart = SBO).
__device__ __forceinline__ uint64_t smem_desc_sw128(uint32_t saddr) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fffu);        // start address
  d |= (uint64_t)1 << 16;                         // leading byte offset (unused for SW128 K-major)
  d |= (uint64_t)(1024u >> 4) << 32;              // stride byte offset: 8 rows x 128 B
  d |= (uint64_t)1 << 46;                         // descriptor version (Blackwell)
  d |= (uint64_t)2 << 61;                         // layout type: SWIZZLE_128B
  return d;
}
// kind::tf32 instruction descriptor: F32 accumulate, TF32 A/B, both K-major, M = 128, N = n
__host__ __device__ constexpr uint32_t idesc_tf32(int n) {
  return (1u << 4) | (2u << 7) | (2u << 10) | ((uint32_t)(n >> 3) << 17) | ((128u >> 4) << 24);
}

// The same swizzled bytes seen MN-major (the "transposed" operand view): 128-byte groups of
// contiguous MN elements are `lbo` bytes apart, consecutive 8-deep K groups `sbo` bytes apart.
// Valid for 16-bit operands (BF16: mlp_bwd.cu); 32-bit (TF32) data needs the BASE32B layout
// instead (scripts/probe/umma_probe.cu).
__device__ __forceinline__ uint64_t smem_desc_sw128_mn(uint32_t saddr, uint32_t lbo, uint32_t sbo) {
  uint64_t d = 0;
  d |= (uint64_t)((saddr >> 4) & 0x3fffu);
  d |= (uint64_t)((lbo >> 4) & 0x3fffu) << 16;
  d |= (uint64_t)((sbo >> 4) & 0x3fffu) << 32;
  d |= (uint64_t)1 << 46;
  d |= (uint64_t)2 << 61;
  return d;
}
// byte offset of 16-byte chunk `chunk` (4 consecutive K elements) of row `row` inside a K-major
// SW128 operand with `rows` rows: K-atom (32 elements) major, then 8-row group, then row, chunk
__device__ __forceinline__ uint32_t sw128_off(int row, int chunk, int rows) {
  const int a = chunk >> 3, c = chunk & 7, g = row >> 3, r8 = row & 7;
  return (uint32_t)(((a * (rows >> 3) + g) << 10) + (r8 << 7) + ((c ^ r8) << 4));
}

// packed K extent of a layer: gather mode puts the C feature channels first (padded to a multiple
// of 4 so the xyz chunk is 16-byte aligned), then dx,dy,dz,0; dense mode is K itself (mult. of 4)
__host__ __device__ inline int packed_k(int Cin, int gather) {
  if (!gather) return (Cin + 3) & ~3;
  const int C = Cin - 3;
  return ((C + 3) & ~3) + 4;
}

// ------------------------------------------------------------------ gathered operand tile --
// Layer-0 input rows of one tile, built on the fly (the reference's QueryAndGroup tail,
// pointnet2_utils.py:347-366): packed row = [feature channels (padded to a multiple of 4),
// (xyz[idx] - new_xyz) (/ radius), 0].  All NT positions of a tile lie in ONE scene `b` (the host
// guarantees NP*NS % NT == 0), so no per-element 64-bit division is needed; feature loads are
// issued in batches of 8 independent 16-byte requests per thread.
struct GatherSrc {
  const float *xyz, *new_xyz, *feat_t;
  int N, NP, NS, C, Cf4;
  int ldf;         // row pitch of feat_t: C, or the whole layer's feature count for a slice
  int chf_shift;   // log2(Cf4/4) when that is a power of two, else -1
  float radius;
  int normalize_xyz;
};

// s_cen != nullptr: compacted position space (csrc/compact.cu): s_idx holds GLOBAL source rows
// and s_cen the global centre of every row (-1 = dead padding -> centre 0); pass b = 0.
template <int NT, int NTHREADS, class OffFn>
__device__ __forceinline__ void build_x_gather(const GatherSrc &g, int b, int in_scene0,
                                               const int *s_idx, uint8_t *s_x, int tid,
                                               OffFn off, const int *s_cen = nullptr) {
  const int C = g.C, CHf = g.Cf4 >> 2;
  // relative xyz chunk: one thread per row, six independent loads
  for (int row = tid; row < NT; row += NTHREADS) {
    const int p = s_idx[row];
    const int j = s_cen != nullptr ? max(s_cen[row], 0) : (in_scene0 + row) / g.NS;
    const float *pp = g.xyz + ((size_t)b * g.N + p) * 3;
    const float *qq = g.new_xyz + ((size_t)b * g.NP + j) * 3;
    const float px = __ldg(pp), py = __ldg(pp + 1), pz = __ldg(pp + 2);
    const float qx = __ldg(qq), qy = __ldg(qq + 1), qz = __ldg(qq + 2);
    float d0 = __fsub_rn(px, qx), d1 = __fsub_rn(py, qy), d2 = __fsub_rn(pz, qz);
    if (g.normalize_xyz) {
      d0 = __fdiv_rn(d0, g.radius);
      d1 = __fdiv_rn(d1, g.radius);
      d2 = __fdiv_rn(d2, g.radius);
    }
    *reinterpret_cast<uint4 *>(s_x + off(row, CHf)) =
        make_uint4(to_tf32(d0), to_tf32(d1), to_tf32(d2), 0u);
  }
  if (CHf == 0) return;
  const float *fb = g.feat_t + (size_t)b * g.N * g.ldf;
  const int total = NT * CHf;
  if ((C & 3) == 0) {
    for (int i0 = tid; i0 < total; i0 += NTHREADS * 8) {
      float4 t[8];
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = i0 + u * NTHREADS;
        if (i < total) {
          const int row = g.chf_shift >= 0 ? (i >> g.chf_shift) : (i / CHf);
          const int ch = i - row * CHf;
          t[u] = __ldg(reinterpret_cast<const float4 *>(fb + (size_t)s_idx[row] * g.ldf) + ch);
        }
      }
#pragma unroll
      for (int u = 0; u < 8; ++u) {
        const int i = i0 + u * NTHREADS;
        if (i < total) {
          const int row = g.chf_shift >= 0 ? (i >> g.chf_shift) : (i / CHf);
          const int ch = i - row * CHf;
          *reinterpret_cast<uint4 *>(s_x + off(row, ch)) =
              make_uint4(to_tf32(t[u].x), to_tf32(t[u].y), to_tf32(t[u].z), to_tf32(t[u].w));
        }
      }
    }
  } else {
    for (int i = tid; i < total; i += NTHREADS) {
      const int row = g.chf_shift >= 0 ? (i >> g.chf_shift) : (i / CHf);
      const int ch = i - row * CHf;
      const float *src = fb + (size_t)s_idx[row] * g.ldf + ch * 4;
      float f[4] = {0.f, 0.f, 0.f, 0.f};
#pragma unroll
      for (int e = 0; e < 4; ++e)
        if (ch * 4 + e < C) f[e] = __ldg(src + e);
      *reinterpret_cast<uint4 *>(s_x + off(row, ch)) =
          make_uint4(to_tf32(f[0]), to_tf32(f[1]), to_tf32(f[2]), to_tf32(f[3]));
    }
  }
}

// ---------------------------------------------------------------- compacted position space --
// Per-tile view of a b2r_compact_plan (csrc/compact.cu).  `m` = the plan's meta words 0..7 (class
// ends, live ends), normally a shared-memory copy; pos0 = first position of the tile (a multiple
// of 32 that never straddles a class).  Everything here is uniform across the CTA.
struct TileClass {
  int ns;      // class size of the tile's centres: 8, 16, 32 or 64 samples
  int live;    // rows [0, live) of the tile are live (<= 0: all dead; may exceed the tile)
  float wx;    // EXTRA weight of a centre's first sample in sums over positions: NS - ns
};
__device__ __forceinline__ TileClass tile_class(const int *m, long long pos0, int NS) {
  const int p = (int)pos0;
  const int c = (p >= m[0]) + (p >= m[1]) + (p >= m[2]);
  TileClass t;
  t.ns = 8 << c;
  t.live = m[4 + c] - p;
  t.wx = (float)(NS - t.ns);
  return t;
}

inline int pow2_shift(int v) {   // log2(v) if v is a power of two (v >= 1), else -1
  if (v < 1 || (v & (v - 1))) return -1;
  int s = 0;
  while ((1 << s) < v) ++s;
  return s;
}

}  // namespace mlp

// CUDA-core streaming variants of the thin first layer (Cin <= 8), mlp_thin.cu
namespace thin {
bool fwd_applicable(const b2r_sa_layer *d);
int fwd_launch(const b2r_sa_layer *d, void *stream);
bool bwd_applicable(const b2r_sa_layer_bwd_desc *d);
int bwd_launch(const b2r_sa_layer_bwd_desc *d, void *stream);
}  // namespace thin
}  // namespace b2r
