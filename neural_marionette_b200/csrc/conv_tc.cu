// Implicit-GEMM 3-D convolution on the 5th-gen tensor cores (tcgen05 + TMEM), operands fed by TMA.
//
// Reference ops replaced: every nn.Conv3d with k in {1, 3} stride 1 and k = 2 stride 2 in
// modules/vox_modules.py:12,26,30,39,53 and model/kypt_detector.py:429,435,444,450.
//
// GEMM view (SURVEY.md §A.1):  D[M = output voxels, N = Cout] = sum_{tap, ci} A[M, (tap, ci)] * W[(tap, ci), N]
//   A  : activations, fp16 channels-last (n, D, H, W, Cin).  For tap (kd, kh, kw) the A tile of a box of
//        128 output voxels is the same box shifted by (kd-p, kh-p, kw-p): one 5-D TMA load per (tap, 64-ch
//        chunk); out-of-bounds coordinates are zero-filled by the TMA unit = the conv's zero padding.
//        k2/s2 ("Pool3DBlock") uses one strided tensor map per tap (base shifted by the tap, strides x2).
//   W  : pre-packed fp16 [tap][Cout][Cin] (K-major B operand), 3-D TMA box (BK, N_tile, 1).
//   D  : fp32 accumulator in TMEM (double-buffered: 2 x N_tile columns), epilogue adds the bias and
//        stores fp16 channels-last.
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM alloc), warps 2-5 = epilogue.
// Persistent: grid = #SMs, static round-robin over output tiles.
#include "common.cuh"
#include "../../include/nm_b200.h"   // the definitions below must match the public declarations
#include <cuda.h>
#include <string.h>
#include <mutex>
#include <vector>

namespace {

constexpr int kTileM = 128;
constexpr int kMaxTaps = 27;
constexpr uint64_t kWatchdogCycles = 8000000000ull;  // ~4 s: turn a protocol bug into a trap, not a hang

struct ConvTcParams {
  CUtensorMap tmap_a[8];
  CUtensorMap tmap_b;
  CUtensorMap tmap_o;            // output (Cout, OW, OH, OD, N), box (32, tw, th, td, tn): TMA-store epilogue
  int taps, kchunks, block_k, n_tile, cout;
  int tw, th, td, tn;            // output-voxel box of one tile (tw*th*td*tn == 128)
  int nw, nh, nd, nn;            // tiles per dimension
  int OW, OH, OD, N;             // output extent
  int stages;
  int8_t dx[kMaxTaps], dy[kMaxTaps], dz[kMaxTaps], map[kMaxTaps];
  const float* bias;
  act_t* out;
  float* stats;                  // optional GroupNorm partials [n][tiles_per_sample*4][Cout][2] (tn == 1 only)
};

// ------------------------------------------------------------------ PTX wrappers
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
  asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
  asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
  asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
  uint32_t ok;
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
      "selp.b32 %0, 1, 0, p;\n\t}"
      : "=r"(ok)
      : "r"(smem_u32(bar)), "r"(parity)
      : "memory");
  return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    if ((uint64_t)(clock64() - t0) > kWatchdogCycles) {
      printf("nm_conv3d_tc: mbarrier watchdog (block %d thread %d)\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
}
// Wait with a short back-off between polls: used by the epilogue warps of the kernels that have producer warps, so
// that eight spinning warps do not take the issue slots the producers need.
__device__ __forceinline__ void mbar_wait_backoff(uint64_t* bar, uint32_t parity, uint32_t ns) {
  if (mbar_try_wait(bar, parity)) return;
  const uint64_t t0 = clock64();
  while (!mbar_try_wait(bar, parity)) {
    __nanosleep(ns);
    if ((uint64_t)(clock64() - t0) > kWatchdogCycles) {
      printf("nm_conv3d_tc: mbarrier watchdog (block %d thread %d)\n", blockIdx.x, threadIdx.x);
      __trap();
    }
  }
}
__device__ __forceinline__ void tma_load_5d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2,
                                            int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5, %6, %7}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void tma_load_3d(void* dst, const CUtensorMap* map, uint64_t* bar, int c0, int c1, int c2) {
  asm volatile(
      "cp.async.bulk.tensor.3d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4, %5}], [%2];"
      ::"r"(smem_u32(dst)), "l"(map), "r"(smem_u32(bar)), "r"(c0), "r"(c1), "r"(c2)
      : "memory");
}
// One elected lane of a converged warp (PTX elect.sync).  Unlike `lane == 0`, ptxas knows that exactly one
// thread executes the guarded region, so it does not wrap every tcgen05.mma in a per-active-thread
// ELECT / BRA.U.ANY serialisation loop.
__device__ __forceinline__ bool elect_one() {
  uint32_t pred;
  asm volatile(
      "{\n\t.reg .pred P;\n\t"
      "elect.sync _|P, 0xffffffff;\n\t"
      "selp.u32 %0, 1, 0, P;\n\t}"
      : "=r"(pred));
  return pred != 0;
}
__device__ __forceinline__ void tma_store_5d(const CUtensorMap* map, const void* src, int c0, int c1, int c2, int c3, int c4) {
  asm volatile(
      "cp.async.bulk.tensor.5d.global.shared::cta.bulk_group [%0, {%2, %3, %4, %5, %6}], [%1];"
      ::"l"(map), "r"(smem_u32(src)), "r"(c0), "r"(c1), "r"(c2), "r"(c3), "r"(c4)
      : "memory");
}
__device__ __forceinline__ void bulk_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
template <int N>
__device__ __forceinline__ void bulk_wait_read() { asm volatile("cp.async.bulk.wait_group.read %0;" ::"n"(N) : "memory"); }
__device__ __forceinline__ void fence_async_smem() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void named_bar_sync(int id, int threads) {
  asm volatile("bar.sync %0, %1;" ::"r"(id), "r"(threads) : "memory");
}
__device__ __forceinline__ uint4 lds128(uint32_t saddr) {
  uint4 v;
  asm volatile("ld.shared.v4.u32 {%0, %1, %2, %3}, [%4];" : "=r"(v.x), "=r"(v.y), "=r"(v.z), "=r"(v.w) : "r"(saddr));
  return v;
}
__device__ __forceinline__ void sts128(uint32_t saddr, const uint4& v) {
  asm volatile("st.shared.v4.u32 [%0], {%1, %2, %3, %4};" ::"r"(saddr), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void umma_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void tmem_ld16(uint32_t addr, uint32_t* r) {
  asm volatile(
      "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15}, [%16];"
      : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]),
        "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
      : "r"(addr));
}
__device__ __forceinline__ void tmem_ld8(uint32_t addr, uint32_t* r) {
  asm volatile("tcgen05.ld.sync.aligned.32x32b.x8.b32 {%0, %1, %2, %3, %4, %5, %6, %7}, [%8];"
               : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7])
               : "r"(addr));
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
__device__ __forceinline__ void tmem_st8(uint32_t addr, const uint32_t* r) {
  asm volatile("tcgen05.st.sync.aligned.32x32b.x8.b32 [%0], {%1, %2, %3, %4, %5, %6, %7, %8};"
               ::"r"(addr), "r"(r[0]), "r"(r[1]), "r"(r[2]), "r"(r[3]), "r"(r[4]), "r"(r[5]), "r"(r[6]), "r"(r[7])
               : "memory");
}
__device__ __forceinline__ void tmem_st_wait() { asm volatile("tcgen05.wait::st.sync.aligned;" ::: "memory"); }

// ---- CTA pairs (cluster of 2, cta_group::2): one MMA of M = 256 reads A rows 128r.. and B rows r*N/2.. from the
// shared memory of CTA r at the same offsets, and writes CTA r's own TMEM lanes (tools/probe/umma2_probe.cu).
__device__ __forceinline__ uint32_t cluster_ctarank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cluster_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
  asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// Arrive on the barrier at the same shared-memory offset in CTA `rank` of the cluster.  Default (CTA-scope release)
// semantics, as CUTLASS's 2-SM pipelines use: what the arrival publishes is consumed by the leader's tcgen05 ops, which
// are ordered by the tcgen05 / async-proxy fences around it.  A .release.cluster arrive (a cluster-scope fence per
// slice in every epilogue and producer warp) made the pair kernels 1.8x slower [measured, B200, 32->32 @ 64^3].
__device__ __forceinline__ void mbar_arrive_remote(uint64_t* bar, uint32_t rank) {
  asm volatile(
      "{\n\t.reg .b32 ra;\n\t"
      "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
      "mbarrier.arrive.shared::cluster.b64 _, [ra];\n\t}"
      ::"r"(smem_u32(bar)), "r"(rank)
      : "memory");
}
__device__ __forceinline__ void umma2_f16(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, %4, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate)
      : "memory");
}
__device__ __forceinline__ void umma2_f16_acc(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, 1, 0;\n\t"
      "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc)
      : "memory");
}
// arrives on the barrier at this offset in both CTAs of the pair once the leader's MMAs issued so far retire
__device__ __forceinline__ void umma2_commit(uint64_t* bar) {
  asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
               ::"r"(smem_u32(bar)), "h"((uint16_t)3) : "memory");
}

// Column sums over the 32 lanes of a warp for 32 per-lane values: recursive halving (31 shuffles instead of
// 160 for a butterfly all-reduce).  On exit lane l holds the total of column l in v[0].
__device__ __forceinline__ void warp_reduce_scatter32(float (&v)[32], int lane) {
#pragma unroll
  for (int half = 16; half >= 1; half >>= 1) {
    const bool upper = (lane & half) != 0;
#pragma unroll
    for (int i = 0; i < half; i++) {
      const float send = upper ? v[i] : v[i + half];
      const float recv = __shfl_xor_sync(0xffffffffu, send, half);
      v[i] = (upper ? v[i + half] : v[i]) + recv;
    }
  }
}

// K-major shared-memory matrix descriptor (cute::UMMA::SmemDescriptor bit layout):
//   [0,14) start address >> 4, [16,30) leading byte offset >> 4 (unused for swizzled K-major),
//   [32,46) stride byte offset >> 4 (= stride between 8-row groups), [46,48) version = 1, [61,64) layout type.
// The MMA-issuing thread is a single lane running scalar code: every instruction between two tcgen05.mma
// costs issue latency (first version: ~30 dependent integer ops per MMA = ~165 cycles per MMA, 10x the
// tensor-pipe time).  Descriptors are therefore split into a loop-invariant high word and a low word that
// advances by plain 32-bit adds of (bytes >> 4).
__device__ __forceinline__ uint32_t desc_hi(uint32_t sbo_bytes, uint32_t layout_type) {
  return (sbo_bytes >> 4) | (1u << 14) | (layout_type << 29);
}
__device__ __forceinline__ uint32_t desc_lo(uint32_t saddr) { return ((saddr & 0x3FFFFu) >> 4) | (1u << 16); }
__device__ __forceinline__ uint64_t desc64(uint32_t hi, uint32_t lo) { return ((uint64_t)hi << 32) | lo; }
__device__ __forceinline__ void umma_f16_acc(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc) {
  asm volatile(
      "{\n\t.reg .pred p;\n\t"
      "setp.ne.b32 p, 1, 0;\n\t"
      "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
      ::"r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc)
      : "memory");
}

// ------------------------------------------------------------------ the kernel
__global__ void __launch_bounds__(192, 1)
conv3d_tc_kernel(const __grid_constant__ ConvTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  // 1024-byte alignment for the swizzled tiles
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int a_bytes = kTileM * p.block_k * 2;
  const int b_bytes = p.n_tile * p.block_k * 2;
  const int stage_bytes = a_bytes + b_bytes;
  uint8_t* tiles = smem;
  uint8_t* s_out = smem + (size_t)p.stages * stage_bytes;             // [2][128 rows x 32 ch fp16] store staging
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_out + 2 * 8192);
  uint64_t* full = bars;
  uint64_t* empty = bars + p.stages;
  uint64_t* tfull = bars + 2 * p.stages;
  uint64_t* tempty = tfull + 2;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tempty + 2);
  float* s_bias = reinterpret_cast<float*>(tmem_slot + 4);      // [n_tile], zero beyond Cout
  for (int i = threadIdx.x; i < p.n_tile; i += blockDim.x) s_bias[i] = i < p.cout ? p.bias[i] : 0.f;

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int total_tiles = p.nw * p.nh * p.nd * p.nn;
  const int k_iters = p.taps * p.kchunks;
  uint32_t tmem_cols = 32;
  while ((int)tmem_cols < 2 * p.n_tile) tmem_cols <<= 1;

  if (warp == 0 && lane == 0) {
    for (int i = 0; i < 8; i++)
      asm volatile("prefetch.tensormap [%0];" ::"l"(&p.tmap_a[i]) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&p.tmap_b) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&p.tmap_o) : "memory");
    for (int s = 0; s < p.stages; s++) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    for (int s = 0; s < 2; s++) {
      mbar_init(&tfull[s], 1);
      mbar_init(&tempty[s], 4);   // one arrive per epilogue warp
    }
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols)
                 : "memory");
    asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
        int t = tile;
        const int iw = t % p.nw; t /= p.nw;
        const int ih = t % p.nh; t /= p.nh;
        const int id = t % p.nd; t /= p.nd;
        const int in_ = t;
        const int w0 = iw * p.tw, h0 = ih * p.th, d0 = id * p.td, n0 = in_ * p.tn;
        for (int tap = 0; tap < p.taps; tap++) {
          const CUtensorMap* ma = &p.tmap_a[p.map[tap]];
          for (int kc = 0; kc < p.kchunks; kc++) {
            mbar_wait(&empty[stage], phase ^ 1);
            uint8_t* sa = tiles + (size_t)stage * stage_bytes;
            mbar_expect_tx(&full[stage], (uint32_t)stage_bytes);
            tma_load_5d(sa, ma, &full[stage], kc * p.block_k, w0 + p.dx[tap], h0 + p.dy[tap], d0 + p.dz[tap], n0);
            tma_load_3d(sa + a_bytes, &p.tmap_b, &full[stage], kc * p.block_k, 0, tap);
            if (++stage == p.stages) { stage = 0; phase ^= 1; }
          }
        }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // instruction descriptor (cute::UMMA::InstrDescriptor): c_format F32 (bit 4), a/b format F16 (0),
    // K-major A and B, N >> 3 at [17,23), M >> 4 at [24,29)
    const uint32_t idesc = (1u << 4) | ((uint32_t)(p.n_tile >> 3) << 17) | ((uint32_t)(kTileM >> 4) << 24);
    const uint32_t row_bytes = p.block_k * 2;                       // 128 (SW128) or 64 (SW64)
    const uint32_t layout = row_bytes == 128 ? 2u : (row_bytes == 64 ? 4u : 6u);
    const uint32_t hi = desc_hi(8 * row_bytes, layout);
    const int ksteps = p.block_k / 16;
    int stage = 0;
    uint32_t phase = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      mbar_wait(&tempty[acc], acc_phase ^ 1);
      tc_fence_after();
      const uint32_t tmem_d = tmem_base + (uint32_t)(acc * p.n_tile);
      for (int it = 0; it < k_iters; it++) {
        mbar_wait(&full[stage], phase);
        tc_fence_after();
        __syncwarp();
        if (elect_one()) {
          const uint32_t sa = smem_u32(tiles + (size_t)stage * stage_bytes);
          const uint32_t alo = desc_lo(sa), blo = desc_lo(sa + a_bytes);
          umma_f16(tmem_d, desc64(hi, alo), desc64(hi, blo), idesc, it > 0 ? 1u : 0u);
          for (int k = 1; k < ksteps; k++) umma_f16_acc(tmem_d, desc64(hi, alo + 2 * k), desc64(hi, blo + 2 * k), idesc);
          umma_commit(&empty[stage]);                // frees the smem slot once these MMAs retire
          if (it == k_iters - 1) umma_commit(&tfull[acc]);
        }
        __syncwarp();
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
  } else {
    // ===================== epilogue (warps 2..5) =====================
    // TMEM -> registers (+bias) -> fp16 -> swizzled smem staging (32 channels x 128 rows) -> one TMA store per
    // 32-channel chunk.  (Per-thread 16-byte global stores of a row each touch a different cache line per lane
    // and ran at ~1 TB/s; the TMA store also clips partial tiles / channel remainders.)
    const int quad = warp & 3;                     // TMEM lane quadrant this warp may access
    const int row = quad * 32 + lane;
    const bool is_issuer = warp == 2 && lane == 0;
    uint32_t n_out = 0;
    int acc = 0;
    uint32_t acc_phase = 0;
    for (int tile = blockIdx.x; tile < total_tiles; tile += gridDim.x) {
      int t = tile;
      const int iw = t % p.nw; t /= p.nw;
      const int ih = t % p.nh; t /= p.nh;
      const int id = t % p.nd; t /= p.nd;
      const int in_ = t;
      mbar_wait(&tfull[acc], acc_phase);
      tc_fence_after();
      const uint32_t taddr = tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(acc * p.n_tile);
      for (int c0 = 0; c0 < p.n_tile; c0 += 32) {
        uint32_t r[32];
        tmem_ld16(taddr + c0, r);
        if (c0 + 16 < p.n_tile) tmem_ld16(taddr + c0 + 16, r + 16);
        tmem_ld_wait();
        if (c0 + 32 >= p.n_tile) {                 // last chunk read: hand the accumulator back to the MMA warp
          tc_fence_before();
          __syncwarp();
          if (lane == 0) mbar_arrive(&tempty[acc]);
        }
        uint8_t* buf = s_out + (n_out & 1) * 8192;
        if (is_issuer) bulk_wait_read<1>();
        named_bar_sync(1, 128);
        float v32[32];
#pragma unroll
        for (int j = 0; j < 32; j++) v32[j] = c0 + j < p.n_tile ? __uint_as_float(r[j]) + s_bias[c0 + j] : 0.f;
#pragma unroll
        for (int h = 0; h < 4; h++) {              // four 16-byte chunks of the row's 64-byte staging line
          const uint32_t off = (uint32_t)row * 64 + h * 16;
          *reinterpret_cast<half8*>(buf + (off ^ (((off >> 7) & 3u) << 4))) = nm_pack8(v32 + h * 8);
        }
        if (p.stats) {
          // fused GroupNorm statistics: per-channel sum / sum of squares over this warp's 32 rows
          float sq32[32];
#pragma unroll
          for (int j = 0; j < 32; j++) sq32[j] = v32[j] * v32[j];
          warp_reduce_scatter32(v32, lane);
          warp_reduce_scatter32(sq32, lane);
          const int ch = c0 + lane;
          if (ch < p.cout) {
            const int tiles_per_sample = p.nw * p.nh * p.nd;
            const long long chunk = (long long)(tile % tiles_per_sample) * 4 + quad;
            float2* dst = reinterpret_cast<float2*>(p.stats) +
                          ((long long)in_ * tiles_per_sample * 4 + chunk) * p.cout + ch;
            *dst = make_float2(v32[0], sq32[0]);
          }
        }
        fence_async_smem();
        named_bar_sync(1, 128);
        if (is_issuer) {
          tma_store_5d(&p.tmap_o, buf, c0, iw * p.tw, ih * p.th, id * p.td, in_ * p.tn);
          bulk_commit();
        }
        n_out++;
      }
      if (++acc == 2) { acc = 0; acc_phase ^= 1; }
    }
    if (is_issuer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(tmem_base), "r"(tmem_cols) : "memory");
  }
}

// ------------------------------------------------------------------ slab-walking kernel (k3, Cout <= 128)
// For Cout <= 64 the tap-streaming kernel above is bound by operand delivery: every tap re-fetches its
// 128 x Cin A tile from L2 (27x re-read; ncu: 7 TB/s L2->SM, tensor pipe 8 %).  Here a CTA owns a column of
// output tiles (16 h x 8 w voxels) and walks it along d: each input slice (18 x 10 halo rows) is fetched ONCE
// by TMA into a ring of slots and reused by all 27 taps - a tap is just a different start address / the same
// 8-row-group stride (10 rows) in the A descriptor (the 128B/64B swizzle is a function of the absolute
// shared-memory address, so a row-shifted start stays consistent with what TMA wrote; verified on B200).
// The weights of all taps stay resident in shared memory.
struct ConvSlabParams {
  CUtensorMap tmap_a;     // (C, W, H, D, N) box (BK, 10, 18, 1, 1)
  CUtensorMap tmap_b;     // (Cin, Cout, 27) box (BK, PN, 1)
  CUtensorMap tmap_o;     // output (Cout, W, H, D, N) box (PN, 8, 16, 1, 1) for the TMA-store epilogue
  int kchunks, block_k, n_tile, cout;
  int nw, nh;             // tiles per (w, h); columns = N * nh * nw
  int D, H, W, N;
  int slot_bytes;         // bytes of one ring slot (kchunks chunks)
  int chunk_bytes;        // bytes of one (slice, k-chunk) = 180 rows, padded to 1 KiB
  int ring;               // ring slots actually used (2..8)
  float* stats;           // optional GroupNorm partials [n][nh*nw*4][Cout][2] (sum, sum of squares)
  const float* in_scale;  // optional fused input transform x <- act(x * in_scale[n][c] + in_shift[n][c]),
  const float* in_shift;  // i.e. the GroupNorm (+LeakyReLU) of the producing layer applied on the halo
  int in_act;             // slice in shared memory (zero padding preserved); (n, Cin) fp32 each
  int cin;
  int cin_off;            // first input channel of this launch (split-K over two launches: Cin = 128)
  int accum;              // add the existing contents of `out` (the partial sum of the previous launch)
  const float* bias;      // may be null (second split-K launch)
  act_t* out;
};

constexpr int kHaloW = 10, kHaloH = 18;

// ------------------------------------------------------------------ slab kernel, 3 depth-taps per MMA (Cout = 32)
// With N = Cout = 32 an MMA is 16 tensor-pipe cycles but costs ~70 cycles to issue from a single thread and
// reads 4 KB of A for 1 KB of B: issue- and smem-bound.  Stack the weights of the three depth taps of a
// (kh, kw) position into one B tile of N = 96 rows: one MMA then multiplies the window of input slice s with
// W(kd=0), W(kd=1), W(kd=2) at once, i.e. it produces the contribution of slice s to the outputs s+1, s, s-1 in
// three 32-column blocks of a TMEM group P(s).  A is read once instead of three times and the MMA count drops
// 3x.  The epilogue forms out(j) = P(j-1)[0:32] + P(j)[32:64] + P(j+1)[64:96] (+ bias) from a ring of four
// groups (4 x 96 TMEM columns).
constexpr int kPGroups = 5;    // 5 x 96 TMEM columns = 480 <= 512

// BK: channels per k-chunk (64 -> 128B swizzle, 32 -> 64B); PN: output channels per CTA "part" (32, or 16 when
// Cin = 128 so that the 27 x kchunks resident weight tiles still fit, or 64 on a CTA pair, which holds half of them);
// MMA N = 3 * PN.
constexpr int kSlab3EpiWarps = 8;
constexpr int kSlab3Threads = 64 + 32 * kSlab3EpiWarps;
constexpr int kSlab3Ring = 8;        // max halo-slice ring depth (Cin = 32 has room for 8 slots, Cin = 64 for 4)
constexpr int kSlab3XformWarps = 6;   // max extra warps (only launched when the input transform is fused); the
                                      // number actually launched comes from blockDim (512 threads x 128 registers)

// UP: the conv input is the 2x trilinear up-sampling (align_corners = False) of a low-resolution tensor that is
// never materialised (tmap_a then describes the low-resolution tensor; BK = 64, one k-chunk).  Everything after the
// input transform is linear and trilinear x2 is separable, so the depth part of the up-sampling is applied to the
// accumulators instead of the operand: TMA brings (10 x 6)-row low-resolution planes into a small ring, the transform
// warps build one halo slice per LOW-resolution plane (h / w interpolation only) directly in the swizzled operand
// layout, the MMAs run over D/2 slices, and the epilogue forms every output slice as a fixed combination of the TMEM
// groups P(i-1), P(i), P(i+1).  Half the MMAs, half the operand traffic; the depth border (clamp + zero padding)
// stays exact and is blended in fp32.
constexpr int kLoRing = 4;
constexpr int kLoRows = 10 * 6;              // low-resolution box: 10 (h) x 6 (w) rows of 64 channels
constexpr int kLoBytes = kLoRows * 128;      // 7680
constexpr int kUpWarps = 4;                  // up-sampling producer warps launched (3 working)

// ACC: split-K second launch - the epilogue adds the partial sum already in `out`.
// PAIR: a cluster of two CTAs that own two adjacent 8-wide w tiles of the same (n, h-tile) column and walk d in
// lockstep.  The leader (rank 0) issues cta_group::2 MMAs of M = 256 x N = 3 * PN; each CTA holds its own halo slices
// and half of the stacked weight rows (CTA r: rows r * 3PN/2 ..), so per CTA the B-operand read of an MMA and the
// resident weights are halved.  The peer's slices, transforms and drained TMEM groups are reported to the leader's
// barriers by remote arrives; the leader's commits arrive on the barriers of both CTAs (multicast).
template <int BK, int PN, bool UP = false, bool ACC = false, bool PAIR = false>
__global__ void __launch_bounds__(kSlab3Threads + 32 * kSlab3XformWarps, 1)
conv3d_slab3_kernel(const __grid_constant__ ConvSlabParams p) {
  static_assert(!UP || PN == 32, "the up-sampling epilogue serves 32-channel parts");
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  constexpr int CG = PAIR ? 2 : 1;                                     // CTAs per MMA
  // TMEM groups P(s) of 3 * PN columns in flight: 5 x 96, or 2 x 192 with PN = 64 (the epilogue then carries the
  // running sums in the remaining 2 x 64 columns)
  constexpr int PG = PN == 64 ? 2 : kPGroups;
  static_assert(PN != 64 || (PAIR && !UP && !ACC), "64-channel parts run on CTA pairs, without up-sampling / split-K");
  constexpr int box_rows = PN / CG;                                    // rows of one weight TMA box
  constexpr int w_tile_bytes = 3 * box_rows * BK * 2;                  // one (kh, kw, k-chunk): this CTA's stacked rows
  const int w_bytes = 9 * p.kchunks * w_tile_bytes;
  const int ring = p.ring;
  uint8_t* s_w = smem;                                                 // [kh*3+kw][kc][3 * PN / CG rows][BK]
  uint8_t* s_ring = smem + w_bytes;
  constexpr int stage_bytes = kTileM * PN * 2;                         // one output tile (128 rows x PN fp16)
  uint8_t* s_lo = s_ring + (size_t)ring * p.slot_bytes;                // UP: [kLoRing][kLoBytes] low-res planes
  uint8_t* s_out = s_lo + (UP ? kLoRing * kLoBytes : 0);               // [2][stage_bytes], 1 KiB aligned
  uint64_t* bars = reinterpret_cast<uint64_t*>(s_out + 2 * stage_bytes);
  uint64_t* full = bars;                  // [ring]   slice landed
  uint64_t* empty = full + kSlab3Ring;     // [ring]   slice consumed
  uint64_t* pfull = empty + kSlab3Ring;    // [groups] P group complete
  uint64_t* pempty = pfull + kPGroups;    // [groups] P group drained
  uint64_t* wfull = pempty + kPGroups;    // [1]
  uint64_t* ready = wfull + 1;            // [ring]   slice transformed (fused input GroupNorm / LeakyReLU)
  uint64_t* full_lo = ready + kSlab3Ring; // [kLoRing] UP: low-res plane landed
  uint64_t* empty_lo = full_lo + kLoRing; // [kLoRing] UP: low-res plane dead
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(empty_lo + kLoRing);
  float* s_ab = reinterpret_cast<float*>(tmem_slot + 4);   // [2][Cin] scale | shift of the current sample
  const bool xform = UP || p.in_scale != nullptr;
  const int nxw = ((int)blockDim.x - kSlab3Threads) >> 5;   // transform / producer warps launched (0, 4 or 6)
  const int n_sl = UP ? p.D >> 1 : p.D;                     // operand slices (= TMEM groups) per column

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int n_cols = p.N * p.nh * p.nw;
  constexpr uint32_t tmem_cols = 512;
  // Cout > PN: the output channels are split into parts of PN; CTA b serves part b % parts with its own
  // resident weights (A is re-read once per part, each pass runs at the N = 3*PN rate)
  // (with PAIR the "unit" is a CTA pair: cluster c = CTAs 2c, 2c+1, column pair (2j, 2j+1))
  const int parts = p.n_tile / PN;
  const int rank = PAIR ? (int)cluster_ctarank() : 0;
  const int unit = blockIdx.x / CG, n_units = gridDim.x / CG;
  const int part = unit % parts;
  const int col0 = (unit / parts) * CG + rank, col_step = (n_units / parts) * CG;
  // barriers of the leader that the peer CTA also arrives on count its arrivals too
  const uint32_t peers = PAIR && rank == 0 ? 2u : 1u;
  // arrival on a barrier the MMA issuer waits on: the leader's copy
  auto arrive_issuer = [&](uint64_t* bar) {
    if constexpr (PAIR) mbar_arrive_remote(bar, 0);
    else mbar_arrive(bar);
  };

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&p.tmap_a) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&p.tmap_b) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&p.tmap_o) : "memory");
    for (int s = 0; s < kSlab3Ring; s++) { mbar_init(&full[s], xform ? 1 : peers); mbar_init(&empty[s], 1); }
    for (int s = 0; s < kPGroups; s++) { mbar_init(&pfull[s], 1); mbar_init(&pempty[s], kSlab3EpiWarps * peers); }
    for (int s = 0; s < kSlab3Ring; s++) mbar_init(&ready[s], nxw * peers);
    for (int s = 0; s < kLoRing; s++) { mbar_init(&full_lo[s], 1); mbar_init(&empty_lo[s], nxw); }
    mbar_init(wfull, peers);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) {
    if constexpr (PAIR) {   // one warp in each CTA of the pair
      asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    } else {
      asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(tmem_cols)
                   : "memory");
      asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) cluster_sync();   // the peer's barriers are initialised before anything arrives on them
  tc_fence_after();
  if (*tmem_slot != 0u) {       // single allocation per SM: base 0 keeps all TMEM addresses warp-uniform
    printf("nm_conv3d_tc(slab3): unexpected TMEM base %u\n", *tmem_slot);
    __trap();
  }

  if (UP && warp >= 2 + kSlab3EpiWarps) {
    // ===================== up-sampling operand producer (warps 10..13) =====================
    // Operand slice d is low-res plane d up-sampled along h and w (the depth part is applied in the epilogue): a
    // full-resolution row blends the low-res rows near and far = near -/+ 1 (clamped) with weights 0.75 / 0.25
    // (PyTorch trilinear, align_corners = False), and the same rule applies along w.  Work item = (pair of halo rows,
    // 16-byte channel chunk c): 12 plane loads -> h blends for the 6 box columns -> the 10 halo columns of both rows,
    // written at the TMA-128B-swizzle position.  Rows / columns outside the tensor are the conv's zero padding.  With
    // a fused prologue the producer's GroupNorm scale/shift (+LeakyReLU) is applied to each plane in place when it
    // lands.
    const int tid = threadIdx.x - 32 * (2 + kSlab3EpiWarps);
    const bool fused = p.in_scale != nullptr;
    const int Hl = p.H >> 1;
    const __half2 q25 = __float2half2_rn(0.25f);
    auto lerp = [&](const uint4& a, const uint4& b) -> uint4 {      // a + 0.25 (b - a)
      uint4 r;
      const __half2* pa = reinterpret_cast<const __half2*>(&a);
      const __half2* pb = reinterpret_cast<const __half2*>(&b);
      __half2* pr = reinterpret_cast<__half2*>(&r);
#pragma unroll
      for (int i = 0; i < 4; i++) pr[i] = __hfma2(q25, __hsub2(pb[i], pa[i]), pa[i]);
      return r;
    };
    const __half2 q75 = __float2half2_rn(0.75f);
    auto scale4 = [&](const uint4& a, const __half2 f) -> uint4 {
      uint4 r;
      const __half2* pa = reinterpret_cast<const __half2*>(&a);
      __half2* pr = reinterpret_cast<__half2*>(&r);
#pragma unroll
      for (int i = 0; i < 4; i++) pr[i] = __hmul2(pa[i], f);
      return r;
    };
    auto add4 = [&](const uint4& a, const uint4& b) -> uint4 {
      uint4 r;
      const __half2* pa = reinterpret_cast<const __half2*>(&a);
      const __half2* pb = reinterpret_cast<const __half2*>(&b);
      __half2* pr = reinterpret_cast<__half2*>(&r);
#pragma unroll
      for (int i = 0; i < 4; i++) pr[i] = __hadd2(pa[i], pb[i]);
      return r;
    };
    uint32_t fill = 0;                                    // slices produced so far (ring position)
    uint32_t planes = 0;                                  // global index of plane 0 of the current column
    int cur_n = -1;
    const uint32_t lo_base = smem_u32(s_lo), ring_base = smem_u32(s_ring);
    for (int col = col0; col < n_cols; col += col_step, planes += n_sl) {
      int t = col;
      const int iw = t % p.nw; t /= p.nw;
      const int ih = t % p.nh; t /= p.nh;
      const int n = t;
      if (fused && n != cur_n) {
        named_bar_sync(2, 32 * nxw);
        for (int i = tid; i < p.cin; i += 32 * nxw) {
          s_ab[i] = p.in_scale[(long long)n * p.cin + i];
          s_ab[p.cin + i] = p.in_shift[(long long)n * p.cin + i];
        }
        named_bar_sync(2, 32 * nxw);
        cur_n = n;
      }
      for (int d = 0; d < n_sl; d++, fill++) {
        const uint32_t g = planes + d;                    // global index of low-res plane d
        const uint32_t lo = lo_base + (g % kLoRing) * kLoBytes;
        mbar_wait(&full_lo[g % kLoRing], (g / kLoRing) & 1);
        if (fused) {
          for (int i = tid; i < kLoRows * 8; i += 32 * nxw) {
            const int c = i & 7;
            const uint32_t addr = lo + i * 16;
            const uint4 raw = lds128(addr);
            const uint32_t in[4] = {raw.x, raw.y, raw.z, raw.w};
            uint32_t o[4];
#pragma unroll
            for (int k = 0; k < 4; k++) {
              const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&in[k]));
              __half2 hv = __floats2half2_rn(fmaf(f.x, s_ab[c * 8 + 2 * k], s_ab[p.cin + c * 8 + 2 * k]),
                                             fmaf(f.y, s_ab[c * 8 + 2 * k + 1], s_ab[p.cin + c * 8 + 2 * k + 1]));
              if (p.in_act) hv = __hmax2(hv, __hmul2(hv, __float2half2_rn(0.01f)));
              o[k] = *reinterpret_cast<uint32_t*>(&hv);
            }
            sts128(addr, make_uint4(o[0], o[1], o[2], o[3]));
          }
          named_bar_sync(2, 32 * nxw);
        }
        const int slot = fill % ring;
        mbar_wait(&empty[slot], ((fill / ring) & 1) ^ 1);
        const uint32_t sbase = ring_base + (uint32_t)slot * p.slot_bytes;
        // item = (pair of halo rows 2j, 2j+1, chunk c): h = ih*16 - 1 + 2j is odd (= 2m+1) and h + 1 = 2m+2, so both
        // rows interpolate between the same low-res rows m and m+1 (near / far swapped): the 12 plane loads are shared.
        // The 72 items go to the first three producer warps.  The fourth (warp 13) shares its SM sub-partition with
        // the MMA-issuing warp and only takes part in the barriers, so that it does not compete for issue slots.
        if (tid < (kHaloH / 2) * 8) {
          const int j = tid >> 3, c = tid & 7;
          const int h0 = ih * 16 - 1 + 2 * j;                        // first row of the pair (may be -1)
          const int m = (h0 + 1) / 2 - 1;                            // h0 = 2m + 1
          const int ma = min(max(m, 0), Hl - 1), mb = min(m + 1, Hl - 1);
          const uint32_t oa = (uint32_t)((ma - (ih * 8 - 1)) * 6) * 128 + c * 16;
          const uint32_t ob = (uint32_t)((mb - (ih * 8 - 1)) * 6) * 128 + c * 16;
          const uint4 zero = make_uint4(0, 0, 0, 0);
          constexpr int NW = 6;                                      // box columns
          uint4 va[NW], vb[NW];                                      // low-res rows m and m+1
#pragma unroll
          for (int w = 0; w < NW; w++) {
            va[w] = lds128(lo + oa + w * 128);
            vb[w] = lds128(lo + ob + w * 128);
          }
#pragma unroll
          for (int r2 = 0; r2 < 2; r2++) {
            const int hh = 2 * j + r2, hf = h0 + r2;
            const uint32_t orow = sbase + (uint32_t)(hh * kHaloW) * 128;
            if ((unsigned)hf >= (unsigned)p.H) {                     // conv padding row
#pragma unroll
              for (int ww = 0; ww < kHaloW; ww++) sts128(orow + ww * 128 + ((c ^ ((hh * kHaloW + ww) & 7)) << 4), zero);
              continue;
            }
            uint4 v[NW];                                             // row 2m+1: near m, far m+1; row 2m+2: near m+1, far m
#pragma unroll
            for (int w = 0; w < NW; w++) v[w] = r2 == 0 ? lerp(va[w], vb[w]) : lerp(vb[w], va[w]);
            // along w every box column is the near operand of two halo columns and the far operand of up to two:
            // 0.75 v and 0.25 v once per column, then one add per output (22 instead of 40 half2 ops per channel pair)
            uint4 t75[NW], t25[NW];
#pragma unroll
            for (int w = 0; w < NW; w++) { t75[w] = scale4(v[w], q75); t25[w] = scale4(v[w], q25); }
#pragma unroll
            for (int ww = 0; ww < kHaloW; ww++) {
              // halo column ww <-> w = iw*8 - 1 + ww: near box column (ww+1)>>1, far = near +1 (ww even) / -1 (ww odd)
              const int nr = (ww + 1) >> 1, fr = (ww & 1) ? nr - 1 : nr + 1;
              uint4 o;
              if ((ww == 0 && iw == 0) || (ww == kHaloW - 1 && iw == p.nw - 1)) o = zero;             // conv padding
              else if ((ww == 1 && iw == 0) || (ww == kHaloW - 2 && iw == p.nw - 1)) o = v[nr];        // clamped far
              else o = add4(t75[nr], t25[fr]);
              sts128(orow + ww * 128 + ((c ^ ((hh * kHaloW + ww) & 7)) << 4), o);
            }
          }
        }
        fence_async_smem();                              // generic-proxy writes -> visible to the UMMA reads
        __syncwarp();
        if (lane == 0) {
          arrive_issuer(&ready[slot]);
          mbar_arrive(&empty_lo[g % kLoRing]);
        }
      }
    }
  } else if (warp >= 2 + kSlab3EpiWarps) {
    // ===================== input transform (warps 10..13, only with a fused prologue) =====================
    // The GroupNorm affine (+LeakyReLU) of the producing layer is applied to each halo slice in place, once,
    // before the 9 x kchunks x BK/16 MMAs read it: the activated tensor never exists in HBM.  Rows outside the
    // tensor stay zero (conv padding applies to the activated tensor).  The 16-byte chunk c of row r sits at
    // position c ^ ((r * row_bytes >> 7) & mask) (TMA 128B / 64B swizzle on a 1 KiB-aligned slot).
    constexpr int row_bytes = BK * 2;
    constexpr int cpr = row_bytes / 16;                  // chunks per row: 8 (SW128) or 4 (SW64)
    const int tid = threadIdx.x - 32 * (2 + kSlab3EpiWarps);
    // thread <-> (logical 16-byte channel chunk lc, rows r0, r0 + rstep, ...): a warp covers whole rows
    const int lc = tid % cpr, r0 = tid / cpr;
    const int rstep = 32 * nxw / cpr;
    uint32_t fill = 0;
    int cur_n = -1;
    for (int col = col0; col < n_cols; col += col_step) {
      int t = col;
      const int iw = t % p.nw; t /= p.nw;
      const int ih = t % p.nh; t /= p.nh;
      const int n = t;
      if (n != cur_n) {                                  // (re)load this sample's scale / shift
        named_bar_sync(2, 32 * nxw);
        for (int i = tid; i < p.cin; i += 32 * nxw) {
          s_ab[i] = p.in_scale[(long long)n * p.cin + i];
          s_ab[p.cin + i] = p.in_shift[(long long)n * p.cin + i];
        }
        named_bar_sync(2, 32 * nxw);
        cur_n = n;
      }
      for (int dz = 0; dz < p.D; dz++, fill++) {
        const int slot = fill % ring;
        mbar_wait(&full[slot], (fill / ring) & 1);
        uint8_t* base = s_ring + (size_t)slot * p.slot_bytes;
        for (int kc = 0; kc < p.kchunks; kc++) {
          // this thread's 8 channels: logical chunk lc of k-chunk kc (scale / shift stay in registers)
          float sc[8], sh[8];
#pragma unroll
          for (int k = 0; k < 8; k++) {
            sc[k] = s_ab[kc * BK + lc * 8 + k];
            sh[k] = s_ab[p.cin + kc * BK + lc * 8 + k];
          }
          const uint32_t cbase = smem_u32(base) + (uint32_t)kc * p.chunk_bytes;   // shared-space address
          // fp32 affine, fp16 LeakyReLU (max(y, 0.01 y) on the rounded value); two rows in flight per thread
          auto xf = [&](uint4 raw) -> uint4 {
            const uint32_t in[4] = {raw.x, raw.y, raw.z, raw.w};
            uint32_t o[4];
#pragma unroll
            for (int k = 0; k < 4; k++) {
              const float2 f = __half22float2(*reinterpret_cast<const __half2*>(&in[k]));
              __half2 hv = __floats2half2_rn(fmaf(f.x, sc[2 * k], sh[2 * k]), fmaf(f.y, sc[2 * k + 1], sh[2 * k + 1]));
              if (p.in_act) hv = __hmax2(hv, __hmul2(hv, __float2half2_rn(0.01f)));
              o[k] = *reinterpret_cast<uint32_t*>(&hv);
            }
            return make_uint4(o[0], o[1], o[2], o[3]);
          };
          auto row_addr = [&](int r, bool& ok) -> uint32_t {
            const int hh = r / kHaloW, ww = r - hh * kHaloW;
            const int h = ih * 16 - 1 + hh, w = iw * 8 - 1 + ww;
            ok = r < kHaloW * kHaloH && (unsigned)h < (unsigned)p.H && (unsigned)w < (unsigned)p.W;
            const int pc = lc ^ (row_bytes == 128 ? (r & 7) : ((r >> 1) & 3));
            return cbase + r * row_bytes + pc * 16;
          };
          for (int r = r0; r < kHaloW * kHaloH; r += 2 * rstep) {
            bool ok0, ok1;
            const uint32_t a0 = row_addr(r, ok0), a1 = row_addr(r + rstep, ok1);
            uint4 v0 = make_uint4(0, 0, 0, 0), v1 = make_uint4(0, 0, 0, 0);
            if (ok0) v0 = lds128(a0);
            if (ok1) v1 = lds128(a1);
            v0 = xf(v0);
            v1 = xf(v1);
            if (ok0) sts128(a0, v0);
            if (ok1) sts128(a1, v1);
          }
        }
        fence_async_smem();                              // generic-proxy writes -> visible to the UMMA reads
        __syncwarp();
        if (lane == 0) arrive_issuer(&ready[slot]);
      }
    }
  } else

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      mbar_expect_tx(wfull, (uint32_t)w_bytes);
      // stacked tile of a (kh, kw, k-chunk): W(kd = 0) | W(kd = 1) | W(kd = 2), PN rows each, in boxes of box_rows;
      // this CTA holds boxes 3 * rank .. 3 * rank + 2
      for (int khw = 0; khw < 9; khw++)
        for (int kc = 0; kc < p.kchunks; kc++)
          for (int b = 0; b < 3; b++) {
            const int jb = 3 * rank + b, kd = jb / CG;
            tma_load_3d(s_w + (size_t)(khw * p.kchunks + kc) * w_tile_bytes + (size_t)b * box_rows * BK * 2, &p.tmap_b,
                        wfull, p.cin_off + kc * BK, part * PN + (jb % CG) * box_rows, kd * 9 + khw);
          }
      uint32_t fill = 0;
      const uint32_t slice_tx = (uint32_t)(kHaloW * kHaloH * BK * 2 * p.kchunks);
      for (int col = col0; col < n_cols; col += col_step) {
        int t = col;
        const int iw = t % p.nw; t /= p.nw;
        const int ih = t % p.nh; t /= p.nh;
        const int n = t;
        if constexpr (UP) {
          for (int pl = 0; pl < (p.D >> 1); pl++, fill++) {
            const int slot = fill % kLoRing;
            mbar_wait(&empty_lo[slot], ((fill / kLoRing) & 1) ^ 1);
            mbar_expect_tx(&full_lo[slot], (uint32_t)kLoBytes);
            tma_load_5d(s_lo + (size_t)slot * kLoBytes, &p.tmap_a, &full_lo[slot], p.cin_off, iw * 4 - 1, ih * 8 - 1, pl, n);
          }
          continue;
        }
        for (int dz = 0; dz < p.D; dz++, fill++) {
          const int slot = fill % ring;
          mbar_wait(&empty[slot], ((fill / ring) & 1) ^ 1);
          mbar_expect_tx(&full[slot], slice_tx);
          for (int kc = 0; kc < p.kchunks; kc++)
            tma_load_5d(s_ring + (size_t)slot * p.slot_bytes + (size_t)kc * p.chunk_bytes, &p.tmap_a, &full[slot],
                        p.cin_off + kc * BK, iw * 8 - 1, ih * 16 - 1, dz, n);
        }
      }
      // a pair's CTA does not exit while the leader's last commits may still arrive on its slot barriers
      if constexpr (PAIR)
        for (int i = 0; i < ring; i++, fill++) mbar_wait(&empty[fill % ring], ((fill / ring) & 1) ^ 1);
    }
  } else if (PAIR && warp == 1 && rank != 0) {
    // ===================== pair peer: forwards its landed weights / slices to the leader's barriers =====================
    if (elect_one()) {
      mbar_wait(wfull, 0);
      mbar_arrive_remote(wfull, 0);
      if (!xform) {                                      // (with a transform the producer warps report `ready`)
        uint32_t q = 0;
        for (int col = col0; col < n_cols; col += col_step)
          for (int sl = 0; sl < p.D; sl++, q++) {
            mbar_wait(&full[q % ring], (q / ring) & 1);
            mbar_arrive_remote(&full[q % ring], 0);
          }
      }
    }
    __syncwarp();
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    constexpr uint32_t idesc = (1u << 4) | ((uint32_t)((3 * PN) >> 3) << 17) | ((uint32_t)(CG * kTileM >> 4) << 24);
    constexpr uint32_t row_bytes = BK * 2;
    constexpr uint32_t layout = row_bytes == 128 ? 2u : 4u;
    const uint32_t hi_a = desc_hi(kHaloW * row_bytes, layout), hi_b = desc_hi(8 * row_bytes, layout);
    const uint32_t ring_lo = desc_lo(smem_u32(s_ring)), w_lo = desc_lo(smem_u32(s_w));
    const uint32_t slot_step = (uint32_t)p.slot_bytes >> 4, chunk_step = (uint32_t)p.chunk_bytes >> 4;
    constexpr uint32_t w_step = (uint32_t)w_tile_bytes >> 4;             // one (khw, kc) B tile = 3 kd tiles
    auto mma = [&](uint32_t tmem_d, uint32_t alo, uint32_t blo, uint32_t accumulate) {
      if constexpr (PAIR) umma2_f16(tmem_d, desc64(hi_a, alo), desc64(hi_b, blo), idesc, accumulate);
      else umma_f16(tmem_d, desc64(hi_a, alo), desc64(hi_b, blo), idesc, accumulate);
    };
    auto mma_acc = [&](uint32_t tmem_d, uint32_t alo, uint32_t blo) {
      if constexpr (PAIR) umma2_f16_acc(tmem_d, desc64(hi_a, alo), desc64(hi_b, blo), idesc);
      else umma_f16_acc(tmem_d, desc64(hi_a, alo), desc64(hi_b, blo), idesc);
    };
    auto commit = [&](uint64_t* bar) {
      if constexpr (PAIR) umma2_commit(bar);
      else umma_commit(bar);
    };
    if (xform) {
      // With an in-kernel operand producer (fused GroupNorm / up-sampling) the plain loop is faster [measured: dec.8
      // with fused up-sampling 9.0 vs 9.4 ms, dec.11 with fused GroupNorm 5.4 vs 6.0 ms]: the burstier stream of the
      // pipelined variant below starves the producer warps.
      mbar_wait(wfull, 0);
      uint32_t q = 0;                                    // global slice counter (ring + P-group position)
      for (int col = col0; col < n_cols; col += col_step) {
        for (int sl = 0; sl < n_sl; sl++, q++) {
          mbar_wait(&ready[q % ring], (q / ring) & 1);
          mbar_wait(&pempty[q % PG], ((q / PG) & 1) ^ 1);
          tc_fence_after();
          __syncwarp();
          if (elect_one()) {
            const uint32_t tmem_d = (q % PG) * (3 * PN);
            const uint32_t slot_lo = ring_lo + (q % ring) * slot_step;
            uint32_t blo = w_lo;
#pragma unroll
            for (int t9 = 0; t9 < 9; t9++) {
              const uint32_t tap_lo = slot_lo + (uint32_t)(((t9 / 3) * kHaloW + (t9 % 3)) * (BK * 2 / 16));
#pragma unroll 1
              for (int kc = 0; kc < p.kchunks; kc++) {
                const uint32_t alo = tap_lo + kc * chunk_step;
                if (t9 == 0 && kc == 0) mma(tmem_d, alo, blo, 0u);
                else mma_acc(tmem_d, alo, blo);
#pragma unroll
                for (int k = 1; k < BK / 16; k++) mma_acc(tmem_d, alo + 2 * k, blo + 2 * k);
                blo += w_step;
              }
            }
            commit(&empty[q % ring]);
            commit(&pfull[q % PG]);
          }
          __syncwarp();
        }
      }
    } else
    // One elected thread runs the whole issue loop.  The waits for slice q+1 (operand slice landed / transformed,
    // TMEM group drained) are taken BEFORE the last tap of slice q is issued, while the tensor pipe still has queued
    // MMAs: the barrier round trip no longer drains the pipe at every slice boundary.
    if (elect_one()) {
      mbar_wait(wfull, 0);
      uint32_t q = 0;                                    // global slice counter (ring + P-group position)
      auto wait_slice = [&](uint32_t qq) {
        mbar_wait(&full[qq % ring], (qq / ring) & 1);
        mbar_wait(&pempty[qq % PG], ((qq / PG) & 1) ^ 1);
        tc_fence_after();
      };
      auto issue_tap = [&](int t9, uint32_t tmem_d, uint32_t slot_lo, uint32_t& blo) {
        const uint32_t tap_lo = slot_lo + (uint32_t)(((t9 / 3) * kHaloW + (t9 % 3)) * (BK * 2 / 16));
#pragma unroll 1
        for (int kc = 0; kc < p.kchunks; kc++) {
          const uint32_t alo = tap_lo + kc * chunk_step;
          if (t9 == 0 && kc == 0) mma(tmem_d, alo, blo, 0u);
          else mma_acc(tmem_d, alo, blo);
#pragma unroll
          for (int k = 1; k < BK / 16; k++) mma_acc(tmem_d, alo + 2 * k, blo + 2 * k);
          blo += w_step;
        }
      };
      // non-blocking variant: true when both barriers of slice qq have already completed
      auto try_slice = [&](uint32_t qq) -> bool {
        if (!mbar_try_wait(&full[qq % ring], (qq / ring) & 1)) return false;
        if (!mbar_try_wait(&pempty[qq % PG], ((qq / PG) & 1) ^ 1)) return false;
        tc_fence_after();
        return true;
      };
      bool ready_now = false;
      for (int col = col0; col < n_cols; col += col_step) {
        for (int sl = 0; sl < p.D; sl++, q++) {
          if (!ready_now) wait_slice(q);
          const uint32_t tmem_d = (q % PG) * (3 * PN);
          const uint32_t slot_lo = ring_lo + (q % ring) * slot_step;
          uint32_t blo = w_lo;
          const bool has_next = sl + 1 < p.D || col + col_step < n_cols;
#pragma unroll
          for (int t9 = 0; t9 < 8; t9++) issue_tap(t9, tmem_d, slot_lo, blo);
          ready_now = has_next && try_slice(q + 1);      // if it is not there yet, block after this slice's commits
          issue_tap(8, tmem_d, slot_lo, blo);
          commit(&empty[q % ring]);
          commit(&pfull[q % PG]);
        }
      }
    }
    __syncwarp();
  } else {
    // ===================== epilogue (warps 2..9) =====================
    // The epilogue (TMEM -> registers, 3-block sum, fp16 pack, store) is what bounds the low-K layers
    // (Cin = 32: 18 MMAs per slice): two warps share each TMEM lane quadrant and split the PN columns.
    constexpr int CW = PN / 2;                           // columns per warp
    const int quad = warp & 3;
    const int chalf = (warp - 2) >> 2;                   // 0: columns [0, CW), 1: [CW, PN)
    const int row = quad * 32 + lane;
    const uint32_t lane_addr = ((uint32_t)(quad * 32) << 16) + (uint32_t)(chalf * CW);
    float bias[CW];
    // UP: the bias is read from shared memory (broadcast), which keeps that epilogue within 128 registers; it sits
    // behind the scale / shift (Cin = 64, well inside the 2 x 256 floats reserved for them)
    float* s_bias = s_ab + 2 * p.cin;
    if constexpr (UP || PN == 64) {
      const int e = threadIdx.x - 64;
      if (e < PN) s_bias[e] = (p.bias && part * PN + e < p.cout) ? __ldg(p.bias + part * PN + e) : 0.f;
      named_bar_sync(1, 32 * kSlab3EpiWarps);
    } else {
#pragma unroll
      for (int j = 0; j < CW; j++) {
        const int ch = part * PN + chalf * CW + j;
        bias[j] = (p.bias && ch < p.cout) ? __ldg(p.bias + ch) : 0.f;
      }
    }
    uint32_t q0 = 0;                                    // global index of slice 0 of the current column
    uint32_t n_out = 0;                                  // output tiles staged so far (staging buffer parity)
    const bool is_issuer = warp == 2 && lane == 0;       // the thread that owns the TMA-store bulk groups
    // this thread's 16-byte chunks in the staging tile (swizzled like the store tensor map): constant per thread
    constexpr int row_b = PN * 2;                        // 128 B (SWIZZLE_128B), 64 B (SWIZZLE_64B) or 32 B (SWIZZLE_32B)
    uint32_t st_off[CW / 8];
#pragma unroll
    for (int c8 = 0; c8 < CW / 8; c8++) {
      const uint32_t off = (uint32_t)row * row_b + (uint32_t)(chalf * CW + c8 * 8) * 2;
      st_off[c8] = off ^ (((off >> 7) & (row_b == 128 ? 7u : (row_b == 64 ? 3u : 1u))) << 4);
    }
    const uint32_t s_out_u32 = smem_u32(s_out);
    for (int col = col0; col < n_cols; col += col_step, q0 += n_sl) {
      int t = col;
      const int iw = t % p.nw; t /= p.nw;
      const int ih = t % p.nh; t /= p.nh;
      const int n = t;
      // Event s = "group P(s) complete".  It finishes out(s-1) (needs P(s)[2]) and starts out(s)
      // (P(s-1)[0] + P(s)[1] + bias); after its TMEM loads P(s-1) is dead and is handed back to the MMA warp
      // BEFORE the arithmetic / stores, so the issue loop runs up to kPGroups-1 slices ahead of the stores.
      float partial[CW];
      float ssum[CW], ssq[CW];                           // fused GroupNorm statistics of this thread's row
#pragma unroll
      for (int c = 0; c < CW; c++) { ssum[c] = 0.f; ssq[c] = 0.f; }
      // statistics, fp16 pack, swizzled staging tile, one TMA store per tile (direct per-thread 16-byte stores
      // touched 16 cache lines per warp instruction and ran at ~1 TB/s)
      // split-K second launch: the partial sum the first launch left in `out` (fp16) is added; its loads are issued
      // one output slice ahead
      using PrevT = uint4[ACC ? CW / 8 : 1];
      PrevT pvq, pvq1;
      auto load_prev = [&](PrevT& pv, int od) {
        const act_t* prev = p.out + ((((long long)n * p.D + od) * p.H + ih * 16 + (row >> 3)) * p.W + iw * 8 + (row & 7)) * p.cout +
                            part * PN + chalf * CW;
#pragma unroll
        for (int c8 = 0; c8 < (ACC ? CW / 8 : 0); c8++) pv[c8] = *reinterpret_cast<const uint4*>(prev + c8 * 8);
      };
      auto emit = [&](float (&f)[CW], int od, const PrevT& pv) {
        if constexpr (ACC) {
#pragma unroll
          for (int c8 = 0; c8 < CW / 8; c8++) {
            float pf[8];
            nm_unpack8(*reinterpret_cast<const half8*>(&pv[c8]), pf);
#pragma unroll
            for (int k = 0; k < 8; k++) f[c8 * 8 + k] += pf[k];
          }
          if (!UP && od + 1 < p.D) load_prev(pvq, od + 1);   // for the next output slice: a whole slice period ahead
        }
#pragma unroll
        for (int c = 0; c < CW; c++) { ssum[c] += f[c]; ssq[c] = fmaf(f[c], f[c], ssq[c]); }
        const uint32_t boff = (n_out & 1) * stage_bytes;
        if (is_issuer) bulk_wait_read<1>();              // the store that last read this buffer has drained
        named_bar_sync(1, 32 * kSlab3EpiWarps);
#pragma unroll
        for (int c8 = 0; c8 < CW / 8; c8++) {
          const half8 hv = nm_pack8(f + c8 * 8);
          sts128(s_out_u32 + boff + st_off[c8], *reinterpret_cast<const uint4*>(&hv));
        }
        fence_async_smem();
        named_bar_sync(1, 32 * kSlab3EpiWarps);
        if (is_issuer) {
          tma_store_5d(&p.tmap_o, s_out + boff, part * PN, iw * 8, ih * 16, od, n);
          bulk_commit();
        }
        n_out++;
      };
      if constexpr (UP) {
        // Event s = "group P(s) complete", P(s)[kd] = W(kd) x(s) with x(s) = low-res plane s up-sampled in h and w.  The
        // depth-up-sampled input is h(2i) = 0.75 x(i) + 0.25 x(max(i-1, 0)), h(2i+1) = 0.75 x(i) + 0.25 x(min(i+1, Dl-1)),
        // h(-1) = h(2 Dl) = 0 (conv padding), and out(m) = sum_kd W(kd) h(m+kd-1):
        //   out(2i)   = 0.75 P(i-1)[0] + 0.25 P(i)[0] + 0.25 P(i-1)[1] + 0.75 P(i)[1] + 0.75 P(i)[2] + 0.25 P(i+1)[2]
        //   out(2i+1) = 0.25 P(i-1)[0] + 0.75 P(i)[0] + 0.75 P(i)[1] + 0.25 P(i+1)[1] + 0.25 P(i)[2] + 0.75 P(i+1)[2]
        // At the first and last slice the clamp and the zero padding only change coefficients.  Event s adds the P(s)
        // terms of pair s-1 and emits it, then starts pair s from P(s-1) and P(s) (P(s-1) is dead after that) and, at
        // the last slice, emits it too.  TMEM blocks are loaded two at a time: the register budget of the 8 warps.
        static_assert(CW == 16, "UP epilogue: 16 columns per warp");
        float part0[CW], part1[CW];                      // out(2i), out(2i+1) of the pair in flight
        for (int s = 0; s < n_sl; s++) {
          const uint32_t q = q0 + s;
          const bool first = s == 0, last = s == n_sl - 1;
          if (ACC && !first) { load_prev(pvq, 2 * s - 2); load_prev(pvq1, 2 * s - 1); }   // in flight during the wait
          mbar_wait_backoff(&pfull[q % kPGroups], (q / kPGroups) & 1, 100u);
          tc_fence_after();
          const uint32_t g_cur = lane_addr + (q % kPGroups) * (3 * PN);
          const uint32_t g_prev = lane_addr + ((q + kPGroups - 1) % kPGroups) * (3 * PN);
          uint32_t ra[CW], rb[CW];
          if (!first) {
            tmem_ld16(g_cur + PN, ra);
            tmem_ld16(g_cur + 2 * PN, rb);
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < CW; c++) {
              part0[c] = fmaf(0.25f, __uint_as_float(rb[c]), part0[c]);
              part1[c] = fmaf(0.75f, __uint_as_float(rb[c]), fmaf(0.25f, __uint_as_float(ra[c]), part1[c]));
            }
            emit(part0, 2 * s - 2, pvq);
            emit(part1, 2 * s - 1, pvq1);
          }
          tmem_ld16(g_cur, ra);
          tmem_ld16(g_cur + PN, rb);
          tmem_ld_wait();
          {
            const float a0 = first ? 0.f : 0.25f, a1 = first ? 1.f : 0.75f;
            const float e0 = first ? 1.f : 0.75f, e1 = last ? 1.f : 0.75f;
#pragma unroll
            for (int c = 0; c < CW; c++) {
              const float b = s_bias[chalf * CW + c];
              part0[c] = fmaf(a1, __uint_as_float(rb[c]), fmaf(a0, __uint_as_float(ra[c]), b));
              part1[c] = fmaf(e1, __uint_as_float(rb[c]), fmaf(e0, __uint_as_float(ra[c]), b));
            }
          }
          tmem_ld16(g_cur + 2 * PN, ra);
          if (!first) tmem_ld16(g_prev, rb);
          tmem_ld_wait();
          {
            const float a2 = last ? 1.f : 0.75f, e2 = last ? 0.f : 0.25f;
#pragma unroll
            for (int c = 0; c < CW; c++) {
              part0[c] = fmaf(a2, __uint_as_float(ra[c]), part0[c]);
              part1[c] = fmaf(e2, __uint_as_float(ra[c]), part1[c]);
            }
          }
          if (!first) {
#pragma unroll
            for (int c = 0; c < CW; c++) {
              part0[c] = fmaf(0.75f, __uint_as_float(rb[c]), part0[c]);
              part1[c] = fmaf(0.25f, __uint_as_float(rb[c]), part1[c]);
            }
            tmem_ld16(g_prev + PN, ra);
            tmem_ld_wait();
#pragma unroll
            for (int c = 0; c < CW; c++) part0[c] = fmaf(0.25f, __uint_as_float(ra[c]), part0[c]);
          }
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (!first) arrive_issuer(&pempty[(q + kPGroups - 1) % kPGroups]);
            if (last) arrive_issuer(&pempty[q % kPGroups]);
          }
          if (last) {
            if (ACC) { load_prev(pvq, 2 * s); load_prev(pvq1, 2 * s + 1); }
            emit(part0, 2 * s, pvq);
            emit(part1, 2 * s + 1, pvq1);
          }
        }
      } else if constexpr (PN == 64) {
        // N = 192: TMEM holds two groups (columns 0 and 192) and two carries: C0 (columns 384..447) = P(s)[0] raw,
        // C1 (448..511) = the partial sum of out(s).  Event s reads all of P(s) and releases it at once:
        //   out(s-1) = C1 + P(s)[2]          (emitted)
        //   C1      <- (P(s)[1] + C0) + bias (C0 = P(s-1)[0]; 0 at s = 0)
        //   C0      <- P(s)[0]
        // the same additions in the same order as the 32-channel epilogue, 8 columns at a time (register budget).
        const uint32_t c0a = lane_addr + 6 * PN, c1a = lane_addr + 7 * PN;
        auto stage = [&](const float (&f)[8], int c8) {
#pragma unroll
          for (int k = 0; k < 8; k++) { ssum[c8 * 8 + k] += f[k]; ssq[c8 * 8 + k] = fmaf(f[k], f[k], ssq[c8 * 8 + k]); }
          const half8 hv = nm_pack8(f);
          sts128(s_out_u32 + (n_out & 1) * stage_bytes + st_off[c8], *reinterpret_cast<const uint4*>(&hv));
        };
        auto store_tile = [&](int od) {
          fence_async_smem();
          named_bar_sync(1, 32 * kSlab3EpiWarps);
          if (is_issuer) {
            tma_store_5d(&p.tmap_o, s_out + (n_out & 1) * stage_bytes, part * PN, iw * 8, ih * 16, od, n);
            bulk_commit();
          }
          n_out++;
        };
        auto claim_staging = [&]() {
          if (is_issuer) bulk_wait_read<1>();              // the store that last read this buffer has drained
          named_bar_sync(1, 32 * kSlab3EpiWarps);
        };
        for (int sl = 0; sl < p.D; sl++) {
          const uint32_t q = q0 + sl;
          if (xform) mbar_wait_backoff(&pfull[q % PG], (q / PG) & 1, 100u);
          else mbar_wait(&pfull[q % PG], (q / PG) & 1);
          tc_fence_after();
          const uint32_t g = lane_addr + (q % PG) * (3 * PN);
          if (sl >= 1) claim_staging();
#pragma unroll
          for (int c8 = 0; c8 < CW / 8; c8++) {
            uint32_t ra[8], rb[8];
            if (sl >= 1) {
              tmem_ld8(g + 2 * PN + c8 * 8, ra);
              tmem_ld8(c1a + c8 * 8, rb);
              tmem_ld_wait();
              float f[8];
#pragma unroll
              for (int k = 0; k < 8; k++) f[k] = __uint_as_float(rb[k]) + __uint_as_float(ra[k]);
              stage(f, c8);
            }
            tmem_ld8(g + PN + c8 * 8, ra);
            if (sl >= 1) tmem_ld8(c0a + c8 * 8, rb);
            tmem_ld_wait();
            if (sl == 0) {
#pragma unroll
              for (int k = 0; k < 8; k++) rb[k] = 0u;
            }
#pragma unroll
            for (int k = 0; k < 8; k++)
              ra[k] = __float_as_uint((__uint_as_float(ra[k]) + __uint_as_float(rb[k])) + s_bias[chalf * CW + c8 * 8 + k]);
            tmem_st8(c1a + c8 * 8, ra);
            tmem_ld8(g + c8 * 8, rb);
            tmem_ld_wait();
            tmem_st8(c0a + c8 * 8, rb);
          }
          tmem_st_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) arrive_issuer(&pempty[q % PG]);
          if (sl >= 1) store_tile(sl - 1);
          if (sl == p.D - 1) {                             // out(D-1) = C1
            claim_staging();
#pragma unroll
            for (int c8 = 0; c8 < CW / 8; c8++) {
              uint32_t ra[8];
              tmem_ld8(c1a + c8 * 8, ra);
              tmem_ld_wait();
              float f[8];
#pragma unroll
              for (int k = 0; k < 8; k++) f[k] = __uint_as_float(ra[k]);
              stage(f, c8);
            }
            store_tile(sl);
          }
        }
      } else {
        if (ACC) load_prev(pvq, 0);
        for (int sl = 0; sl < p.D; sl++) {
          const uint32_t q = q0 + sl;
          // with producer warps in the CTA the eight epilogue warps back off between polls (isolated launch of the
          // fused 32->32 layer: 5.97 -> 5.12 ms; inside the full step the effect is within run-to-run noise)
          if (xform) mbar_wait_backoff(&pfull[q % kPGroups], (q / kPGroups) & 1, 100u);
          else mbar_wait(&pfull[q % kPGroups], (q / kPGroups) & 1);
          tc_fence_after();
          const uint32_t g_cur = lane_addr + (q % kPGroups) * (3 * PN);
          const uint32_t g_prev = lane_addr + ((q + kPGroups - 1) % kPGroups) * (3 * PN);
          uint32_t ra[CW], rb[CW], rc[CW];
          if (sl >= 1) {
            if constexpr (CW == 16) { tmem_ld16(g_cur + 2 * PN, ra); tmem_ld16(g_prev, rc); }
            else { tmem_ld8(g_cur + 2 * PN, ra); tmem_ld8(g_prev, rc); }
          } else {
#pragma unroll
            for (int c = 0; c < CW; c++) { ra[c] = 0u; rc[c] = 0u; }
          }
          if constexpr (CW == 16) tmem_ld16(g_cur + PN, rb);
          else tmem_ld8(g_cur + PN, rb);
          tmem_ld_wait();
          tc_fence_before();
          __syncwarp();
          if (lane == 0) {
            if (sl >= 1) arrive_issuer(&pempty[(q + kPGroups - 1) % kPGroups]);
            if (sl == p.D - 1) arrive_issuer(&pempty[q % kPGroups]);
          }
          // out(sl-1) is complete now; out(D-1) completes together with the last event
          if (sl >= 1) {
            float f[CW];
#pragma unroll
            for (int c = 0; c < CW; c++) f[c] = partial[c] + __uint_as_float(ra[c]);
            emit(f, sl - 1, pvq);
          }
#pragma unroll
          for (int c = 0; c < CW; c++) partial[c] = (__uint_as_float(rb[c]) + __uint_as_float(rc[c])) + bias[c];
          if (sl == p.D - 1) {
            emit(partial, sl, pvq);
          }
        }
      }
      if (p.stats) {
        // column done: fold the 32 rows of this warp (fixed butterfly order -> deterministic) and emit one
        // partial per (sample, tile column, TMEM quadrant): chunk = (ih * nw + iw) * 4 + quad
#pragma unroll
        for (int c = 0; c < CW; c++) {
#pragma unroll
          for (int o = 16; o > 0; o >>= 1) {
            ssum[c] += __shfl_xor_sync(0xffffffffu, ssum[c], o);
            ssq[c] += __shfl_xor_sync(0xffffffffu, ssq[c], o);
          }
        }
        const int chunks = p.nh * p.nw * 4;
        const long long chunk = (long long)(ih * p.nw + iw) * 4 + quad;
#pragma unroll
        for (int c = 0; c < CW; c++) {
          const int ch = part * PN + chalf * CW + c;
          if (lane == c && ch < p.cout)
            reinterpret_cast<float2*>(p.stats)[((long long)n * chunks + chunk) * p.cout + ch] = make_float2(ssum[c], ssq[c]);
        }
      }
    }
    if (is_issuer) asm volatile("cp.async.bulk.wait_group 0;" ::: "memory");
  }
  tc_fence_before();
  __syncthreads();
  if constexpr (PAIR) cluster_sync();   // no CTA of the pair leaves while the other may still arrive on its barriers
  if (warp == 1) {
    tc_fence_after();
    if constexpr (PAIR)
      asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" ::"r"(0u), "r"(tmem_cols) : "memory");
    else
      asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(0u), "r"(tmem_cols) : "memory");
  }
}

// ------------------------------------------------------------------ weight pre-pack
// nn.Conv3d weight (Cout, Cin, k, k, k) fp32 -> [tap][Cout][Cin] fp16
__global__ void pack_weights_kernel(const float* __restrict__ w, act_t* __restrict__ out, int Cout, int Cin, int taps) {
  const long long total = (long long)taps * Cout * Cin;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int ci = (int)(i % Cin);
    const int co = (int)((i / Cin) % Cout);
    const int tap = (int)(i / ((long long)Cin * Cout));
    out[i] = __float2half_rn(w[((long long)co * Cin + ci) * taps + tap]);
  }
}

typedef CUresult (*EncodeTiledFn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                  const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                  CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

EncodeTiledFn get_encode_fn() {
  static EncodeTiledFn fn = nullptr;
  if (!fn) {
    void* ptr = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &ptr, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (EncodeTiledFn)ptr;
  }
  return fn;
}

}  // namespace

extern "C" int nm_pack_conv_weights(const float* weight, void* packed, int Cout, int Cin, int k, void* stream) {
  NM_CHECK_ARG(weight && packed, "nm_pack_conv_weights: null pointer");
  const int taps = k * k * k;
  const long long total = (long long)taps * Cout * Cin;
  pack_weights_kernel<<<(int)min((total + 255) / 256, 4096LL), 256, 0, (cudaStream_t)stream>>>(weight, (act_t*)packed,
                                                                                              Cout, Cin, taps);
  NM_CHECK_LAUNCH("pack_conv_weights");
  return NM_OK;
}

// x: (n, D, H, W, Cin) fp16; packed_w: [k^3][Cout][Cin] fp16; out: (n, OD, OH, OW, Cout) fp16.
// Supported: (k=1|3, stride 1, pad (k-1)/2) and (k=2, stride 2, pad 0); Cin, Cout multiples of 8; Cout <= 256.
namespace {
// Which kernel serves this conv (slab3: conv3d_slab3_kernel, else conv3d_tc_kernel), and how many GroupNorm partial
// chunks per sample it can emit (0 = none).
struct ConvPlan { bool slab3, pair; int bk, kch, ntile, pn, ring, chunk_bytes; size_t need, w_bytes, extra; int stats_chunks; };
// wide64: a pair may serve 64 output channels per part (not for the up-sampling and split-K launches)
ConvPlan plan_conv(int n, int D, int H, int W, int Cin, int Cout, int k, int stride, bool wide64 = true) {
  ConvPlan pl;
  memset(&pl, 0, sizeof(pl));
  pl.bk = Cin >= 64 ? 64 : 32;
  pl.kch = (Cin + pl.bk - 1) / pl.bk;
  pl.ntile = ((Cout + 15) / 16) * 16;
  pl.pn = pl.kch == 1 ? 32 : 16;
  const size_t w_bytes = (size_t)27 * pl.kch * pl.pn * pl.bk * 2;
  pl.chunk_bytes = ((kHaloW * kHaloH * pl.bk * 2 + 1023) / 1024) * 1024;
  pl.ring = kSlab3Ring;
  const size_t extra = 1024 + 48 * 8 + 16 + 2 * 256 * 4 + (size_t)2 * kTileM * pl.pn * 2;
  while (pl.ring > 2 && w_bytes + (size_t)pl.ring * pl.kch * pl.chunk_bytes + extra > 227 * 1024) pl.ring--;
  pl.need = w_bytes + (size_t)pl.ring * pl.kch * pl.chunk_bytes + extra;
  pl.w_bytes = w_bytes; pl.extra = extra;
  // Measured (B200, 320 frames): with N = Cout >= 128 the tap-streaming kernel amortises the shared-memory A-operand
  // read over a wide MMA and wins over 16-channel slab3 parts: 128->128 @16^3 1.17 vs 1.32 ms, @32^3 (64 clips) 1.87
  // vs 2.11 ms.  (128->64: 8.0 vs 5.1 ms, 64->128: 0.63 vs 0.51 ms - those stay on slab3.)
  const bool wide = Cin >= 128 && Cout >= 128;
  pl.slab3 = pl.kch <= 2 && Cout % pl.pn == 0 && Cout <= 128 && !wide && k == 3 && stride == 1 && Cin >= 32 &&
             Cin % pl.bk == 0 && W % 8 == 0 && H % 16 == 0 && pl.need <= 227 * 1024;
  if (pl.slab3) {
    pl.stats_chunks = (H / 16) * (W / 8) * 4;
    // CTA pairs own two adjacent 8-wide w tiles; each CTA holds half of the weights, the freed room deepens the ring.
    // (Cin = 128 parts, PN = 16, stay on single CTAs: no pair instantiation.)
    pl.pair = pl.pn == 32 && W % 16 == 0;
    if (pl.pair) {
      // Cout % 64 == 0: one 64-channel part per pair, N = 192 (the full MMA rate; each slice is fetched, transformed and
      // read as A once per 64 channels instead of once per 32).  Each CTA then holds 96 of the 192 stacked weight rows.
      if (wide64 && Cout % 64 == 0) pl.pn = 64;
      pl.w_bytes = (size_t)27 * pl.kch * pl.pn * pl.bk;
      pl.extra = 1024 + 48 * 8 + 16 + 2 * 256 * 4 + (size_t)2 * kTileM * pl.pn * 2;
      pl.ring = kSlab3Ring;
      while (pl.ring > 2 && pl.w_bytes + (size_t)pl.ring * pl.kch * pl.chunk_bytes + pl.extra > 227 * 1024) pl.ring--;
      pl.need = pl.w_bytes + (size_t)pl.ring * pl.kch * pl.chunk_bytes + pl.extra;
      if (pl.need > 227 * 1024) pl.pair = false;   // (cannot happen for kch == 1; kept as the fit condition)
    }
  } else {
    const int OD = D / stride, OH = H / stride, OW = W / stride;
    const int tw = OW < 8 ? OW : 8, th = OH < 4 ? OH : 4, td = OD < 4 ? OD : 4;
    const bool one_sample = tw * th * td == kTileM && OW % tw == 0 && OH % th == 0 && OD % td == 0;
    pl.stats_chunks = one_sample ? (OW / tw) * (OH / th) * (OD / td) * 4 : 0;
  }
  (void)n;
  return pl;
}
}  // namespace

// Number of GroupNorm partial chunks per sample nm_conv3d_tc writes when `stats_partial` is given (0: this shape
// cannot fuse the statistics; use nm_groupnorm_scale_shift on the output instead).
extern "C" int nm_conv3d_stats_chunks(int n, int D, int H, int W, int Cin, int Cout, int k, int stride) {
  return plan_conv(n, D, H, W, Cin, Cout, k, stride).stats_chunks;
}

// 1 when nm_conv3d_tc_fused can apply the producer's GroupNorm scale/shift (+LeakyReLU) to its input on the fly
extern "C" int nm_conv3d_can_fuse_input(int n, int D, int H, int W, int Cin, int Cout, int k, int stride) {
  // Measured on B200 (320 frames): the in-smem transform pays off when the slice is not repeated by many
  // output-channel parts: 32->32 @64^3 4.95 ms plain + 2.23 ms affine pass vs 5.59 ms fused; 64->64 @32^3 1.95 + 0.69 vs
  // 2.05.  For Cin = 128 (8 parts of 16 channels) the separate HBM-bound affine pass is faster.
  const ConvPlan pl = plan_conv(n, D, H, W, Cin, Cout, k, stride);
  if (pl.slab3 && pl.kch == 1 && pl.bk == 32 && Cout <= 32) return 1;
  return pl.slab3 && pl.kch == 1 && pl.bk == 64 && Cout <= 64 ? 1 : 0;
}

extern "C" int nm_conv3d_tc_fused(const void* x, const void* packed_w, const float* bias, void* out, int n, int D,
                                  int H, int W, int Cin, int Cout, int k, int stride, const float* in_scale,
                                  const float* in_shift, int in_act, float* stats_partial, void* stream);

extern "C" int nm_conv3d_tc(const void* x, const void* packed_w, const float* bias, void* out, int n, int D, int H,
                            int W, int Cin, int Cout, int k, int stride, float* stats_partial, void* stream) {
  return nm_conv3d_tc_fused(x, packed_w, bias, out, n, D, H, W, Cin, Cout, k, stride, nullptr, nullptr, 0,
                            stats_partial, stream);
}

namespace {
int conv3d_tc_impl(const void* x, const void* packed_w, const float* bias, void* out, int n, int D, int H, int W,
                   int Cin, int Cout, int k, int stride, const float* in_scale, const float* in_shift, int in_act,
                   float* stats_partial, void* stream, bool up, int cin_total = 0, int cin_off = 0, int accum = 0);
// up-sampling mode needs the slab3<64, 32> kernel with 3 slice slots + the low-resolution plane ring
bool up2x_ok(int n, int D, int H, int W, int Cin, int Cout) {
  if ((D | H | W) & 1) return false;
  if (Cin == 128) Cin = 64;   // split-K: two launches over 64-channel slices of the low-resolution tensor
  const ConvPlan pl = plan_conv(n, D, H, W, Cin, Cout, 3, 1, false);
  return pl.slab3 && pl.bk == 64 && pl.kch == 1 && pl.pn == 32 &&
         pl.w_bytes + (size_t)3 * pl.chunk_bytes + kLoRing * kLoBytes + pl.extra <= 227 * 1024;
}
}  // namespace

extern "C" int nm_conv3d_tc_fused(const void* x, const void* packed_w, const float* bias, void* out, int n, int D,
                                  int H, int W, int Cin, int Cout, int k, int stride, const float* in_scale,
                                  const float* in_shift, int in_act, float* stats_partial, void* stream) {
  return conv3d_tc_impl(x, packed_w, bias, out, n, D, H, W, Cin, Cout, k, stride, in_scale, in_shift, in_act,
                        stats_partial, stream, false);
}

// 1 when nm_conv3d_tc_up2x serves a k3 conv with (D, H, W) OUTPUT extent
extern "C" int nm_conv3d_up2x_supported(int n, int D, int H, int W, int Cin, int Cout) {
  return up2x_ok(n, D, H, W, Cin, Cout) ? 1 : 0;
}

// out = conv3d_k3(upsample2x_trilinear(act(x_lo * in_scale + in_shift))), x_lo: (n, D/2, H/2, W/2, Cin); the
// up-sampled tensor is never written (reference: nn.Upsample(scale_factor=2, mode='trilinear') followed by
// nn.Conv3d(k3) in build_voxel_decoder, model/kypt_detector.py:385-396).  in_scale / in_shift may be null.
extern "C" int nm_conv3d_tc_up2x(const void* x_lo, const void* packed_w, const float* bias, void* out, int n, int D,
                                 int H, int W, int Cin, int Cout, const float* in_scale, const float* in_shift,
                                 int in_act, float* stats_partial, void* stream) {
  NM_CHECK_ARG(up2x_ok(n, D, H, W, Cin, Cout), "nm_conv3d_tc_up2x: unsupported shape n=%d out %dx%dx%d Cin=%d Cout=%d", n,
               D, H, W, Cin, Cout);
  if (Cin == 128) {
    // split-K (see conv3d_tc_impl): both launches interpolate their 64-channel slice of the low-resolution tensor
    NM_CHECK_ARG(!in_scale, "nm_conv3d_tc_up2x: the fused input transform is not implemented for Cin = 128");
    if (n == 0) return NM_OK;
    const int rc = conv3d_tc_impl(x_lo, packed_w, bias, out, n, D, H, W, 64, Cout, 3, 1, nullptr, nullptr, 0, nullptr, stream,
                                  true, 128, 0, 0);
    if (rc != NM_OK) return rc;
    return conv3d_tc_impl(x_lo, packed_w, nullptr, out, n, D, H, W, 64, Cout, 3, 1, nullptr, nullptr, 0, stats_partial,
                          stream, true, 128, 64, 1);
  }
  return conv3d_tc_impl(x_lo, packed_w, bias, out, n, D, H, W, Cin, Cout, 3, 1, in_scale, in_shift, in_act,
                        stats_partial, stream, true);
}

namespace {
// Clusters of two CTAs of `kern` that can be resident at once with this block size and shared memory.  It depends on
// how the SMs group into TPCs and GPCs, so it is asked of the runtime rather than taken as #SMs / 2; cached per
// (device, kernel, block size, shared memory).
cudaError_t max_resident_pairs(const void* kern, const cudaLaunchConfig_t& cfg, int* out) {
  struct Entry { int dev; const void* kern; unsigned threads; size_t smem; int pairs; };
  static std::mutex mu;
  static std::vector<Entry> cache;
  int dev = 0;
  cudaError_t e = cudaGetDevice(&dev);
  if (e != cudaSuccess) return e;
  std::lock_guard<std::mutex> lock(mu);
  for (const Entry& c : cache)
    if (c.dev == dev && c.kern == kern && c.threads == cfg.blockDim.x && c.smem == cfg.dynamicSmemBytes) {
      *out = c.pairs;
      return cudaSuccess;
    }
  cudaLaunchConfig_t probe = cfg;
  probe.gridDim = dim3(2 * nm_num_sms());
  int pairs = 0;
  e = cudaOccupancyMaxActiveClusters(&pairs, kern, &probe);
  if (e != cudaSuccess) return e;
  cache.push_back({dev, kern, cfg.blockDim.x, cfg.dynamicSmemBytes, pairs});
  *out = pairs;
  return cudaSuccess;
}

int conv3d_tc_impl(const void* x, const void* packed_w, const float* bias, void* out, int n, int D, int H, int W,
                   int Cin, int Cout, int k, int stride, const float* in_scale, const float* in_shift, int in_act,
                   float* stats_partial, void* stream, bool up, int cin_total, int cin_off, int accum) {
  NM_CHECK_ARG(x && packed_w && (bias || accum) && out, "nm_conv3d_tc: null pointer");
  if (cin_total == 0) cin_total = Cin;
  // Split-K over two launches for Cin = 128 -> Cout <= 64 (dec.1): with both 64-channel chunks of the weights
  // resident a CTA can only serve 16 output channels (N = 48 per MMA, 58 cycles for 24 cycles of tensor work); one
  // chunk at a time allows 32-channel parts (N = 96, 92 cycles for 48).  The second launch adds the fp16 partial sum
  // the first one left in `out`; GroupNorm statistics come from the second.
  if (!up && !in_scale && cin_total == Cin && Cin == 128 && Cout % 32 == 0 && Cout <= 64 && k == 3 && stride == 1 && n > 0) {
    const ConvPlan half = plan_conv(n, D, H, W, 64, Cout, k, stride, false);
    if (half.slab3 && half.pn == 32) {
      const int rc = conv3d_tc_impl(x, packed_w, bias, out, n, D, H, W, 64, Cout, k, stride, nullptr, nullptr, 0, nullptr,
                                    stream, false, 128, 0, 0);
      if (rc != NM_OK) return rc;
      return conv3d_tc_impl(x, packed_w, nullptr, out, n, D, H, W, 64, Cout, k, stride, nullptr, nullptr, 0,
                            stats_partial, stream, false, 128, 64, 1);
    }
  }
  NM_CHECK_ARG((stride == 1 && (k == 1 || k == 3)) || (stride == 2 && k == 2), "nm_conv3d_tc: k=%d stride=%d unsupported",
               k, stride);
  NM_CHECK_ARG(Cin % 8 == 0 && Cout % 8 == 0 && Cout <= 256 && Cin >= 16, "nm_conv3d_tc: Cin=%d Cout=%d unsupported", Cin,
               Cout);
  NM_CHECK_ARG(stride == 1 || (D % 2 == 0 && H % 2 == 0 && W % 2 == 0), "nm_conv3d_tc: odd extent with stride 2");
  if (n == 0) return NM_OK;
  EncodeTiledFn encode = get_encode_fn();
  if (!encode) {
    nm_set_error("nm_conv3d_tc: cuTensorMapEncodeTiled entry point not available");
    return NM_ERR_DRIVER;
  }
  // ---- slab-walking kernel: k3, weights resident in smem
  ConvPlan pl = plan_conv(n, D, H, W, Cin, Cout, k, stride, !up && cin_total == Cin);
  if (up) {
    pl.ring = 3;
    pl.need = pl.w_bytes + (size_t)3 * pl.chunk_bytes + kLoRing * kLoBytes + pl.extra;
  }
  NM_CHECK_ARG(!stats_partial || pl.stats_chunks > 0, "nm_conv3d_tc: this shape cannot fuse GroupNorm statistics");
  NM_CHECK_ARG((in_scale == nullptr) == (in_shift == nullptr), "nm_conv3d_tc: in_scale and in_shift go together");
  NM_CHECK_ARG(!in_scale || (pl.slab3 && Cin <= 256),
               "nm_conv3d_tc: this shape cannot fuse the input transform (see nm_conv3d_can_fuse_input)");
  if (pl.slab3) {
    const int bk = pl.bk, kch = pl.kch, ntile = pl.ntile, pn = pl.pn, ring = pl.ring, chunk_bytes = pl.chunk_bytes;
    const size_t need = pl.need;
    ConvSlabParams q;
    memset(&q, 0, sizeof(q));
    q.kchunks = kch; q.block_k = bk; q.n_tile = ntile; q.cout = Cout;
    q.nw = W / 8; q.nh = H / 16; q.D = D; q.H = H; q.W = W; q.N = n;
    q.chunk_bytes = chunk_bytes; q.slot_bytes = kch * chunk_bytes; q.ring = ring;
    q.bias = bias; q.out = (act_t*)out; q.stats = stats_partial;
    q.in_scale = in_scale; q.in_shift = in_shift; q.in_act = in_act; q.cin = Cin;
    q.cin_off = cin_off; q.accum = accum;
    const CUtensorMapSwizzle swz = bk == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B;
    const cuuint64_t ct = (cuuint64_t)cin_total;
    cuuint64_t dims[5] = {ct, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)n};
    cuuint64_t strides[4] = {ct * 2, (cuuint64_t)W * ct * 2, (cuuint64_t)H * W * ct * 2, (cuuint64_t)D * H * W * ct * 2};
    cuuint32_t box[5] = {(cuuint32_t)bk, kHaloW, kHaloH, 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    if (up) {   // the low-resolution tensor, (10 x 6)-row planes, linear rows (read by the transform warps)
      dims[1] = W / 2; dims[2] = H / 2; dims[3] = D / 2;
      strides[1] = (cuuint64_t)(W / 2) * ct * 2; strides[2] = (cuuint64_t)(H / 2) * (W / 2) * ct * 2;
      strides[3] = (cuuint64_t)(D / 2) * (H / 2) * (W / 2) * ct * 2;
      box[1] = 6; box[2] = 10;
    }
    CUresult r = encode(&q.tmap_a, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, (void*)x, dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, up ? CU_TENSOR_MAP_SWIZZLE_NONE : swz,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { nm_set_error("nm_conv3d_tc(slab3): cuTensorMapEncodeTiled(A) failed with %d", (int)r); return NM_ERR_DRIVER; }
    cuuint64_t wdims[3] = {ct, (cuuint64_t)Cout, 27};
    cuuint64_t wstrides[2] = {ct * 2, ct * Cout * 2};
    cuuint32_t wbox[3] = {(cuuint32_t)bk, (cuuint32_t)(pl.pair ? pn / 2 : pn), 1};
    cuuint32_t westr[3] = {1, 1, 1};
    r = encode(&q.tmap_b, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, (void*)packed_w, wdims, wstrides, wbox, westr,
               CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { nm_set_error("nm_conv3d_tc(slab3): cuTensorMapEncodeTiled(W) failed with %d", (int)r); return NM_ERR_DRIVER; }
    cuuint64_t odims[5] = {(cuuint64_t)Cout, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)n};
    cuuint64_t ostrides[4] = {(cuuint64_t)Cout * 2, (cuuint64_t)W * Cout * 2, (cuuint64_t)H * W * Cout * 2,
                              (cuuint64_t)D * H * W * Cout * 2};
    cuuint32_t obox[5] = {(cuuint32_t)pn, 8, 16, 1, 1};
    r = encode(&q.tmap_o, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, out, odims, ostrides, obox, estr,
               CU_TENSOR_MAP_INTERLEAVE_NONE,
               pn == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : (pn == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B),
               CU_TENSOR_MAP_L2_PROMOTION_NONE, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { nm_set_error("nm_conv3d_tc(slab3): cuTensorMapEncodeTiled(out) failed with %d", (int)r); return NM_ERR_DRIVER; }
    const int cols = n * q.nh * q.nw;
    const int parts = ntile / pn;
    NM_PER_DEVICE_ONCE({
      NM_CHECK_CUDA(cudaFuncSetAttribute(conv3d_slab3_kernel<64, 16>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      NM_CHECK_CUDA(cudaFuncSetAttribute(conv3d_slab3_kernel<64, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      NM_CHECK_CUDA(cudaFuncSetAttribute(conv3d_slab3_kernel<32, 32>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      NM_CHECK_CUDA(cudaFuncSetAttribute(conv3d_slab3_kernel<64, 32, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      NM_CHECK_CUDA(cudaFuncSetAttribute(conv3d_slab3_kernel<64, 32, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      NM_CHECK_CUDA(cudaFuncSetAttribute(conv3d_slab3_kernel<64, 32, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      NM_CHECK_CUDA(cudaFuncSetAttribute(conv3d_slab3_kernel<64, 32, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      NM_CHECK_CUDA(cudaFuncSetAttribute(conv3d_slab3_kernel<32, 32, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      NM_CHECK_CUDA(cudaFuncSetAttribute(conv3d_slab3_kernel<64, 64, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      NM_CHECK_CUDA(cudaFuncSetAttribute(conv3d_slab3_kernel<32, 64, false, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      NM_CHECK_CUDA(cudaFuncSetAttribute(conv3d_slab3_kernel<64, 32, true, false, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      NM_CHECK_CUDA(cudaFuncSetAttribute(conv3d_slab3_kernel<64, 32, false, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
      NM_CHECK_CUDA(cudaFuncSetAttribute(conv3d_slab3_kernel<64, 32, true, true, true>, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
    });
    // the up-sampling producer runs on 4 warps (3 working): with 6 (5 working, 144 finer items) dec.8 got slower
    // [measured, same GPU: 20.4 -> 24.6 ms per 640 frames] - more producer threads take issue slots and shared-memory
    // bandwidth from the MMA / epilogue warps; the in-place transform gains from 6 (13.2 -> 11.6 ms)
    const int threads3 = kSlab3Threads + (up ? 32 * kUpWarps : (in_scale ? 32 * kSlab3XformWarps : 0));
    NM_CHECK_ARG(!accum || (bk == 64 && pn == 32 && !in_scale), "nm_conv3d_tc: split-K accumulation needs slab3<64, 32>");
    cudaLaunchConfig_t cfg = {};
    cfg.blockDim = dim3(threads3);
    cfg.dynamicSmemBytes = need;
    cfg.stream = (cudaStream_t)stream;
    cudaLaunchAttribute cluster;
    cluster.id = cudaLaunchAttributeClusterDimension;
    cluster.val.clusterDim.x = 2; cluster.val.clusterDim.y = 1; cluster.val.clusterDim.z = 1;
    // persistent grid: one unit (CTA or CTA pair) per column and part, at most as many as can be resident
    auto launch = [&](auto kern, bool pair) -> int {
      if (!pair) {
        cfg.gridDim = dim3(cols * parts < nm_num_sms() ? cols * parts : (nm_num_sms() / parts) * parts);
        NM_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, q));
        return NM_OK;
      }
      cfg.attrs = &cluster;
      cfg.numAttrs = 1;
      int max_pairs = 0;
      NM_CHECK_ARG(max_resident_pairs((const void*)kern, cfg, &max_pairs) == cudaSuccess && max_pairs >= parts,
                   "nm_conv3d_tc(slab3): no resident CTA pairs for %d parts", parts);
      const int units = (cols / 2) * parts;
      cfg.gridDim = dim3(2 * (units < max_pairs ? units : (max_pairs / parts) * parts));
      NM_CHECK_CUDA(cudaLaunchKernelEx(&cfg, kern, q));
      return NM_OK;
    };
    int rc;
    if (pl.pair) {
      if (accum && up) rc = launch(conv3d_slab3_kernel<64, 32, true, true, true>, true);
      else if (accum) rc = launch(conv3d_slab3_kernel<64, 32, false, true, true>, true);
      else if (up) rc = launch(conv3d_slab3_kernel<64, 32, true, false, true>, true);
      else if (pn == 64 && bk == 64) rc = launch(conv3d_slab3_kernel<64, 64, false, false, true>, true);
      else if (pn == 64) rc = launch(conv3d_slab3_kernel<32, 64, false, false, true>, true);
      else if (bk == 64) rc = launch(conv3d_slab3_kernel<64, 32, false, false, true>, true);
      else rc = launch(conv3d_slab3_kernel<32, 32, false, false, true>, true);
    } else {
      if (accum && up) rc = launch(conv3d_slab3_kernel<64, 32, true, true>, false);
      else if (accum) rc = launch(conv3d_slab3_kernel<64, 32, false, true>, false);
      else if (up) rc = launch(conv3d_slab3_kernel<64, 32, true>, false);
      else if (pn == 16) rc = launch(conv3d_slab3_kernel<64, 16>, false);
      else if (bk == 64) rc = launch(conv3d_slab3_kernel<64, 32>, false);
      else rc = launch(conv3d_slab3_kernel<32, 32>, false);
    }
    if (rc != NM_OK) return rc;
    NM_CHECK_LAUNCH("conv3d_slab3");
    return NM_OK;
  }
  NM_CHECK_ARG(cin_total == Cin, "nm_conv3d_tc: split-K needs the slab3 kernel");
  ConvTcParams p;
  memset(&p, 0, sizeof(p));
  const int pad = stride == 1 ? (k - 1) / 2 : 0;
  p.taps = k * k * k;
  p.OD = D / stride; p.OH = H / stride; p.OW = W / stride; p.N = n;
  p.block_k = Cin >= 64 ? 64 : (Cin >= 32 ? 32 : 16);
  p.kchunks = (Cin + p.block_k - 1) / p.block_k;
  p.n_tile = ((Cout + 15) / 16) * 16;
  p.cout = Cout;
  p.tw = p.OW < 8 ? p.OW : 8;
  p.th = p.OH < 4 ? p.OH : 4;
  p.td = p.OD < 4 ? p.OD : 4;
  NM_CHECK_ARG(kTileM % (p.tw * p.th * p.td) == 0, "nm_conv3d_tc: output extent (%d,%d,%d) cannot be tiled", p.OD, p.OH, p.OW);
  p.tn = kTileM / (p.tw * p.th * p.td);
  NM_CHECK_ARG(p.tn <= 256, "nm_conv3d_tc: tile batch extent too large");
  p.nw = nm_cdiv(p.OW, p.tw); p.nh = nm_cdiv(p.OH, p.th); p.nd = nm_cdiv(p.OD, p.td); p.nn = nm_cdiv(n, p.tn);
  p.bias = bias;
  p.out = (act_t*)out;
  p.stats = stats_partial;
  {
    int t = 0;
    for (int a = 0; a < k; a++)
      for (int b = 0; b < k; b++)
        for (int c = 0; c < k; c++, t++) {
          if (stride == 1) { p.dz[t] = (int8_t)(a - pad); p.dy[t] = (int8_t)(b - pad); p.dx[t] = (int8_t)(c - pad); p.map[t] = 0; }
          else { p.dz[t] = p.dy[t] = p.dx[t] = 0; p.map[t] = (int8_t)t; }
        }
  }
  const CUtensorMapSwizzle swz = p.block_k == 64 ? CU_TENSOR_MAP_SWIZZLE_128B
                                 : (p.block_k == 32 ? CU_TENSOR_MAP_SWIZZLE_64B : CU_TENSOR_MAP_SWIZZLE_32B);
  // activation maps
  const int n_maps = stride == 1 ? 1 : 8;
  for (int m = 0; m < 8; m++) {
    const int mm = m < n_maps ? m : 0;
    const int a = (mm >> 2) & 1, b = (mm >> 1) & 1, c = mm & 1;
    const char* base = (const char*)x + (stride == 2 ? ((((size_t)a * H + b) * W + c) * Cin * 2) : 0);
    cuuint64_t dims[5] = {(cuuint64_t)Cin, (cuuint64_t)p.OW, (cuuint64_t)p.OH, (cuuint64_t)p.OD, (cuuint64_t)n};
    cuuint64_t strides[4] = {(cuuint64_t)stride * Cin * 2, (cuuint64_t)stride * W * Cin * 2,
                             (cuuint64_t)stride * H * W * Cin * 2, (cuuint64_t)D * H * W * Cin * 2};
    cuuint32_t box[5] = {(cuuint32_t)p.block_k, (cuuint32_t)p.tw, (cuuint32_t)p.th, (cuuint32_t)p.td, (cuuint32_t)p.tn};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = encode(&p.tmap_a[m], CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, (void*)base, dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      nm_set_error("nm_conv3d_tc: cuTensorMapEncodeTiled(A, map %d) failed with %d", m, (int)r);
      return NM_ERR_DRIVER;
    }
  }
  {
    cuuint64_t dims[3] = {(cuuint64_t)Cin, (cuuint64_t)Cout, (cuuint64_t)p.taps};
    cuuint64_t strides[2] = {(cuuint64_t)Cin * 2, (cuuint64_t)Cin * Cout * 2};
    cuuint32_t box[3] = {(cuuint32_t)p.block_k, (cuuint32_t)p.n_tile, 1};
    cuuint32_t estr[3] = {1, 1, 1};
    CUresult r = encode(&p.tmap_b, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 3, (void*)packed_w, dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, swz, CU_TENSOR_MAP_L2_PROMOTION_L2_256B,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      nm_set_error("nm_conv3d_tc: cuTensorMapEncodeTiled(W) failed with %d", (int)r);
      return NM_ERR_DRIVER;
    }
  }
  {
    cuuint64_t dims[5] = {(cuuint64_t)Cout, (cuuint64_t)p.OW, (cuuint64_t)p.OH, (cuuint64_t)p.OD, (cuuint64_t)n};
    cuuint64_t strides[4] = {(cuuint64_t)Cout * 2, (cuuint64_t)p.OW * Cout * 2, (cuuint64_t)p.OH * p.OW * Cout * 2,
                             (cuuint64_t)p.OD * p.OH * p.OW * Cout * 2};
    cuuint32_t box[5] = {32, (cuuint32_t)p.tw, (cuuint32_t)p.th, (cuuint32_t)p.td, (cuuint32_t)p.tn};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = encode(&p.tmap_o, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, out, dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_64B, CU_TENSOR_MAP_L2_PROMOTION_NONE,
                        CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) {
      nm_set_error("nm_conv3d_tc: cuTensorMapEncodeTiled(out) failed with %d", (int)r);
      return NM_ERR_DRIVER;
    }
  }
  const int stage_bytes = kTileM * p.block_k * 2 + p.n_tile * p.block_k * 2;
  int stages = (184 * 1024) / stage_bytes;
  if (stages > 8) stages = 8;
  if (stages < 2) stages = 2;
  p.stages = stages;
  const size_t smem = (size_t)stages * stage_bytes + 2 * 8192 + 1024 /*align*/ + (2 * stages + 4) * 8 + 16 + 256 * 4;
  NM_PER_DEVICE_ONCE({
    NM_CHECK_CUDA(cudaFuncSetAttribute(conv3d_tc_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, 227 * 1024));
  });
  const int total_tiles = p.nw * p.nh * p.nd * p.nn;
  const int grid = total_tiles < nm_num_sms() ? total_tiles : nm_num_sms();
  conv3d_tc_kernel<<<grid, 192, smem, (cudaStream_t)stream>>>(p);
  NM_CHECK_LAUNCH("conv3d_tc");
  return NM_OK;
}
}  // namespace
