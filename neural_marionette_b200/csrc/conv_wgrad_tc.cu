// Weight gradient of the stride-1 3x3x3 "same" convolutions on the 5th-gen tensor cores (tcgen05 + TMEM), operands fed
// by TMA - the dense third of the training step's FLOPs (config #4; autograd through modules/vox_modules.py:26,30 and
// model/kypt_detector.py:429-450).
//
//   dW[co][ci][kd][kh][kw] = sum over voxels (n, d, h, w) of  dY[n, d, h, w][co] * X[n, d+kd-1, h+kh-1, w+kw-1][ci]
//
// GEMM view: the reduction (K) runs over voxels, and both tensors are voxel-major with channels contiguous - exactly the
// MN-major operand form of tcgen05.mma.  A tile that TMA drops into shared memory (rows = voxels along w, 64 or 128
// bytes of channels per row, hardware swizzle) is consumed as it lands; nothing is transposed or copied.
//   * Taps are stacked inside one instruction through the descriptor strides:
//       A (M = 128) = X[w + jw][ci] for jw = 0.. (2 kw-shifts of 64 channels or 4 of 32): the atoms of the M dimension
//         start one voxel row (128 / 64 bytes) apart - a shifted window of the same rows;
//       B (N = 3 * CO) = dY[h + jh][co] for the three rows h-1, h, h+1 (kh = 2, 1, 0): the atoms of the N dimension
//         start one w-row of the dY tile apart.
//     One M128 x N96/192 x K16 instruction therefore produces 6 (or 9 incl. one idle slot) taps at once.
//   * A CTA owns one kd, one 32/64-channel block of Cin and of Cout and a contiguous share of the (n, d, h-tile) units;
//     its accumulators (1 or 2 groups of N columns) live in TMEM for its whole life and are written once at the end;
//     a second kernel sums the partials of all CTAs in a fixed order (bit-reproducible) into (Cout, Cin, 3, 3, 3) fp32.
//   * Zero padding of the convolution = TMA out-of-bounds fill, for X and for dY alike.
// Warp roles (192 threads): warp 0 = TMA producer, warp 1 = MMA issuer (+ TMEM alloc), warps 2-5 = epilogue.
#include "common.cuh"
#include "tc_ptx.cuh"
#include "../../include/nm_b200.h"
#include <string.h>

namespace {

using namespace tcx;

struct WgTcParams {
  CUtensorMap tmap_x;            // (Cin, W, H, D, N), box (CI, W + 3, HT, 1, 1)
  CUtensorMap tmap_y;            // (Cout, W, H, D, N), box (CO, W, HT + 2, 1, 1)
  int N, D, H, W, ht;            // ht rows of X per unit (ht * W = 256 voxels)
  int ci, co;                    // channel block sizes (32 or 64)
  int ci_blocks, co_blocks;
  int stages, x_bytes, y_bytes;
  int tmem_cols;
  float* partial;                // [split][group][mg][128][3 * co]
};

// CI / CO: channel block sizes (32 -> 64-byte rows, SW64; 64 -> 128-byte rows, SW128); KS = W / 16 K steps per w-row.
// Everything the MMA-issuing lane needs per instruction is a compile-time offset from two per-stage base words: one
// thread issues all MMAs, so every scalar instruction between two tcgen05.mma is exposed issue latency (the first,
// runtime-indexed loop spent ~160 cycles per MMA on descriptor arithmetic; the tensor work is 50-100).
template <int CI, int CO, int KS>
__global__ void __launch_bounds__(192, 1)
conv_wgrad_tc_kernel(const __grid_constant__ WgTcParams p) {
  extern __shared__ uint8_t smem_raw[];
  uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~(uintptr_t)1023);
  const int stage_bytes = (p.x_bytes + p.y_bytes + 1023) & ~1023;
  uint64_t* bars = reinterpret_cast<uint64_t*>(smem + (size_t)p.stages * stage_bytes);
  uint64_t* full = bars;
  uint64_t* empty = bars + p.stages;
  uint64_t* tfull = bars + 2 * p.stages;
  uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(tfull + 1);

  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int group = blockIdx.y;
  const int kd = group % 3, cib = (group / 3) % p.ci_blocks, cob = group / (3 * p.ci_blocks);
  const int htiles = p.H / p.ht;
  const long long units = (long long)p.N * p.D * htiles;              // < 2^31 (checked by the host)
  const int u0 = (int)(units * blockIdx.x / gridDim.x), u1 = (int)(units * (blockIdx.x + 1) / gridDim.x);
  constexpr int slots = 128 / CI;                  // kw shifts stacked along M
  constexpr int gm = (3 + slots - 1) / slots;      // M groups: 1 (CI = 32) or 2 (CI = 64)
  constexpr int ncols = 3 * CO;
  constexpr int HT = 16 / KS;                      // X rows per unit (HT * W = 256 voxels)

  if (warp == 0 && lane == 0) {
    asm volatile("prefetch.tensormap [%0];" ::"l"(&p.tmap_x) : "memory");
    asm volatile("prefetch.tensormap [%0];" ::"l"(&p.tmap_y) : "memory");
    for (int s = 0; s < p.stages; s++) {
      mbar_init(&full[s], 1);
      mbar_init(&empty[s], 1);
    }
    mbar_init(tfull, 1);
    asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
  }
  if (warp == 1) tmem_alloc(tmem_slot, (uint32_t)p.tmem_cols);
  tc_fence_before();
  __syncthreads();
  tc_fence_after();
  const uint32_t tmem_base = *tmem_slot;

  if (warp == 0) {
    // ===================== TMA producer =====================
    if (lane == 0) {
      int stage = 0;
      uint32_t phase = 0;
      for (int u = u0; u < u1; u++) {
        const int ht = u % htiles;
        const int d = (u / htiles) % p.D;
        const int n = u / (htiles * p.D);
        const int dy = d - kd + 1;                                   // plane of dY paired with X plane d
        if ((unsigned)dy >= (unsigned)p.D) continue;                 // all-zero operand: nothing to add
        mbar_wait(&empty[stage], phase ^ 1, "nm_conv3d_k3_wgrad_tc(producer)");
        uint8_t* sx = smem + (size_t)stage * stage_bytes;
        mbar_expect_tx(&full[stage], (uint32_t)(p.x_bytes + p.y_bytes));
        tma_load_5d(sx, &p.tmap_x, &full[stage], cib * p.ci, -1, ht * p.ht, d, n);
        tma_load_5d(sx + p.x_bytes, &p.tmap_y, &full[stage], cob * p.co, 0, ht * p.ht - 1, dy, n);
        if (++stage == p.stages) { stage = 0; phase ^= 1; }
      }
    }
  } else if (warp == 1) {
    // ===================== MMA issuer =====================
    // instruction descriptor: D = F32 (bit 4), A = B = F16, A and B MN-major (bits 15, 16), N >> 3 at [17,23), M >> 4 at [24,29)
    constexpr uint32_t idesc = (1u << 4) | (1u << 15) | (1u << 16) | ((uint32_t)(ncols >> 3) << 17) | ((uint32_t)(128 >> 4) << 24);
    constexpr uint32_t row_a = CI * 2, row_b = CO * 2;               // bytes per voxel row: 128 (SW128) or 64 (SW64)
    constexpr uint32_t lay_a = row_a == 128 ? 2u : 4u, lay_b = row_b == 128 ? 2u : 4u;
    const uint32_t xrow16 = ((uint32_t)(p.W + 3) * row_a) >> 4, yrow16 = ((uint32_t)p.W * row_b) >> 4;
    // descriptor words: hi = SBO (8 voxel rows) | version | layout, lo = start >> 4 | LBO << 16
    constexpr uint32_t hi_a = ((8 * row_a) >> 4) | (1u << 14) | (lay_a << 29);
    constexpr uint32_t hi_b = ((8 * row_b) >> 4) | (1u << 14) | (lay_b << 29);
    const uint32_t lbo_a = (row_a >> 4) << 16;                      // next kw shift = next voxel row
    const uint32_t lbo_b = yrow16 << 16;                            // next kh = next w-row of the dY tile
    int stage = 0;
    uint32_t phase = 0, accum = 0;
    for (int u = u0; u < u1; u++) {
      const int d = (u / htiles) % p.D;
      if ((unsigned)(d - kd + 1) >= (unsigned)p.D) continue;
      mbar_wait(&full[stage], phase, "nm_conv3d_k3_wgrad_tc(mma)");
      tc_fence_after();
      __syncwarp();
      if (elect_one()) {
        const uint32_t sx = smem_u32(smem + (size_t)stage * stage_bytes);
        uint32_t a_r = lbo_a | ((sx & 0x3FFFFu) >> 4);
        uint32_t b_r = lbo_b | (((sx + (uint32_t)p.x_bytes) & 0x3FFFFu) >> 4);
#pragma unroll
        for (int r = 0; r < HT; r++) {
#pragma unroll
          for (int ks = 0; ks < KS; ks++) {
            // B: dY rows h-1, h, h+1 (the tile starts at row h0 - 1) of the 16 voxels w = 16 ks ...
            const uint64_t db = ((uint64_t)hi_b << 32) | (b_r + (uint32_t)(ks * ((16 * row_b) >> 4)));
#pragma unroll
            for (int mg = 0; mg < gm; mg++) {
              // A: X rows (w + 1) = 16 ks + jw .. for the kw shifts jw = mg * slots + (0 .. slots - 1)
              const uint64_t da = ((uint64_t)hi_a << 32) | (a_r + (uint32_t)(((16 * ks + mg * slots) * row_a) >> 4));
              umma_f16(tmem_base + (uint32_t)(mg * ncols), da, db, idesc, (r | ks) == 0 ? accum : 1u);
            }
          }
          a_r += xrow16;
          b_r += yrow16;
        }
        umma_commit(&empty[stage]);
      }
      __syncwarp();
      accum = 1;
      if (++stage == p.stages) { stage = 0; phase ^= 1; }
    }
    if (elect_one()) umma_commit(tfull);
    __syncwarp();
  } else {
    // ===================== epilogue (warps 2..5): TMEM -> fp32 partial =====================
    const int quad = warp & 3;
    const int row = quad * 32 + lane;
    bool any = false;
    for (int u = u0; u < u1 && !any; u++) {
      const int d = (u / htiles) % p.D;
      any = (unsigned)(d - kd + 1) < (unsigned)p.D;
    }
    mbar_wait(tfull, 0, "nm_conv3d_k3_wgrad_tc(epilogue)");
    tc_fence_after();
    float* out = p.partial + (((long long)blockIdx.x * gridDim.y + group) * gm) * 128 * ncols;
    for (int mg = 0; mg < gm; mg++) {
      for (int c0 = 0; c0 < ncols; c0 += 16) {
        uint32_t v[16];
        if (any) {
          tmem_ld16(tmem_base + ((uint32_t)(quad * 32) << 16) + (uint32_t)(mg * ncols + c0), v);
          tmem_ld_wait();
        } else {
#pragma unroll
          for (int i = 0; i < 16; i++) v[i] = 0u;
        }
        float4* o = reinterpret_cast<float4*>(out + ((long long)mg * 128 + row) * ncols + c0);
#pragma unroll
        for (int i = 0; i < 4; i++)
          o[i] = make_float4(__uint_as_float(v[4 * i]), __uint_as_float(v[4 * i + 1]), __uint_as_float(v[4 * i + 2]),
                             __uint_as_float(v[4 * i + 3]));
      }
    }
  }
  tc_fence_before();
  __syncthreads();
  if (warp == 1) {
    tc_fence_after();
    tmem_dealloc(tmem_base, (uint32_t)p.tmem_cols);
  }
}

// dW[co][ci][kd][kh][kw] = out_scale * sum over the splits (fixed order)
__global__ void conv_wgrad_tc_reduce_kernel(const float* __restrict__ partial, int splits, int groups, int ci_blk, int co_blk,
                                            int ci_blocks, int Cin, int Cout, float out_scale, float* __restrict__ dw) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= (long long)Cout * Cin * 27) return;
  const int tap = (int)(i % 27), ci = (int)((i / 27) % Cin), co = (int)(i / (27LL * Cin));
  const int kd = tap / 9, kh = (tap / 3) % 3, kw = tap % 3;
  const int slots = 128 / ci_blk, gm = (3 + slots - 1) / slots, ncols = 3 * co_blk;
  const int group = kd + 3 * ((ci / ci_blk) + ci_blocks * (co / co_blk));
  const int mg = kw / slots, m = (kw % slots) * ci_blk + ci % ci_blk, ncol = (2 - kh) * co_blk + co % co_blk;
  const long long off = (((long long)group * gm + mg) * 128 + m) * ncols + ncol;
  const long long stride = (long long)groups * gm * 128 * ncols;
  float s = 0.f;
  for (int sp = 0; sp < splits; sp++) s += partial[sp * stride + off];
  dw[i] = s * out_scale;
}

struct WgPlan {
  int ci, co, ci_blocks, co_blocks, groups, splits, gm, ncols, ht, stages, x_bytes, y_bytes, tmem_cols;
  size_t smem, ws_bytes;
};

constexpr long long kWgMaxUnits = 2048;  // units (256 voxels) one CTA accumulates at most

bool wg_plan(int N, int D, int H, int W, int Cin, int Cout, WgPlan* q) {
  if (N <= 0 || D <= 0 || H <= 0 || Cin % 32 || Cout % 32 || Cin > 256 || Cout > 256 || Cin <= 0 || Cout <= 0) return false;
  if (!(W == 16 || W == 32 || W == 64 || W == 128)) return false;
  const int ht = 256 / W;
  if (H % ht) return false;
  q->ci = Cin % 64 == 0 ? 64 : 32;
  q->co = Cout % 64 == 0 ? 64 : 32;
  q->ci_blocks = Cin / q->ci;
  q->co_blocks = Cout / q->co;
  q->groups = 3 * q->ci_blocks * q->co_blocks;
  const int slots = 128 / q->ci;
  q->gm = (3 + slots - 1) / slots;
  q->ncols = 3 * q->co;
  q->ht = ht;
  q->x_bytes = ht * (W + 3) * q->ci * 2;
  q->y_bytes = (ht + 2) * W * q->co * 2;
  const int stage_bytes = (q->x_bytes + q->y_bytes + 1023) & ~1023;
  q->stages = (200 * 1024) / stage_bytes;
  if (q->stages > 4) q->stages = 4;
  if (q->stages < 2) return false;
  q->smem = (size_t)q->stages * stage_bytes + 1024 /* alignment */ + 256 /* barriers */;
  int cols = 32;
  while (cols < q->gm * q->ncols) cols <<= 1;
  q->tmem_cols = cols;
  const long long units = (long long)N * D * (H / ht);
  if (units >= (1LL << 31)) return false;
  // one wave of CTAs, repeated until no CTA sums more than kWgMaxUnits units: the tensor cores do not round the fp32
  // accumulator to nearest, so a chain's error grows with its length (~1e-9 of the largest dW entry per voxel - 1.3e-3
  // at the 64^3 layers of a 240-frame step with one wave); the splits are summed in fixed order by the reduce kernel
  long long splits = nm_num_sms() / q->groups;
  if (splits < 1) splits = 1;
  splits *= (units + splits * kWgMaxUnits - 1) / (splits * kWgMaxUnits);
  if (splits > units) splits = units;
  q->splits = (int)splits;
  q->ws_bytes = (size_t)q->splits * q->groups * q->gm * 128 * q->ncols * sizeof(float);
  return true;
}

}  // namespace

extern "C" int nm_conv3d_k3_wgrad_tc_supported(int n, int D, int H, int W, int Cin, int Cout) {
  WgPlan q;
  return wg_plan(n, D, H, W, Cin, Cout, &q) ? 1 : 0;
}

extern "C" size_t nm_conv3d_k3_wgrad_tc_workspace_bytes(int n, int D, int H, int W, int Cin, int Cout) {
  WgPlan q;
  return wg_plan(n, D, H, W, Cin, Cout, &q) ? q.ws_bytes : 0;
}

extern "C" int nm_conv3d_k3_wgrad_tc(const void* x, const void* grad_out, int n, int D, int H, int W, int Cin, int Cout,
                                     float out_scale, float* dw, void* workspace, void* stream) {
  NM_CHECK_ARG(x && grad_out && dw && workspace, "nm_conv3d_k3_wgrad_tc: null pointer");
  WgPlan q;
  NM_CHECK_ARG(wg_plan(n, D, H, W, Cin, Cout, &q),
               "nm_conv3d_k3_wgrad_tc: need Cin, Cout multiples of 32 (<= 256), W in {16, 32, 64, 128}, H a multiple of 256 / W "
               "(got %d -> %d, %d x %d x %d)", Cin, Cout, D, H, W);
  EncodeTiledFn encode = get_encode_fn();
  if (!encode) {
    nm_set_error("nm_conv3d_k3_wgrad_tc: cuTensorMapEncodeTiled entry point not available");
    return NM_ERR_DRIVER;
  }
  WgTcParams p;
  memset(&p, 0, sizeof(p));
  p.N = n; p.D = D; p.H = H; p.W = W; p.ht = q.ht; p.ci = q.ci; p.co = q.co; p.ci_blocks = q.ci_blocks; p.co_blocks = q.co_blocks;
  p.stages = q.stages; p.x_bytes = q.x_bytes; p.y_bytes = q.y_bytes; p.tmem_cols = q.tmem_cols;
  p.partial = reinterpret_cast<float*>(workspace);
  {
    const cuuint64_t c = (cuuint64_t)Cin;
    cuuint64_t dims[5] = {c, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)n};
    cuuint64_t strides[4] = {c * 2, (cuuint64_t)W * c * 2, (cuuint64_t)H * W * c * 2, (cuuint64_t)D * H * W * c * 2};
    cuuint32_t box[5] = {(cuuint32_t)q.ci, (cuuint32_t)(W + 3), (cuuint32_t)q.ht, 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = encode(&p.tmap_x, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, const_cast<void*>(x), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, q.ci == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { nm_set_error("nm_conv3d_k3_wgrad_tc: cuTensorMapEncodeTiled(x) failed with %d", (int)r); return NM_ERR_DRIVER; }
  }
  {
    const cuuint64_t c = (cuuint64_t)Cout;
    cuuint64_t dims[5] = {c, (cuuint64_t)W, (cuuint64_t)H, (cuuint64_t)D, (cuuint64_t)n};
    cuuint64_t strides[4] = {c * 2, (cuuint64_t)W * c * 2, (cuuint64_t)H * W * c * 2, (cuuint64_t)D * H * W * c * 2};
    cuuint32_t box[5] = {(cuuint32_t)q.co, (cuuint32_t)W, (cuuint32_t)(q.ht + 2), 1, 1};
    cuuint32_t estr[5] = {1, 1, 1, 1, 1};
    CUresult r = encode(&p.tmap_y, CU_TENSOR_MAP_DATA_TYPE_FLOAT16, 5, const_cast<void*>(grad_out), dims, strides, box, estr,
                        CU_TENSOR_MAP_INTERLEAVE_NONE, q.co == 64 ? CU_TENSOR_MAP_SWIZZLE_128B : CU_TENSOR_MAP_SWIZZLE_64B,
                        CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
    if (r != CUDA_SUCCESS) { nm_set_error("nm_conv3d_k3_wgrad_tc: cuTensorMapEncodeTiled(grad_out) failed with %d", (int)r); return NM_ERR_DRIVER; }
  }
  cudaStream_t st = (cudaStream_t)stream;
  const dim3 grid(q.splits, q.groups);
  int rc = NM_OK;
#define NM_WG_LAUNCH(CI_, CO_, KS_)                                                                                              \
  do {                                                                                                                           \
    cudaError_t e_ = cudaFuncSetAttribute(conv_wgrad_tc_kernel<CI_, CO_, KS_>, cudaFuncAttributeMaxDynamicSharedMemorySize,      \
                                          (int)q.smem);                                                                          \
    if (e_ != cudaSuccess) { nm_set_error("nm_conv3d_k3_wgrad_tc: cudaFuncSetAttribute: %s", cudaGetErrorString(e_)); rc = NM_ERR_CUDA; } \
    else conv_wgrad_tc_kernel<CI_, CO_, KS_><<<grid, 192, q.smem, st>>>(p);                                                      \
  } while (0)
#define NM_WG_KS(CI_, CO_)                                          \
  do {                                                              \
    if (W == 16) NM_WG_LAUNCH(CI_, CO_, 1);                         \
    else if (W == 32) NM_WG_LAUNCH(CI_, CO_, 2);                    \
    else if (W == 64) NM_WG_LAUNCH(CI_, CO_, 4);                    \
    else NM_WG_LAUNCH(CI_, CO_, 8);                                 \
  } while (0)
  if (q.ci == 32 && q.co == 32) NM_WG_KS(32, 32);
  else if (q.ci == 32) NM_WG_KS(32, 64);
  else if (q.co == 32) NM_WG_KS(64, 32);
  else NM_WG_KS(64, 64);
#undef NM_WG_KS
#undef NM_WG_LAUNCH
  if (rc != NM_OK) return rc;
  NM_CHECK_LAUNCH("conv_wgrad_tc_kernel");
  conv_wgrad_tc_reduce_kernel<<<nm_cdiv((long long)Cout * Cin * 27, 256), 256, 0, st>>>(
      reinterpret_cast<const float*>(workspace), q.splits, q.groups, q.ci, q.co, q.ci_blocks, Cin, Cout, out_scale, dw);
  NM_CHECK_LAUNCH("conv_wgrad_tc_reduce_kernel");
  return NM_OK;
}
