// Heat-map heads, soft-argmax keypoints, Gaussian re-rendering and the decoder's
// 1x1 "adjust" convolution over the (never materialised) 179-channel concat.
//
// Reference:
//   heads            model/kypt_detector.py:273-297, 336-343   (LeakyReLU(1x1 conv) -> 2->1 conv -> Softplus;
//                    there is NO softmax: marginals of (hm + 1e-6) are sum-normalised)
//   soft-argmax      utils/kypt_detector_utils.py:28-55
//   Gaussian render  utils/kypt_detector_utils.py:57-90 (called per keypoint, kypt_detector.py:349-353)
//   adjust conv      model/kypt_detector.py:381,404-408 (cat[gauss_t, first_feature, gauss_0, coords] -> 128)
//
// One CTA per frame.  Shared-memory staging of the head weights, warp-shuffle reductions for
// the marginals; the feature map is read once (HBM-bound: g^3*C fp16 per frame).
#include "common.cuh"
#include "../../include/nm_b200.h"   // the definitions below must match the public declarations

namespace {

// Keypoint capacity of a kernel instantiation (compile-time bound of register and shared arrays).  K <= 24 (the shipped
// configuration) runs the kTunedK instantiations; 24 < K <= kMaxK runs a second set compiled for kMaxK.
constexpr int kTunedK = 24, kMaxK = 64;

__device__ __forceinline__ float softplus1(float x) {
  // nn.Softplus(beta=1, threshold=20)
  return x > 20.f ? x : log1pf(expf(x));
}

// Phase 1 (parallel over voxels): heat-map values on mma.sync (m16n8k16, fp16 operands, fp32 accumulate).
// grid = (g^3 / 512, n); a warp owns M-tiles of 16 consecutive voxels, K = C feature channels, N = the keypoint capacity
// (NB n-blocks).  The K order is permuted so that the 8 consecutive channels a lane loads with one 16-byte load are the
// K slots it owns in two k-steps (as in conv_pw.cu); the 1x1 conv weights are packed into B fragments once per block.
//   mode 0: heat = lrelu(w1 f + b1);  mode 1: heat = softplus(pw0 * lrelu(w1 f + b1) + pw1 * prev[clip] + pb)
__device__ __forceinline__ void head_mma(float (&c)[4], const uint32_t a0, const uint32_t a1, const uint32_t a2,
                                         const uint32_t a3, const uint2 b) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b.x), "r"(b.y));
}

// NB: n-blocks of 8 keypoints (3 for K <= 24, 8 for K <= 64).  The 3-block fragments fit in static shared memory; the
// 8-block ones (64 KB at C = 256) are dynamic (smem bytes = head_frag_bytes<C, 8>()).
template <int C, int NB>
constexpr int head_frag_bytes() { return 2 * (C / 16) * NB * 32 * (int)sizeof(uint2); }

template <int C, int NB>
__global__ void __launch_bounds__(256)
head_heat_kernel(const act_t* __restrict__ feature, const float* __restrict__ w1, const float* __restrict__ b1,
                 int K, int S, int mode, const float* __restrict__ prev, int frames_per_clip, float pw0, float pw1,
                 float pb, const float* __restrict__ prop_dev, float* __restrict__ heat) {
  if (prop_dev) { pw0 = __ldg(prop_dev); pw1 = __ldg(prop_dev + 1); pb = __ldg(prop_dev + 2); }   // live parameters
  constexpr int KS = C / 16, KC = NB * 8;
  constexpr bool kStatic = KC <= kTunedK;
  // the fp32 weights are split into fp16 hi + lo parts (two MMAs per k-step): the heat-maps keep fp32-weight accuracy
  __shared__ __align__(16) uint2 s_frag_st[kStatic ? KS * NB * 32 : 1];
  __shared__ __align__(16) uint2 s_frag_lo_st[kStatic ? KS * NB * 32 : 1];
  extern __shared__ __align__(16) uint2 s_frag_dyn[];
  uint2* s_frag = kStatic ? s_frag_st : s_frag_dyn;
  uint2* s_frag_lo = kStatic ? s_frag_lo_st : s_frag_dyn + KS * NB * 32;
  __shared__ float s_b[KC];
  const int n = blockIdx.y;
  // k-step ks = 2m + s of the 32-channel group m: slot (2t + j + 8 hi) <-> channel m*32 + t*8 + s*4 + hi*2 + j
  for (int i = threadIdx.x; i < KS * NB * 32; i += 256) {
    const int lane = i & 31, nb = (i >> 5) % NB, ks = (i >> 5) / NB;
    const int g = lane >> 2, t = lane & 3, k = nb * 8 + g;
    const int c0 = (ks >> 1) * 32 + t * 8 + (ks & 1) * 4;
    float v[4] = {0.f, 0.f, 0.f, 0.f};
    if (k < K) {
#pragma unroll
      for (int e = 0; e < 4; e++) v[e] = w1[k * C + c0 + e];
    }
    __half2 h0 = __floats2half2_rn(v[0], v[1]), h1 = __floats2half2_rn(v[2], v[3]);
    s_frag[i] = make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
    const float2 f0 = __half22float2(h0), f1 = __half22float2(h1);
    __half2 l0 = __floats2half2_rn(v[0] - f0.x, v[1] - f0.y), l1 = __floats2half2_rn(v[2] - f1.x, v[3] - f1.y);
    s_frag_lo[i] = make_uint2(*reinterpret_cast<uint32_t*>(&l0), *reinterpret_cast<uint32_t*>(&l1));
  }
  for (int i = threadIdx.x; i < KC; i += 256) s_b[i] = i < K ? b1[i] : 0.f;
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, g = lane >> 2, t = lane & 3;
  const float* pv = prev ? prev + (long long)(n / frames_per_clip) * K * S : nullptr;
  float* hm_out = heat + (long long)n * K * S;
#pragma unroll 1
  for (int it = 0; it < 4; it++) {
    const int s0 = ((blockIdx.x * 4 + it) * 8 + warp) * 16;
    if (s0 >= S) break;
    float c[NB][4];
#pragma unroll
    for (int nb = 0; nb < NB; nb++)
#pragma unroll
      for (int j = 0; j < 2; j++) c[nb][j] = c[nb][2 + j] = s_b[nb * 8 + 2 * t + j];
    const uint4* f0 = reinterpret_cast<const uint4*>(feature + ((long long)n * S + s0 + g) * C + t * 8);
    const uint4* f1 = f0 + 8 * (C / 8);
#pragma unroll
    for (int m = 0; m < C / 32; m++) {
      const uint4 r0 = __ldg(f0 + m * 4), r1 = __ldg(f1 + m * 4);
      const uint2* fr = s_frag + (2 * m) * NB * 32 + lane;
      const uint2* fl = s_frag_lo + (2 * m) * NB * 32 + lane;
#pragma unroll
      for (int nb = 0; nb < NB; nb++) {
        head_mma(c[nb], r0.x, r1.x, r0.y, r1.y, fl[nb * 32]);
        head_mma(c[nb], r0.z, r1.z, r0.w, r1.w, fl[(NB + nb) * 32]);
        head_mma(c[nb], r0.x, r1.x, r0.y, r1.y, fr[nb * 32]);
        head_mma(c[nb], r0.z, r1.z, r0.w, r1.w, fr[(NB + nb) * 32]);
      }
    }
#pragma unroll
    for (int nb = 0; nb < NB; nb++)
#pragma unroll
      for (int e = 0; e < 4; e++) {
        const int k = nb * 8 + 2 * t + (e & 1), s = s0 + g + (e >> 1) * 8;
        if (k < K) {
          float h = nm_lrelu(c[nb][e]);
          if (mode == 1) h = softplus1(fmaf(pw0, h, fmaf(pw1, pv[(long long)k * S + s], pb)));
          hm_out[(long long)k * S + s] = h;
        }
      }
  }
}

// Phase 2 (one CTA per frame): marginals of the heat-maps -> soft-argmax keypoints -> Gaussian re-render.
// heat: (n, K, g^3) fp32 written by head_heat_kernel, g in {8, 16, 32}.  Per keypoint a thread reads z rows of g
// floats (16-byte loads): the row sum feeds the x and y marginals, the row itself is accumulated into per-thread z
// partials that are folded through shared memory in a fixed order.  No float atomics: bit-reproducible run to run.
template <int KMAX>
__global__ void __launch_bounds__(256)
head_reduce_kernel(int K, int g, const float* __restrict__ lin, float gauss_width, const float* __restrict__ heat,
                   float* __restrict__ keypoints, float* __restrict__ gaussians, float* __restrict__ heat_mean) {
  extern __shared__ float smem[];
  float* s_m = smem;                       // [3][K][32] raw marginal sums along x, y, z
  float* s_kp = s_m + 3 * KMAX * 32;       // [K][4]
  float* s_e = s_kp + KMAX * 4;            // [K][3][32] separable gaussian factors
  float* s_row = s_e + KMAX * 3 * 32;      // [g*g] row sums of the current keypoint
  float* s_part = s_row + 32 * 32;         // [256 / g][g] partial z marginals
  float* s_z = s_part + 256;               // [256][g + 1] per-thread z partials, rows padded by one float
  const int n = blockIdx.x;
  const int S = g * g * g, GG = g * g, gp = g + 1;
  const int lg = g == 8 ? 3 : (g == 16 ? 4 : 5);
  const int parts = 256 >> lg;             // thread groups per z value in the z-marginal fold
  for (int k = 0; k < K; k++) {
    const float* vol = heat + ((long long)n * K + k) * S;
    float zacc[32];
#pragma unroll
    for (int i = 0; i < 32; i++) zacc[i] = 0.f;
    for (int r = threadIdx.x; r < GG; r += 256) {
      const float4* row = reinterpret_cast<const float4*>(vol + (long long)r * g);
      float sum = 0.f;
#pragma unroll
      for (int q = 0; q < 8; q++) {
        if (q < g / 4) {
          const float4 v = row[q];                                 // written by head_heat_kernel
          sum += v.x; sum += v.y; sum += v.z; sum += v.w;
          zacc[4 * q] += v.x; zacc[4 * q + 1] += v.y; zacc[4 * q + 2] += v.z; zacc[4 * q + 3] += v.w;
        }
      }
      s_row[r] = sum;
    }
#pragma unroll
    for (int i = 0; i < 32; i++)
      if (i < g) s_z[threadIdx.x * gp + i] = zacc[i];
    __syncthreads();
    {
      // z marginal: thread (part, z) folds the partials of threads part, part + parts, ...; x / y from the row sums
      const int z = threadIdx.x & (g - 1), part = threadIdx.x >> lg;
      float t = 0.f;
      for (int u = part; u < 256; u += parts) t += s_z[u * gp + z];
      s_part[part * g + z] = t;
      if (threadIdx.x < g) {
        float mx = 0.f, my = 0.f;
        for (int j = 0; j < g; j++) {
          mx += s_row[threadIdx.x * g + j];                        // x = threadIdx.x, sum over y
          my += s_row[j * g + threadIdx.x];                        // y = threadIdx.x, sum over x
        }
        s_m[(0 * KMAX + k) * 32 + threadIdx.x] = mx;
        s_m[(1 * KMAX + k) * 32 + threadIdx.x] = my;
      }
    }
    __syncthreads();
    if (threadIdx.x < g) {
      float t = 0.f;
      for (int q = 0; q < parts; q++) t += s_part[q * g + threadIdx.x];
      s_m[(2 * KMAX + k) * 32 + threadIdx.x] = t;
    }
    __syncthreads();
  }

  // ---- soft-argmax (utils/kypt_detector_utils.py:28-55)
  if (threadIdx.x < K) {
    const int k = threadIdx.x;
    float total = 0.f;
    for (int i = 0; i < g; i++) total += s_m[(0 * KMAX + k) * 32 + i];
    s_kp[k * 4 + 3] = total / (float)S;                         // mean (intensity numerator)
    if (heat_mean) heat_mean[(long long)n * K + k] = total / (float)S;   // get_keypoint_sparsity_loss input
    const float plane = (float)(g * g) * 1e-6f;                 // the +1e-6 summed over the other two axes
    for (int a = 0; a < 3; a++) {
      const float* m = s_m + (a * KMAX + k) * 32;
      float den = 0.f;
      for (int i = 0; i < g; i++) den += m[i] + plane;
      float c = 0.f;
      for (int i = 0; i < g; i++) c += ((m[i] + plane) / den) * lin[i];
      s_kp[k * 4 + a] = c;
    }
  }
  __syncthreads();
  float inten = 0.f;
  if (threadIdx.x < K) {
    float mx = -INFINITY;
    for (int k = 0; k < K; k++) mx = fmaxf(mx, s_kp[k * 4 + 3]);
    inten = s_kp[threadIdx.x * 4 + 3] / (mx + 1e-6f);
  }
  __syncthreads();
  if (threadIdx.x < K) s_kp[threadIdx.x * 4 + 3] = inten;
  __syncthreads();
  for (int i = threadIdx.x; i < K * 4; i += 256) keypoints[(long long)n * K * 4 + i] = s_kp[i];
  if (!gaussians) return;
  // ---- Gaussian re-render (utils/kypt_detector_utils.py:57-90): ((1*ex)*ey)*ez*I
  for (int i = threadIdx.x; i < K * 3 * g; i += 256) {
    const int k = i / (3 * g), a = (i / g) % 3, j = i % g;
    const float d = lin[j] - s_kp[k * 4 + a];
    s_e[(k * 3 + a) * 32 + j] = expf(-(d * d) / gauss_width);
  }
  __syncthreads();
  float* go = gaussians + (long long)n * K * S;
  // one z row (k, x, y) per thread iteration, 16-byte stores; same multiplication order as before: ((ex*ey)*ez)*I
  for (int r = threadIdx.x; r < K * GG; r += 256) {
    const int k = r / GG, xy = r - k * GG, x = xy >> lg, y = xy & (g - 1);
    const float exy = s_e[(k * 3 + 0) * 32 + x] * s_e[(k * 3 + 1) * 32 + y];
    const float inten_k = s_kp[k * 4 + 3];
    const float* ez = s_e + (k * 3 + 2) * 32;
    float4* dst = reinterpret_cast<float4*>(go + (long long)r * g);
    for (int q = 0; q < g / 4; q++)
      dst[q] = make_float4((exy * ez[4 * q]) * inten_k, (exy * ez[4 * q + 1]) * inten_k, (exy * ez[4 * q + 2]) * inten_k,
                           (exy * ez[4 * q + 3]) * inten_k);
  }
}

// Standalone render for decode_from_dyna (model/kypt_detector.py:213-231): keypoints (n,K,4) -> (n,K,g^3)
template <int KMAX>
__global__ void __launch_bounds__(256)
gaussian_render_kernel(const float* __restrict__ keypoints, int K, int g, const float* __restrict__ lin,
                       float gauss_width, float* __restrict__ gaussians) {
  __shared__ float s_e[KMAX * 3 * 32];
  __shared__ float s_i[KMAX];
  const int n = blockIdx.x;
  const int S = g * g * g;
  const float* kp = keypoints + (long long)n * K * 4;
  for (int i = threadIdx.x; i < K * 3 * g; i += 256) {
    const int k = i / (3 * g), a = (i / g) % 3, j = i % g;
    const float d = lin[j] - kp[k * 4 + a];
    s_e[(k * 3 + a) * 32 + j] = expf(-(d * d) / gauss_width);
  }
  for (int i = threadIdx.x; i < K; i += 256) s_i[i] = kp[i * 4 + 3];
  __syncthreads();
  float* go = gaussians + (long long)n * K * S;
  // one z row (k, x, y) per thread iteration, 16-byte stores; multiplication order ((ex*ey)*ez)*I as in the reference
  const int GG = g * g;
  for (int r = threadIdx.x; r < K * GG; r += 256) {
    const int k = r / GG, xy = r - k * GG, x = xy / g, y = xy - x * g;
    const float exy = (1.0f * s_e[(k * 3 + 0) * 32 + x]) * s_e[(k * 3 + 1) * 32 + y];
    const float inten = s_i[k];
    const float* ez = s_e + (k * 3 + 2) * 32;
    float4* dst = reinterpret_cast<float4*>(go + (long long)r * g);
    for (int q = 0; q < g / 4; q++)
      dst[q] = make_float4((exy * ez[4 * q]) * inten, (exy * ez[4 * q + 1]) * inten, (exy * ez[4 * q + 2]) * inten,
                           (exy * ez[4 * q + 3]) * inten);
  }
}

// ------------------------------------------------------------------ decoder adjust conv
// combined = cat[gauss_t (K), first_feature (F=128), gauss_0 (K), coords (3)]; out = lrelu(W comb + b), W (CO, 2K+F+3).
// Everything but gauss_t is constant over the frames of a clip, so it is hoisted:
//   base[clip][s][co] = b[co] + W[:,K:K+F] ff[clip][s] + W[:,K+F:2K+F] gauss_0[clip][s] + W[:,2K+F:] coords(s)
//   out[frame][s][co] = lrelu(base[clip][s][co] + W[:, :K] gauss_t[frame][s])
// Gaussians are recomputed from the keypoints (separable exps) unless a gaussians tensor is passed.
// Both parts run on mma.sync (m16n8k16, fp16 operands, fp32 accumulate) with the fragment tricks of conv_pw.cu: the
// K order is permuted so that the 8 consecutive feature channels a lane loads with one 16-byte load are the K slots
// it owns in two k-steps, and the fragment columns are permuted so that a lane owns 4 consecutive output channels
// (16-byte base loads / stores, 8-byte fp16 stores).  The Gaussian operand is evaluated straight into the A fragment
// from the separable exp tables.  coords and bias stay fp32 (CUDA cores).
constexpr int kAdjCO = 128, kAdjFD = 128, kAdjNB = kAdjCO / 8;
// uint2 per Gaussian weight block: one k-step per 16 keypoints of the capacity (2 for kTunedK, 4 for kMaxK)
template <int KMAX>
constexpr int adj_frag_g() { return (KMAX + 15) / 16 * kAdjNB * 32; }
constexpr int kAdjFragFF = (kAdjFD / 16) * kAdjNB * 32;    // first-feature block (8 k-steps)

// output channel of fragment column c (0..7) of n-block nb
__host__ __device__ inline int adj_channel(int nb, int c) { return (nb >> 1) * 16 + (c >> 1) * 4 + (nb & 1) * 2 + (c & 1); }

// frags: [gauss_t (GS k-steps)][gauss_0 (GS)][first_feature (8)] x [16 n-blocks][32 lanes]; xyzb[co] = (Wx, Wy, Wz, bias)
template <int KMAX>
__global__ void adjust_pack_kernel(const float* __restrict__ w, const float* __restrict__ bias, int K, int ld,
                                   uint2* __restrict__ frags, float4* __restrict__ xyzb) {
  constexpr int GS = (KMAX + 15) / 16;
  const int total = 2 * adj_frag_g<KMAX>() + kAdjFragFF;
  for (int i = blockIdx.x * blockDim.x + threadIdx.x; i < total; i += gridDim.x * blockDim.x) {
    const int lane = i & 31, g = lane >> 2, t = lane & 3;
    int rest = i >> 5;
    const int nb = rest % kAdjNB; rest /= kAdjNB;          // rest = k-step over the three blocks
    const int co = adj_channel(nb, g);
    float v[4];
#pragma unroll
    for (int e = 0; e < 4; e++) {
      const int j = e & 1, hi = e >> 1;
      int col;
      bool ok = true;
      if (rest < 2 * GS) {                                 // Gaussian blocks: k = s*16 + 2t + j + 8*hi
        const int k = (rest & (GS - 1)) * 16 + 2 * t + j + 8 * hi;
        ok = k < K;
        col = (rest < GS ? 0 : K + kAdjFD) + k;
      } else {                                             // first feature: ci = m*32 + t*8 + s*4 + hi*2 + j
        const int ks = rest - 2 * GS, m = ks >> 1, sst = ks & 1;
        col = K + m * 32 + t * 8 + sst * 4 + hi * 2 + j;
      }
      v[e] = ok ? w[(long long)co * ld + col] : 0.f;
    }
    __half2 b0 = __floats2half2_rn(v[0], v[1]), b1 = __floats2half2_rn(v[2], v[3]);
    frags[i] = make_uint2(*reinterpret_cast<uint32_t*>(&b0), *reinterpret_cast<uint32_t*>(&b1));
  }
  for (int co = blockIdx.x * blockDim.x + threadIdx.x; co < kAdjCO; co += gridDim.x * blockDim.x) {
    const float* wr = w + (long long)co * ld + 2 * K + kAdjFD;
    xyzb[co] = make_float4(wr[0], wr[1], wr[2], bias[co]);
  }
}

__device__ __forceinline__ void adj_mma(float (&c)[4], const uint32_t a0, const uint32_t a1, const uint32_t a2,
                                        const uint32_t a3, const uint2 b) {
  asm volatile("mma.sync.aligned.m16n8k16.row.col.f32.f16.f16.f32 {%0,%1,%2,%3}, {%4,%5,%6,%7}, {%8,%9}, {%0,%1,%2,%3};"
               : "+f"(c[0]), "+f"(c[1]), "+f"(c[2]), "+f"(c[3])
               : "r"(a0), "r"(a1), "r"(a2), "r"(a3), "r"(b.x), "r"(b.y));
}

// Gaussian A fragments (GS k-steps) of one M-tile: rows r0 / r1 are voxels s0 / s1 of frame `gn`
struct GaussSrc {
  const float* s_e;     // [K][3][32] separable exps (keypoint mode)
  const float* s_i;     // [K] intensities
  const float* gs;      // gaussians tensor of this frame (K, S) or null
  int K, g, S;
};
template <int GS>
__device__ __forceinline__ void gauss_frags(const GaussSrc& q, int s0, int s1, int t, uint32_t (&a)[GS][4]) {
  const int z0 = s0 % q.g, y0 = (s0 / q.g) % q.g, x0 = s0 / (q.g * q.g);
  const int z1 = s1 % q.g, y1 = (s1 / q.g) % q.g, x1 = s1 / (q.g * q.g);
#pragma unroll
  for (int st = 0; st < GS; st++)
#pragma unroll
    for (int hi = 0; hi < 2; hi++) {
      float v[2][2];
#pragma unroll
      for (int j = 0; j < 2; j++) {
        const int k = st * 16 + 2 * t + j + 8 * hi;
        if (k < q.K) {
          if (q.gs) {
            v[0][j] = q.gs[(long long)k * q.S + s0];
            v[1][j] = q.gs[(long long)k * q.S + s1];
          } else {
            const float* e = q.s_e + k * 96;
            v[0][j] = ((1.0f * e[x0]) * e[32 + y0]) * e[64 + z0] * q.s_i[k];
            v[1][j] = ((1.0f * e[x1]) * e[32 + y1]) * e[64 + z1] * q.s_i[k];
          }
        } else {
          v[0][j] = v[1][j] = 0.f;
        }
      }
      __half2 h0 = __floats2half2_rn(v[0][0], v[0][1]), h1 = __floats2half2_rn(v[1][0], v[1][1]);
      a[st][hi * 2] = *reinterpret_cast<uint32_t*>(&h0);       // a0 / a2: row g
      a[st][hi * 2 + 1] = *reinterpret_cast<uint32_t*>(&h1);   // a1 / a3: row g + 8
    }
}

__device__ __forceinline__ void stage_exps(const float* kp /* (K,4) of one frame */, int K, int g, const float* lin,
                                           float gauss_width, float* s_e, float* s_i) {
  for (int i = threadIdx.x; i < K * 3 * g; i += 256) {
    const int k = i / (3 * g), a = (i / g) % 3, j = i % g;
    const float d = lin[j] - kp[k * 4 + a];
    s_e[(k * 3 + a) * 32 + j] = expf(-(d * d) / gauss_width);
  }
  for (int i = threadIdx.x; i < K; i += 256) s_i[i] = kp[i * 4 + 3];
}

// base[clip][s][co] (fp32): one block = 128 voxels of one clip, one M-tile per warp
template <int KMAX>
__global__ void __launch_bounds__(256)
adjust_base_kernel(const act_t* __restrict__ ff /* (clips, S, 128) */, const float* __restrict__ kp /* (n,K,4) */,
                   const float* __restrict__ gs /* optional (n,K,S) */, int frames_per_clip,
                   const uint2* __restrict__ frags, const float4* __restrict__ xyzb, int K, int g,
                   const float* __restrict__ lin, float gauss_width, float* __restrict__ base) {
  extern __shared__ __align__(16) uint2 s_frag[];          // [gauss_0 (2)][first_feature (8)] k-steps
  __shared__ float s_e[KMAX * 3 * 32];
  __shared__ float s_i[KMAX];
  const int clip = blockIdx.y;
  const int S = g * g * g;
  for (int i = threadIdx.x; i < adj_frag_g<KMAX>() + kAdjFragFF; i += 256) s_frag[i] = __ldg(frags + adj_frag_g<KMAX>() + i);
  // gauss_0 = the gaussians of the clip's first frame (kypt_detector.py:406: gaussians[:, 0])
  if (!gs) stage_exps(kp + (long long)clip * frames_per_clip * K * 4, K, g, lin, gauss_width, s_e, s_i);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, gr = lane >> 2, t = lane & 3;
  const int s0 = (blockIdx.x * 8 + warp) * 16 + gr, s1 = s0 + 8;
  if (s0 - gr >= S) return;
  // accumulators start as bias + W_xyz coords
  float c[kAdjNB][4];
  {
    const float cx0 = lin[s0 / (g * g)], cy0 = lin[(s0 / g) % g], cz0 = lin[s0 % g];
    const float cx1 = lin[s1 / (g * g)], cy1 = lin[(s1 / g) % g], cz1 = lin[s1 % g];
#pragma unroll
    for (int nb = 0; nb < kAdjNB; nb++)
#pragma unroll
      for (int j = 0; j < 2; j++) {
        const float4 k = __ldg(xyzb + adj_channel(nb, 2 * t + j));
        c[nb][j] = fmaf(cx0, k.x, fmaf(cy0, k.y, fmaf(cz0, k.z, k.w)));
        c[nb][2 + j] = fmaf(cx1, k.x, fmaf(cy1, k.y, fmaf(cz1, k.z, k.w)));
      }
  }
  GaussSrc q{s_e, s_i, gs ? gs + (long long)clip * frames_per_clip * K * S : nullptr, K, g, S};
  constexpr int GS = (KMAX + 15) / 16;
  uint32_t a[GS][4];
  gauss_frags<GS>(q, s0, s1, t, a);
#pragma unroll
  for (int st = 0; st < GS; st++)
#pragma unroll
    for (int nb = 0; nb < kAdjNB; nb++) adj_mma(c[nb], a[st][0], a[st][1], a[st][2], a[st][3], s_frag[(st * kAdjNB + nb) * 32 + lane]);
  const uint4* f0 = reinterpret_cast<const uint4*>(ff + ((long long)clip * S + s0) * kAdjFD + t * 8);
  const uint4* f1 = reinterpret_cast<const uint4*>(ff + ((long long)clip * S + s1) * kAdjFD + t * 8);
#pragma unroll
  for (int m = 0; m < kAdjFD / 32; m++) {
    const uint4 r0 = __ldg(f0 + m * 4), r1 = __ldg(f1 + m * 4);
    const uint2* fr = s_frag + adj_frag_g<KMAX>() + (2 * m) * kAdjNB * 32 + lane;
#pragma unroll
    for (int nb = 0; nb < kAdjNB; nb++) {
      adj_mma(c[nb], r0.x, r1.x, r0.y, r1.y, fr[nb * 32]);
      adj_mma(c[nb], r0.z, r1.z, r0.w, r1.w, fr[(kAdjNB + nb) * 32]);
    }
  }
  float* b0 = base + ((long long)clip * S + s0) * kAdjCO + t * 4;
#pragma unroll
  for (int m = 0; m < kAdjNB / 2; m++) {
    *reinterpret_cast<float4*>(b0 + m * 16) = make_float4(c[2 * m][0], c[2 * m][1], c[2 * m + 1][0], c[2 * m + 1][1]);
    *reinterpret_cast<float4*>(b0 + 8 * kAdjCO + m * 16) = make_float4(c[2 * m][2], c[2 * m][3], c[2 * m + 1][2], c[2 * m + 1][3]);
  }
}

// out[frame][s][co] = lrelu(base[clip][s][co] + W[:, :K] gauss_t[frame][s]); one block = TILES*128 voxels of a frame
template <int KMAX>
__global__ void __launch_bounds__(256)
adjust_frame_kernel(const float* __restrict__ base, const float* __restrict__ kp /* (n,K,4) */,
                    const float* __restrict__ gs /* optional (n,K,S) */, const uint2* __restrict__ frags, int K, int g,
                    int frames_per_clip, int tiles_per_warp, const float* __restrict__ lin, float gauss_width,
                    act_t* __restrict__ out) {
  __shared__ __align__(16) uint2 s_frag[adj_frag_g<KMAX>()];
  __shared__ float s_e[KMAX * 3 * 32];
  __shared__ float s_i[KMAX];
  const int n = blockIdx.y, clip = n / frames_per_clip;
  const int S = g * g * g;
  for (int i = threadIdx.x; i < adj_frag_g<KMAX>(); i += 256) s_frag[i] = __ldg(frags + i);
  if (!gs) stage_exps(kp + (long long)n * K * 4, K, g, lin, gauss_width, s_e, s_i);
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31, gr = lane >> 2, t = lane & 3;
  GaussSrc q{s_e, s_i, gs ? gs + (long long)n * K * S : nullptr, K, g, S};
  for (int it = 0; it < tiles_per_warp; it++) {
    const int tile = (blockIdx.x * tiles_per_warp + it) * 8 + warp;
    if (tile * 16 >= S) break;
    const int s0 = tile * 16 + gr, s1 = s0 + 8;
    float c[kAdjNB][4];
    const float* b0 = base + ((long long)clip * S + s0) * kAdjCO + t * 4;
#pragma unroll
    for (int m = 0; m < kAdjNB / 2; m++) {
      const float4 v0 = __ldg(reinterpret_cast<const float4*>(b0 + m * 16));
      const float4 v1 = __ldg(reinterpret_cast<const float4*>(b0 + 8 * kAdjCO + m * 16));
      c[2 * m][0] = v0.x; c[2 * m][1] = v0.y; c[2 * m + 1][0] = v0.z; c[2 * m + 1][1] = v0.w;
      c[2 * m][2] = v1.x; c[2 * m][3] = v1.y; c[2 * m + 1][2] = v1.z; c[2 * m + 1][3] = v1.w;
    }
    constexpr int GS = (KMAX + 15) / 16;
    uint32_t a[GS][4];
    gauss_frags<GS>(q, s0, s1, t, a);
#pragma unroll
    for (int st = 0; st < GS; st++)
#pragma unroll
      for (int nb = 0; nb < kAdjNB; nb++)
        adj_mma(c[nb], a[st][0], a[st][1], a[st][2], a[st][3], s_frag[(st * kAdjNB + nb) * 32 + lane]);
    act_t* o0 = out + ((long long)n * S + s0) * kAdjCO + t * 4;
    const __half2 slope = __float2half2_rn(0.01f);
#pragma unroll
    for (int m = 0; m < kAdjNB / 2; m++) {
      __half2 h[4] = {__floats2half2_rn(c[2 * m][0], c[2 * m][1]), __floats2half2_rn(c[2 * m + 1][0], c[2 * m + 1][1]),
                      __floats2half2_rn(c[2 * m][2], c[2 * m][3]), __floats2half2_rn(c[2 * m + 1][2], c[2 * m + 1][3])};
#pragma unroll
      for (int e = 0; e < 4; e++) h[e] = __hmax2(h[e], __hmul2(h[e], slope));
      *reinterpret_cast<uint2*>(o0 + m * 16) = make_uint2(*reinterpret_cast<uint32_t*>(&h[0]), *reinterpret_cast<uint32_t*>(&h[1]));
      *reinterpret_cast<uint2*>(o0 + 8 * kAdjCO + m * 16) = make_uint2(*reinterpret_cast<uint32_t*>(&h[2]), *reinterpret_cast<uint32_t*>(&h[3]));
    }
  }
}

// ------------------------------------------------------------------ launchers, one per keypoint capacity
template <int C, int NB>
int launch_head_heat(dim3 grid, cudaStream_t st, const act_t* feature, const float* w1, const float* b1, int K, int S,
                      int mode, const float* prev, int frames_per_clip, float pw0, float pw1, float pb,
                      const float* prop_dev, float* heat) {
  size_t smem = 0;
  if (NB * 8 > kTunedK) {
    smem = head_frag_bytes<C, NB>();
    NM_PER_DEVICE_ONCE({
      NM_CHECK_CUDA(cudaFuncSetAttribute(head_heat_kernel<C, NB>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    });
  }
  head_heat_kernel<C, NB><<<grid, 256, smem, st>>>(feature, w1, b1, K, S, mode, prev, frames_per_clip, pw0, pw1, pb,
                                                   prop_dev, heat);
  return NM_OK;
}

template <int KMAX>
void launch_head_reduce(int n, cudaStream_t st, int K, int g, const float* lin, float gauss_width, const float* heat,
                        float* keypoints, float* gaussians, float* heat_mean) {
  const size_t smem2 = (size_t)(3 * KMAX * 32 + KMAX * 4 + KMAX * 3 * 32 + 32 * 32 + 256 + 256 * 33) * sizeof(float);
  NM_PER_DEVICE_ONCE({
    cudaFuncSetAttribute(head_reduce_kernel<KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize,
                         KMAX <= kTunedK ? 64 * 1024 : (int)smem2);
  });
  head_reduce_kernel<KMAX><<<n, 256, smem2, st>>>(K, g, lin, gauss_width, heat, keypoints, gaussians, heat_mean);
}

template <int KMAX>
int launch_adjust(const act_t* ff, const float* kp, const float* gaussians, const float* weight, const float* bias,
                  int n_clips, int frames_per_clip, int g, int K, const float* lin, float width, float* base_ws, act_t* out,
                  cudaStream_t st) {
  const int S = g * g * g;
  // workspace: [base fp32 (n_clips, S, 128)][packed weight fragments][(Wx, Wy, Wz, bias) per channel]
  uint2* frags = reinterpret_cast<uint2*>(base_ws + (size_t)n_clips * S * kAdjCO);
  float4* xyzb = reinterpret_cast<float4*>(frags + 2 * adj_frag_g<KMAX>() + kAdjFragFF);
  adjust_pack_kernel<KMAX><<<8, 256, 0, st>>>(weight, bias, K, 2 * K + kAdjFD + 3, frags, xyzb);
  NM_CHECK_LAUNCH("decoder_adjust(pack)");
  const size_t smem = (size_t)(adj_frag_g<KMAX>() + kAdjFragFF) * sizeof(uint2);
  NM_PER_DEVICE_ONCE({
    NM_CHECK_CUDA(cudaFuncSetAttribute(adjust_base_kernel<KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, 64 * 1024));
  });
  const int n = n_clips * frames_per_clip;
  adjust_base_kernel<KMAX><<<dim3(S / 128, n_clips), 256, smem, st>>>(ff, kp, gaussians, frames_per_clip, frags, xyzb, K,
                                                                       g, lin, width, base_ws);
  NM_CHECK_LAUNCH("decoder_adjust(base)");
  const int tiles_per_warp = S >= 4096 ? 4 : 1;
  adjust_frame_kernel<KMAX><<<dim3(S / (128 * tiles_per_warp), n), 256, 0, st>>>(base_ws, kp, gaussians, frags, K, g,
                                                                                  frames_per_clip, tiles_per_warp, lin,
                                                                                  width, out);
  NM_CHECK_LAUNCH("decoder_adjust(frame)");
  return NM_OK;
}

}  // namespace

extern "C" int nm_heatmap_head(const void* feature, const float* w1, const float* b1, int n, int g, int C, int K,
                               int mode, const float* prev, int frames_per_clip, float pw0, float pw1, float pb, const float* prop_dev,
                               const float* linspace, float gauss_width, float* heat, float* keypoints,
                               float* gaussians, float* heat_mean, void* stream) {
  NM_CHECK_ARG(feature && w1 && b1 && heat && linspace, "nm_heatmap_head: null pointer");
  NM_CHECK_ARG(K <= kMaxK && (g == 8 || g == 16 || g == 32), "nm_heatmap_head: K=%d g=%d unsupported", K, g);
  NM_CHECK_ARG(mode == 0 || (prev && keypoints), "nm_heatmap_head: mode 1 needs prev and keypoints");
  if (n == 0) return NM_OK;
  NM_CHECK_ARG(C == 128 || C == 256, "nm_heatmap_head: C=%d unsupported", C);
  cudaStream_t st = (cudaStream_t)stream;
  const int S = g * g * g;
  dim3 grid1(nm_cdiv(S, 512), n);
  const act_t* f = (const act_t*)feature;
  int rc;
  if (K <= kTunedK) {
    if (C == 128) rc = launch_head_heat<128, kTunedK / 8>(grid1, st, f, w1, b1, K, S, mode, prev, frames_per_clip, pw0, pw1, pb, prop_dev, heat);
    else rc = launch_head_heat<256, kTunedK / 8>(grid1, st, f, w1, b1, K, S, mode, prev, frames_per_clip, pw0, pw1, pb, prop_dev, heat);
  } else {
    if (C == 128) rc = launch_head_heat<128, kMaxK / 8>(grid1, st, f, w1, b1, K, S, mode, prev, frames_per_clip, pw0, pw1, pb, prop_dev, heat);
    else rc = launch_head_heat<256, kMaxK / 8>(grid1, st, f, w1, b1, K, S, mode, prev, frames_per_clip, pw0, pw1, pb, prop_dev, heat);
  }
  if (rc) return rc;
  NM_CHECK_LAUNCH("heatmap_head(heat)");
  if (mode == 0) return NM_OK;
  if (K <= kTunedK) launch_head_reduce<kTunedK>(n, st, K, g, linspace, gauss_width, heat, keypoints, gaussians, heat_mean);
  else launch_head_reduce<kMaxK>(n, st, K, g, linspace, gauss_width, heat, keypoints, gaussians, heat_mean);
  NM_CHECK_LAUNCH("heatmap_head(reduce)");
  return NM_OK;
}

extern "C" int nm_gaussian_render(const float* keypoints, int n, int K, int g, const float* linspace,
                                  float gauss_width, float* gaussians, void* stream) {
  NM_CHECK_ARG(keypoints && linspace && gaussians, "nm_gaussian_render: null pointer");
  NM_CHECK_ARG(K <= kMaxK && g <= 32 && g % 4 == 0, "nm_gaussian_render: K=%d g=%d unsupported", K, g);
  if (n == 0) return NM_OK;
  const float width = gauss_width;
  if (K <= kTunedK)
    gaussian_render_kernel<kTunedK><<<n, 256, 0, (cudaStream_t)stream>>>(keypoints, K, g, linspace, width, gaussians);
  else
    gaussian_render_kernel<kMaxK><<<n, 256, 0, (cudaStream_t)stream>>>(keypoints, K, g, linspace, width, gaussians);
  NM_CHECK_LAUNCH("gaussian_render");
  return NM_OK;
}

// sized for the kMaxK layout (the larger one) whatever K is, since the size does not take K
extern "C" size_t nm_decoder_adjust_workspace_bytes(int n_clips, int g) {
  return (size_t)n_clips * g * g * g * kAdjCO * sizeof(float) + (size_t)(2 * adj_frag_g<kMaxK>() + kAdjFragFF) * sizeof(uint2) +
         (size_t)kAdjCO * sizeof(float4);
}

extern "C" int nm_decoder_adjust(const void* first_feature, const float* keypoints, const float* gaussians,
                                 const float* weight, const float* bias, int n_clips, int frames_per_clip, int g,
                                 int K, const float* linspace, float gauss_width, float* base_ws, void* out,
                                 void* stream) {
  NM_CHECK_ARG(first_feature && weight && bias && base_ws && out && linspace, "nm_decoder_adjust: null pointer");
  NM_CHECK_ARG(keypoints || gaussians, "nm_decoder_adjust: need keypoints or gaussians");
  NM_CHECK_ARG(K <= kMaxK && (g == 8 || g == 16 || g == 32), "nm_decoder_adjust: K=%d g=%d unsupported", K, g);
  if (n_clips == 0) return NM_OK;
  const float* kp = gaussians ? nullptr : keypoints;
  const act_t* ff = (const act_t*)first_feature;
  if (K <= kTunedK)
    return launch_adjust<kTunedK>(ff, kp, gaussians, weight, bias, n_clips, frames_per_clip, g, K, linspace, gauss_width,
                                  base_ws, (act_t*)out, (cudaStream_t)stream);
  return launch_adjust<kMaxK>(ff, kp, gaussians, weight, bias, n_clips, frames_per_clip, g, K, linspace, gauss_width,
                              base_ws, (act_t*)out, (cudaStream_t)stream);
}
