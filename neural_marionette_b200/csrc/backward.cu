// Backward kernels of the detector's non-convolution stages and of its first layer (config #4 training step).
// What torch.autograd computes for the reference, restated per stage:
//   trilinear x2 up-sampling      model/kypt_detector.py:427,441           -> nm_upsample2x_backward
//   decoder tail + BCE            model/kypt_detector.py:410,453-457,91-92 -> nm_final_recon_backward
//   heat-map heads + soft-argmax  model/kypt_detector.py:273-297,336-343; utils/kypt_detector_utils.py:28-55
//                                                                          -> nm_heatmap_head_backward
//   Gaussian render + adjust conv utils/kypt_detector_utils.py:57-90; model/kypt_detector.py:381,404-408
//                                                                          -> nm_decoder_adjust_backward
//   chamfer volume-fitting loss   utils/kypt_detector_utils.py:141-157     -> nm_chamfer_vol_fit_backward
//   CoordConv first layer         utils/kypt_detector_utils.py:4-26 + modules/vox_modules.py:12 -> nm_first_conv_wgrad
//   Adam                          train.py:380-409 (torch.optim.Adam defaults) -> nm_adam_step
// Activation gradients travel as fp16 multiplied by a loss scale (`grad_scale`); every fp32 output (parameter and
// keypoint gradients) is divided by it again (`inv_scale`).  All reductions run in a fixed order: bit-reproducible.
#include "common.cuh"
#include "../../include/nm_b200.h"

namespace {

// Keypoint capacity of the heat-map / adjust / chamfer backward kernels: K <= kTunedK (the shipped 24) runs the tuned
// instantiations, 24 < K <= kMaxK a set compiled for kMaxK (template parameter KMAX).
constexpr int kTunedK = 24, kMaxK = 64;

// ------------------------------------------------------------------ trilinear x2 backward
// d_in[i] = sum_{j in -1..2} w_j * g[clamp(2i + j)], w = (.25, .75, .75, .25) per axis (the transpose of PyTorch's
// align_corners=False rule incl. its index clamping at the borders).  The 64-tap stencil is separable: three passes
// (w, then h, then d), each halving one axis with 4 taps per output: [outer][2L][inner] -> [outer][L][inner] in 16-byte
// units of 8 channels.  A one-pass version reads every gradient value 8 x (64 GB through L2 for the decoder's 64^3 layer,
// 9.6 ms); the passes move 8 + 4 + 4 + 2 + 2 + 1 = 21 GB.  fp32 arithmetic inside a pass, fp16 between passes.
// POW2: L and inner8 are powers of two (every shape of the model): the index decomposition is two shifts and two masks
// instead of four 64-bit divisions per 16-byte output (which held the passes at 4.9 TB/s).
template <bool POW2>
__global__ void __launch_bounds__(256)
upsample2x_bwd_axis_kernel(const __half* __restrict__ g, __half* __restrict__ out, long long outer, int L, long long inner8,
                           long long total8, int log_inner8, int log_L) {
#pragma unroll 2
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total8; i += (long long)gridDim.x * 256) {
    long long in8, o;
    int l;
    if (POW2) {
      in8 = i & (inner8 - 1);
      const long long r = i >> log_inner8;
      l = (int)(r & (L - 1));
      o = r >> log_L;
    } else {
      in8 = i % inner8;
      const long long r = i / inner8;
      l = (int)(r % L);
      o = r / L;
    }
    const half8* base = reinterpret_cast<const half8*>(g) + (o * (2LL * L)) * inner8 + in8;
    const int j0 = max(2 * l - 1, 0), j3 = min(2 * l + 2, 2 * L - 1);
    float f0[8], f1[8], f2[8], f3[8], acc[8];
    nm_unpack8(base[(long long)j0 * inner8], f0);
    nm_unpack8(base[(long long)(2 * l) * inner8], f1);
    nm_unpack8(base[(long long)(2 * l + 1) * inner8], f2);
    nm_unpack8(base[(long long)j3 * inner8], f3);
#pragma unroll
    for (int k = 0; k < 8; k++) acc[k] = 0.25f * (f0[k] + f3[k]) + 0.75f * (f1[k] + f2[k]);
    reinterpret_cast<half8*>(out)[i] = nm_pack8(acc);
  }
}

// ------------------------------------------------------------------ depth-to-space (k2/s2 transposed conv as a 1x1 conv)
// The data gradient of a k2/s2 "pool" conv is a transposed conv: out[2v + t][ci] = sum_co W[co][ci][t] dy[v][co].  For
// wide layers it runs as a 1x1 convolution dy -> (taps, ci) on the tensor cores (nm_conv3d_tc); this kernel scatters the
// tap-major result y (n, D, H, W, ntaps, C) of taps tap0 .. tap0 + ntaps - 1 to their voxels of out (n, 2D, 2H, 2W, C).
__global__ void __launch_bounds__(256)
depth_to_space2_kernel(const __half* __restrict__ y, __half* __restrict__ out, int D, int H, int W, int C, int tap0, int ntaps,
                       long long total8) {
  const int c8n = C >> 3;
  for (long long i = (long long)blockIdx.x * 256 + threadIdx.x; i < total8; i += (long long)gridDim.x * 256) {
    int c8, tl, w, h, d;
    long long n;
    if (total8 <= 0x7fffffffLL) {                 // 32-bit index arithmetic (a 64-bit division costs ~4x as much)
      unsigned r = (unsigned)i;
      c8 = (int)(r % (unsigned)c8n); r /= (unsigned)c8n;
      tl = (int)(r % (unsigned)ntaps); r /= (unsigned)ntaps;
      w = (int)(r % (unsigned)W); r /= (unsigned)W;
      h = (int)(r % (unsigned)H); r /= (unsigned)H;
      d = (int)(r % (unsigned)D);
      n = r / (unsigned)D;
    } else {
      c8 = (int)(i % c8n);
      long long r = i / c8n;
      tl = (int)(r % ntaps); r /= ntaps;
      w = (int)(r % W); r /= W;
      h = (int)(r % H); r /= H;
      d = (int)(r % D);
      n = r / D;
    }
    const int t = tap0 + tl;
    const long long o = (((n * (2 * D) + 2 * d + (t >> 2)) * (2 * H) + 2 * h + ((t >> 1) & 1)) * (2 * W) + 2 * w + (t & 1)) * C + c8 * 8;
    *reinterpret_cast<uint4*>(out + o) = reinterpret_cast<const uint4*>(y)[i];
  }
}

// ------------------------------------------------------------------ decoder tail backward
// forward: act = lrelu(x*a + b); x14 = w . act + bias; p = sigmoid(sharp * (tanh(x14) + ff - trans)); bce = mean BCE(p, y)
// backward (PyTorch's binary_cross_entropy_backward: (p - y) / max(p (1 - p), 1e-12)):
//   dx14 = gbce[n] / S * (p - y) * [p(1-p) / max(p(1-p), 1e-12)] * sharp * (1 - tanh^2(x14))
//   dact[c] = w[c] * dx14 (written fp16, times grad_scale);  dw[c] = sum act[c] * dx14;  dbias = sum dx14
constexpr int kFrbBlocks = 64;
__global__ void __launch_bounds__(256)
final_recon_bwd_kernel(const __half* __restrict__ x, const float* __restrict__ a, const float* __restrict__ b,
                       const float* __restrict__ w, float bias, const float* __restrict__ bias_dev,
                       const float* __restrict__ first_frame, int frames_per_clip,
                       float sharp, float trans, const float* __restrict__ recon, const float* __restrict__ target,
                       const float* __restrict__ gbce, float grad_scale, __half* __restrict__ dact,
                       float* __restrict__ partial /* [n][blocks][33] */, int S) {
  constexpr int C = 32;
  if (bias_dev) bias = __ldg(bias_dev);
  const int n = blockIdx.y;
  __shared__ float sa[C], sb[C], sw[C];
  __shared__ float red[8][C + 1];
  if (threadIdx.x < C) {
    sa[threadIdx.x] = a[(long long)n * C + threadIdx.x];
    sb[threadIdx.x] = b[(long long)n * C + threadIdx.x];
    sw[threadIdx.x] = w[threadIdx.x];
  }
  __syncthreads();
  const int clip = n / frames_per_clip;
  const float gn = gbce[n] / (float)S;
  float dw[C], db = 0.f;
#pragma unroll
  for (int c = 0; c < C; c++) dw[c] = 0.f;
  const half8* base = reinterpret_cast<const half8*>(x + (long long)n * S * C);
  half8* obase = reinterpret_cast<half8*>(dact + (long long)n * S * C);
  for (int s = blockIdx.x * 256 + threadIdx.x; s < S; s += gridDim.x * 256) {
    half8 raw[4];
#pragma unroll
    for (int j = 0; j < 4; j++) raw[j] = base[(long long)s * 4 + j];
    float act[C];
    float x14 = bias;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      float f[8];
      nm_unpack8(raw[j], f);
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const int c = j * 8 + k;
        act[c] = nm_lrelu(fmaf(f[k], sa[c], sb[c]));
        x14 = fmaf(act[c], sw[c], x14);
      }
    }
    const float t = tanhf(x14);
    const float p = recon[(long long)n * S + s], y = target[(long long)n * S + s];
    (void)first_frame; (void)clip; (void)trans;                         // p already contains them (saved forward output)
    const float pq = p * (1.f - p);
    const float dx14 = gn * (p - y) * (pq / fmaxf(pq, 1e-12f)) * sharp * (1.f - t * t);
    db += dx14;
    const float ds = dx14 * grad_scale;
#pragma unroll
    for (int j = 0; j < 4; j++) {
      float o[8];
#pragma unroll
      for (int k = 0; k < 8; k++) {
        const int c = j * 8 + k;
        dw[c] = fmaf(act[c], dx14, dw[c]);
        o[k] = sw[c] * ds;
      }
      obase[(long long)s * 4 + j] = nm_pack8(o);
    }
  }
  // block reduction: butterfly inside the warp, then the 8 warps in order
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
#pragma unroll
  for (int c = 0; c < C; c++) {
    const float v = nm_warp_sum(dw[c]);
    if (lane == 0) red[warp][c] = v;
  }
  db = nm_warp_sum(db);
  if (lane == 0) red[warp][C] = db;
  __syncthreads();
  if (threadIdx.x <= C) {
    float tot = 0.f;
    for (int k = 0; k < 8; k++) tot += red[k][threadIdx.x];
    partial[((long long)n * gridDim.x + blockIdx.x) * (C + 1) + threadIdx.x] = tot;
  }
}

// out[j] = scale * sum_r partial[r * ld + j], j < cols: fp64, fixed order (8 interleaved row groups per column, combined
// in order).  Launch with blockDim (32, 8).
__global__ void __launch_bounds__(256)
reduce_cols_kernel(const float* __restrict__ partial, long long rows, int ld, int cols, float scale, float* __restrict__ out) {
  __shared__ double red[8][32];
  const int j = blockIdx.x * 32 + threadIdx.x;
  double acc = 0.0;
  if (j < cols)
    for (long long r = threadIdx.y; r < rows; r += 8) acc += (double)partial[r * ld + j];
  red[threadIdx.y][threadIdx.x] = acc;
  __syncthreads();
  if (threadIdx.y == 0 && j < cols) {
    double t = 0.0;
#pragma unroll
    for (int y = 0; y < 8; y++) t += red[y][threadIdx.x];
    out[j] = (float)(t * (double)scale);
  }
}

// ------------------------------------------------------------------ heat-map head backward
// mode 1 (per-frame head): u = w1 f + b1; h = lrelu(u); q = pw0 h + pw1 prev + pb; hm = softplus(q);
//   keypoints / heat_mean are functions of hm:  d hm[k][s] = A_k + sum_a B_ka lin[s_a]  (+ dheat[k][s]) with
//     den_k = S (mean_k + 1e-6),  B_ka = dkp[k][a] / den_k,  A_k = dmean_k / S - sum_a B_ka kp[k][a],
//     dmean_k = dkp[k][3] / (mx + 1e-6) + dmean_up[k] - [k == argmax] sum_j dkp[j][3] mean_j / (mx + 1e-6)^2
//   dq = dhm * (1 - exp(-hm));  du = pw0 dq lrelu'(u)
// mode 0 (spatio-temporal head): h = lrelu(u) is the output; dh[k][s] = pw1 * sum_t dq[clip*T + t][k][s]
// outputs: dfeat = grad_scale * W1^T du (fp16), dq (mode 1), per-frame partials of dW1, db1, (dpw0, dpw1, dpb).
// Work split: grid (frame, voxel split); a CTA walks its share of the S / 64 voxel tiles.  All three contractions are
// register-tiled over shared memory (the first version did one FMA per two shared loads and was bound by the LDS pipe:
// 2.05 ms for 240 frames, 2.7 ms for the 24 clips of the 256-channel head on 24 CTAs):
//   u  [k][s] = w1 f      thread = (voxel, 6 keypoints): per 4 channels 1 LDS.128 of f + 6 broadcast LDS.128 of w1, 24 FMA
//   dfeat[s][c] = W1^T du thread = (4 voxels, 8 channels): per keypoint 1 + 2 LDS.128, 32 FMA
//   dW1[k][c] += du f^T   thread = (channel, 12 or 24 keypoints): per voxel 1 LDS + 3 or 6 broadcast LDS.128, 12 or 24 FMA
// At capacity 64 the dW1 tile is split over blockIdx.z: block z owns keypoints [KW z, KW z + KW) of dW1 (KW = 32 at
// C = 128, 16 at C = 256: 16 accumulators per thread instead of 32 or 64, which spill); every z computes u and du for all
// keypoints, only z = 0 writes dfeat, dq, db1 and the propagation partials.
template <int C, int KMAX>
constexpr int head_bwd_kw() { return KMAX <= kTunedK ? KMAX : (C == 256 ? 16 : 32); }

template <int C, int KMAX>
__global__ void __launch_bounds__(256)
head_bwd_kernel(const __half* __restrict__ feature, const float* __restrict__ w1, const float* __restrict__ b1, int K, int g,
                int mode, const float* __restrict__ prev, int frames_per_clip, float pw0, float pw1, float pb,
                const float* __restrict__ prop_dev,
                const float* __restrict__ lin, const float* __restrict__ heat, const float* __restrict__ kp,
                const float* __restrict__ heat_mean, const float* __restrict__ dkp, const float* __restrict__ dmean_up,
                const float* __restrict__ dheat, const float* __restrict__ dq_in, float grad_scale,
                __half* __restrict__ dfeat, float* __restrict__ dq_out, float* __restrict__ pw_partial /* [n*splits][K][C] */,
                float* __restrict__ pb_partial /* [n*splits][K] */, float* __restrict__ pp_partial /* [n*splits][3] */) {
  if (prop_dev) { pw0 = __ldg(prop_dev); pw1 = __ldg(prop_dev + 1); pb = __ldg(prop_dev + 2); }   // live parameters
  constexpr int TS = 64;                                   // voxels per tile
  constexpr int FS = C + 4;                                // fp32 feature row stride: 16-byte aligned rows, conflict-free LDS.128
  constexpr int KW = head_bwd_kw<C, KMAX>();               // keypoints of dW1 per block
  constexpr int KPT = KW * C / 256;                        // dW1 accumulators per thread (12 or 24; 16 at 64)
  const bool lead = KW == KMAX || blockIdx.z == 0;         // writes dfeat, dq, db1 and the propagation partials
  constexpr int NC8 = C / 8, VPT = TS / (256 / NC8);       // dfeat: voxels per thread (4 or 8, in rounds of 4)
  extern __shared__ __align__(16) float smem[];
  float* s_w = smem;                                       // [KMAX][C]
  float* s_f = s_w + KMAX * C;                             // [TS][FS]
  float* s_du = s_f + TS * FS;                             // [KMAX][TS]
  float* s_duT = s_du + KMAX * TS;                         // [TS][KMAX]
  float* s_co = s_duT + TS * KMAX;                         // [KMAX][4]: A, Bx, By, Bz
  float* s_red = s_co + KMAX * 4;                          // [256][3]
  const int n = blockIdx.x, S = g * g * g;
  const int tiles = (S / TS) / gridDim.y, tile0 = blockIdx.y * tiles;
  const long long part = (long long)n * gridDim.y + blockIdx.y;
  const int clip = n / frames_per_clip;
  for (int i = threadIdx.x; i < KMAX * C; i += 256) s_w[i] = (i / C) < K ? w1[i] : 0.f;
  if (mode == 1 && threadIdx.x < KMAX) {
    const int k = threadIdx.x;
    float A = 0.f, B[3] = {0.f, 0.f, 0.f};
    if (k < K) {
      const float* hmn = heat_mean + (long long)n * K;
      float mx = -INFINITY;
      int jm = 0;
      for (int j = 0; j < K; j++)
        if (hmn[j] > mx) { mx = hmn[j]; jm = j; }            // first maximum, as torch.max
      const float inv = 1.f / (mx + 1e-6f);
      float dmean = dmean_up ? dmean_up[(long long)n * K + k] : 0.f;
      if (dkp) {
        dmean += dkp[((long long)n * K + k) * 4 + 3] * inv;
        if (k == jm) {
          float t = 0.f;
          for (int j = 0; j < K; j++) t += dkp[((long long)n * K + j) * 4 + 3] * hmn[j];
          dmean -= t * inv * inv;
        }
      }
      const float den = (float)S * (hmn[k] + 1e-6f);
      A = dmean / (float)S;
      if (dkp)
        for (int a = 0; a < 3; a++) {
          B[a] = dkp[((long long)n * K + k) * 4 + a] / den;
          A -= B[a] * kp[((long long)n * K + k) * 4 + a];
        }
    }
    s_co[k * 4] = A; s_co[k * 4 + 1] = B[0]; s_co[k * 4 + 2] = B[1]; s_co[k * 4 + 3] = B[2];
  }
  __syncthreads();
  float accw[KPT];
#pragma unroll
  for (int i = 0; i < KPT; i++) accw[i] = 0.f;
  float accb = 0.f, sp0 = 0.f, sp1 = 0.f, sp2 = 0.f;
  const int wc = threadIdx.x % C, wk0 = (KW == KMAX ? 0 : blockIdx.z * KW) + (threadIdx.x / C) * KPT;   // dW1: channel wc, keypoints wk0..
  const __half* fbase = feature + (long long)n * S * C;
  for (int tile = tile0; tile < tile0 + tiles; tile++) {
    const int s0 = tile * TS;
    // feature tile -> fp32 shared (4 channels per thread: conflict-free 16-byte stores)
    for (int i = threadIdx.x; i < TS * (C / 4); i += 256) {
      const int sl = i / (C / 4), c4 = i % (C / 4);
      const uint2 raw = *reinterpret_cast<const uint2*>(fbase + (long long)(s0 + sl) * C + c4 * 4);
      const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&raw.x));
      const float2 hi = __half22float2(*reinterpret_cast<const __half2*>(&raw.y));
      *reinterpret_cast<float4*>(s_f + sl * FS + c4 * 4) = make_float4(lo.x, lo.y, hi.x, hi.y);
    }
    __syncthreads();
    {
      // u, dq, du for 6 keypoints of one voxel
      constexpr int KG = KMAX / 4;
      const int sl = threadIdx.x % TS, kg = threadIdx.x / TS, s = s0 + sl;
      float u[KG];
#pragma unroll
      for (int j = 0; j < KG; j++) u[j] = kg * KG + j < K ? b1[kg * KG + j] : 0.f;
      const float* fr = s_f + sl * FS;
      const float* wr = s_w + kg * KG * C;
#pragma unroll 2
      for (int c = 0; c < C; c += 4) {
        const float4 f = *reinterpret_cast<const float4*>(fr + c);
#pragma unroll
        for (int j = 0; j < KG; j++) {
          const float4 w = *reinterpret_cast<const float4*>(wr + j * C + c);
          u[j] = fmaf(w.x, f.x, fmaf(w.y, f.y, fmaf(w.z, f.z, fmaf(w.w, f.w, u[j]))));
        }
      }
      const int x = s / (g * g), y = (s / g) % g, z = s % g;
      const float lx = lin[x], ly = lin[y], lz = lin[z];
#pragma unroll
      for (int j = 0; j < KG; j++) {
        const int k = kg * KG + j;
        float du = 0.f;
        if (k < K) {
          const float slope = u[j] > 0.f ? 1.f : 0.01f;
          float dh;
          if (mode == 1) {
            const float h = u[j] > 0.f ? u[j] : 0.01f * u[j];
            const float pv = prev[((long long)clip * K + k) * S + s];
            const float hm = heat[((long long)n * K + k) * S + s];
            float dhm = s_co[k * 4] + s_co[k * 4 + 1] * lx + s_co[k * 4 + 2] * ly + s_co[k * 4 + 3] * lz;
            if (dheat) dhm += dheat[((long long)n * K + k) * S + s];
            const float dq = dhm * (1.f - expf(-hm));
            if (lead) dq_out[((long long)n * K + k) * S + s] = dq;
            sp0 = fmaf(dq, h, sp0);
            sp1 = fmaf(dq, pv, sp1);
            sp2 += dq;
            dh = pw0 * dq;
          } else {
            dh = dheat ? dheat[((long long)n * K + k) * S + s] : 0.f;
            if (dq_in) {
              float t = 0.f;
              for (int tt = 0; tt < frames_per_clip; tt++) t += dq_in[(((long long)n * frames_per_clip + tt) * K + k) * S + s];
              dh = fmaf(pw1, t, dh);
            }
          }
          du = dh * slope;
        }
        s_du[k * TS + sl] = du;
        s_duT[sl * KMAX + k] = du;
      }
    }
    __syncthreads();
    // dfeat[s][c] = grad_scale * sum_k du[k][s] w1[k][c]: thread = (4 voxels, channels c8*4 .. +3 and C/2 + c8*4 .. +3)
    if (lead) {
      const int c8 = threadIdx.x % NC8, slg = threadIdx.x / NC8;
#pragma unroll 1
      for (int v0 = 0; v0 < VPT; v0 += 4) {
        const int slb = slg * VPT + v0;
        float o[4][8];
#pragma unroll
        for (int i = 0; i < 4; i++)
#pragma unroll
          for (int e = 0; e < 8; e++) o[i][e] = 0.f;
        for (int k = 0; k < K; k++) {
          const float4 d = *reinterpret_cast<const float4*>(s_du + k * TS + slb);
          const float4 w0 = *reinterpret_cast<const float4*>(s_w + k * C + c8 * 4);
          const float4 w1v = *reinterpret_cast<const float4*>(s_w + k * C + C / 2 + c8 * 4);
          const float dv[4] = {d.x, d.y, d.z, d.w};
          const float wv[8] = {w0.x, w0.y, w0.z, w0.w, w1v.x, w1v.y, w1v.z, w1v.w};
#pragma unroll
          for (int i = 0; i < 4; i++)
#pragma unroll
            for (int e = 0; e < 8; e++) o[i][e] = fmaf(dv[i], wv[e], o[i][e]);
        }
#pragma unroll
        for (int i = 0; i < 4; i++) {
          __half2 h[4];
#pragma unroll
          for (int e = 0; e < 4; e++) h[e] = __floats2half2_rn(o[i][2 * e] * grad_scale, o[i][2 * e + 1] * grad_scale);
          __half* dst = dfeat + ((long long)n * S + s0 + slb + i) * C + c8 * 4;
          *reinterpret_cast<uint2*>(dst) = make_uint2(*reinterpret_cast<uint32_t*>(&h[0]), *reinterpret_cast<uint32_t*>(&h[1]));
          *reinterpret_cast<uint2*>(dst + C / 2) = make_uint2(*reinterpret_cast<uint32_t*>(&h[2]), *reinterpret_cast<uint32_t*>(&h[3]));
        }
      }
    }
    // dW1[k][c] += sum_s du[k][s] f[s][c];  db1[k] += sum_s du[k][s]
#pragma unroll 2
    for (int sl = 0; sl < TS; sl++) {
      const float f = s_f[sl * FS + wc];
      const float4* dr = reinterpret_cast<const float4*>(s_duT + sl * KMAX + wk0);
#pragma unroll
      for (int q = 0; q < KPT / 4; q++) {
        const float4 d = dr[q];
        accw[q * 4] = fmaf(d.x, f, accw[q * 4]);
        accw[q * 4 + 1] = fmaf(d.y, f, accw[q * 4 + 1]);
        accw[q * 4 + 2] = fmaf(d.z, f, accw[q * 4 + 2]);
        accw[q * 4 + 3] = fmaf(d.w, f, accw[q * 4 + 3]);
      }
    }
    if (lead && threadIdx.x < KMAX) {
      const float4* dr = reinterpret_cast<const float4*>(s_du + threadIdx.x * TS);
      float t = 0.f;
#pragma unroll 4
      for (int q = 0; q < TS / 4; q++) {
        const float4 d = dr[q];
        t += (d.x + d.y) + (d.z + d.w);
      }
      accb += t;
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < KPT; i++)
    if (wk0 + i < K) pw_partial[(part * K + wk0 + i) * C + wc] = accw[i];
  if (!lead) return;
  if (threadIdx.x < K) pb_partial[part * K + threadIdx.x] = accb;
  if (mode == 1) {
    s_red[threadIdx.x * 3] = sp0; s_red[threadIdx.x * 3 + 1] = sp1; s_red[threadIdx.x * 3 + 2] = sp2;
    __syncthreads();
    if (threadIdx.x < 3) {
      float t = 0.f;
      for (int i = 0; i < 256; i++) t += s_red[i * 3 + threadIdx.x];
      pp_partial[part * 3 + threadIdx.x] = t;
    }
  }
}

// ------------------------------------------------------------------ decoder adjust + Gaussian render backward
// forward: y = lrelu(W cat[G_t (K), ff (128), G_0 (K), coords (3)] + b), G[k][s] = ex[x] ey[y] ez[z] I_k
// dz = dy / grad_scale * lrelu'(y).  Per frame: dG_t = W[:, :K]^T dz -> d keypoints (render backward), dW[:, :K], db.
// Per clip (on sum_t dz): d first_feature, d keypoints of frame 0 (through G_0), dW[:, K:].
// All contractions are register-tiled over shared memory (the first version issued two shared loads per FMA and was
// bound by the LDS pipe: 1.4 + 1.3 ms per step); dz lives in shared memory in both orientations.
constexpr int kAdjC = 128;
constexpr int kAdjTS = 64;
constexpr int kAdjDS = kAdjTS + 4;     // s_dz  [co][68]: 16-byte aligned rows (broadcast LDS.128 over voxels)
constexpr int kAdjDT = kAdjC + 4;      // s_dzT [sl][132]: conflict-free 16-byte stores with lanes over voxels

__device__ __forceinline__ void adj_stage_exps(const float* kp, int K, int g, const float* lin, float width, float* s_e, float* s_kp) {
  for (int i = threadIdx.x; i < K * 3 * g; i += 256) {
    const int k = i / (3 * g), a = (i / g) % 3, j = i % g;
    const float d = lin[j] - kp[k * 4 + a];
    s_e[(k * 3 + a) * 32 + j] = expf(-(d * d) / width);
  }
  for (int i = threadIdx.x; i < K * 4; i += 256) s_kp[i] = kp[i];
}

// dz tile -> shared as s_dz [co][kAdjDS] and s_dzT [sl][kAdjDT]; frames = 1 (per-frame kernel) or T (sum over the clip's
// frames).  Lanes run over voxels: both shared stores are conflict-free, the 8-byte global loads of a lane walk its
// voxel's 256-byte channel row (sectors are reused from L1 by the next channel groups).
__device__ __forceinline__ void adj_load_dz(const __half* dy, const __half* y, long long frame0, int frames, int S, int s0,
                                            float inv_scale, float* s_dz, float* s_dzT) {
  for (int i = threadIdx.x; i < kAdjTS * (kAdjC / 4); i += 256) {
    const int sl = i % kAdjTS, c4 = i / kAdjTS;
    float acc[4] = {0.f, 0.f, 0.f, 0.f};
    for (int t = 0; t < frames; t++) {
      const long long off = ((frame0 + t) * S + s0 + sl) * kAdjC + c4 * 4;
      const uint2 rd = *reinterpret_cast<const uint2*>(dy + off), ro = *reinterpret_cast<const uint2*>(y + off);
      const float2 d0 = __half22float2(*reinterpret_cast<const __half2*>(&rd.x)), d1 = __half22float2(*reinterpret_cast<const __half2*>(&rd.y));
      const float2 o0 = __half22float2(*reinterpret_cast<const __half2*>(&ro.x)), o1 = __half22float2(*reinterpret_cast<const __half2*>(&ro.y));
      acc[0] += o0.x > 0.f ? d0.x : 0.01f * d0.x;
      acc[1] += o0.y > 0.f ? d0.y : 0.01f * d0.y;
      acc[2] += o1.x > 0.f ? d1.x : 0.01f * d1.x;
      acc[3] += o1.y > 0.f ? d1.y : 0.01f * d1.y;
    }
#pragma unroll
    for (int e = 0; e < 4; e++) {
      acc[e] *= inv_scale;
      s_dz[(c4 * 4 + e) * kAdjDS + sl] = acc[e];
    }
    *reinterpret_cast<float4*>(s_dzT + sl * kAdjDT + c4 * 4) = make_float4(acc[0], acc[1], acc[2], acc[3]);
  }
}

// render backward accumulation for the keypoints owned by this thread (6 of them, one voxel)
template <int KMAX>
struct RenderAcc { float v[KMAX / 4][4]; };

// Gaussians of the tile, voxel-major: s_GT[sl][KMAX]
template <int KMAX>
__device__ __forceinline__ void adj_gauss_tile(const float* s_e, const float* s_kp, int K, int g, int s0, float* s_GT) {
  for (int i = threadIdx.x; i < KMAX * kAdjTS; i += 256) {
    const int k = i / kAdjTS, sl = i % kAdjTS, s = s0 + sl;
    float v = 0.f;
    if (k < K) {
      const int x = s / (g * g), yy = (s / g) % g, z = s % g;
      v = ((1.0f * s_e[(k * 3) * 32 + x]) * s_e[(k * 3 + 1) * 32 + yy]) * s_e[(k * 3 + 2) * 32 + z] * s_kp[k * 4 + 3];
    }
    s_GT[sl * KMAX + k] = v;
  }
}

// dG[k][s] = sum_co W[co][col0 + k] dz[co][s] for this thread's 6 keypoints (per co: one LDS of dz, three broadcast
// LDS.64 of the weights, 6 FMA), accumulated into the render gradient
template <int KMAX>
__device__ __forceinline__ void adj_render_bwd(const float* s_wg /* [128][KMAX] */, const float* s_dz, const float* s_e,
                                               const float* s_kp, const float* lin, int K, int g, int s0, float width,
                                               RenderAcc<KMAX>& r) {
  constexpr int KG = KMAX / 4;
  const int sl = threadIdx.x % kAdjTS, kg = threadIdx.x / kAdjTS, s = s0 + sl;
  const int x = s / (g * g), yy = (s / g) % g, z = s % g;
  const float lx = lin[x], ly = lin[yy], lz = lin[z];
  float dG[KG];
#pragma unroll
  for (int j = 0; j < KG; j++) dG[j] = 0.f;
  const float* wr = s_wg + kg * KG;
#pragma unroll 4
  for (int co = 0; co < kAdjC; co++) {
    const float d = s_dz[co * kAdjDS + sl];
    const float2* w2 = reinterpret_cast<const float2*>(wr + co * KMAX);
#pragma unroll
    for (int j = 0; j < KG / 2; j++) {
      const float2 w = w2[j];
      dG[2 * j] = fmaf(w.x, d, dG[2 * j]);
      dG[2 * j + 1] = fmaf(w.y, d, dG[2 * j + 1]);
    }
  }
#pragma unroll
  for (int kk = 0; kk < KG; kk++) {
    const int k = kg * KG + kk;
    if (k < K) {
      const float E = ((1.0f * s_e[(k * 3) * 32 + x]) * s_e[(k * 3 + 1) * 32 + yy]) * s_e[(k * 3 + 2) * 32 + z];
      const float gG = dG[kk] * E * s_kp[k * 4 + 3] * (2.f / width);
      r.v[kk][0] = fmaf(gG, lx - s_kp[k * 4], r.v[kk][0]);
      r.v[kk][1] = fmaf(gG, ly - s_kp[k * 4 + 1], r.v[kk][1]);
      r.v[kk][2] = fmaf(gG, lz - s_kp[k * 4 + 2], r.v[kk][2]);
      r.v[kk][3] = fmaf(dG[kk], E, r.v[kk][3]);
    }
  }
}

// dWg[co][k0 .. k0+KMAX/2-1] += sum_s dz[co][s] G[k][s] (thread = output channel co, half the keypoints; per voxel one LDS of
// dz and KMAX/8 broadcast LDS.128 of the Gaussians); returns sum_s dz[co][s] through `dsum`
template <int KMAX>
__device__ __forceinline__ void adj_wg_accumulate(const float* s_dzT, const float* s_GT, int co, int k0, float (&acc)[KMAX / 2], float& dsum) {
#pragma unroll 2
  for (int sl = 0; sl < kAdjTS; sl++) {
    const float d = s_dzT[sl * kAdjDT + co];
    const float4* gr = reinterpret_cast<const float4*>(s_GT + sl * KMAX + k0);
#pragma unroll
    for (int q = 0; q < KMAX / 8; q++) {
      const float4 gv = gr[q];
      acc[q * 4] = fmaf(d, gv.x, acc[q * 4]);
      acc[q * 4 + 1] = fmaf(d, gv.y, acc[q * 4 + 1]);
      acc[q * 4 + 2] = fmaf(d, gv.z, acc[q * 4 + 2]);
      acc[q * 4 + 3] = fmaf(d, gv.w, acc[q * 4 + 3]);
    }
    dsum += d;
  }
}

// fold the per-thread render accumulators over the 64 voxel lanes of each keypoint group (fixed order)
template <int KMAX>
__device__ __forceinline__ void adj_render_store(const RenderAcc<KMAX>& r, float* s_tmp /* [256][KMAX] */, int K, float* out /* [K][4] */) {
#pragma unroll
  for (int kk = 0; kk < KMAX / 4; kk++)
#pragma unroll
    for (int q = 0; q < 4; q++) s_tmp[threadIdx.x * KMAX + kk * 4 + q] = r.v[kk][q];
  __syncthreads();
  if (threadIdx.x < KMAX * 4) {
    const int k = threadIdx.x / 4, q = threadIdx.x % 4, kg = k / (KMAX / 4), kk = k % (KMAX / 4);
    float t = 0.f;
    for (int sl = 0; sl < kAdjTS; sl++) t += s_tmp[(kg * kAdjTS + sl) * KMAX + kk * 4 + q];
    if (k < K) out[k * 4 + q] = t;
  }
  __syncthreads();
}

// shared-memory floats: frame kernel / extra of the clip kernel (s_tmp of adj_render_store aliases s_dz .. s_dzT).  At
// capacity 64 the clip kernel would need 237 KB with the first-feature weights staged; it reads them from L2 instead.
template <int KMAX>
constexpr int adj_frame_floats() { return kAdjC * KMAX + kAdjC * kAdjDS + kAdjTS * kAdjDT + kAdjTS * KMAX + KMAX * 96 + KMAX * 4; }
template <int KMAX>
constexpr bool adj_wff_shared() { return KMAX <= kTunedK; }
template <int KMAX>
constexpr int adj_clip_floats() {
  return adj_frame_floats<KMAX>() + (adj_wff_shared<KMAX>() ? kAdjC * kAdjC : 0) + kAdjTS * kAdjC + kAdjTS * 4;
}
static_assert(256 * kMaxK <= kAdjC * kAdjDS + kAdjTS * kAdjDT, "s_tmp must fit in the dz buffers");
static_assert(adj_clip_floats<kMaxK>() * 4 <= 227 * 1024, "adjust_bwd_clip_kernel<64> must fit in shared memory");

template <int KMAX>
__global__ void __launch_bounds__(256)
adjust_bwd_frame_kernel(const __half* __restrict__ dy, const __half* __restrict__ y, const float* __restrict__ kp,
                        const float* __restrict__ W, int ld, int K, int g, const float* __restrict__ lin, float width,
                        float inv_scale, float* __restrict__ dkp /* [n][K][4] */, float* __restrict__ pwg /* [n][128][KMAX] */,
                        float* __restrict__ pbias /* [n][128] */) {
  extern __shared__ __align__(16) float smem[];
  float* s_wg = smem;                                     // [128][KMAX]
  float* s_dz = s_wg + kAdjC * KMAX;                      // [128][kAdjDS]
  float* s_dzT = s_dz + kAdjC * kAdjDS;                   // [TS][kAdjDT]
  float* s_GT = s_dzT + kAdjTS * kAdjDT;                  // [TS][KMAX]
  float* s_e = s_GT + kAdjTS * KMAX;                      // [KMAX][3][32]
  float* s_kp = s_e + KMAX * 96;                          // [KMAX][4]
  float* s_tmp = s_dz;                                    // [256][KMAX], after the tile loop
  const int n = blockIdx.x, S = g * g * g;
  for (int i = threadIdx.x; i < kAdjC * KMAX; i += 256) {
    const int co = i / KMAX, k = i % KMAX;
    s_wg[i] = k < K ? W[(long long)co * ld + k] : 0.f;
  }
  adj_stage_exps(kp + (long long)n * K * 4, K, g, lin, width, s_e, s_kp);
  __syncthreads();
  RenderAcc<KMAX> r;
#pragma unroll
  for (int kk = 0; kk < KMAX / 4; kk++)
#pragma unroll
    for (int q = 0; q < 4; q++) r.v[kk][q] = 0.f;
  constexpr int KH = KMAX / 2;                            // keypoints of dW per thread
  float accw[KH], accb = 0.f;
#pragma unroll
  for (int i = 0; i < KH; i++) accw[i] = 0.f;
  const int wco = threadIdx.x % kAdjC, wk0 = (threadIdx.x / kAdjC) * KH;
  for (int s0 = 0; s0 < S; s0 += kAdjTS) {
    adj_load_dz(dy, y, n, 1, S, s0, inv_scale, s_dz, s_dzT);
    adj_gauss_tile<KMAX>(s_e, s_kp, K, g, s0, s_GT);
    __syncthreads();
    adj_render_bwd<KMAX>(s_wg, s_dz, s_e, s_kp, lin, K, g, s0, width, r);
    // dW[co][k] += sum_s dz[co][s] G[k][s];  db[co] += sum_s dz[co][s]
    adj_wg_accumulate<KMAX>(s_dzT, s_GT, wco, wk0, accw, accb);
    __syncthreads();
  }
  adj_render_store<KMAX>(r, s_tmp, K, dkp + (long long)n * K * 4);
#pragma unroll
  for (int i = 0; i < KH; i++) pwg[((long long)n * kAdjC + wco) * KMAX + wk0 + i] = accw[i];
  if (threadIdx.x < kAdjC) pbias[(long long)n * kAdjC + threadIdx.x] = accb;
}

// per clip, split over `splits` voxel ranges: works on dzs = sum over the clip's frames of dz
template <int KMAX>
__global__ void __launch_bounds__(256)
adjust_bwd_clip_kernel(const __half* __restrict__ dy, const __half* __restrict__ y, const __half* __restrict__ ff,
                       const float* __restrict__ kp, const float* __restrict__ W, int ld, int K, int g, int frames_per_clip,
                       const float* __restrict__ lin, float width, float inv_scale, float grad_scale,
                       __half* __restrict__ dff /* [clips][S][128] */, float* __restrict__ dkp0 /* [clips][splits][K][4] */,
                       float* __restrict__ pw /* [clips][splits][128][128 + KMAX + 3] */) {
  extern __shared__ __align__(16) float smem[];
  float* s_wg = smem;                                     // [128][KMAX]  (gauss_0 columns)
  float* s_dz = s_wg + kAdjC * KMAX;                      // [128][kAdjDS]
  float* s_dzT = s_dz + kAdjC * kAdjDS;                   // [TS][kAdjDT]
  float* s_GT = s_dzT + kAdjTS * kAdjDT;                  // [TS][KMAX]
  float* s_e = s_GT + kAdjTS * KMAX;                      // [KMAX][3][32]
  float* s_kp = s_e + KMAX * 96;                          // [KMAX][4]
  constexpr bool kWff = adj_wff_shared<KMAX>();
  float* s_wff = s_kp + KMAX * 4;                         // [128 co][128 c] (capacity 24 only)
  float* s_ff = s_wff + (kWff ? kAdjC * kAdjC : 0);       // [TS][128]
  float* s_xyz = s_ff + kAdjTS * kAdjC;                   // [TS][4]: lin[x], lin[y], lin[z] of the tile's voxels
  float* s_tmp = s_dz;                                    // [256][KMAX], after the tile loop
  const int clip = blockIdx.x, split = blockIdx.y, splits = gridDim.y, S = g * g * g;
  const int per = S / splits;                             // multiple of TS (checked by the host)
  if (kWff)
    for (int i = threadIdx.x; i < kAdjC * kAdjC; i += 256) s_wff[i] = W[(long long)(i / kAdjC) * ld + K + i % kAdjC];
  for (int i = threadIdx.x; i < kAdjC * KMAX; i += 256) {
    const int co = i / KMAX, k = i % KMAX;
    s_wg[i] = k < K ? W[(long long)co * ld + K + kAdjC + k] : 0.f;
  }
  adj_stage_exps(kp + (long long)clip * frames_per_clip * K * 4, K, g, lin, width, s_e, s_kp);
  __syncthreads();
  RenderAcc<KMAX> r;
#pragma unroll
  for (int kk = 0; kk < KMAX / 4; kk++)
#pragma unroll
    for (int q = 0; q < 4; q++) r.v[kk][q] = 0.f;
  // dW[:, K:K+128]: thread = (4 feature channels fc4*4.., 16 output channels cog*16..)
  constexpr int KH = KMAX / 2;
  float accf[16][4], accg[KH], accx[3] = {0.f, 0.f, 0.f}, dsum = 0.f;
#pragma unroll
  for (int i = 0; i < 16; i++)
#pragma unroll
    for (int e = 0; e < 4; e++) accf[i][e] = 0.f;
#pragma unroll
  for (int i = 0; i < KH; i++) accg[i] = 0.f;
  const int wc = threadIdx.x % kAdjC, half_id = threadIdx.x / kAdjC;   // half_id: 0 / 1
  const int fc4 = threadIdx.x % 32, cog = threadIdx.x / 32;            // cog doubles as the voxel group of d first_feature
  for (int s0 = split * per; s0 < (split + 1) * per; s0 += kAdjTS) {
    adj_load_dz(dy, y, (long long)clip * frames_per_clip, frames_per_clip, S, s0, inv_scale, s_dz, s_dzT);
    adj_gauss_tile<KMAX>(s_e, s_kp, K, g, s0, s_GT);
    for (int i = threadIdx.x; i < kAdjTS * (kAdjC / 4); i += 256) {
      const int sl = i / (kAdjC / 4), c4 = i % (kAdjC / 4);
      const uint2 raw = *reinterpret_cast<const uint2*>(ff + ((long long)clip * S + s0 + sl) * kAdjC + c4 * 4);
      const float2 lo = __half22float2(*reinterpret_cast<const __half2*>(&raw.x));
      const float2 hi = __half22float2(*reinterpret_cast<const __half2*>(&raw.y));
      *reinterpret_cast<float4*>(s_ff + sl * kAdjC + c4 * 4) = make_float4(lo.x, lo.y, hi.x, hi.y);
    }
    if (threadIdx.x < kAdjTS) {
      const int s = s0 + threadIdx.x;
      *reinterpret_cast<float4*>(s_xyz + threadIdx.x * 4) = make_float4(lin[s / (g * g)], lin[(s / g) % g], lin[s % g], 0.f);
    }
    __syncthreads();
    adj_render_bwd<KMAX>(s_wg, s_dz, s_e, s_kp, lin, K, g, s0, width, r);
    // d first_feature[s][c] = grad_scale * sum_co W[co][K + c] dzs[co][s]: thread = (channels fc4*4.., voxels cog*8..);
    // per co one LDS.128 of the weights and two broadcast LDS.128 of dzs for 32 FMA
    {
      float o[8][4];
#pragma unroll
      for (int v = 0; v < 8; v++)
#pragma unroll
        for (int e = 0; e < 4; e++) o[v][e] = 0.f;
#pragma unroll 2
      for (int co = 0; co < kAdjC; co++) {
        float4 w;
        if (kWff) {
          w = *reinterpret_cast<const float4*>(s_wff + co * kAdjC + fc4 * 4);
        } else {
          const float* wr = W + (long long)co * ld + K + fc4 * 4;
          w = make_float4(__ldg(wr), __ldg(wr + 1), __ldg(wr + 2), __ldg(wr + 3));
        }
        const float4 d0 = *reinterpret_cast<const float4*>(s_dz + co * kAdjDS + cog * 8);
        const float4 d1 = *reinterpret_cast<const float4*>(s_dz + co * kAdjDS + cog * 8 + 4);
        const float dv[8] = {d0.x, d0.y, d0.z, d0.w, d1.x, d1.y, d1.z, d1.w};
#pragma unroll
        for (int v = 0; v < 8; v++) {
          o[v][0] = fmaf(w.x, dv[v], o[v][0]);
          o[v][1] = fmaf(w.y, dv[v], o[v][1]);
          o[v][2] = fmaf(w.z, dv[v], o[v][2]);
          o[v][3] = fmaf(w.w, dv[v], o[v][3]);
        }
      }
#pragma unroll
      for (int v = 0; v < 8; v++) {
        __half2 h0 = __floats2half2_rn(o[v][0] * grad_scale, o[v][1] * grad_scale);
        __half2 h1 = __floats2half2_rn(o[v][2] * grad_scale, o[v][3] * grad_scale);
        *reinterpret_cast<uint2*>(dff + ((long long)clip * S + s0 + cog * 8 + v) * kAdjC + fc4 * 4) =
            make_uint2(*reinterpret_cast<uint32_t*>(&h0), *reinterpret_cast<uint32_t*>(&h1));
      }
    }
    // dW[co][K + c] += sum_s dzs[co][s] ff[s][c]: per voxel one LDS.128 of ff and four broadcast LDS.128 of dzs for 64 FMA
#pragma unroll 2
    for (int sl = 0; sl < kAdjTS; sl++) {
      const float4 f = *reinterpret_cast<const float4*>(s_ff + sl * kAdjC + fc4 * 4);
      const float4* dr = reinterpret_cast<const float4*>(s_dzT + sl * kAdjDT + cog * 16);
#pragma unroll
      for (int q = 0; q < 4; q++) {
        const float4 d = dr[q];
        const float dv[4] = {d.x, d.y, d.z, d.w};
#pragma unroll
        for (int e = 0; e < 4; e++) {
          accf[q * 4 + e][0] = fmaf(dv[e], f.x, accf[q * 4 + e][0]);
          accf[q * 4 + e][1] = fmaf(dv[e], f.y, accf[q * 4 + e][1]);
          accf[q * 4 + e][2] = fmaf(dv[e], f.z, accf[q * 4 + e][2]);
          accf[q * 4 + e][3] = fmaf(dv[e], f.w, accf[q * 4 + e][3]);
        }
      }
    }
    // dW[co][K + 128 + k] += sum_s dzs[co][s] G0[k][s]  (co = wc, KMAX / 2 keypoints);  coords: thread co = wc of half 0
    adj_wg_accumulate<KMAX>(s_dzT, s_GT, wc, half_id * KH, accg, dsum);
    if (half_id == 0) {
#pragma unroll 4
      for (int sl = 0; sl < kAdjTS; sl++) {
        const float d = s_dzT[sl * kAdjDT + wc];
        const float4 c = *reinterpret_cast<const float4*>(s_xyz + sl * 4);
        accx[0] = fmaf(d, c.x, accx[0]);
        accx[1] = fmaf(d, c.y, accx[1]);
        accx[2] = fmaf(d, c.z, accx[2]);
      }
    }
    __syncthreads();
  }
  const long long part = (long long)clip * splits + split;
  adj_render_store<KMAX>(r, s_tmp, K, dkp0 + part * K * 4);
  constexpr int LDP = kAdjC + KMAX + 3;
  float* o = pw + part * kAdjC * LDP;
#pragma unroll
  for (int i = 0; i < 16; i++)
#pragma unroll
    for (int e = 0; e < 4; e++) o[(long long)(cog * 16 + i) * LDP + fc4 * 4 + e] = accf[i][e];
#pragma unroll
  for (int i = 0; i < KH; i++) o[(long long)wc * LDP + kAdjC + half_id * KH + i] = accg[i];
  if (half_id == 0)
    for (int a = 0; a < 3; a++) o[(long long)wc * LDP + kAdjC + KMAX + a] = accx[a];
}

// dW (128, 2K + 131) and db (128) from the per-frame / per-clip partials; dkp[clip's frame 0] += sum over splits of dkp0
template <int KMAX>
__global__ void adjust_bwd_finalize_kernel(const float* __restrict__ pwg, const float* __restrict__ pbias, const float* __restrict__ pw,
                                           const float* __restrict__ dkp0, int n, int parts, int clips, int splits,
                                           int frames_per_clip, int K, float* __restrict__ dW, float* __restrict__ db,
                                           float* __restrict__ dkp) {
  const int ld = 2 * K + kAdjC + 3;
  constexpr int LDP = kAdjC + KMAX + 3;
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i < kAdjC * ld) {
    const int co = i / ld, col = i % ld;
    double acc = 0.0;
    if (col < K) {
      for (int f = 0; f < n; f++) acc += (double)pwg[((long long)f * kAdjC + co) * KMAX + col];
    } else {
      const int pc = col < K + kAdjC ? col - K : (col < 2 * K + kAdjC ? kAdjC + (col - K - kAdjC) : kAdjC + KMAX + (col - 2 * K - kAdjC));
      for (int p = 0; p < parts; p++) acc += (double)pw[((long long)p * kAdjC + co) * LDP + pc];
    }
    dW[i] = (float)acc;
  } else if (i < kAdjC * ld + kAdjC) {
    const int co = i - kAdjC * ld;
    double acc = 0.0;
    for (int f = 0; f < n; f++) acc += (double)pbias[(long long)f * kAdjC + co];
    db[co] = (float)acc;
  } else if (i < kAdjC * ld + kAdjC + clips * K * 4) {
    const int j = i - kAdjC * ld - kAdjC, clip = j / (K * 4), e = j % (K * 4);
    float acc = 0.f;
    for (int sp = 0; sp < splits; sp++) acc += dkp0[((long long)clip * splits + sp) * K * 4 + e];
    dkp[(long long)clip * frames_per_clip * K * 4 + e] += acc;
  }
}

// ------------------------------------------------------------------ chamfer volume-fitting loss backward
// loss_n = sum_v o_v min_k |c_v - kp_k|^2 / sum_v o_v  ->  d kp_k = g_n / sum o * sum_{v: argmin = k} o_v 2 (kp_k - c_v)
constexpr int kChbBlocks = 32;
template <int KMAX>
__global__ void __launch_bounds__(256)
chamfer_bwd_kernel(const float* __restrict__ seq, const float* __restrict__ kp, int K, int G, const float* __restrict__ lin,
                   float* __restrict__ partial /* [n][blocks][K*3 + 1] */) {
  extern __shared__ float sm[];
  float* s_kp = sm;                       // [K][3]
  float* s_acc = sm + KMAX * 3;           // [K*3][256] thread-private columns
  const int n = blockIdx.y;
  for (int i = threadIdx.x; i < K * 3; i += 256) s_kp[i] = kp[((long long)n * K + i / 3) * 4 + i % 3];
  for (int i = 0; i < K * 3; i++) s_acc[i * 256 + threadIdx.x] = 0.f;
  __syncthreads();
  const int S = G * G * G;
  float osum = 0.f;
  for (int s = blockIdx.x * 256 + threadIdx.x; s < S; s += gridDim.x * 256) {
    const float o = seq[(long long)n * S + s];
    if (o != 0.f) {
      const float cx = lin[s / (G * G)], cy = lin[(s / G) % G], cz = lin[s % G];
      float best = INFINITY;
      int kb = 0;
      for (int k = 0; k < K; k++) {
        const float dx = cx - s_kp[k * 3], dy = cy - s_kp[k * 3 + 1], dz = cz - s_kp[k * 3 + 2];
        const float d = dx * dx + dy * dy + dz * dz;
        if (d < best) { best = d; kb = k; }                                // first minimum, as torch.min
      }
      s_acc[(kb * 3) * 256 + threadIdx.x] += o * 2.f * (s_kp[kb * 3] - cx);
      s_acc[(kb * 3 + 1) * 256 + threadIdx.x] += o * 2.f * (s_kp[kb * 3 + 1] - cy);
      s_acc[(kb * 3 + 2) * 256 + threadIdx.x] += o * 2.f * (s_kp[kb * 3 + 2] - cz);
      osum += o;
    }
  }
  __syncthreads();
  float* out = partial + ((long long)n * gridDim.x + blockIdx.x) * (K * 3 + 1);
  for (int i = threadIdx.x; i < K * 3; i += 256) {
    float t = 0.f;
    for (int j = 0; j < 256; j++) t += s_acc[i * 256 + j];
    out[i] = t;
  }
  __shared__ float red[8];
  osum = nm_warp_sum(osum);
  if ((threadIdx.x & 31) == 0) red[threadIdx.x >> 5] = osum;
  __syncthreads();
  if (threadIdx.x == 0) {
    float t = 0.f;
    for (int k = 0; k < 8; k++) t += red[k];
    out[K * 3] = t;
  }
}

__global__ void chamfer_bwd_finalize_kernel(const float* __restrict__ partial, const float* __restrict__ gout, int n, int K,
                                            int blocks, float* __restrict__ dkp /* [n][K][4] */) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n * K * 4) return;
  const int f = i / (K * 4), k = (i / 4) % K, a = i % 4;
  if (a == 3) { dkp[i] = 0.f; return; }
  double acc = 0.0, os = 0.0;
  for (int b = 0; b < blocks; b++) {
    const float* p = partial + ((long long)f * blocks + b) * (K * 3 + 1);
    acc += (double)p[k * 3 + a];
    os += (double)p[K * 3];
  }
  dkp[i] = (float)((double)gout[f] * acc / os);
}

// ------------------------------------------------------------------ CoordConv first layer: weight gradient
// dW[co][c][t] = sum_v dY[v][co] in_c[v + t - 2], t = (tx, ty, tz) in 0..4, in = cat[occ, x, y, z] zero-padded by 2.
// Coordinate channels: in_a[v + t - 2] = lin[v_a + t_a - 2] inside the volume -> affine in the voxel index, so the sums
// over the tap's in-bounds box follow from 125 bins (5 position classes per axis: 0, 1, interior, G-2, G-1) of the
// moments (sum dY, sum x dY, sum y dY, sum z dY).  Occupancy channel: a gather over the occupied voxels.
// One pass over the CTA's x slab in memory order.  Rows (x, y) are grouped by their (x class, y class); inside a row
// lane = (z lane, 16-byte channel chunk) and only the lanes that meet z = 0, 1, G-2, G-1 (in the first / last load of the
// row) keep a second accumulator set, so a group's five z bins come out of one sweep.  A group ends with a butterfly over
// the z lanes and a fixed-order fold of the 8 warps.  (The first version swept the slab once per bin: 125 block-wide
// reductions per CTA, 1.9 TB/s.)
template <int C>
__global__ void __launch_bounds__(256, 2)
first_wgrad_moments_kernel(const __half* __restrict__ dy, int G, float* __restrict__ bins /* [n][parts][125][4][C] */) {
  constexpr int CC = C / 8, ZL = 32 / CC;                    // channel chunks per voxel, lanes along z
  __shared__ float red[8][5][4][C];
  const int n = blockIdx.x, part = blockIdx.y, parts = gridDim.y;
  const int xs = G * part / parts, xe = G * (part + 1) / parts;        // this CTA's x slab
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cc = lane % CC, zl = lane / CC;
  const int nj = G / ZL;                                     // loads per row and lane
  const __half* base = dy + (long long)n * G * G * G * C + cc * 8;
  float* out = bins + ((long long)n * parts + part) * 125 * 4 * C;
  // z class of this lane's boundary slot (first load: zl = 0, 1; last load: zl = ZL-2, ZL-1), -1: interior lanes only
  const int bcls = zl == 0 ? 0 : (zl == 1 ? 1 : (zl == ZL - 2 ? 3 : (zl == ZL - 1 ? 4 : -1)));
  const float bz = bcls == 0 ? 0.f : (bcls == 1 ? 1.f : (bcls == 3 ? (float)(G - 2) : (float)(G - 1)));
  for (int grp = 0; grp < 25; grp++) {
    const int cxc = grp / 5, cyc = grp % 5;
    int lo[2], cnt[2];
    const int cl2[2] = {cxc, cyc};
#pragma unroll
    for (int a = 0; a < 2; a++) {
      lo[a] = cl2[a] == 0 ? 0 : (cl2[a] == 1 ? 1 : (cl2[a] == 2 ? 2 : (cl2[a] == 3 ? G - 2 : G - 1)));
      cnt[a] = cl2[a] == 2 ? G - 4 : 1;
    }
    {
      const int a0 = max(lo[0], xs), a1 = min(lo[0] + cnt[0], xe);
      lo[0] = a0;
      cnt[0] = max(0, a1 - a0);
    }
    const int rows = cnt[0] * cnt[1];
    float* og = out + (long long)grp * 5 * 4 * C;            // bins (cxc, cyc, 0..4)
    if (rows == 0) {                                         // block-uniform: the group lies outside the slab
      for (int i = threadIdx.x; i < 5 * 4 * C; i += 256) og[i] = 0.f;
      continue;
    }
    float s0[8], sx[8], sy[8], sz[8], b0[8], bx[8], by[8];
#pragma unroll
    for (int k = 0; k < 8; k++) s0[k] = sx[k] = sy[k] = sz[k] = b0[k] = bx[k] = by[k] = 0.f;
    for (int r = warp; r < rows; r += 8) {
      const int x = lo[0] + r / cnt[1], y = lo[1] + r % cnt[1];
      const float fx = (float)x, fy = (float)y;
      const __half* row = base + (((long long)x * G + y) * G + zl) * C;
      // x and y are constant along a row: the row's plain sum r0 gives three of the four moments with 24 FMAs per row
      float r0[8], rz[8];
#pragma unroll
      for (int k = 0; k < 8; k++) r0[k] = rz[k] = 0.f;
      // loads are issued in batches of 8 ahead of the (divergent) accumulation so that they overlap
#pragma unroll 1
      for (int j0 = 0; j0 < nj; j0 += 8) {
        half8 v[8];
#pragma unroll
        for (int u = 0; u < 8; u++)
          if (j0 + u < nj) v[u] = *reinterpret_cast<const half8*>(row + (long long)(j0 + u) * ZL * C);
#pragma unroll
        for (int u = 0; u < 8; u++) {
          const int j = j0 + u;
          if (j >= nj) break;
          float f[8];
          nm_unpack8(v[u], f);
          const bool bnd = (j == 0 && zl < 2) || (j == nj - 1 && zl >= ZL - 2);
          if (bnd) {
#pragma unroll
            for (int k = 0; k < 8; k++) {
              b0[k] += f[k];
              bx[k] = fmaf(fx, f[k], bx[k]);
              by[k] = fmaf(fy, f[k], by[k]);
            }
          } else {
            const float fz = (float)(zl + j * ZL);
#pragma unroll
            for (int k = 0; k < 8; k++) {
              r0[k] += f[k];
              rz[k] = fmaf(fz, f[k], rz[k]);
            }
          }
        }
      }
#pragma unroll
      for (int k = 0; k < 8; k++) {
        s0[k] += r0[k];
        sx[k] = fmaf(fx, r0[k], sx[k]);
        sy[k] = fmaf(fy, r0[k], sy[k]);
        sz[k] += rz[k];
      }
    }
    // interior z bin: butterfly over the z lanes (fixed order); boundary z bins: one lane each
#pragma unroll
    for (int k = 0; k < 8; k++) {
#pragma unroll
      for (int o = CC; o < 32; o <<= 1) {
        s0[k] += __shfl_xor_sync(0xffffffffu, s0[k], o);
        sx[k] += __shfl_xor_sync(0xffffffffu, sx[k], o);
        sy[k] += __shfl_xor_sync(0xffffffffu, sy[k], o);
        sz[k] += __shfl_xor_sync(0xffffffffu, sz[k], o);
      }
    }
    if (zl == 0) {
#pragma unroll
      for (int k = 0; k < 8; k++) {
        red[warp][2][0][cc * 8 + k] = s0[k];
        red[warp][2][1][cc * 8 + k] = sx[k];
        red[warp][2][2][cc * 8 + k] = sy[k];
        red[warp][2][3][cc * 8 + k] = sz[k];
      }
    }
    if (bcls >= 0) {
#pragma unroll
      for (int k = 0; k < 8; k++) {
        red[warp][bcls][0][cc * 8 + k] = b0[k];
        red[warp][bcls][1][cc * 8 + k] = bx[k];
        red[warp][bcls][2][cc * 8 + k] = by[k];
        red[warp][bcls][3][cc * 8 + k] = bz * b0[k];
      }
    }
    __syncthreads();
    for (int i = threadIdx.x; i < 5 * 4 * C; i += 256) {
      float t = 0.f;
#pragma unroll
      for (int w = 0; w < 8; w++) t += (&red[w][0][0][0])[i];
      og[i] = t;
    }
    __syncthreads();
  }
}

// occupancy channel: partial[n][parts][125][C] = sum over this part's occupied u of occ[u] * dY[u - (t - 2)].
// The volume is walked in 8^3 cores; a core without occupied voxels (most of them: the occupancy is a surface) costs one
// 2 KB read.  For the others the 12^3 dY voxels the core's taps can reach are staged once in shared memory (cp.async,
// zero fill outside the volume = the conv's padding), 32 channels at a time, and every occupied voxel gathers its 125
// rows from there: lane = channel, warp w owns taps w, w + 8, ... (16 accumulators per lane, carried over all cores of the
// CTA).  The first version gathered the 64-byte rows straight from L2 (40 MB per frame, latency-bound: 6.3 + 2.5 ms per step).
constexpr int kFoCore = 8, kFoReg = kFoCore + 4;
template <int C>
__global__ void __launch_bounds__(256)
first_wgrad_occ_kernel(const float* __restrict__ occ, const __half* __restrict__ dy, int G, float* __restrict__ partial) {
  extern __shared__ __align__(16) uint8_t fo_smem[];
  __half* s_dy = reinterpret_cast<__half*>(fo_smem);                       // [12^3][32]
  int* s_idx = reinterpret_cast<int*>(fo_smem + (size_t)kFoReg * kFoReg * kFoReg * 64);   // [512] local voxel index
  float* s_val = reinterpret_cast<float*>(s_idx + 512);                     // [512]
  int* s_cnt = reinterpret_cast<int*>(s_val + 512);                         // [9]
  constexpr int HALVES = C / 32;
  const int n = blockIdx.x, part = blockIdx.y, parts = gridDim.y, S = G * G * G;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int cpa = G / kFoCore, cores = cpa * cpa * cpa;
  float acc[HALVES][16];
#pragma unroll
  for (int hh = 0; hh < HALVES; hh++)
#pragma unroll
    for (int i = 0; i < 16; i++) acc[hh][i] = 0.f;
  const float* on = occ + (long long)n * S;
  const __half* dyn = dy + (long long)n * S * C;
  // this warp's taps t = warp + 8 i as offsets inside the staged region (in halfs): the gather's address is one subtraction
  int toff[16];
#pragma unroll
  for (int i = 0; i < 16; i++) {
    const int t = warp + 8 * i;
    toff[i] = (((t / 25) * kFoReg + (t / 5) % 5) * kFoReg + t % 5) * 32;
  }
  // the core's two occupancy values of this thread (2 consecutive z): read one core ahead of their use
  auto occ_pair = [&](int core) -> float2 {
    const int cx = (core / (cpa * cpa)) * kFoCore, cy = ((core / cpa) % cpa) * kFoCore, cz = (core % cpa) * kFoCore;
    const int l = threadIdx.x * 2;
    return *reinterpret_cast<const float2*>(on + ((long long)(cx + (l >> 6)) * G + cy + ((l >> 3) & 7)) * G + cz + (l & 7));
  };
  float2 nextv = make_float2(0.f, 0.f);
  if (part < cores) nextv = occ_pair(part);
  for (int core = part; core < cores; core += parts) {
    const int cx = (core / (cpa * cpa)) * kFoCore, cy = ((core / cpa) % cpa) * kFoCore, cz = (core % cpa) * kFoCore;
    // ordered compaction of the core's non-zero voxels (2 consecutive z per thread)
    __syncthreads();                                                        // previous core's list / tile are consumed
    const float v[2] = {nextv.x, nextv.y};
    if (core + parts < cores) nextv = occ_pair(core + parts);
    int mine = 0;
#pragma unroll
    for (int j = 0; j < 2; j++) mine += v[j] != 0.f;
    int incl = mine;
#pragma unroll
    for (int o = 1; o < 32; o <<= 1) {
      const int t = __shfl_up_sync(0xffffffffu, incl, o);
      if (lane >= o) incl += t;
    }
    if (lane == 31) s_cnt[warp + 1] = incl;
    __syncthreads();
    if (threadIdx.x == 0) {
      s_cnt[0] = 0;
      for (int k = 1; k <= 8; k++) s_cnt[k] += s_cnt[k - 1];
    }
    __syncthreads();
    const int count = s_cnt[8];
    if (count == 0) continue;                                               // block-uniform
    int pos = s_cnt[warp] + incl - mine;
#pragma unroll
    for (int j = 0; j < 2; j++)
      if (v[j] != 0.f) { s_idx[pos] = threadIdx.x * 2 + j; s_val[pos] = v[j]; pos++; }
#pragma unroll
    for (int hh = 0; hh < HALVES; hh++) {
      if (hh > 0) __syncthreads();                                          // the previous half's tile is consumed
      // stage the 12^3 x 32-channel dY region around the core
      for (int i = threadIdx.x; i < kFoReg * kFoReg * kFoReg * 4; i += 256) {
        const int c = i & 3, r = i >> 2;
        const int rz = r % kFoReg, ry = (r / kFoReg) % kFoReg, rx = r / (kFoReg * kFoReg);
        const int gx = cx - 2 + rx, gy = cy - 2 + ry, gz = cz - 2 + rz;
        const bool ok = (unsigned)gx < (unsigned)G && (unsigned)gy < (unsigned)G && (unsigned)gz < (unsigned)G;
        const __half* src = ok ? dyn + (((long long)gx * G + gy) * G + gz) * C + hh * 32 + c * 8 : dyn;
        asm volatile("cp.async.cg.shared.global [%0], [%1], 16, %2;" ::"r"((uint32_t)__cvta_generic_to_shared(s_dy + r * 32 + c * 8)),
                     "l"(src), "r"(ok ? 16 : 0) : "memory");
      }
      asm volatile("cp.async.commit_group;\n\tcp.async.wait_group 0;" ::: "memory");
      __syncthreads();
      for (int e = 0; e < count; e++) {
        const int l = s_idx[e];
        const float val = s_val[e];
        // region coordinates of dY[u - (t - 2)]: (l + 4 - t) per axis, always inside the staged region
        const int bx = (l >> 6) + 4, by = ((l >> 3) & 7) + 4, bz = (l & 7) + 4;
        const __half* pe = s_dy + ((bx * kFoReg + by) * kFoReg + bz) * 32 + lane;
#pragma unroll
        for (int i = 0; i < 16; i++)
          if (warp + 8 * i < 125) acc[hh][i] = fmaf(val, __half2float(pe[-toff[i]]), acc[hh][i]);
      }
    }
  }
#pragma unroll
  for (int hh = 0; hh < HALVES; hh++)
#pragma unroll
    for (int i = 0; i < 16; i++) {
      const int t = warp + 8 * i;
      if (t < 125) partial[(((long long)n * parts + part) * 125 + t) * C + hh * 32 + lane] = acc[hh][i];
    }
}

// dW (C, 4, 5, 5, 5) from the per-frame bins and occupancy partials (fixed order over the frames, fp64)
__global__ void first_wgrad_finalize_kernel(const float* __restrict__ bins, const float* __restrict__ occp, int n, int C, int G,
                                            const float* __restrict__ lin, float out_scale, float* __restrict__ dw) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= C * 4 * 125) return;
  const int t = i % 125, ch = (i / 125) % 4, co = i / 500;
  double acc = 0.0;
  if (ch == 0) {
    for (int f = 0; f < n; f++) acc += (double)occp[((long long)f * 125 + t) * C + co];
  } else {
    const int a = ch - 1;
    const int tap[3] = {t / 25, (t / 5) % 5, t % 5};
    const double l0 = lin[0], delta = ((double)lin[G - 1] - (double)lin[0]) / (double)(G - 1);
    double m0 = 0.0, ma = 0.0;
    for (int f = 0; f < n; f++)
      for (int bx = max(0, 2 - tap[0]); bx <= min(4, 6 - tap[0]); bx++)
        for (int by = max(0, 2 - tap[1]); by <= min(4, 6 - tap[1]); by++)
          for (int bz = max(0, 2 - tap[2]); bz <= min(4, 6 - tap[2]); bz++) {
            const float* b = bins + (((long long)f * 125 + (bx * 25 + by * 5 + bz)) * 4) * C;
            m0 += (double)b[co];
            ma += (double)b[(1 + a) * C + co];
          }
    acc = (l0 + delta * (double)(tap[a] - 2)) * m0 + delta * ma;
  }
  dw[i] = (float)(acc * (double)out_scale);
}

// ------------------------------------------------------------------ Adam (torch.optim.Adam defaults: no amsgrad, no decay)
__global__ void grad_nonfinite_kernel(const float* __restrict__ g, long long n, int* __restrict__ flag) {
  bool bad = false;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float v = g[i];
    bad |= !(fabsf(v) <= 3.0e38f);
  }
  if (__syncthreads_or(bad) && threadIdx.x == 0) atomicOr(flag, 1);
}

__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                            long long n, float lr, float beta1, float beta2, float eps, float bc1, float bc2_sqrt,
                            float grad_mul, const int* __restrict__ skip_flag) {
  if (skip_flag && *skip_flag) return;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i] * grad_mul;
    const float mi = fmaf(beta1, m[i], (1.f - beta1) * gi);
    const float vi = fmaf(beta2, v[i], (1.f - beta2) * gi * gi);
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}

// The same step with the step count kept on the device (*step_dev = number of steps applied so far): nothing about the
// launch depends on host state, so a captured CUDA graph of a whole training step can be replayed.  The bias corrections
// are evaluated per thread in double, exactly as the host does for adam_kernel.
__global__ void adam_dev_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m, float* __restrict__ v,
                                long long n, float lr, float beta1, float beta2, float eps, const int* __restrict__ step_dev,
                                float grad_mul, const int* __restrict__ skip_flag) {
  if (skip_flag && *skip_flag) return;
  const double step = (double)(*step_dev + 1);
  const float bc1 = (float)(1.0 - pow((double)beta1, step));
  const float bc2_sqrt = (float)sqrt(1.0 - pow((double)beta2, step));
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < n; i += (long long)gridDim.x * blockDim.x) {
    const float gi = g[i] * grad_mul;
    const float mi = fmaf(beta1, m[i], (1.f - beta1) * gi);
    const float vi = fmaf(beta2, v[i], (1.f - beta2) * gi * gi);
    m[i] = mi;
    v[i] = vi;
    const float denom = sqrtf(vi) / bc2_sqrt + eps;
    p[i] -= (lr / bc1) * (mi / denom);
  }
}
// counters[0] += 1 when the step was applied, counters[1] += 1 when it was skipped (runs after adam_dev_kernel)
__global__ void adam_advance_kernel(int* __restrict__ counters, const int* __restrict__ skip_flag) {
  if (threadIdx.x == 0 && blockIdx.x == 0) counters[(skip_flag && *skip_flag) ? 1 : 0] += 1;
}

}  // namespace

// =================================================================== C ABI
extern "C" size_t nm_upsample2x_backward_workspace_bytes(int n, int D, int H, int W, int C) {
  // the two intermediates: (n, 2D, 2H, W, C) and (n, 2D, H, W, C) fp16
  return ((size_t)n * 2 * D * 2 * H * W * C + (size_t)n * 2 * D * H * W * C) * sizeof(__half) + 256;
}

extern "C" int nm_upsample2x_backward(const void* grad_out, void* grad_in, int n, int D, int H, int W, int C, void* workspace,
                                      void* stream) {
  NM_CHECK_ARG(grad_out && grad_in && workspace, "nm_upsample2x_backward: null pointer");
  NM_CHECK_ARG(C % 8 == 0 && n > 0 && D > 0 && H > 0 && W > 0, "nm_upsample2x_backward: bad shape");
  cudaStream_t st = (cudaStream_t)stream;
  __half* t1 = reinterpret_cast<__half*>(workspace);                              // (n, 2D, 2H, W, C)
  __half* t2 = t1 + (((size_t)n * 2 * D * 2 * H * W * C + 127) & ~(size_t)127);   // (n, 2D, H, W, C)
  const long long c8 = C / 8;
  struct Pass { const __half* in; __half* out; long long outer; int L; long long inner8; };
  const Pass passes[3] = {
      {reinterpret_cast<const __half*>(grad_out), t1, (long long)n * 2 * D * 2 * H, W, c8},
      {t1, t2, (long long)n * 2 * D, H, (long long)W * c8},
      {t2, reinterpret_cast<__half*>(grad_in), (long long)n, D, (long long)H * W * c8}};
  for (const Pass& p : passes) {
    const long long total8 = p.outer * p.L * p.inner8;
    const int blocks = (int)min((long long)nm_num_sms() * 16, (total8 + 255) / 256);
    auto lg = [](long long v) { int l = 0; while ((1LL << l) < v) l++; return l; };
    const bool pow2 = !(p.L & (p.L - 1)) && !(p.inner8 & (p.inner8 - 1));
    if (pow2)
      upsample2x_bwd_axis_kernel<true><<<blocks, 256, 0, st>>>(p.in, p.out, p.outer, p.L, p.inner8, total8, lg(p.inner8), lg(p.L));
    else
      upsample2x_bwd_axis_kernel<false><<<blocks, 256, 0, st>>>(p.in, p.out, p.outer, p.L, p.inner8, total8, 0, 0);
    NM_CHECK_LAUNCH("upsample2x_bwd_axis_kernel");
  }
  return NM_OK;
}

extern "C" int nm_depth_to_space2(const void* y, void* out, int n, int D, int H, int W, int C, int tap0, int ntaps, void* stream) {
  NM_CHECK_ARG(y && out, "nm_depth_to_space2: null pointer");
  NM_CHECK_ARG(C % 8 == 0 && tap0 >= 0 && ntaps >= 1 && tap0 + ntaps <= 8 && n > 0 && D > 0 && H > 0 && W > 0,
               "nm_depth_to_space2: bad shape");
  const long long total8 = (long long)n * D * H * W * ntaps * (C / 8);
  const int blocks = (int)min((long long)nm_num_sms() * 16, (total8 + 255) / 256);
  depth_to_space2_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(reinterpret_cast<const __half*>(y), reinterpret_cast<__half*>(out),
                                                                   D, H, W, C, tap0, ntaps, total8);
  NM_CHECK_LAUNCH("depth_to_space2_kernel");
  return NM_OK;
}

extern "C" size_t nm_final_recon_backward_workspace_bytes(int n) { return ((size_t)n * kFrbBlocks * 33 + 64) * sizeof(float); }

extern "C" int nm_final_recon_backward(const void* x, const float* a, const float* b, const float* w, float bias,
                                       const float* bias_dev,
                                       const float* first_frame, int frames_per_clip, float sharpness, float translation,
                                       const float* recon, const float* target, const float* grad_bce, float grad_scale,
                                       void* grad_act, float* dw, float* dbias, void* workspace, int n, int S, int C,
                                       void* stream) {
  NM_CHECK_ARG(x && a && b && w && recon && target && grad_bce && grad_act && dw && dbias && workspace,
               "nm_final_recon_backward: null pointer");
  NM_CHECK_ARG(C == 32, "nm_final_recon_backward: C=%d unsupported (decoder tail is 32 channels)", C);
  if (n == 0) return NM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  float* partial = reinterpret_cast<float*>(workspace);
  final_recon_bwd_kernel<<<dim3(kFrbBlocks, n), 256, 0, st>>>(reinterpret_cast<const __half*>(x), a, b, w, bias, bias_dev, first_frame,
                                                             frames_per_clip, sharpness, translation, recon, target, grad_bce,
                                                             grad_scale, reinterpret_cast<__half*>(grad_act), partial, S);
  NM_CHECK_LAUNCH("final_recon_bwd_kernel");
  // columns 0..31 -> dw, column 32 -> dbias
  reduce_cols_kernel<<<1, dim3(32, 8), 0, st>>>(partial, (long long)n * kFrbBlocks, 33, 32, 1.0f, dw);
  NM_CHECK_LAUNCH("final_recon_bwd(reduce dw)");
  reduce_cols_kernel<<<1, dim3(32, 8), 0, st>>>(partial + 32, (long long)n * kFrbBlocks, 33, 1, 1.0f, dbias);
  NM_CHECK_LAUNCH("final_recon_bwd(reduce dbias)");
  return NM_OK;
}

// voxel splits per frame: enough CTAs for ~4 per SM, at most 8 (a 8^3 heat-map has 8 tiles of 64 voxels)
static int head_bwd_splits(int n) {
  int splits = 1;
  while (splits < 8 && (long long)n * splits < 592) splits *= 2;
  return splits;
}

template <int C, int KMAX>
static int launch_head_bwd(int n, int splits, cudaStream_t st, const __half* feature, const float* w1, const float* b1, int K, int g,
                           int mode, const float* prev, int frames_per_clip, float pw0, float pw1, float pb, const float* prop_dev,
                           const float* lin, const float* heat, const float* kp, const float* heat_mean, const float* dkp,
                           const float* dmean_up, const float* dheat, const float* dq_in, float grad_scale, __half* dfeat,
                           float* dq_out, float* pwp, float* pbp, float* ppp) {
  const size_t smem = (size_t)(KMAX * C + 64 * (C + 4) + 2 * KMAX * 64 + KMAX * 4 + 256 * 3) * sizeof(float);
  const dim3 grid(n, splits, KMAX / head_bwd_kw<C, KMAX>());
  NM_CHECK_CUDA(cudaFuncSetAttribute(head_bwd_kernel<C, KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  head_bwd_kernel<C, KMAX><<<grid, 256, smem, st>>>(feature, w1, b1, K, g, mode, prev, frames_per_clip, pw0, pw1, pb, prop_dev, lin,
                                                    heat, kp, heat_mean, dkp, dmean_up, dheat, dq_in, grad_scale, dfeat, dq_out,
                                                    pwp, pbp, ppp);
  return NM_OK;
}

extern "C" size_t nm_heatmap_head_backward_workspace_bytes(int n, int C, int K) {
  const size_t rows = (size_t)n * head_bwd_splits(n);
  return (rows * K * C + rows * K + rows * 3) * sizeof(float);
}

extern "C" int nm_heatmap_head_backward(const void* feature, const float* w1, const float* b1, int n, int g, int C, int K, int mode,
                                        const float* prev, int frames_per_clip, float pw0, float pw1, float pb,
                                        const float* prop_dev,
                                        const float* linspace, const float* heat, const float* keypoints,
                                        const float* heat_mean, const float* grad_keypoints, const float* grad_heat_mean,
                                        const float* grad_heat, const float* dq_in, float grad_scale, void* grad_feature,
                                        float* dq_out, float* dw1, float* db1, float* dprop, void* workspace, void* stream) {
  NM_CHECK_ARG(feature && w1 && b1 && linspace && grad_feature && dw1 && db1 && workspace, "nm_heatmap_head_backward: null pointer");
  NM_CHECK_ARG(K <= kMaxK && (g == 8 || g == 16 || g == 32), "nm_heatmap_head_backward: K=%d g=%d unsupported", K, g);
  NM_CHECK_ARG(mode == 0 || (prev && heat && keypoints && heat_mean && dq_out && dprop),
               "nm_heatmap_head_backward: mode 1 needs prev, heat, keypoints, heat_mean, dq_out and dprop");
  NM_CHECK_ARG(C == 128 || C == 256, "nm_heatmap_head_backward: C=%d unsupported", C);
  if (n == 0) return NM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int splits = head_bwd_splits(n);
  const long long rows = (long long)n * splits;
  float* pwp = reinterpret_cast<float*>(workspace);
  float* pbp = pwp + (size_t)rows * K * C;
  float* ppp = pbp + (size_t)rows * K;
  const __half* f = reinterpret_cast<const __half*>(feature);
  __half* gf = reinterpret_cast<__half*>(grad_feature);
  int rc;
  if (K <= kTunedK)
    rc = C == 128 ? launch_head_bwd<128, kTunedK>(n, splits, st, f, w1, b1, K, g, mode, prev, frames_per_clip, pw0, pw1, pb, prop_dev, linspace, heat, keypoints, heat_mean, grad_keypoints, grad_heat_mean, grad_heat, dq_in, grad_scale, gf, dq_out, pwp, pbp, ppp)
                  : launch_head_bwd<256, kTunedK>(n, splits, st, f, w1, b1, K, g, mode, prev, frames_per_clip, pw0, pw1, pb, prop_dev, linspace, heat, keypoints, heat_mean, grad_keypoints, grad_heat_mean, grad_heat, dq_in, grad_scale, gf, dq_out, pwp, pbp, ppp);
  else
    rc = C == 128 ? launch_head_bwd<128, kMaxK>(n, splits, st, f, w1, b1, K, g, mode, prev, frames_per_clip, pw0, pw1, pb, prop_dev, linspace, heat, keypoints, heat_mean, grad_keypoints, grad_heat_mean, grad_heat, dq_in, grad_scale, gf, dq_out, pwp, pbp, ppp)
                  : launch_head_bwd<256, kMaxK>(n, splits, st, f, w1, b1, K, g, mode, prev, frames_per_clip, pw0, pw1, pb, prop_dev, linspace, heat, keypoints, heat_mean, grad_keypoints, grad_heat_mean, grad_heat, dq_in, grad_scale, gf, dq_out, pwp, pbp, ppp);
  if (rc) return rc;
  NM_CHECK_LAUNCH("head_bwd_kernel");
  reduce_cols_kernel<<<nm_cdiv(K * C, 32), dim3(32, 8), 0, st>>>(pwp, rows, K * C, K * C, 1.0f, dw1);
  NM_CHECK_LAUNCH("head_bwd(reduce dw1)");
  reduce_cols_kernel<<<nm_cdiv(K, 32), dim3(32, 8), 0, st>>>(pbp, rows, K, K, 1.0f, db1);
  NM_CHECK_LAUNCH("head_bwd(reduce db1)");
  if (mode == 1) {
    reduce_cols_kernel<<<1, dim3(32, 8), 0, st>>>(ppp, rows, 3, 3, 1.0f, dprop);
    NM_CHECK_LAUNCH("head_bwd(reduce dprop)");
  }
  return NM_OK;
}

constexpr int kAdjSplits = 8;

template <int KMAX>
size_t adjust_bwd_ws_bytes(size_t n, size_t n_clips) {
  return (n * kAdjC * KMAX + n * kAdjC + n_clips * kAdjSplits * kAdjC * (kAdjC + KMAX + 3) + n_clips * kAdjSplits * KMAX * 4) *
         sizeof(float);
}

template <int KMAX>
static int launch_adjust_bwd(const __half* dy, const __half* y, const __half* ff, const float* keypoints, const float* weight,
                             int n_clips, int frames_per_clip, int g, int K, const float* linspace, float gauss_width,
                             float grad_scale, __half* dff, float* grad_keypoints, float* dweight, float* dbias, float* ws,
                             cudaStream_t st) {
  const int n = n_clips * frames_per_clip, ld = 2 * K + kAdjC + 3;
  float* pwg = ws;
  float* pbias = pwg + (size_t)n * kAdjC * KMAX;
  float* pw = pbias + (size_t)n * kAdjC;
  float* dkp0 = pw + (size_t)n_clips * kAdjSplits * kAdjC * (kAdjC + KMAX + 3);
  const float inv_scale = 1.0f / grad_scale;
  const size_t smem_f = (size_t)adj_frame_floats<KMAX>() * sizeof(float);
  NM_CHECK_CUDA(cudaFuncSetAttribute(adjust_bwd_frame_kernel<KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_f));
  adjust_bwd_frame_kernel<KMAX><<<n, 256, smem_f, st>>>(dy, y, keypoints, weight, ld, K, g, linspace, gauss_width, inv_scale,
                                                        grad_keypoints, pwg, pbias);
  NM_CHECK_LAUNCH("adjust_bwd_frame_kernel");
  const size_t smem_c = (size_t)adj_clip_floats<KMAX>() * sizeof(float);
  NM_CHECK_CUDA(cudaFuncSetAttribute(adjust_bwd_clip_kernel<KMAX>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem_c));
  adjust_bwd_clip_kernel<KMAX><<<dim3(n_clips, kAdjSplits), 256, smem_c, st>>>(dy, y, ff, keypoints, weight, ld, K, g,
                                                                               frames_per_clip, linspace, gauss_width, inv_scale,
                                                                               grad_scale, dff, dkp0, pw);
  NM_CHECK_LAUNCH("adjust_bwd_clip_kernel");
  const int total = kAdjC * ld + kAdjC + n_clips * K * 4;
  adjust_bwd_finalize_kernel<KMAX><<<nm_cdiv(total, 128), 128, 0, st>>>(pwg, pbias, pw, dkp0, n, n_clips * kAdjSplits, n_clips,
                                                                        kAdjSplits, frames_per_clip, K, dweight, dbias,
                                                                        grad_keypoints);
  NM_CHECK_LAUNCH("adjust_bwd_finalize_kernel");
  return NM_OK;
}

// sized for the kMaxK layout (the larger one) whatever K is, since the size does not take K
extern "C" size_t nm_decoder_adjust_backward_workspace_bytes(int n_clips, int frames_per_clip) {
  return adjust_bwd_ws_bytes<kMaxK>((size_t)n_clips * frames_per_clip, (size_t)n_clips);
}

extern "C" int nm_decoder_adjust_backward(const void* grad_out, const void* out, const void* first_feature, const float* keypoints,
                                          const float* weight, int n_clips, int frames_per_clip, int g, int K,
                                          const float* linspace, float gauss_width, float grad_scale, void* grad_first_feature,
                                          float* grad_keypoints, float* dweight, float* dbias, void* workspace, void* stream) {
  NM_CHECK_ARG(grad_out && out && first_feature && keypoints && weight && linspace && grad_first_feature && grad_keypoints &&
               dweight && dbias && workspace, "nm_decoder_adjust_backward: null pointer");
  NM_CHECK_ARG(K <= kMaxK && (g == 8 || g == 16 || g == 32), "nm_decoder_adjust_backward: K=%d g=%d unsupported", K, g);
  if (n_clips == 0) return NM_OK;
  const __half* dy = reinterpret_cast<const __half*>(grad_out);
  const __half* y = reinterpret_cast<const __half*>(out);
  const __half* ff = reinterpret_cast<const __half*>(first_feature);
  __half* dff = reinterpret_cast<__half*>(grad_first_feature);
  float* ws = reinterpret_cast<float*>(workspace);
  if (K <= kTunedK)
    return launch_adjust_bwd<kTunedK>(dy, y, ff, keypoints, weight, n_clips, frames_per_clip, g, K, linspace, gauss_width,
                                      grad_scale, dff, grad_keypoints, dweight, dbias, ws, (cudaStream_t)stream);
  return launch_adjust_bwd<kMaxK>(dy, y, ff, keypoints, weight, n_clips, frames_per_clip, g, K, linspace, gauss_width,
                                  grad_scale, dff, grad_keypoints, dweight, dbias, ws, (cudaStream_t)stream);
}

extern "C" size_t nm_chamfer_vol_fit_backward_workspace_bytes(int n, int K) { return (size_t)n * kChbBlocks * (K * 3 + 1) * sizeof(float); }

extern "C" int nm_chamfer_vol_fit_backward(const float* seq, const float* keypoints, const float* linspace, const float* grad_out,
                                           int n, int K, int G, float* grad_keypoints, void* workspace, void* stream) {
  NM_CHECK_ARG(seq && keypoints && linspace && grad_out && grad_keypoints && workspace, "nm_chamfer_vol_fit_backward: null pointer");
  NM_CHECK_ARG(K <= kMaxK, "nm_chamfer_vol_fit_backward: K=%d unsupported", K);
  if (n == 0) return NM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  float* ws = reinterpret_cast<float*>(workspace);
  if (K <= kTunedK) {
    const size_t smem = (size_t)(kTunedK * 3 + kTunedK * 3 * 256) * sizeof(float);
    NM_CHECK_CUDA(cudaFuncSetAttribute(chamfer_bwd_kernel<kTunedK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    chamfer_bwd_kernel<kTunedK><<<dim3(kChbBlocks, n), 256, smem, st>>>(seq, keypoints, K, G, linspace, ws);
  } else {
    // 196 KB: one CTA per SM
    const size_t smem = (size_t)(kMaxK * 3 + kMaxK * 3 * 256) * sizeof(float);
    NM_CHECK_CUDA(cudaFuncSetAttribute(chamfer_bwd_kernel<kMaxK>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    chamfer_bwd_kernel<kMaxK><<<dim3(kChbBlocks, n), 256, smem, st>>>(seq, keypoints, K, G, linspace, ws);
  }
  NM_CHECK_LAUNCH("chamfer_bwd_kernel");
  chamfer_bwd_finalize_kernel<<<nm_cdiv((long long)n * K * 4, 128), 128, 0, st>>>(reinterpret_cast<const float*>(workspace), grad_out, n, K,
                                                                                 kChbBlocks, grad_keypoints);
  NM_CHECK_LAUNCH("chamfer_bwd_finalize_kernel");
  return NM_OK;
}

// CTAs per frame: the once-per-clip branch has few (dense) frames, the per-frame encoder many sparse ones
static int first_wgrad_parts(int n) {
  int p = (12 * nm_num_sms() + n - 1) / n;                 // >= 6 waves of 2 CTAs per SM: the x slabs are uneven work
  return p < 1 ? 1 : (p > 8 ? 8 : p);
}
// the occupancy gather is latency-bound (64-byte rows from L2): several resident CTAs per SM keep more loads in flight
static int first_wgrad_occ_parts(int n) {
  int p = (6 * nm_num_sms() + n - 1) / n;
  return p < 1 ? 1 : (p > 16 ? 16 : p);
}

extern "C" size_t nm_first_conv_wgrad_workspace_bytes(int n, int Cout) {
  return ((size_t)n * first_wgrad_parts(n) * 4 + (size_t)n * first_wgrad_occ_parts(n) + 5) * 125 * Cout * sizeof(float);
}

extern "C" int nm_first_conv_wgrad(const float* occ, const void* grad_out, const float* linspace, int n, int G, int Cout,
                                   float out_scale, float* dw, void* workspace, void* stream) {
  NM_CHECK_ARG(occ && grad_out && linspace && dw && workspace, "nm_first_conv_wgrad: null pointer");
  NM_CHECK_ARG((Cout == 32 || Cout == 64) && G >= 8 && G % 16 == 0, "nm_first_conv_wgrad: Cout=%d G=%d unsupported", Cout, G);
  if (n == 0) return NM_OK;
  cudaStream_t st = (cudaStream_t)stream;
  const int parts = first_wgrad_parts(n), oparts = first_wgrad_occ_parts(n);
  const long long rows = (long long)n * parts, orows = (long long)n * oparts;
  float* bins = reinterpret_cast<float*>(workspace);
  float* occp = bins + (size_t)rows * 125 * 4 * Cout;
  const __half* dy = reinterpret_cast<const __half*>(grad_out);
  const dim3 grid(n, parts), ogrid(n, oparts);
  const size_t fo_smem_bytes = (size_t)kFoReg * kFoReg * kFoReg * 64 + 512 * 8 + 64;
  if (Cout == 32) {
    first_wgrad_moments_kernel<32><<<grid, 256, 0, st>>>(dy, G, bins);
    NM_CHECK_LAUNCH("first_wgrad_moments_kernel");
    NM_CHECK_CUDA(cudaFuncSetAttribute(first_wgrad_occ_kernel<32>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fo_smem_bytes));
    first_wgrad_occ_kernel<32><<<ogrid, 256, fo_smem_bytes, st>>>(occ, dy, G, occp);
  } else {
    first_wgrad_moments_kernel<64><<<grid, 256, 0, st>>>(dy, G, bins);
    NM_CHECK_LAUNCH("first_wgrad_moments_kernel");
    NM_CHECK_CUDA(cudaFuncSetAttribute(first_wgrad_occ_kernel<64>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)fo_smem_bytes));
    first_wgrad_occ_kernel<64><<<ogrid, 256, fo_smem_bytes, st>>>(occ, dy, G, occp);
  }
  NM_CHECK_LAUNCH("first_wgrad_occ_kernel");
  // sum over the frames and parts first (fixed order), then assemble the (Cout, 4, 5, 5, 5) tensor
  float* rbins = occp + (size_t)orows * 125 * Cout;
  float* roccp = rbins + (size_t)125 * 4 * Cout;
  reduce_cols_kernel<<<nm_cdiv(500 * Cout, 32), dim3(32, 8), 0, st>>>(bins, rows, 500 * Cout, 500 * Cout, 1.0f, rbins);
  NM_CHECK_LAUNCH("first_wgrad(reduce bins)");
  reduce_cols_kernel<<<nm_cdiv(125 * Cout, 32), dim3(32, 8), 0, st>>>(occp, orows, 125 * Cout, 125 * Cout, 1.0f, roccp);
  NM_CHECK_LAUNCH("first_wgrad(reduce occ)");
  first_wgrad_finalize_kernel<<<nm_cdiv(Cout * 500, 128), 128, 0, st>>>(rbins, roccp, 1, Cout, G, linspace, out_scale, dw);
  NM_CHECK_LAUNCH("first_wgrad_finalize_kernel");
  return NM_OK;
}

extern "C" int nm_grad_nonfinite(const float* grad, long long count, int* flag, void* stream) {
  NM_CHECK_ARG(grad && flag, "nm_grad_nonfinite: null pointer");
  if (count <= 0) return NM_OK;
  const int blocks = (int)min((long long)nm_num_sms() * 4, (count + 255) / 256);
  grad_nonfinite_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(grad, count, flag);
  NM_CHECK_LAUNCH("grad_nonfinite_kernel");
  return NM_OK;
}

extern "C" int nm_adam_step_dev(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long count, float lr,
                                float beta1, float beta2, float eps, int* counters, float grad_mul, const int* skip_flag,
                                void* stream) {
  NM_CHECK_ARG(param && grad && exp_avg && exp_avg_sq && counters, "nm_adam_step_dev: null pointer");
  if (count <= 0) return NM_OK;
  const int blocks = (int)min((long long)nm_num_sms() * 8, (count + 255) / 256);
  adam_dev_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(param, grad, exp_avg, exp_avg_sq, count, lr, beta1, beta2, eps, counters,
                                                            grad_mul, skip_flag);
  NM_CHECK_LAUNCH("adam_dev_kernel");
  adam_advance_kernel<<<1, 32, 0, (cudaStream_t)stream>>>(counters, skip_flag);
  NM_CHECK_LAUNCH("adam_advance_kernel");
  return NM_OK;
}

extern "C" int nm_adam_step(float* param, const float* grad, float* exp_avg, float* exp_avg_sq, long long count, float lr,
                            float beta1, float beta2, float eps, int step, float grad_mul, const int* skip_flag, void* stream) {
  NM_CHECK_ARG(param && grad && exp_avg && exp_avg_sq, "nm_adam_step: null pointer");
  NM_CHECK_ARG(step >= 1, "nm_adam_step: step counts from 1");
  if (count <= 0) return NM_OK;
  const double bc1 = 1.0 - pow((double)beta1, (double)step), bc2 = 1.0 - pow((double)beta2, (double)step);
  const int blocks = (int)min((long long)nm_num_sms() * 8, (count + 255) / 256);
  adam_kernel<<<blocks, 256, 0, (cudaStream_t)stream>>>(param, grad, exp_avg, exp_avg_sq, count, lr, beta1, beta2, eps, (float)bc1,
                                                        (float)sqrt(bc2), grad_mul, skip_flag);
  NM_CHECK_LAUNCH("adam_kernel");
  return NM_OK;
}
