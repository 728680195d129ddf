// One fused kernel per HSVRNN time step (reference: model/hsvrnn_bvh.py:89-135 / 171-225,
// extract_kypt_from_latent_and_state :255-286, utils/geo_utils.py:3-78, nn.GRUCell :57-58).
//
// The reference spends a step in ~4.7k ATen launches and ~750 host syncs; the arithmetic is
// ~6 MFLOP/sample over 6.1 MB of fp32 weights, i.e. latency / L2-bound.  Here a CTA owns NB
// batch elements and walks the whole step in shared memory:
//   prior MLP (optional) -> posterior MLP -> z_s = mu + sigma*eps_s -> decoders for all S
//   samples -> 6-D rotations + forward kinematics down the skeleton -> nearest-sample pick
//   -> GRU cell.
// All matrices are stored transposed ([in][out], prepared once by the host) so that a thread
// owns an output column: weight reads are coalesced across the CTA, activations are
// shared-memory broadcasts, no shuffles.  fp32 throughout (the nearest-sample pick is a
// discrete decision; keep it as close to the reference arithmetic as possible).
#include "common.cuh"
#include "../../include/nm_b200.h"

namespace {

constexpr int kThreads = 256;
constexpr int H = 512, Z = 128, HID = 128;
// Keypoint capacity of a kernel instantiation: K <= kTunedK (the shipped 24) runs the tuned kernels, 24 < K <= kMaxK a
// set compiled for kMaxK.  Shared-memory rows sized by the capacity KC:
template <int KC>
struct KpDims {
  static constexpr int K4 = 4 * KC;                  // flat pose (x, y, z, intensity) per keypoint
  static constexpr int XW = 4 * KC + 128;            // GRU input: pose | z
  static constexpr int JO = (3 + KC + 7) / 8 * 8;    // decoder row: root / intensity (3 + K) at 0, joint 6-D (6K) at JO
  static constexpr int DW = JO + 6 * KC;
};
constexpr int kTunedK = 24, kMaxK = 64;
constexpr int VC = 8;  // vectors per register chunk

__device__ __forceinline__ float softplus_d(float x) { return x > 20.f ? x : log1pf(expf(x)); }
__device__ __forceinline__ float sigmoid_d(float x) { return 1.0f / (1.0f + expf(-x)); }

// out[v][c] = act(bias[c] + sum_i WT[i][col0 + c] * x[v][i]) for v < nvec, c < ncols.
// x rows beyond nvec (up to the next multiple of VC) must be readable (zero padded).
// act: 0 none, 1 leaky relu, 2 tanh.  `add` (optional, [v / add_div][c]) is added before act.
__device__ void cols_matvec(const float* __restrict__ WT, int ldw, int col0, int ncols, int I,
                            const float* x, int xstride, int nvec, const float* __restrict__ bias,
                            const float* add, int add_stride, int add_div, int act, float* out, int ostride) {
  for (int c = threadIdx.x; c < ncols; c += kThreads) {
    const float* w = WT + col0 + c;
    for (int v0 = 0; v0 < nvec; v0 += VC) {
      float acc[VC];
#pragma unroll
      for (int u = 0; u < VC; u++) acc[u] = 0.f;
#pragma unroll 4
      for (int i = 0; i < I; i++) {
        const float wi = __ldg(w + (long long)i * ldw);
#pragma unroll
        for (int u = 0; u < VC; u++) acc[u] = fmaf(wi, x[(v0 + u) * xstride + i], acc[u]);
      }
#pragma unroll
      for (int u = 0; u < VC; u++) {
        const int v = v0 + u;
        if (v < nvec) {
          float r = acc[u] + (bias ? bias[c] : 0.f);
          if (add) r += add[(v / add_div) * add_stride + c];
          if (act == 1) r = nm_lrelu(r);
          else if (act == 2) r = tanhf(r);
          out[v * ostride + c] = r;
        }
      }
    }
  }
}

// 6-D -> rotation (geo_utils.py:56-78): x = a/|a|, z = (x × b)/|x × b|, y = z × x; columns (x, y, z)
__device__ __forceinline__ void rot6d(const float* p, float* R /* row-major 3x3 */) {
  const float na = sqrtf(p[0] * p[0] + p[1] * p[1] + p[2] * p[2]) + 1e-10f;
  const float x0 = p[0] / na, x1 = p[1] / na, x2 = p[2] / na;
  float z0 = x1 * p[5] - x2 * p[4], z1 = x2 * p[3] - x0 * p[5], z2 = x0 * p[4] - x1 * p[3];
  const float nz = sqrtf(z0 * z0 + z1 * z1 + z2 * z2) + 1e-10f;
  z0 /= nz; z1 /= nz; z2 /= nz;
  const float y0 = z1 * x2 - z2 * x1, y1 = z2 * x0 - z0 * x2, y2 = z0 * x1 - z1 * x0;
  R[0] = x0; R[1] = y0; R[2] = z0;
  R[3] = x1; R[4] = y1; R[5] = z1;
  R[6] = x2; R[7] = y2; R[8] = z2;
}

// Forward kinematics for one (batch element, sample): hsvrnn_bvh.py:264-281.
// root_raw: 3 + K tanh outputs; rot: K*6; offset: K*3; Rg scratch K*9; flat out K*4.
__device__ void fk_pose(const float* root_raw, const float* rot, const float* offset, const int* order,
                        const int* parents, int K, float* Rg, float* flat) {
  const int root = order[0];
  rot6d(rot + root * 6, Rg + root * 9);
  flat[root * 4 + 0] = root_raw[0];
  flat[root * 4 + 1] = root_raw[1];
  flat[root * 4 + 2] = root_raw[2];
  for (int j = 1; j < K; j++) {
    const int i = order[j], pa = parents[i];
    float Rl[9];
    rot6d(rot + i * 6, Rl);
    const float* Rp = Rg + pa * 9;
    float* Ri = Rg + i * 9;
#pragma unroll
    for (int r = 0; r < 3; r++)
#pragma unroll
      for (int c = 0; c < 3; c++) Ri[r * 3 + c] = Rp[r * 3] * Rl[c] + Rp[r * 3 + 1] * Rl[3 + c] + Rp[r * 3 + 2] * Rl[6 + c];
    const float* o = offset + i * 3;
#pragma unroll
    for (int r = 0; r < 3; r++) flat[i * 4 + r] = Ri[r * 3] * o[0] + Ri[r * 3 + 1] * o[1] + Ri[r * 3 + 2] * o[2] + flat[pa * 4 + r];
  }
  for (int i = 0; i < K; i++) flat[i * 4 + 3] = (root_raw[3 + i] + 1.0f) * 0.5f;
}

struct StepArgs {
  nm_hsvrnn_weights w;
  const float* h_in;      // (B, 512)
  const float* kp;        // (B, 4K) detected keypoints (posterior mode) or null
  const float* eps;       // (S, B, 128)
  const float* offset;    // (B, K, 3)
  const int* order;       // (K)
  const int* parents;     // (K)
  float* h_out;           // (B, 512)
  float* kp_out;          // (B, 4K)
  float* z_out;           // (B, 128) or null
  float* R_out;           // (B, K, 9) or null
  float* post_out;        // (B, 256) posterior mean | std, or null
  float* prior_out;       // (B, 256) prior mean | std, or null
  int* pick_out;          // (B) index of the sample fed to the GRU, or null
  int B, K, S, posterior;
};

template <int NB, int KC>
__global__ void __launch_bounds__(kThreads)
hsvrnn_step_kernel(const StepArgs a) {
  using D = KpDims<KC>;
  extern __shared__ float sm[];
  const int K = a.K, S = a.S, K4 = 4 * a.K;
  const int b0 = blockIdx.x * NB;
  const int nb = min(NB, a.B - b0);
  const int nvs = nb * S;                       // live (element, sample) vectors
  const int NVS = ((NB * S + VC - 1) / VC) * VC;  // padded
  constexpr int NBP = ((NB + VC - 1) / VC) * VC;
  // ---- shared-memory carve-up (floats)
  float* s_in = sm;                         // [NBP][H + D::K4]  h | kp   (posterior MLP input)
  const int IN = H + K4;
  float* s_hid = s_in + NBP * (H + D::K4);     // [NBP][HID]
  float* s_dist = s_hid + NBP * HID;        // [NBP][2Z]  mean | std (posterior, or prior in prior mode)
  float* s_z = s_dist + NBP * 2 * Z;        // [NVS][Z]
  float* s_ah = s_z + NVS * Z;              // [NBP][2 HID]  W0[:, :H] h + b0 for (root | joint) decoders
  float* s_h2 = s_ah + NBP * 2 * HID;       // [NVS][2 HID]
  float* s_dec = s_h2 + NVS * 2 * HID;      // [NVS][D::DW]  root(3+K) at 0, joint(6K) at JO
  float* s_flat = s_dec + NVS * D::DW;      // [NVS][D::K4]
  float* s_rg = s_flat + NVS * D::K4;          // [NVS][K*9]
  float* s_x = s_rg + NVS * KC * 9;     // [NBP][D::XW]  GRU input
  float* s_off = s_x + NBP * D::XW;           // [NB][K*3]
  int* s_tree = reinterpret_cast<int*>(s_off + NB * KC * 3);  // order[K] | parents[K] | best[NB]
  int* s_best = s_tree + 2 * KC;

  // ---- stage 0: load, zero the padding rows
  for (int i = threadIdx.x; i < NBP * (H + D::K4); i += kThreads) {
    const int v = i / (H + D::K4), j = i % (H + D::K4);
    float val = 0.f;
    if (v < nb) {
      if (j < H) val = a.h_in[(long long)(b0 + v) * H + j];
      else if (a.posterior && j - H < K4) val = a.kp[(long long)(b0 + v) * K4 + (j - H)];
    }
    s_in[i] = val;
  }
  for (int i = threadIdx.x; i < NVS * Z; i += kThreads) s_z[i] = 0.f;
  for (int i = threadIdx.x; i < NBP * HID; i += kThreads) s_hid[i] = 0.f;
  for (int i = threadIdx.x; i < NBP * D::XW; i += kThreads) s_x[i] = 0.f;
  for (int i = threadIdx.x; i < nb * K * 3; i += kThreads) s_off[(i / (K * 3)) * KC * 3 + i % (K * 3)] = a.offset[(long long)b0 * K * 3 + i];
  for (int i = threadIdx.x; i < K; i += kThreads) {
    s_tree[i] = a.order[i];
    s_tree[KC + i] = a.parents[i];
  }
  __syncthreads();

  // ---- prior MLP (hsvrnn_bvh.py:92-96 / 210-214): 512 -> 128 -> 256
  if (a.prior_out || !a.posterior) {
    cols_matvec(a.w.prior0_wt, HID, 0, HID, H, s_in, H + D::K4, nb, a.w.prior0_b, nullptr, 0, 1, 1, s_hid, HID);
    __syncthreads();
    cols_matvec(a.w.prior2_wt, 2 * Z, 0, 2 * Z, HID, s_hid, HID, nb, a.w.prior2_b, nullptr, 0, 1, 0, s_dist, 2 * Z);
    __syncthreads();
    for (int i = threadIdx.x; i < nb * Z; i += kThreads) {
      const int v = i / Z, j = i % Z;
      const float sd = softplus_d(s_dist[v * 2 * Z + Z + j]) + 1e-4f;
      s_dist[v * 2 * Z + Z + j] = sd;
    }
    __syncthreads();
    if (a.prior_out)
      for (int i = threadIdx.x; i < nb * 2 * Z; i += kThreads) a.prior_out[(long long)b0 * 2 * Z + i] = s_dist[i];
    __syncthreads();
  }
  // ---- posterior MLP (hsvrnn_bvh.py:99-104): (512 + 4K) -> 128 -> 256
  if (a.posterior) {
    cols_matvec(a.w.post0_wt, HID, 0, HID, IN, s_in, H + D::K4, nb, a.w.post0_b, nullptr, 0, 1, 1, s_hid, HID);
    __syncthreads();
    cols_matvec(a.w.post2_wt, 2 * Z, 0, 2 * Z, HID, s_hid, HID, nb, a.w.post2_b, nullptr, 0, 1, 0, s_dist, 2 * Z);
    __syncthreads();
    for (int i = threadIdx.x; i < nb * Z; i += kThreads) {
      const int v = i / Z, j = i % Z;
      s_dist[v * 2 * Z + Z + j] = softplus_d(s_dist[v * 2 * Z + Z + j]) + 1e-4f;
    }
    __syncthreads();
    if (a.post_out)
      for (int i = threadIdx.x; i < nb * 2 * Z; i += kThreads) a.post_out[(long long)b0 * 2 * Z + i] = s_dist[i];
  }
  // ---- reparameterised samples z = mean + std * eps (Normal.rsample, :107 / :216); vector index v*S + s
  for (int i = threadIdx.x; i < nvs * Z; i += kThreads) {
    const int vs = i / Z, j = i % Z, v = vs / S, s = vs % S;
    const float e = a.eps[((long long)s * a.B + b0 + v) * Z + j];
    s_z[vs * Z + j] = s_dist[v * 2 * Z + j] + s_dist[v * 2 * Z + Z + j] * e;
  }
  // ---- decoders, first layer split: W0 [h; z] = W0[:, :H] h (shared by the S samples) + W0[:, H:] z
  cols_matvec(a.w.root0_wt, HID, 0, HID, H, s_in, H + D::K4, nb, a.w.root0_b, nullptr, 0, 1, 0, s_ah, 2 * HID);
  cols_matvec(a.w.joint0_wt, HID, 0, HID, H, s_in, H + D::K4, nb, a.w.joint0_b, nullptr, 0, 1, 0, s_ah + HID, 2 * HID);
  __syncthreads();
  cols_matvec(a.w.root0_wt + (long long)H * HID, HID, 0, HID, Z, s_z, Z, nvs, nullptr, s_ah, 2 * HID, S, 1, s_h2, 2 * HID);
  cols_matvec(a.w.joint0_wt + (long long)H * HID, HID, 0, HID, Z, s_z, Z, nvs, nullptr, s_ah + HID, 2 * HID, S, 1,
              s_h2 + HID, 2 * HID);
  __syncthreads();
  // second layers: root/intensity (3+K, tanh), joint (6K)
  cols_matvec(a.w.root2_wt, 3 + K, 0, 3 + K, HID, s_h2, 2 * HID, nvs, a.w.root2_b, nullptr, 0, 1, 2, s_dec, D::DW);
  cols_matvec(a.w.joint2_wt, 6 * K, 0, 6 * K, HID, s_h2 + HID, 2 * HID, nvs, a.w.joint2_b, nullptr, 0, 1, 0, s_dec + D::JO, D::DW);
  __syncthreads();
  // ---- rotations + forward kinematics, one thread per (element, sample)
  if ((int)threadIdx.x < nvs) {
    const int vs = threadIdx.x, v = vs / S;
    fk_pose(s_dec + vs * D::DW, s_dec + vs * D::DW + D::JO, s_off + v * KC * 3, s_tree, s_tree + KC, K,
            s_rg + vs * KC * 9, s_flat + vs * D::K4);
  }
  __syncthreads();
  // ---- nearest sample to the detected keypoints (:116-123); prior mode: the single sample
  if ((int)threadIdx.x < nb) {
    const int v = threadIdx.x;
    int best = 0;
    if (a.posterior) {
      float bd = INFINITY;
      for (int s = 0; s < S; s++) {
        float d = 0.f;
        for (int j = 0; j < K4; j++) {
          const float t = s_in[v * (H + D::K4) + H + j] - s_flat[(v * S + s) * D::K4 + j];
          d += t * t;
        }
        if (d < bd) { bd = d; best = s; }
      }
    }
    s_best[v] = best;
    if (a.pick_out) a.pick_out[b0 + v] = best;
  }
  __syncthreads();
  for (int i = threadIdx.x; i < nb * (K4 + Z); i += kThreads) {
    const int v = i / (K4 + Z), j = i % (K4 + Z);
    const int vs = v * S + s_best[v];
    const float val = j < K4 ? s_flat[vs * D::K4 + j] : s_z[vs * Z + (j - K4)];
    s_x[v * D::XW + j] = val;
    if (j < K4) a.kp_out[(long long)(b0 + v) * K4 + j] = val;
    else if (a.z_out) a.z_out[(long long)(b0 + v) * Z + (j - K4)] = val;
  }
  if (a.R_out)
    for (int i = threadIdx.x; i < nb * K * 9; i += kThreads) {
      const int v = i / (K * 9), j = i % (K * 9);
      a.R_out[(long long)(b0 + v) * K * 9 + j] = s_rg[(v * S + s_best[v]) * KC * 9 + j];
    }
  __syncthreads();
  // ---- GRU cell (gate order r, z, n); thread per hidden unit
  const int XI = K4 + Z;
  for (int j = threadIdx.x; j < H; j += kThreads) {
    float gi[3][NB], gh[3][NB];
#pragma unroll
    for (int g = 0; g < 3; g++)
#pragma unroll
      for (int v = 0; v < NB; v++) { gi[g][v] = 0.f; gh[g][v] = 0.f; }
    for (int i = 0; i < XI; i++) {
      const float w0 = __ldg(a.w.gru_ih_wt + (long long)i * 3 * H + j);
      const float w1 = __ldg(a.w.gru_ih_wt + (long long)i * 3 * H + H + j);
      const float w2 = __ldg(a.w.gru_ih_wt + (long long)i * 3 * H + 2 * H + j);
#pragma unroll
      for (int v = 0; v < NB; v++) {
        const float xv = s_x[v * D::XW + i];
        gi[0][v] = fmaf(w0, xv, gi[0][v]);
        gi[1][v] = fmaf(w1, xv, gi[1][v]);
        gi[2][v] = fmaf(w2, xv, gi[2][v]);
      }
    }
    for (int i = 0; i < H; i++) {
      const float w0 = __ldg(a.w.gru_hh_wt + (long long)i * 3 * H + j);
      const float w1 = __ldg(a.w.gru_hh_wt + (long long)i * 3 * H + H + j);
      const float w2 = __ldg(a.w.gru_hh_wt + (long long)i * 3 * H + 2 * H + j);
#pragma unroll
      for (int v = 0; v < NB; v++) {
        const float hv = s_in[v * (H + D::K4) + i];
        gh[0][v] = fmaf(w0, hv, gh[0][v]);
        gh[1][v] = fmaf(w1, hv, gh[1][v]);
        gh[2][v] = fmaf(w2, hv, gh[2][v]);
      }
    }
#pragma unroll
    for (int v = 0; v < NB; v++) {
      if (v < nb) {
        const float r = sigmoid_d(gi[0][v] + a.w.gru_ih_b[j] + gh[0][v] + a.w.gru_hh_b[j]);
        const float zg = sigmoid_d(gi[1][v] + a.w.gru_ih_b[H + j] + gh[1][v] + a.w.gru_hh_b[H + j]);
        const float ng = tanhf(gi[2][v] + a.w.gru_ih_b[2 * H + j] + r * (gh[2][v] + a.w.gru_hh_b[2 * H + j]));
        a.h_out[(long long)(b0 + v) * H + j] = (1.0f - zg) * ng + zg * s_in[v * (H + D::K4) + j];
      }
    }
  }
}

template <int NB, int KC>
size_t step_smem_bytes(int S) {
  using D = KpDims<KC>;
  const int NVS = ((NB * S + VC - 1) / VC) * VC;
  const int NBP = ((NB + VC - 1) / VC) * VC;
  size_t f = (size_t)NBP * (H + D::K4) + NBP * HID + NBP * 2 * Z + (size_t)NVS * Z + NBP * 2 * HID + (size_t)NVS * 2 * HID +
             (size_t)NVS * D::DW + (size_t)NVS * D::K4 + (size_t)NVS * KC * 9 + NBP * D::XW + NB * KC * 3;
  return f * sizeof(float) + (2 * KC + NB + 8) * sizeof(int);
}

// ------------------------------------------------------------------ small batches: one thread-block cluster per element
// With one CTA per batch element a single SM walks the 6.1 MB of weights alone (296 us per step at B <= 148: 21 GB/s).
// Here a cluster of kCl = 8 CTAs shares one element: the output columns of the big mat-vecs (the four first layers that
// read h, the GRU's hidden-state half - 3.4 MB - and its input half) are split over the cluster ranks, every thread owns
// a quad of columns and a slice of the input (16-byte weight loads, 8 in flight per thread), the 512 hidden values and
// the 512 distribution parameters are broadcast into every CTA's shared memory through DSMEM, and two cluster barriers
// order the three phases.  The small tail (z-part of the decoders, second layers from a shared-memory copy that is
// prefetched with cp.async during the first phases, rotations, forward kinematics, nearest-sample pick) runs redundantly
// in every CTA; each rank then finishes its 64 hidden units of the GRU.
constexpr int kCl = 8;
constexpr int kGruSlice = H / kCl;             // 64 hidden units per rank

__device__ __forceinline__ uint32_t cl_rank() {
  uint32_t r;
  asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
  return r;
}
__device__ __forceinline__ void cl_sync() {
  asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
// store v at the same shared-memory offset in every CTA of the cluster
__device__ __forceinline__ void cl_bcast(float* local_ptr, float v) {
  const uint32_t la = (uint32_t)__cvta_generic_to_shared(local_ptr);
#pragma unroll
  for (int r = 0; r < kCl; r++) {
    uint32_t ra;
    asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(ra) : "r"(la), "r"(r));
    asm volatile("st.shared::cluster.f32 [%0], %1;" ::"r"(ra), "f"(v) : "memory");
  }
}
__device__ __forceinline__ void cl_cp_async16(void* dst_smem, const void* src) {
  asm volatile("cp.async.cg.shared.global [%0], [%1], 16;" ::"r"((uint32_t)__cvta_generic_to_shared(dst_smem)), "l"(src) : "memory");
}

// acc[v][0..3] += sum_{i in [i0, i1)} WT[i][col .. col+3] * x[v][i]; 16-byte weight loads, U rows in flight per thread
// (the mat-vecs are L2-latency bound: 16 rows = 64 KB in flight per CTA for the single-vector phases)
template <int NV>
__device__ __forceinline__ void quad_dot(const float* __restrict__ WT, int ldw, int col, int i0, int i1, const float* x,
                                         int xstride, float (&acc)[NV][4]) {
  constexpr int U = NV == 1 ? 16 : 8;
  const float* w = WT + (long long)i0 * ldw + col;
  int i = i0;
  for (; i + U <= i1; i += U) {
    float4 q[U];
#pragma unroll
    for (int u = 0; u < U; u++) q[u] = __ldg(reinterpret_cast<const float4*>(w + (long long)u * ldw));
    w += (long long)U * ldw;
#pragma unroll
    for (int u = 0; u < U; u++)
#pragma unroll
      for (int v = 0; v < NV; v++) {
        const float xv = x[v * xstride + i + u];
        acc[v][0] = fmaf(q[u].x, xv, acc[v][0]);
        acc[v][1] = fmaf(q[u].y, xv, acc[v][1]);
        acc[v][2] = fmaf(q[u].z, xv, acc[v][2]);
        acc[v][3] = fmaf(q[u].w, xv, acc[v][3]);
      }
  }
  for (; i < i1; i++) {
    const float4 q = __ldg(reinterpret_cast<const float4*>(w));
    w += ldw;
#pragma unroll
    for (int v = 0; v < NV; v++) {
      const float xv = x[v * xstride + i];
      acc[v][0] = fmaf(q.x, xv, acc[v][0]);
      acc[v][1] = fmaf(q.y, xv, acc[v][1]);
      acc[v][2] = fmaf(q.z, xv, acc[v][2]);
      acc[v][3] = fmaf(q.w, xv, acc[v][3]);
    }
  }
}

// The cluster kernel serves K <= kTunedK only: its layout keeps both decoders' second layers resident, which at
// kMaxK (231 KB for them alone) exceeds the 227 KB a CTA can have.  Larger K runs the per-element kernel.
constexpr int kClK = kTunedK;
using ClD = KpDims<kClK>;
struct ClSmem {   // offsets in floats
  int in, hid, ah, gh, dist, part, z, h2, dec, flat, rl, rg, x, off, w2, tree, total;
};
__host__ __device__ inline ClSmem cl_layout(int SV) {
  ClSmem m;
  int o = 0;
  m.in = o;   o += H + ClD::K4;
  m.hid = o;  o += 2 * HID;                 // prior0 | post0 outputs
  m.ah = o;   o += 2 * HID;                 // root0 | joint0 applied to h (+ bias)
  m.gh = o;   o += 3 * kGruSlice;           // this rank's W_hh h (3 gates x 64 units)
  m.dist = o; o += 4 * Z;                   // prior mean | std, posterior mean | std
  m.part = o; o += 4 * SV * 256 > 1024 ? 4 * SV * 256 : 1024;
  m.z = o;    o += SV * Z;
  m.h2 = o;   o += SV * 2 * HID;
  m.dec = o;  o += SV * ClD::DW;
  m.flat = o; o += SV * ClD::K4;
  m.rl = o;   o += SV * kClK * 9;
  m.rg = o;   o += SV * kClK * 9;
  m.x = o;    o += ClD::XW;
  m.off = o;  o += kClK * 3;
  m.w2 = o;   o += HID * (3 + kClK) + HID * 6 * kClK;
  m.tree = o; o += 2 * kClK + 8;
  m.total = o;
  return m;
}

template <int SV>
__global__ void __cluster_dims__(kCl, 1, 1) __launch_bounds__(kThreads, 1)
hsvrnn_step_cluster_kernel(const StepArgs a) {
  extern __shared__ __align__(16) float sm[];
  const ClSmem L = cl_layout(SV);
  float* s_in = sm + L.in;
  float* s_hid = sm + L.hid;
  float* s_ah = sm + L.ah;
  float* s_gh = sm + L.gh;
  float* s_dist = sm + L.dist;
  float* s_part = sm + L.part;
  float* s_z = sm + L.z;
  float* s_h2 = sm + L.h2;
  float* s_dec = sm + L.dec;
  float* s_flat = sm + L.flat;
  float* s_rl = sm + L.rl;
  float* s_rg = sm + L.rg;
  float* s_x = sm + L.x;
  float* s_off = sm + L.off;
  float* s_w2r = sm + L.w2;                              // root2^T [HID][3 + K]
  int* s_tree = reinterpret_cast<int*>(sm + L.tree);
  const int K = a.K, S = a.S, K4 = 4 * a.K, R2 = 3 + a.K, J2 = 6 * a.K;
  float* s_w2j = s_w2r + HID * R2;                       // joint2^T [HID][6 K]
  const int b = blockIdx.x / kCl;
  const int rank = (int)cl_rank();
  const int tid = threadIdx.x;
  const bool need_prior = a.prior_out != nullptr || !a.posterior;
  const int IN = H + K4;

  // ---- stage 0: inputs; the second-layer weights start streaming into shared memory (16-byte aligned segments)
  {
    const int nr = HID * R2, nj = HID * J2;
    const int head = (int)(((16 - ((uintptr_t)a.w.root2_wt & 15)) & 15) >> 2);   // floats until 16-byte alignment (0 in practice)
    for (int i = tid * 4; i + 4 <= nr - head; i += kThreads * 4) cl_cp_async16(s_w2r + head + i, a.w.root2_wt + head + i);
    for (int i = tid; i < head; i += kThreads) s_w2r[i] = a.w.root2_wt[i];
    for (int i = head + ((nr - head) & ~3) + tid; i < nr; i += kThreads) s_w2r[i] = a.w.root2_wt[i];
    // joint2: HID * 6K floats; s_w2j may start off 16-byte alignment when HID * R2 is odd -> plain loads
    if ((((uintptr_t)s_w2j | (uintptr_t)a.w.joint2_wt) & 15) == 0) {
      for (int i = tid * 4; i + 4 <= nj; i += kThreads * 4) cl_cp_async16(s_w2j + i, a.w.joint2_wt + i);
      for (int i = (nj & ~3) + tid; i < nj; i += kThreads) s_w2j[i] = a.w.joint2_wt[i];
    } else {
      for (int i = tid; i < nj; i += kThreads) s_w2j[i] = __ldg(a.w.joint2_wt + i);
    }
    asm volatile("cp.async.commit_group;" ::: "memory");
  }
  for (int j = tid; j < H + ClD::K4; j += kThreads) {
    float val = 0.f;
    if (j < H) val = a.h_in[(long long)b * H + j];
    else if (a.posterior && j - H < K4) val = a.kp[(long long)b * K4 + (j - H)];
    s_in[j] = val;
  }
  for (int i = tid; i < K * 3; i += kThreads) s_off[i] = a.offset[(long long)b * K * 3 + i];
  for (int i = tid; i < K; i += kThreads) {
    s_tree[i] = a.order[i];
    s_tree[kClK + i] = a.parents[i];
  }
  __syncthreads();

  // ---- phase A: everything that reads h (and kp).  256 columns per rank = 64 quads x 4 input slices.
  //   quads 0-3 prior0, 4-7 post0, 8-11 root0[:H], 12-15 joint0[:H] (16 columns each), 16-63 GRU hidden half (3 x 64)
  {
    const int qd = tid & 63, ks = tid >> 6;
    float acc[1][4] = {{0.f, 0.f, 0.f, 0.f}};
    if (qd < 16) {
      const int job = qd >> 2, col = rank * 16 + (qd & 3) * 4;
      const float* WT = job == 0 ? a.w.prior0_wt : (job == 1 ? a.w.post0_wt : (job == 2 ? a.w.root0_wt : a.w.joint0_wt));
      const int I = job == 1 ? IN : H;
      const bool live = job == 0 ? need_prior : (job == 1 ? a.posterior != 0 : true);
      if (live) {
        const int per = (I + 3) / 4;
        quad_dot<1>(WT, HID, col, min(I, ks * per), min(I, (ks + 1) * per), s_in, 0, acc);
      }
    } else {
      const int g = (qd - 16) >> 4, col = g * H + rank * kGruSlice + ((qd - 16) & 15) * 4;
      quad_dot<1>(a.w.gru_hh_wt, 3 * H, col, ks * (H / 4), (ks + 1) * (H / 4), s_in, 0, acc);
    }
#pragma unroll
    for (int e = 0; e < 4; e++) s_part[ks * 256 + qd * 4 + e] = acc[0][e];
  }
  __syncthreads();
  {
    const int c = tid;                                      // local column 0..255
    const float v = s_part[c] + s_part[256 + c] + s_part[512 + c] + s_part[768 + c];
    if (c < 64) {
      const int job = c >> 4, col = rank * 16 + (c & 15);
      if (job == 0) { if (need_prior) cl_bcast(s_hid + col, nm_lrelu(v + a.w.prior0_b[col])); }
      else if (job == 1) { if (a.posterior) cl_bcast(s_hid + HID + col, nm_lrelu(v + a.w.post0_b[col])); }
      else if (job == 2) cl_bcast(s_ah + col, v + a.w.root0_b[col]);
      else cl_bcast(s_ah + HID + col, v + a.w.joint0_b[col]);
    } else {
      s_gh[c - 64] = v;                                    // [gate][unit]
    }
  }
  cl_sync();

  // ---- phase B: second layers of the prior / posterior MLPs: 512 columns, 64 per rank = 16 quads x 16 input slices
  {
    const int qd = tid & 15, ks = tid >> 4;
    const int job = qd >> 3, col = rank * 32 + (qd & 7) * 4;   // job 0: prior2, 1: post2; 32 columns of each per rank
    float acc[1][4] = {{0.f, 0.f, 0.f, 0.f}};
    const bool live = job == 0 ? need_prior : a.posterior != 0;
    if (live) quad_dot<1>(job == 0 ? a.w.prior2_wt : a.w.post2_wt, 2 * Z, col, ks * 8, ks * 8 + 8, s_hid + job * HID, 0, acc);
#pragma unroll
    for (int e = 0; e < 4; e++) s_part[ks * 64 + qd * 4 + e] = acc[0][e];
  }
  __syncthreads();
  if (tid < 64) {
    float v = 0.f;
    for (int ks = 0; ks < 16; ks++) v += s_part[ks * 64 + tid];
    const int job = tid >> 5, col = rank * 32 + (tid & 31);
    const bool live = job == 0 ? need_prior : a.posterior != 0;
    if (live) {
      v += job == 0 ? a.w.prior2_b[col] : a.w.post2_b[col];
      if (col >= Z) v = softplus_d(v) + 1e-4f;
      cl_bcast(s_dist + job * 2 * Z + col, v);
      float* gout = job == 0 ? a.prior_out : a.post_out;
      if (gout) gout[(long long)b * 2 * Z + col] = v;
    }
  }
  cl_sync();

  // ---- from here on every rank works on its own copy.  z = mean + std * eps
  const float* dsel = s_dist + (a.posterior ? 2 * Z : 0);
  for (int i = tid; i < SV * Z; i += kThreads) {
    const int sidx = i / Z, j = i % Z;
    s_z[i] = sidx < S ? dsel[j] + dsel[Z + j] * a.eps[((long long)sidx * a.B + b) * Z + j] : 0.f;
  }
  __syncthreads();
  // decoders, first layer, z part: 256 columns (root | joint) = 64 quads x 4 input slices, all samples at once
  {
    const int qd = tid & 63, ks = tid >> 6;
    float acc[SV][4];
#pragma unroll
    for (int v = 0; v < SV; v++) acc[v][0] = acc[v][1] = acc[v][2] = acc[v][3] = 0.f;
    const bool joint = qd >= 32;
    const int col = (qd & 31) * 4;
    quad_dot<SV>((joint ? a.w.joint0_wt : a.w.root0_wt) + (long long)H * HID, HID, col, ks * (Z / 4), (ks + 1) * (Z / 4), s_z, Z, acc);
#pragma unroll
    for (int v = 0; v < SV; v++)
#pragma unroll
      for (int e = 0; e < 4; e++) s_part[(ks * SV + v) * 256 + qd * 4 + e] = acc[v][e];
  }
  __syncthreads();
  for (int i = tid; i < S * 256; i += kThreads) {
    const int v = i >> 8, c = i & 255;
    const float t = s_part[(0 * SV + v) * 256 + c] + s_part[(1 * SV + v) * 256 + c] + s_part[(2 * SV + v) * 256 + c] +
                    s_part[(3 * SV + v) * 256 + c];
    s_h2[v * 2 * HID + c] = nm_lrelu(t + s_ah[c]);
  }
  asm volatile("cp.async.wait_all;" ::: "memory");
  __syncthreads();
  // second layers from shared memory: root / intensity (3 + K, tanh) at s_dec[0..], joint 6-D rotations at s_dec[JO..]
  for (int i = tid; i < S * (R2 + J2); i += kThreads) {
    const int v = i / (R2 + J2), c = i % (R2 + J2);
    float t;
    if (c < R2) {
      t = a.w.root2_b[c];
      const float* hv = s_h2 + v * 2 * HID;
      for (int k = 0; k < HID; k++) t = fmaf(s_w2r[k * R2 + c], hv[k], t);
      s_dec[v * ClD::DW + c] = tanhf(t);
    } else {
      const int cj = c - R2;
      t = a.w.joint2_b[cj];
      const float* hv = s_h2 + v * 2 * HID + HID;
      for (int k = 0; k < HID; k++) t = fmaf(s_w2j[k * J2 + cj], hv[k], t);
      s_dec[v * ClD::DW + ClD::JO + cj] = t;
    }
  }
  __syncthreads();
  // rotations in parallel over (sample, joint), then the kinematic chain per sample
  for (int i = tid; i < S * K; i += kThreads) rot6d(s_dec + (i / K) * ClD::DW + ClD::JO + (i % K) * 6, s_rl + (i / K) * kClK * 9 + (i % K) * 9);
  __syncthreads();
  if (tid < S) {
    const int v = tid;
    const float* raw = s_dec + v * ClD::DW;
    float* Rg = s_rg + v * kClK * 9;
    float* flat = s_flat + v * ClD::K4;
    const float* Rl0 = s_rl + v * kClK * 9;
    const int root = s_tree[0];
    for (int e = 0; e < 9; e++) Rg[root * 9 + e] = Rl0[root * 9 + e];
    flat[root * 4] = raw[0]; flat[root * 4 + 1] = raw[1]; flat[root * 4 + 2] = raw[2];
    for (int j = 1; j < K; j++) {
      const int i = s_tree[j], pa = s_tree[kClK + i];
      const float* Rl = Rl0 + i * 9;
      const float* Rp = Rg + pa * 9;
      float* Ri = Rg + i * 9;
#pragma unroll
      for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = 0; c < 3; c++) Ri[r * 3 + c] = Rp[r * 3] * Rl[c] + Rp[r * 3 + 1] * Rl[3 + c] + Rp[r * 3 + 2] * Rl[6 + c];
      const float* o = s_off + i * 3;
#pragma unroll
      for (int r = 0; r < 3; r++) flat[i * 4 + r] = Ri[r * 3] * o[0] + Ri[r * 3 + 1] * o[1] + Ri[r * 3 + 2] * o[2] + flat[pa * 4 + r];
    }
    for (int i = 0; i < K; i++) flat[i * 4 + 3] = (raw[3 + i] + 1.0f) * 0.5f;
  }
  __syncthreads();
  if (tid == 0) {
    int best = 0;
    if (a.posterior) {
      float bd = INFINITY;
      for (int sidx = 0; sidx < S; sidx++) {
        float d = 0.f;
        for (int j = 0; j < K4; j++) {
          const float t = s_in[H + j] - s_flat[sidx * ClD::K4 + j];
          d += t * t;
        }
        if (d < bd) { bd = d; best = sidx; }
      }
    }
    s_tree[2 * kClK] = best;
    if (rank == 0 && a.pick_out) a.pick_out[b] = best;
  }
  __syncthreads();
  const int best = s_tree[2 * kClK];
  for (int j = tid; j < ClD::XW; j += kThreads) {
    float val = 0.f;
    if (j < K4) val = s_flat[best * ClD::K4 + j];
    else if (j < K4 + Z) val = s_z[best * Z + (j - K4)];
    s_x[j] = val;
    if (rank == 0) {
      if (j < K4) a.kp_out[(long long)b * K4 + j] = val;
      else if (j < K4 + Z && a.z_out) a.z_out[(long long)b * Z + (j - K4)] = val;
    }
  }
  if (rank == 0 && a.R_out)
    for (int j = tid; j < K * 9; j += kThreads) a.R_out[(long long)b * K * 9 + j] = s_rg[best * kClK * 9 + j];
  __syncthreads();
  // ---- GRU: this rank's 64 hidden units; input half W_ih x: 192 columns = 48 quads x 4 input slices
  {
    const int XI = K4 + Z;
    const int qd = tid & 63, ks = tid >> 6;
    float acc[1][4] = {{0.f, 0.f, 0.f, 0.f}};
    if (qd < 48) {
      const int g = qd >> 4, col = g * H + rank * kGruSlice + (qd & 15) * 4;
      const int per = (XI + 3) / 4;
      quad_dot<1>(a.w.gru_ih_wt, 3 * H, col, min(XI, ks * per), min(XI, (ks + 1) * per), s_x, 0, acc);
    }
#pragma unroll
    for (int e = 0; e < 4; e++) s_part[ks * 256 + qd * 4 + e] = acc[0][e];
  }
  __syncthreads();
  if (tid < kGruSlice) {
    const int j = rank * kGruSlice + tid;
    float gi[3];
#pragma unroll
    for (int g = 0; g < 3; g++) {
      const int c = g * kGruSlice + tid;
      gi[g] = s_part[c] + s_part[256 + c] + s_part[512 + c] + s_part[768 + c];
    }
    const float r = sigmoid_d(gi[0] + a.w.gru_ih_b[j] + s_gh[tid] + a.w.gru_hh_b[j]);
    const float zg = sigmoid_d(gi[1] + a.w.gru_ih_b[H + j] + s_gh[kGruSlice + tid] + a.w.gru_hh_b[H + j]);
    const float ng = tanhf(gi[2] + a.w.gru_ih_b[2 * H + j] + r * (s_gh[2 * kGruSlice + tid] + a.w.gru_hh_b[2 * H + j]));
    a.h_out[(long long)b * H + j] = (1.0f - zg) * ng + zg * s_in[j];
  }
}

// Pose decoding on its own (extract_kypt_from_latent_and_state, hsvrnn_bvh.py:255-286) for callers that
// drive the sub-modules by hand (vis_generation.py:108-113).
template <int KC>
__global__ void __launch_bounds__(kThreads)
decode_pose_kernel(nm_hsvrnn_weights w, const float* __restrict__ dec_in /* (B, H+Z) */,
                   const float* __restrict__ offset, const int* __restrict__ order, const int* __restrict__ parents,
                   int B, int K, float* __restrict__ flat_out, float* __restrict__ R_out) {
  __shared__ float s_in[VC * (H + Z)];
  __shared__ float s_hid[VC * 2 * HID];
  __shared__ float s_dec[KpDims<KC>::DW];
  __shared__ float s_rg[KC * 9];
  __shared__ float s_flat[KpDims<KC>::K4];
  __shared__ int s_tree[2 * KC];
  const int b = blockIdx.x;
  for (int i = threadIdx.x; i < VC * (H + Z); i += kThreads) s_in[i] = i < H + Z ? dec_in[(long long)b * (H + Z) + i] : 0.f;
  for (int i = threadIdx.x; i < K; i += kThreads) { s_tree[i] = order[i]; s_tree[KC + i] = parents[i]; }
  __syncthreads();
  cols_matvec(w.root0_wt, HID, 0, HID, H + Z, s_in, H + Z, 1, w.root0_b, nullptr, 0, 1, 1, s_hid, 2 * HID);
  cols_matvec(w.joint0_wt, HID, 0, HID, H + Z, s_in, H + Z, 1, w.joint0_b, nullptr, 0, 1, 1, s_hid + HID, 2 * HID);
  __syncthreads();
  cols_matvec(w.root2_wt, 3 + K, 0, 3 + K, HID, s_hid, 2 * HID, 1, w.root2_b, nullptr, 0, 1, 2, s_dec, KpDims<KC>::DW);
  cols_matvec(w.joint2_wt, 6 * K, 0, 6 * K, HID, s_hid + HID, 2 * HID, 1, w.joint2_b, nullptr, 0, 1, 0, s_dec + KpDims<KC>::JO, KpDims<KC>::DW);
  __syncthreads();
  if (threadIdx.x == 0)
    fk_pose(s_dec, s_dec + KpDims<KC>::JO, offset + (long long)b * K * 3, s_tree, s_tree + KC, K, s_rg, s_flat);
  __syncthreads();
  for (int i = threadIdx.x; i < 4 * K; i += kThreads) flat_out[(long long)b * 4 * K + i] = s_flat[i];
  if (R_out)
    for (int i = threadIdx.x; i < 9 * K; i += kThreads) R_out[(long long)b * 9 * K + i] = s_rg[i];
}

// Bone offsets (get_offset, hsvrnn_bvh.py:236-253): lower median over T of |kp_k - kp_parent(k)| times the
// unit offset_param direction.  One thread per (b, k); T <= 64.
__global__ void bone_offset_kernel(const float* __restrict__ kp /* (B,T,K,4) */, const int* __restrict__ parents,
                                   const float* __restrict__ offset_param /* (K,3) */, int B, int T, int K,
                                   float* __restrict__ out /* (B,K,3) */) {
  const int idx = blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= B * K) return;
  const int b = idx / K, k = idx % K, pa = parents[k];
  float d[64];
  for (int t = 0; t < T; t++) {
    const float* p = kp + (((long long)b * T + t) * K + k) * 4;
    const float* q = kp + (((long long)b * T + t) * K + pa) * 4;
    const float dx = p[0] - q[0], dy = p[1] - q[1], dz = p[2] - q[2];
    d[t] = sqrtf(dx * dx + dy * dy + dz * dz);
  }
  // insertion sort, lower median = element (T-1)/2 (torch.median semantics)
  for (int i = 1; i < T; i++) {
    const float v = d[i];
    int j = i - 1;
    while (j >= 0 && d[j] > v) { d[j + 1] = d[j]; j--; }
    d[j + 1] = v;
  }
  const float med = d[(T - 1) / 2];
  const float* o = offset_param + k * 3;
  const float nrm = sqrtf(o[0] * o[0] + o[1] * o[1] + o[2] * o[2]) + 1e-10f;
  for (int c = 0; c < 3; c++) out[(long long)idx * 3 + c] = (o[c] / nrm) * med;
}

}  // namespace

// one CTA per NB elements; NB = 4 only for batches that fill the GPU four times over and when its layout fits
// (at kMaxK it does for S = 1, not for S = 10: 22 KB + 4 S x 6.8 KB)
template <int KC>
static int launch_step(const StepArgs& a, cudaStream_t st) {
  if (a.B >= 4 * nm_num_sms() && step_smem_bytes<4, KC>(a.S) <= 227 * 1024) {
    const size_t smem = step_smem_bytes<4, KC>(a.S);
    NM_CHECK_CUDA(cudaFuncSetAttribute(hsvrnn_step_kernel<4, KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    hsvrnn_step_kernel<4, KC><<<nm_cdiv(a.B, 4), kThreads, smem, st>>>(a);
  } else {
    const size_t smem = step_smem_bytes<1, KC>(a.S);
    NM_CHECK_CUDA(cudaFuncSetAttribute(hsvrnn_step_kernel<1, KC>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    hsvrnn_step_kernel<1, KC><<<a.B, kThreads, smem, st>>>(a);
  }
  NM_CHECK_LAUNCH("hsvrnn_step");
  return NM_OK;
}

static int hsvrnn_step_impl(const nm_hsvrnn_weights* w, const float* h_in, const float* kp, const float* eps,
                            const float* offset, const int* order, const int* parents, int B, int K, int S, int posterior,
                            float* h_out, float* kp_out, float* z_out, float* R_out, float* post_out, float* prior_out,
                            int* pick_out, void* stream) {
  NM_CHECK_ARG(w && h_in && eps && offset && order && parents && h_out && kp_out, "nm_hsvrnn_step: null pointer");
  NM_CHECK_ARG(!posterior || kp, "nm_hsvrnn_step: posterior step needs detected keypoints");
  NM_CHECK_ARG(K > 0 && K <= kMaxK && S >= 1 && S <= 16, "nm_hsvrnn_step: K=%d S=%d unsupported", K, S);
  NM_CHECK_ARG(posterior || S == 1, "nm_hsvrnn_step: prior step draws one sample");
  if (B == 0) return NM_OK;
  StepArgs a;
  a.w = *w; a.h_in = h_in; a.kp = kp; a.eps = eps; a.offset = offset; a.order = order; a.parents = parents;
  a.h_out = h_out; a.kp_out = kp_out; a.z_out = z_out; a.R_out = R_out; a.post_out = post_out; a.prior_out = prior_out;
  a.pick_out = pick_out;
  a.B = B; a.K = K; a.S = S; a.posterior = posterior;
  cudaStream_t st = (cudaStream_t)stream;
  // small and medium batches: a cluster of 8 CTAs per element (weights split over the ranks, DSMEM broadcasts)
  // measured, cluster vs one-CTA-per-element kernel (us per step): B = 1: 30 vs 216, B = 16: 59 vs 228, B = 64: 144 vs 235, B = 256: 510 vs 240
  if (K <= kClK && S <= 10 && B <= 96) {
    const int SV = S == 1 ? 1 : 10;
    const size_t smem = (size_t)cl_layout(SV).total * sizeof(float);
    if (SV == 1) {
      NM_CHECK_CUDA(cudaFuncSetAttribute(hsvrnn_step_cluster_kernel<1>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      hsvrnn_step_cluster_kernel<1><<<B * kCl, kThreads, smem, st>>>(a);
    } else {
      NM_CHECK_CUDA(cudaFuncSetAttribute(hsvrnn_step_cluster_kernel<10>, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
      hsvrnn_step_cluster_kernel<10><<<B * kCl, kThreads, smem, st>>>(a);
    }
    NM_CHECK_LAUNCH("hsvrnn_step(cluster)");
    return NM_OK;
  }
  if (K <= kTunedK) return launch_step<kTunedK>(a, st);
  return launch_step<kMaxK>(a, st);
}

extern "C" int nm_hsvrnn_step(const nm_hsvrnn_weights* w, const float* h_in, const float* kp, const float* eps,
                              const float* offset, const int* order, const int* parents, int B, int K, int S,
                              int posterior, float* h_out, float* kp_out, float* z_out, float* R_out,
                              float* post_out, float* prior_out, void* stream) {
  return hsvrnn_step_impl(w, h_in, kp, eps, offset, order, parents, B, K, S, posterior, h_out, kp_out, z_out, R_out,
                          post_out, prior_out, nullptr, stream);
}

extern "C" int nm_hsvrnn_step_record(const nm_hsvrnn_weights* w, const float* h_in, const float* kp, const float* eps,
                                     const float* offset, const int* order, const int* parents, int B, int K, int S,
                                     int posterior, float* h_out, float* kp_out, float* z_out, float* R_out,
                                     float* post_out, float* prior_out, int* pick_out, void* stream) {
  return hsvrnn_step_impl(w, h_in, kp, eps, offset, order, parents, B, K, S, posterior, h_out, kp_out, z_out, R_out,
                          post_out, prior_out, pick_out, stream);
}

extern "C" int nm_hsvrnn_decode_pose(const nm_hsvrnn_weights* w, const float* dec_in, const float* offset,
                                     const int* order, const int* parents, int B, int K, float* flat_out,
                                     float* R_out, void* stream) {
  NM_CHECK_ARG(w && dec_in && offset && order && parents && flat_out, "nm_hsvrnn_decode_pose: null pointer");
  NM_CHECK_ARG(K > 0 && K <= kMaxK, "nm_hsvrnn_decode_pose: K=%d unsupported", K);
  if (B == 0) return NM_OK;
  if (K <= kTunedK)
    decode_pose_kernel<kTunedK><<<B, kThreads, 0, (cudaStream_t)stream>>>(*w, dec_in, offset, order, parents, B, K, flat_out, R_out);
  else
    decode_pose_kernel<kMaxK><<<B, kThreads, 0, (cudaStream_t)stream>>>(*w, dec_in, offset, order, parents, B, K, flat_out, R_out);
  NM_CHECK_LAUNCH("hsvrnn_decode_pose");
  return NM_OK;
}

extern "C" int nm_hsvrnn_bone_offsets(const float* keypoints, const int* parents, const float* offset_param, int B,
                                      int T, int K, float* out, void* stream) {
  NM_CHECK_ARG(keypoints && parents && offset_param && out, "nm_hsvrnn_bone_offsets: null pointer");
  NM_CHECK_ARG(T >= 1 && T <= 64, "nm_hsvrnn_bone_offsets: T=%d unsupported (1..64)", T);
  if (B == 0) return NM_OK;
  bone_offset_kernel<<<nm_cdiv(B * K, 128), 128, 0, (cudaStream_t)stream>>>(keypoints, parents, offset_param, B, T, K, out);
  NM_CHECK_LAUNCH("hsvrnn_bone_offsets");
  return NM_OK;
}

// ================================================================== stage-2 training: backward of a conditioned step
// The reverse loop launches nm_hsvrnn_step_backward once per step, t = T-1 .. 0.  Only the picked sample of each
// element feeds anything downstream (the other S-1 decodes do not), so the backward decodes one pose per element.  It
// saves nothing from the forward beyond the pick: the hidden layers, the decoder outputs and the GRU gates are recomputed
// from h_t, kp_t and the picked (z, f) that encode() already returns.  The work is a chain of small batched mat-vecs over
// all B elements at once; every one of them splits its output columns over CTAs (32 columns x 16 elements per CTA, the
// reduction split 32 ways inside the CTA), so the 6.1 MB of weights stream through many SMs whatever B is.  Forward
// recomputes read the cached [in][out] copies, the transposed products dx = W^T dy read the fp32 parameters in their own
// [out][in] layout: both are coalesced along the output columns.  Every reduction runs in a fixed order.
namespace {

// Per-(t, b) row record (floats): forward recomputes, then every d pre-activation the weight gradients need.  One layout
// at capacity kMaxK serves every K: nm_hsvrnn_backward_workspace_bytes does not take K.
using RD = KpDims<kMaxK>;
enum : int {
  RW_AP = 0, RW_AQ = RW_AP + HID, RW_AR = RW_AQ + HID, RW_AJ = RW_AR + HID,       // first-layer pre-activations
  RW_GI = RW_AJ + HID, RW_GH = RW_GI + 3 * H,                                      // W_ih x + b_ih, W_hh h + b_hh
  RW_OP = RW_GH + 3 * H, RW_OQ = RW_OP + 2 * Z,                                    // prior / posterior raw outputs
  RW_OR = RW_OQ + 2 * Z, RW_OJ = RW_OR + RD::JO,                                   // tanh(root) (3+K), joint 6-D (6K)
  RW_DGI = RW_OJ + 6 * kMaxK, RW_DGH = RW_DGI + 3 * H,                             // d gates (input / hidden side)
  RW_DXG = RW_DGH + 3 * H, RW_DH1 = RW_DXG + RD::XW,                               // W_ih^T dgi (then df | dz), W_hh^T dgh
  RW_DOR = RW_DH1 + H, RW_DOJ = RW_DOR + RD::JO,                                   // d pre-tanh root, d joint 6-D
  RW_DAR = RW_DOJ + 6 * kMaxK, RW_DAJ = RW_DAR + HID,                              // d first-layer pre-activations
  RW_DXDR = RW_DAJ + HID, RW_DXDJ = RW_DXDR + H + Z,                               // W0^T da of the decoders ([h | z])
  RW_DOP = RW_DXDJ + H + Z, RW_DOQ = RW_DOP + 2 * Z,                               // d prior / posterior raw outputs
  RW_DAP = RW_DOQ + 2 * Z, RW_DAQ = RW_DAP + HID,
  RW_DXP = RW_DAQ + HID, RW_DXQ = RW_DXP + H, RW_DHD = RW_DXQ + H,                 // h parts; GRU's direct dh' * z
  RW = RW_DHD + H
};

constexpr int GR = 16;        // elements per CTA
constexpr int GC = 32;        // output columns per CTA (8 quads)
constexpr int GKS = 32;       // reduction slices per CTA (4 per warp)
constexpr int kMaxGemmJobs = 6;

// Y[b][c] = epi(sum_k X[b][k] M[k][c]),  X[b] = [x0[b][0:k0] | x1[b][0:K-k0]] (LeakyReLU applied on load when xlrelu),
// M[k][c] = m[k * ldm + c]; epi: + bias[c], then tanh, then * LeakyReLU'(gate[b][c]) - each optional.
struct GemmJob {
  const float* x0; const float* x1; const float* m; const float* bias; const float* gate; float* y;
  int ldx0, ldx1, k0, K, ldm, N, ldgate, ldy, xlrelu, tanh_out;
};
struct GemmJobs {
  GemmJob j[kMaxGemmJobs];
  int tile_end[kMaxGemmJobs];
  int n, B;
};

__global__ void __launch_bounds__(kThreads)
rows_gemm_kernel(const __grid_constant__ GemmJobs js) {
  extern __shared__ float sm[];
  int tile = blockIdx.x, ji = 0;
  while (tile >= js.tile_end[ji]) ji++;
  const GemmJob& J = js.j[ji];
  const int c0 = (tile - (ji ? js.tile_end[ji - 1] : 0)) * GC;
  const int b0 = blockIdx.y * GR, nb = min(GR, js.B - b0);
  const int K = J.K;
  float* sx = sm;                 // [GR][K]
  float* sred = sm + GR * K;      // [8 warps][GR][GC]
  for (int i = threadIdx.x; i < GR * K; i += kThreads) {
    const int r = i / K, k = i % K;
    float v = 0.f;
    if (r < nb) {
      v = k < J.k0 ? J.x0[(long long)(b0 + r) * J.ldx0 + k] : J.x1[(long long)(b0 + r) * J.ldx1 + (k - J.k0)];
      if (J.xlrelu) v = nm_lrelu(v);
    }
    sx[i] = v;
  }
  __syncthreads();
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int q = lane & 7, s = lane >> 3, ks = warp * 4 + s;
  const int col = c0 + q * 4;
  const int per = (K + GKS - 1) / GKS;
  const int klo = min(K, ks * per), khi = min(K, klo + per);
  float acc[GR][4];
#pragma unroll
  for (int r = 0; r < GR; r++) acc[r][0] = acc[r][1] = acc[r][2] = acc[r][3] = 0.f;
#pragma unroll 4
  for (int k = klo; k < khi; k++) {      // four rows of weight loads in flight
    const float* mr = J.m + (long long)k * J.ldm;
    float w[4];
#pragma unroll
    for (int e = 0; e < 4; e++) w[e] = col + e < J.N ? __ldg(mr + col + e) : 0.f;
    const float* xk = sx + k;
#pragma unroll
    for (int r = 0; r < GR; r++) {
      const float xv = xk[r * K];
#pragma unroll
      for (int e = 0; e < 4; e++) acc[r][e] = fmaf(w[e], xv, acc[r][e]);
    }
  }
#pragma unroll
  for (int r = 0; r < GR; r++)
#pragma unroll
    for (int e = 0; e < 4; e++) {
      float v = acc[r][e];
      v += __shfl_xor_sync(0xffffffffu, v, 8);
      v += __shfl_xor_sync(0xffffffffu, v, 16);
      acc[r][e] = v;
    }
  if (s == 0)
#pragma unroll
    for (int r = 0; r < GR; r++)
#pragma unroll
      for (int e = 0; e < 4; e++) sred[(warp * GR + r) * GC + q * 4 + e] = acc[r][e];
  __syncthreads();
  for (int i = threadIdx.x; i < GR * GC; i += kThreads) {
    const int r = i / GC, c = i % GC;
    if (r >= nb || c0 + c >= J.N) continue;
    float v = 0.f;
#pragma unroll
    for (int w = 0; w < 8; w++) v += sred[(w * GR + r) * GC + c];
    if (J.bias) v += J.bias[c0 + c];
    if (J.tanh_out) v = tanhf(v);
    if (J.gate) v *= J.gate[(long long)(b0 + r) * J.ldgate + c0 + c] > 0.f ? 1.f : 0.01f;
    J.y[(long long)(b0 + r) * J.ldy + c0 + c] = v;
  }
}

__device__ __forceinline__ float ld_or0(const float* p, long long i) { return p ? p[i] : 0.f; }
// d softplus(x) / dx with torch's threshold (softplus(x) = x above 20)
__device__ __forceinline__ float dsoftplus_d(float x) { return x > 20.f ? 1.f : sigmoid_d(x); }

// GRU cell backward (gate order r, z, n): dgi, dgh and the direct part dh' * z of dh.  One CTA per element.
__global__ void __launch_bounds__(kThreads)
gru_bwd_kernel(const float* __restrict__ h, const float* __restrict__ dh_next, float* __restrict__ rows) {
  const int b = blockIdx.x;
  float* rec = rows + (long long)b * RW;
  for (int j = threadIdx.x; j < H; j += kThreads) {
    const float* gi = rec + RW_GI;
    const float* gh = rec + RW_GH;
    const float r = sigmoid_d(gi[j] + gh[j]);
    const float zg = sigmoid_d(gi[H + j] + gh[H + j]);
    const float ghn = gh[2 * H + j];
    const float n = tanhf(gi[2 * H + j] + r * ghn);
    const float d = dh_next[(long long)b * H + j];
    const float dan = d * (1.f - zg) * (1.f - n * n);
    const float dar = dan * ghn * r * (1.f - r);
    const float daz = d * (h[(long long)b * H + j] - n) * zg * (1.f - zg);
    rec[RW_DGI + j] = dar; rec[RW_DGI + H + j] = daz; rec[RW_DGI + 2 * H + j] = dan;
    rec[RW_DGH + j] = dar; rec[RW_DGH + H + j] = daz; rec[RW_DGH + 2 * H + j] = dan * r;
    rec[RW_DHD + j] = d * zg;
  }
}

// 6-D -> rotation backward: dR (row-major 3x3, columns x, y, z) -> dp (6)
__device__ void rot6d_bwd(const float* p, const float* dR, float* dp) {
  const float a0 = p[0], a1 = p[1], a2 = p[2], b0 = p[3], b1 = p[4], b2 = p[5];
  const float la = sqrtf(a0 * a0 + a1 * a1 + a2 * a2), na = la + 1e-10f;
  const float x0 = a0 / na, x1 = a1 / na, x2 = a2 / na;
  const float c0 = x1 * b2 - x2 * b1, c1 = x2 * b0 - x0 * b2, c2 = x0 * b1 - x1 * b0;
  const float lc = sqrtf(c0 * c0 + c1 * c1 + c2 * c2), nc = lc + 1e-10f;
  const float z0 = c0 / nc, z1 = c1 / nc, z2 = c2 / nc;
  float dx0 = dR[0], dx1 = dR[3], dx2 = dR[6];
  const float dy0 = dR[1], dy1 = dR[4], dy2 = dR[7];
  float dz0 = dR[2], dz1 = dR[5], dz2 = dR[8];
  // y = z x x
  dz0 += x1 * dy2 - x2 * dy1; dz1 += x2 * dy0 - x0 * dy2; dz2 += x0 * dy1 - x1 * dy0;
  dx0 += dy1 * z2 - dy2 * z1; dx1 += dy2 * z0 - dy0 * z2; dx2 += dy0 * z1 - dy1 * z0;
  // z = c / (|c| + 1e-10)
  const float cdz = (c0 * dz0 + c1 * dz1 + c2 * dz2) / (lc > 0.f ? lc * nc * nc : 1.f);
  const float dc0 = dz0 / nc - c0 * cdz, dc1 = dz1 / nc - c1 * cdz, dc2 = dz2 / nc - c2 * cdz;
  // c = x x b
  dx0 += b1 * dc2 - b2 * dc1; dx1 += b2 * dc0 - b0 * dc2; dx2 += b0 * dc1 - b1 * dc0;
  dp[3] = dc1 * x2 - dc2 * x1; dp[4] = dc2 * x0 - dc0 * x2; dp[5] = dc0 * x1 - dc1 * x0;
  // x = a / (|a| + 1e-10)
  const float adx = (a0 * dx0 + a1 * dx1 + a2 * dx2) / (la > 0.f ? la * na * na : 1.f);
  dp[0] = dx0 / na - a0 * adx; dp[1] = dx1 / na - a1 * adx; dp[2] = dx2 / na - a2 * adx;
}

// Pose backward of the picked decode: forward kinematics down `order` in reverse, then the 6-D rotations and the tanh.
// df = W_ih^T dgi [:4K] + external d kypt_recon; dR external d R; accumulates d offset.  One CTA of 64 threads per element.
template <int KC>
__global__ void __launch_bounds__(64)
pose_bwd_kernel(const float* __restrict__ Rg_all /* (B, K, 9) */, const float* __restrict__ offset, const int* __restrict__ order,
                const int* __restrict__ parents, const float* __restrict__ df_ext, const float* __restrict__ dR_ext,
                const float* __restrict__ dz_ext, int K, float* __restrict__ doffset, float* __restrict__ rows) {
  __shared__ float s_rl[KC * 9], s_drg[KC * 9], s_dpos[KC * 3], s_doff[KC * 3], s_dint[KC];
  const int b = blockIdx.x, K4 = 4 * K;
  float* rec = rows + (long long)b * RW;
  const float* Rg = Rg_all + (long long)b * K * 9;
  for (int k = threadIdx.x; k < K; k += 64) rot6d(rec + RW_OJ + k * 6, s_rl + k * 9);
  for (int i = threadIdx.x; i < K * 9; i += 64) s_drg[i] = ld_or0(dR_ext, (long long)b * K * 9 + i);
  for (int i = threadIdx.x; i < K4; i += 64) {
    const float d = rec[RW_DXG + i] + ld_or0(df_ext, (long long)b * K4 + i);
    if ((i & 3) == 3) s_dint[i >> 2] = d;
    else s_dpos[(i >> 2) * 3 + (i & 3)] = d;
  }
  for (int i = threadIdx.x; i < K * 3; i += 64) s_doff[i] = 0.f;
  for (int i = threadIdx.x; i < Z; i += 64) rec[RW_DXG + K4 + i] += ld_or0(dz_ext, (long long)b * Z + i);   // dz
  __syncthreads();
  if (threadIdx.x == 0) {
    for (int j = K - 1; j >= 1; j--) {
      const int i = order[j], pa = parents[i];
      const float* Ri = Rg + i * 9;
      const float* Rp = Rg + pa * 9;
      const float* Rl = s_rl + i * 9;
      const float* o = offset + ((long long)b * K + i) * 3;
      float* dRi = s_drg + i * 9;
      float* dRp = s_drg + pa * 9;
      const float dp0 = s_dpos[i * 3], dp1 = s_dpos[i * 3 + 1], dp2 = s_dpos[i * 3 + 2];
      s_dpos[pa * 3] += dp0; s_dpos[pa * 3 + 1] += dp1; s_dpos[pa * 3 + 2] += dp2;
#pragma unroll
      for (int c = 0; c < 3; c++) {
        s_doff[i * 3 + c] = Ri[c] * dp0 + Ri[3 + c] * dp1 + Ri[6 + c] * dp2;
        dRi[c] += dp0 * o[c]; dRi[3 + c] += dp1 * o[c]; dRi[6 + c] += dp2 * o[c];
      }
      float dl[9];
#pragma unroll
      for (int r = 0; r < 3; r++)
#pragma unroll
        for (int c = 0; c < 3; c++) {
          dRp[r * 3 + c] += dRi[r * 3] * Rl[c * 3] + dRi[r * 3 + 1] * Rl[c * 3 + 1] + dRi[r * 3 + 2] * Rl[c * 3 + 2];
          dl[r * 3 + c] = Rp[r] * dRi[c] + Rp[3 + r] * dRi[3 + c] + Rp[6 + r] * dRi[6 + c];
        }
#pragma unroll
      for (int e = 0; e < 9; e++) dRi[e] = dl[e];      // d Rl_i from here on
    }
  }
  __syncthreads();
  // the root's global rotation is its local one: s_drg[root] already holds d Rl_root
  for (int k = threadIdx.x; k < K; k += 64) {
    float dp[6];
    rot6d_bwd(rec + RW_OJ + k * 6, s_drg + k * 9, dp);
#pragma unroll
    for (int e = 0; e < 6; e++) rec[RW_DOJ + k * 6 + e] = dp[e];
  }
  const int root = order[0];
  for (int c = threadIdx.x; c < 3 + K; c += 64) {
    const float y = rec[RW_OR + c];
    const float d = c < 3 ? s_dpos[root * 3 + c] : 0.5f * s_dint[c - 3];
    rec[RW_DOR + c] = d * (1.f - y * y);
  }
  for (int i = threadIdx.x; i < K * 3; i += 64) doffset[(long long)b * K * 3 + i] += s_doff[i];
}

// z = qm + qs * eps_pick: d of the posterior / prior raw outputs (std = softplus(raw) + 1e-4).  One CTA per element.
__global__ void __launch_bounds__(Z)
dist_bwd_kernel(const float* __restrict__ eps, const int* __restrict__ pick, const float* __restrict__ dpost,
                const float* __restrict__ dprior, int B, int K, float* __restrict__ rows) {
  const int b = blockIdx.x, i = threadIdx.x;
  float* rec = rows + (long long)b * RW;
  const float dz = rec[RW_DXG + 4 * K + i] + rec[RW_DXDR + H + i] + rec[RW_DXDJ + H + i];
  const float e = eps[((long long)pick[b] * B + b) * Z + i];
  rec[RW_DOQ + i] = dz + ld_or0(dpost, (long long)b * 2 * Z + i);
  rec[RW_DOQ + Z + i] = (dz * e + ld_or0(dpost, (long long)b * 2 * Z + Z + i)) * dsoftplus_d(rec[RW_OQ + Z + i]);
  rec[RW_DOP + i] = ld_or0(dprior, (long long)b * 2 * Z + i);
  rec[RW_DOP + Z + i] = ld_or0(dprior, (long long)b * 2 * Z + Z + i) * dsoftplus_d(rec[RW_OP + Z + i]);
}

// dh_t = GRU direct part + W_hh^T dgh + decoders' h parts + posterior / prior h parts + external d h_kypts[:, t]
__global__ void __launch_bounds__(kThreads)
dh_sum_kernel(const float* __restrict__ rows, const float* __restrict__ dh_ext, float* __restrict__ dh_out) {
  const int b = blockIdx.x;
  const float* rec = rows + (long long)b * RW;
  for (int j = threadIdx.x; j < H; j += kThreads) {
    float v = rec[RW_DHD + j] + rec[RW_DH1 + j];
    v += rec[RW_DXDR + j] + rec[RW_DXDJ + j];
    v += rec[RW_DXQ + j] + rec[RW_DXP + j];
    dh_out[(long long)b * H + j] = v + ld_or0(dh_ext, (long long)b * H + j);
  }
}

GemmJob gemm_job(const float* x0, int ldx0, int k0, const float* x1, int ldx1, int K, const float* m, int ldm, int N,
                 float* y, int ldy) {
  GemmJob j;
  j.x0 = x0; j.ldx0 = ldx0; j.k0 = k0; j.x1 = x1; j.ldx1 = ldx1; j.K = K;
  j.m = m; j.ldm = ldm; j.N = N; j.bias = nullptr; j.gate = nullptr; j.ldgate = 0; j.y = y; j.ldy = ldy;
  j.xlrelu = 0; j.tanh_out = 0;
  return j;
}

int launch_gemm(GemmJobs& js, int n, int B, cudaStream_t st) {
  js.n = n; js.B = B;
  int tiles = 0, kmax = 0;
  for (int i = 0; i < n; i++) {
    tiles += nm_cdiv(js.j[i].N, GC);
    js.tile_end[i] = tiles;
    kmax = max(kmax, js.j[i].K);
  }
  const size_t smem = ((size_t)GR * kmax + 8 * GR * GC) * sizeof(float);
  NM_CHECK_CUDA(cudaFuncSetAttribute(rows_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
  rows_gemm_kernel<<<dim3(tiles, nm_cdiv(B, GR)), kThreads, smem, st>>>(js);
  NM_CHECK_LAUNCH("hsvrnn_step_backward(gemm)");
  return NM_OK;
}

// ------------------------------------------------------------------ weight gradients over the T*B rows, fixed order
// dW[o][i] = sum_r dY[r][o] X[r][i] (X == null: a column of ones -> bias / init-state sums); 64 x 64 tiles, each thread a
// 4 x 4 block, rows streamed through shared memory 16 at a time in ascending order.  No atomics: bit-reproducible.
constexpr int kMaxWgJobs = 24;
struct WgJob {
  const float* dy; const float* x0; const float* x1; float* dw;
  int lddy, O, ldx0, ldx1, k0, I, xlrelu, R, ldw;
};
struct WgJobs {
  WgJob j[kMaxWgJobs];
  int tile_end[kMaxWgJobs];
  int n;
  const float* offset; const float* doffset; const float* offset_param; float* d_offset_param;
  int B, K;
};

__global__ void __launch_bounds__(kThreads)
hsvrnn_wgrad_kernel(const __grid_constant__ WgJobs js) {
  __shared__ float s_dy[16][64], s_x[16][64];
  const int tid = threadIdx.x;
  const int tile = blockIdx.x;
  if (tile >= js.tile_end[js.n - 1]) {
    // offset_param: offset[b, k] = op_k / (|op_k| + 1e-10) * scale[b, k]  (scale = the bone-length median)
    const int k = tid;
    if (k >= js.K) return;
    const float* op = js.offset_param + k * 3;
    const float lo = sqrtf(op[0] * op[0] + op[1] * op[1] + op[2] * op[2]), n = lo + 1e-10f;
    const float u0 = op[0] / n, u1 = op[1] / n, u2 = op[2] / n, uu = u0 * u0 + u1 * u1 + u2 * u2;
    float du0 = 0.f, du1 = 0.f, du2 = 0.f;
    for (int b = 0; b < js.B; b++) {
      const float* o = js.offset + ((long long)b * js.K + k) * 3;
      const float* d = js.doffset + ((long long)b * js.K + k) * 3;
      const float scale = uu > 0.f ? (o[0] * u0 + o[1] * u1 + o[2] * u2) / uu : 0.f;
      du0 = fmaf(scale, d[0], du0); du1 = fmaf(scale, d[1], du1); du2 = fmaf(scale, d[2], du2);
    }
    const float od = (op[0] * du0 + op[1] * du1 + op[2] * du2) / (lo > 0.f ? lo * n * n : 1.f);
    js.d_offset_param[k * 3] = du0 / n - op[0] * od;
    js.d_offset_param[k * 3 + 1] = du1 / n - op[1] * od;
    js.d_offset_param[k * 3 + 2] = du2 / n - op[2] * od;
    return;
  }
  int ji = 0;
  while (tile >= js.tile_end[ji]) ji++;
  const WgJob& J = js.j[ji];
  const int local = tile - (ji ? js.tile_end[ji - 1] : 0);
  const int ti = (J.I + 63) / 64;
  const int o0 = (local / ti) * 64, i0 = (local % ti) * 64;
  const int tx = tid & 15, ty = tid >> 4;
  float acc[4][4];
#pragma unroll
  for (int e = 0; e < 4; e++) acc[e][0] = acc[e][1] = acc[e][2] = acc[e][3] = 0.f;
  for (int r0 = 0; r0 < J.R; r0 += 16) {
    for (int i = tid; i < 16 * 64; i += kThreads) {
      const int rr = i >> 6, c = i & 63, r = r0 + rr;
      float dy = 0.f, x = 0.f;
      if (r < J.R) {
        if (o0 + c < J.O) dy = J.dy[(long long)r * J.lddy + o0 + c];
        const int ii = i0 + c;
        if (ii < J.I) {
          if (!J.x0) x = 1.f;
          else {
            x = ii < J.k0 ? J.x0[(long long)r * J.ldx0 + ii] : J.x1[(long long)r * J.ldx1 + (ii - J.k0)];
            if (J.xlrelu) x = nm_lrelu(x);
          }
        }
      }
      s_dy[rr][c] = dy;
      s_x[rr][c] = x;
    }
    __syncthreads();
#pragma unroll 4
    for (int rr = 0; rr < 16; rr++) {
      float a[4], v[4];
#pragma unroll
      for (int e = 0; e < 4; e++) { a[e] = s_dy[rr][ty * 4 + e]; v[e] = s_x[rr][tx * 4 + e]; }
#pragma unroll
      for (int e = 0; e < 4; e++)
#pragma unroll
        for (int f = 0; f < 4; f++) acc[e][f] = fmaf(a[e], v[f], acc[e][f]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int e = 0; e < 4; e++) {
    const int o = o0 + ty * 4 + e;
    if (o >= J.O) continue;
#pragma unroll
    for (int f = 0; f < 4; f++) {
      const int i = i0 + tx * 4 + f;
      if (i < J.I) J.dw[(long long)o * J.ldw + i] = acc[e][f];
    }
  }
}

}  // namespace

extern "C" size_t nm_hsvrnn_backward_workspace_bytes(int B, int T) { return (size_t)B * T * RW * sizeof(float); }

extern "C" int nm_hsvrnn_step_backward(const nm_hsvrnn_weights* wt, const nm_hsvrnn_weights* w, const float* h,
                                       const float* kp, const float* eps, const int* pick, const float* f, const float* z,
                                       const float* R, const float* offset, const int* order, const int* parents, int B,
                                       int K, int S, const float* dh_next, const float* dh_ext, const float* df,
                                       const float* dR, const float* dz, const float* dpost, const float* dprior,
                                       float* dh_out, float* doffset, float* rows, void* stream) {
  NM_CHECK_ARG(wt && w && h && kp && eps && pick && f && z && R && offset && order && parents && dh_next && dh_out &&
                   doffset && rows, "nm_hsvrnn_step_backward: null pointer");
  NM_CHECK_ARG(K > 0 && K <= kMaxK && S >= 1 && S <= 16, "nm_hsvrnn_step_backward: K=%d S=%d unsupported", K, S);
  if (B == 0) return NM_OK;
  (void)S;
  cudaStream_t st = (cudaStream_t)stream;
  const int K4 = 4 * K, R2 = 3 + K, J2 = 6 * K;
  GemmJobs js;
  // 1. forward recompute, first layers and both GRU halves (everything that reads h, kp, f, z)
  js.j[0] = gemm_job(h, H, H, nullptr, 0, H, wt->prior0_wt, HID, HID, rows + RW_AP, RW);
  js.j[0].bias = wt->prior0_b;
  js.j[1] = gemm_job(h, H, H, kp, K4, H + K4, wt->post0_wt, HID, HID, rows + RW_AQ, RW);
  js.j[1].bias = wt->post0_b;
  js.j[2] = gemm_job(h, H, H, z, Z, H + Z, wt->root0_wt, HID, HID, rows + RW_AR, RW);
  js.j[2].bias = wt->root0_b;
  js.j[3] = gemm_job(h, H, H, z, Z, H + Z, wt->joint0_wt, HID, HID, rows + RW_AJ, RW);
  js.j[3].bias = wt->joint0_b;
  js.j[4] = gemm_job(h, H, H, nullptr, 0, H, wt->gru_hh_wt, 3 * H, 3 * H, rows + RW_GH, RW);
  js.j[4].bias = wt->gru_hh_b;
  js.j[5] = gemm_job(f, K4, K4, z, Z, K4 + Z, wt->gru_ih_wt, 3 * H, 3 * H, rows + RW_GI, RW);
  js.j[5].bias = wt->gru_ih_b;
  if (int rc = launch_gemm(js, 6, B, st)) return rc;
  // 2. forward recompute, second layers (raw outputs; tanh for the root / intensity decoder)
  js.j[0] = gemm_job(rows + RW_AP, RW, HID, nullptr, 0, HID, wt->prior2_wt, 2 * Z, 2 * Z, rows + RW_OP, RW);
  js.j[1] = gemm_job(rows + RW_AQ, RW, HID, nullptr, 0, HID, wt->post2_wt, 2 * Z, 2 * Z, rows + RW_OQ, RW);
  js.j[2] = gemm_job(rows + RW_AR, RW, HID, nullptr, 0, HID, wt->root2_wt, R2, R2, rows + RW_OR, RW);
  js.j[3] = gemm_job(rows + RW_AJ, RW, HID, nullptr, 0, HID, wt->joint2_wt, J2, J2, rows + RW_OJ, RW);
  js.j[0].bias = wt->prior2_b; js.j[1].bias = wt->post2_b; js.j[2].bias = wt->root2_b; js.j[3].bias = wt->joint2_b;
  for (int i = 0; i < 4; i++) js.j[i].xlrelu = 1;
  js.j[2].tanh_out = 1;
  if (int rc = launch_gemm(js, 4, B, st)) return rc;
  // 3. GRU backward
  gru_bwd_kernel<<<B, kThreads, 0, st>>>(h, dh_next, rows);
  NM_CHECK_LAUNCH("hsvrnn_step_backward(gru)");
  js.j[0] = gemm_job(rows + RW_DGI, RW, 3 * H, nullptr, 0, 3 * H, w->gru_ih_wt, K4 + Z, K4 + Z, rows + RW_DXG, RW);
  js.j[1] = gemm_job(rows + RW_DGH, RW, 3 * H, nullptr, 0, 3 * H, w->gru_hh_wt, H, H, rows + RW_DH1, RW);
  if (int rc = launch_gemm(js, 2, B, st)) return rc;
  // 4. forward kinematics, 6-D rotations, tanh
  if (K <= kTunedK) pose_bwd_kernel<kTunedK><<<B, 64, 0, st>>>(R, offset, order, parents, df, dR, dz, K, doffset, rows);
  else pose_bwd_kernel<kMaxK><<<B, 64, 0, st>>>(R, offset, order, parents, df, dR, dz, K, doffset, rows);
  NM_CHECK_LAUNCH("hsvrnn_step_backward(pose)");
  // 5. decoders: second layers (times LeakyReLU' of the first), then the first layers' [h | z] parts
  js.j[0] = gemm_job(rows + RW_DOR, RW, R2, nullptr, 0, R2, w->root2_wt, HID, HID, rows + RW_DAR, RW);
  js.j[1] = gemm_job(rows + RW_DOJ, RW, J2, nullptr, 0, J2, w->joint2_wt, HID, HID, rows + RW_DAJ, RW);
  js.j[0].gate = rows + RW_AR; js.j[1].gate = rows + RW_AJ;
  js.j[0].ldgate = js.j[1].ldgate = RW;
  if (int rc = launch_gemm(js, 2, B, st)) return rc;
  js.j[0] = gemm_job(rows + RW_DAR, RW, HID, nullptr, 0, HID, w->root0_wt, H + Z, H + Z, rows + RW_DXDR, RW);
  js.j[1] = gemm_job(rows + RW_DAJ, RW, HID, nullptr, 0, HID, w->joint0_wt, H + Z, H + Z, rows + RW_DXDJ, RW);
  if (int rc = launch_gemm(js, 2, B, st)) return rc;
  // 6. posterior / prior distributions, then their MLPs (the posterior's kp columns are not needed)
  dist_bwd_kernel<<<B, Z, 0, st>>>(eps, pick, dpost, dprior, B, K, rows);
  NM_CHECK_LAUNCH("hsvrnn_step_backward(dist)");
  js.j[0] = gemm_job(rows + RW_DOQ, RW, 2 * Z, nullptr, 0, 2 * Z, w->post2_wt, HID, HID, rows + RW_DAQ, RW);
  js.j[1] = gemm_job(rows + RW_DOP, RW, 2 * Z, nullptr, 0, 2 * Z, w->prior2_wt, HID, HID, rows + RW_DAP, RW);
  js.j[0].gate = rows + RW_AQ; js.j[1].gate = rows + RW_AP;
  js.j[0].ldgate = js.j[1].ldgate = RW;
  if (int rc = launch_gemm(js, 2, B, st)) return rc;
  js.j[0] = gemm_job(rows + RW_DAQ, RW, HID, nullptr, 0, HID, w->post0_wt, H + K4, H, rows + RW_DXQ, RW);
  js.j[1] = gemm_job(rows + RW_DAP, RW, HID, nullptr, 0, HID, w->prior0_wt, H, H, rows + RW_DXP, RW);
  if (int rc = launch_gemm(js, 2, B, st)) return rc;
  // 7. dh_t
  dh_sum_kernel<<<B, kThreads, 0, st>>>(rows, dh_ext, dh_out);
  NM_CHECK_LAUNCH("hsvrnn_step_backward(dh)");
  return NM_OK;
}

extern "C" int nm_hsvrnn_weight_grads(const float* rows, const float* h, const float* kp, const float* f, const float* z,
                                      const float* dh0, const float* offset, const float* doffset,
                                      const float* offset_param, int B, int T, int K, const nm_hsvrnn_grads* g,
                                      void* stream) {
  NM_CHECK_ARG(rows && h && kp && f && z && dh0 && g, "nm_hsvrnn_weight_grads: null pointer");
  NM_CHECK_ARG(K > 0 && K <= kMaxK && T >= 1, "nm_hsvrnn_weight_grads: K=%d T=%d unsupported", K, T);
  NM_CHECK_ARG(!g->offset_param || (offset && doffset && offset_param), "nm_hsvrnn_weight_grads: offset_param needs offsets");
  if (B == 0) return NM_OK;
  const int K4 = 4 * K, R = T * B;
  WgJobs js;
  int n = 0;
  auto add = [&](const float* dy, int O, const float* x0, int ldx0, int k0, const float* x1, int ldx1, int I, int xl,
                 float* dw, float* db) {
    WgJob j;
    j.dy = dy; j.lddy = RW; j.O = O; j.x0 = x0; j.ldx0 = ldx0; j.k0 = k0; j.x1 = x1; j.ldx1 = ldx1; j.I = I;
    j.xlrelu = xl; j.R = R; j.dw = dw; j.ldw = I;
    js.j[n++] = j;
    j.x0 = j.x1 = nullptr; j.I = 1; j.ldw = 1; j.dw = db;
    js.j[n++] = j;
  };
  add(rows + RW_DAQ, HID, h, H, H, kp, K4, H + K4, 0, g->post0_w, g->post0_b);
  add(rows + RW_DOQ, 2 * Z, rows + RW_AQ, RW, HID, nullptr, 0, HID, 1, g->post2_w, g->post2_b);
  add(rows + RW_DAP, HID, h, H, H, nullptr, 0, H, 0, g->prior0_w, g->prior0_b);
  add(rows + RW_DOP, 2 * Z, rows + RW_AP, RW, HID, nullptr, 0, HID, 1, g->prior2_w, g->prior2_b);
  add(rows + RW_DAR, HID, h, H, H, z, Z, H + Z, 0, g->root0_w, g->root0_b);
  add(rows + RW_DOR, 3 + K, rows + RW_AR, RW, HID, nullptr, 0, HID, 1, g->root2_w, g->root2_b);
  add(rows + RW_DAJ, HID, h, H, H, z, Z, H + Z, 0, g->joint0_w, g->joint0_b);
  add(rows + RW_DOJ, 6 * K, rows + RW_AJ, RW, HID, nullptr, 0, HID, 1, g->joint2_w, g->joint2_b);
  add(rows + RW_DGI, 3 * H, f, K4, K4, z, Z, K4 + Z, 0, g->gru_ih_w, g->gru_ih_b);
  add(rows + RW_DGH, 3 * H, h, H, H, nullptr, 0, H, 0, g->gru_hh_w, g->gru_hh_b);
  {  // d init_kypt_rnn_state = sum over b of dh_0
    WgJob j;
    j.dy = dh0; j.lddy = H; j.O = H; j.x0 = j.x1 = nullptr; j.ldx0 = j.ldx1 = j.k0 = 0; j.I = 1; j.xlrelu = 0; j.R = B;
    j.dw = g->init_state; j.ldw = 1;
    js.j[n++] = j;
  }
  int tiles = 0;
  for (int i = 0; i < n; i++) {
    tiles += nm_cdiv(js.j[i].O, 64) * nm_cdiv(js.j[i].I, 64);
    js.tile_end[i] = tiles;
  }
  js.n = n; js.B = B; js.K = K;
  js.offset = offset; js.doffset = doffset; js.offset_param = offset_param; js.d_offset_param = g->offset_param;
  hsvrnn_wgrad_kernel<<<tiles + (g->offset_param ? 1 : 0), kThreads, 0, (cudaStream_t)stream>>>(js);
  NM_CHECK_LAUNCH("hsvrnn_weight_grads");
  return NM_OK;
}
