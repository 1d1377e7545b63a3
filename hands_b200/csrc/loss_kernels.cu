// Key-point loss and metric partial sums on the head's outputs (SURVEY.md 8(f) f2), one hand side per call.
//   loss terms   : src/callbacks/loss/loss_arctic_sf.py:70-92,131-136 with src/utils/loss_modules.py:62-73,88-125
//                  (hand_kp3d_loss = root-relative MSE, joints_loss = MSE, both masked by joints_valid and gated per sample,
//                  reduced with .mean() over all B*21*D elements);
//   metrics      : common/metrics.py:23-45 as consumed by src/utils/eval_modules.py:95-118,407-421 (root-relative per-joint
//                  L2 averaged per hand, pixel L2 per joint after data_utils.unormalize_kp2d), and :47-55 (MRRPE).
// One warp per hand, lane = joint; per-hand partial sums land in a (B, 8) scratch and are folded by a fixed-order
// single-block reduction, so the sums are bit-reproducible and can be added straight into the packed all-reduce buffer.
#include "hb_common.cuh"

namespace hb {

constexpr int KS = HB_KP_SUMS;           // 8

struct KpArgs {
  const float* j3d; const float* j2d; const float* gt3; const float* gt2; const float* jv; const float* hv; const float* gate3; const float* gate2;
  int B; float img_res;
};

__device__ __forceinline__ float warp_sum(float v) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}

__global__ void __launch_bounds__(128) kp_loss_fwd_kernel(KpArgs a, float* __restrict__ partial) {
  const int b = blockIdx.x * 4 + (threadIdx.x >> 5), j = threadIdx.x & 31;
  if (b >= a.B) return;
  const bool live = j < NOJ;
  float d3[3] = {0.f, 0.f, 0.f}, d2[2] = {0.f, 0.f};
  float v = 0.f;
  if (live) {
    const size_t o3 = ((size_t)b * NOJ + j) * 3, o2 = ((size_t)b * NOJ + j) * 2;
#pragma unroll
    for (int k = 0; k < 3; ++k) d3[k] = __ldg(a.j3d + o3 + k) - __ldg(a.gt3 + o3 + k);
#pragma unroll
    for (int k = 0; k < 2; ++k) d2[k] = __ldg(a.j2d + o2 + k) - __ldg(a.gt2 + o2 + k);
    v = __ldg(a.jv + (size_t)b * NOJ + j);
  }
  // root-relative: (pred - pred_root) - (gt - gt_root) = d - d_root
#pragma unroll
  for (int k = 0; k < 3; ++k) d3[k] -= __shfl_sync(0xffffffffu, d3[k], 0);
  const float g3 = a.gate3 ? __ldg(a.gate3 + b) : 1.0f, g2 = a.gate2 ? __ldg(a.gate2 + b) : 1.0f, hv = a.hv ? __ldg(a.hv + b) : 1.0f;
  const float sq3 = d3[0] * d3[0] + d3[1] * d3[1] + d3[2] * d3[2], sq2 = d2[0] * d2[0] + d2[1] * d2[1];
  const float s0 = warp_sum(live ? sq3 * v * g3 : 0.f);
  const float s1 = warp_sum(live ? sq2 * v * g2 : 0.f);
  const float s2 = warp_sum(live ? sqrtf(sq3) : 0.f);                                   // compute_joint3d_error: per-hand validity only
  const float half = 0.5f * a.img_res;                                                   // unormalize_kp2d: 0.5 * img_res * (x + 1)
  const float s4 = warp_sum(live ? sqrtf(sq2) * half * v * hv : 0.f);
  const float s5 = warp_sum(live ? v * hv : 0.f);
  if (j == 0) {
    float* p = partial + (size_t)b * KS;
    p[0] = s0; p[1] = s1; p[2] = hv * (s2 / (float)NOJ); p[3] = hv; p[4] = s4; p[5] = s5; p[6] = 0.f; p[7] = 0.f;
  }
}

// sums[k] = sum_b partial[b][k], fixed order: thread t adds rows t, t+1024, ... then a shared-memory tree
__global__ void __launch_bounds__(1024) kp_reduce_kernel(const float* __restrict__ partial, int B, float* __restrict__ sums) {
  __shared__ float sh[1024];
  for (int k = 0; k < KS; ++k) {
    float acc = 0.f;
    for (int b = threadIdx.x; b < B; b += 1024) acc += partial[(size_t)b * KS + k];
    sh[threadIdx.x] = acc;
    __syncthreads();
    for (int m = 512; m > 0; m >>= 1) {
      if (threadIdx.x < m) sh[threadIdx.x] += sh[threadIdx.x + m];
      __syncthreads();
    }
    if (threadIdx.x == 0) sums[k] = sh[0];
    __syncthreads();
  }
}

__global__ void __launch_bounds__(128) kp_loss_bwd_kernel(KpArgs a, const float* __restrict__ g_loss3, const float* __restrict__ g_loss2,
                                                          float* __restrict__ g_j3d, float* __restrict__ g_j2d) {
  const int b = blockIdx.x * 4 + (threadIdx.x >> 5), j = threadIdx.x & 31;
  if (b >= a.B) return;
  const bool live = j < NOJ;
  float d3[3] = {0.f, 0.f, 0.f}, d2[2] = {0.f, 0.f};
  float v = 0.f;
  const size_t o3 = ((size_t)b * NOJ + (live ? j : 0)) * 3, o2 = ((size_t)b * NOJ + (live ? j : 0)) * 2;
  if (live) {
#pragma unroll
    for (int k = 0; k < 3; ++k) d3[k] = __ldg(a.j3d + o3 + k) - __ldg(a.gt3 + o3 + k);
#pragma unroll
    for (int k = 0; k < 2; ++k) d2[k] = __ldg(a.j2d + o2 + k) - __ldg(a.gt2 + o2 + k);
    v = __ldg(a.jv + (size_t)b * NOJ + j);
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) d3[k] -= __shfl_sync(0xffffffffu, d3[k], 0);
  const float g3 = a.gate3 ? __ldg(a.gate3 + b) : 1.0f, g2 = a.gate2 ? __ldg(a.gate2 + b) : 1.0f;
  // loss3 = sum / (B*21*3), loss2 = sum / (B*21*2)
  const float c3 = (g_loss3 ? __ldg(g_loss3) : 0.f) * 2.0f / ((float)a.B * (float)(NOJ * 3)) * v * g3;
  const float c2 = (g_loss2 ? __ldg(g_loss2) : 0.f) * 2.0f / ((float)a.B * (float)(NOJ * 2)) * v * g2;
  float gr[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) { gr[k] = live ? c3 * d3[k] : 0.f; }
  // the root joint also receives minus the sum over all joints (every joint is taken relative to it)
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float tot = warp_sum(gr[k]);
    if (j == 0) gr[k] -= tot;
  }
  if (live) {
    if (g_j3d) {
#pragma unroll
      for (int k = 0; k < 3; ++k) g_j3d[o3 + k] = gr[k];
    }
    if (g_j2d) {
#pragma unroll
      for (int k = 0; k < 2; ++k) g_j2d[o2 + k] = c2 * d2[k];
    }
  }
}

// MRRPE (common/metrics.py:47-55): || (root_l - root_r)_pred - (root_l - root_r)_gt ||, roots = joint 0 of (B,21,3) arrays
__global__ void mrrpe_kernel(const float* __restrict__ pr, const float* __restrict__ pl, const float* __restrict__ gr, const float* __restrict__ gl,
                             const float* __restrict__ valid, int B, float* __restrict__ partial) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const size_t o = (size_t)b * NOJ * 3;
  float sq = 0.f;
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float d = (__ldg(pl + o + k) - __ldg(pr + o + k)) - (__ldg(gl + o + k) - __ldg(gr + o + k));
    sq += d * d;
  }
  const float v = valid ? __ldg(valid + b) : 1.0f;
  float* p = partial + (size_t)b * KS;
  p[0] = v * sqrtf(sq); p[1] = v;
#pragma unroll
  for (int k = 2; k < KS; ++k) p[k] = 0.f;
}

// Procrustes-aligned and root-relative point errors per hand (the HMR / ARCTIC compute_similarity_transform metric,
// src/utils/eval_modules.py:136-219, which runs a numpy SVD per sample on the host; the contract is restated in
// include/hands_b200.h and tests/procrustes_oracle.py::procrustes_errors).  One warp per hand, lane = point (strided):
//   pass 1: moments of a_i = p_i - p_0, b_i = q_i - q_0 in fp64 (shifted by point 0, so camera-space offsets of metres
//           cancel exactly in fp32 before anything is accumulated), folded into the centred C and var;
//   solve : Horn's symmetric 4x4 matrix of C, cyclic Jacobi with a fixed sweep count in fp64 -> the unit quaternion of
//           the proper rotation maximising trace(R C) (= V Z U^T of the SVD form, determinant correction included),
//           computed redundantly by every lane (no broadcast, no divergence);
//   pass 2: the row again (L1/L2), residuals s R X_i - Y_i in centred fp32 coordinates, `aligned`, the per-hand means.
// Every reduction is a fixed butterfly: per-hand results do not depend on the batch they are computed in.
constexpr int PA_SWEEPS = 6;   // quadratic convergence: the 4x4 off-diagonal is at rounding level after 4-5 sweeps

__device__ __forceinline__ double warp_sum_d(double v) {
#pragma unroll
  for (int m = 16; m > 0; m >>= 1) v += __shfl_xor_sync(0xffffffffu, v, m);
  return v;
}

struct ProcArgs {
  const float* pred; const float* gt; const float* root_pred; const float* root_gt; const float* hv;
  int B; int N; float* per_hand; float* aligned;
};

__global__ void __launch_bounds__(128) procrustes_kernel(ProcArgs a, float* __restrict__ partial) {
  const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= a.B) return;
  const int N = a.N;
  const float* P = a.pred + (size_t)b * N * 3;
  const float* Q = a.gt + (size_t)b * N * 3;
  const float p0[3] = {__ldg(P), __ldg(P + 1), __ldg(P + 2)}, q0[3] = {__ldg(Q), __ldg(Q + 1), __ldg(Q + 2)};

  // pass 1: sum a, sum b, sum a b^T, sum |a|^2
  double sa[3] = {0, 0, 0}, sb[3] = {0, 0, 0}, sab[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0}, saa = 0;
  for (int i = lane; i < N; i += 32) {
    double x[3], y[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) { x[k] = (double)(__ldg(P + 3 * i + k) - p0[k]); y[k] = (double)(__ldg(Q + 3 * i + k) - q0[k]); }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      sa[k] += x[k]; sb[k] += y[k]; saa = fma(x[k], x[k], saa);
#pragma unroll
      for (int l = 0; l < 3; ++l) sab[3 * k + l] = fma(x[k], y[l], sab[3 * k + l]);
    }
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) { sa[k] = warp_sum_d(sa[k]); sb[k] = warp_sum_d(sb[k]); }
#pragma unroll
  for (int k = 0; k < 9; ++k) sab[k] = warp_sum_d(sab[k]);
  saa = warp_sum_d(saa);
  const double inv_n = 1.0 / (double)N;
  double ma[3], mb[3], C[9];
#pragma unroll
  for (int k = 0; k < 3; ++k) { ma[k] = sa[k] * inv_n; mb[k] = sb[k] * inv_n; }
#pragma unroll
  for (int k = 0; k < 3; ++k)
#pragma unroll
    for (int l = 0; l < 3; ++l) C[3 * k + l] = sab[3 * k + l] - sa[k] * mb[l];   // sum X_k Y_l
  const double var = saa - (sa[0] * ma[0] + sa[1] * ma[1] + sa[2] * ma[2]);       // sum |X|^2
  const bool degenerate = !(var > 0.0);

  // solve: Horn's matrix, Jacobi eigen-decomposition, quaternion of the largest eigenvalue
  float sR[9] = {0, 0, 0, 0, 0, 0, 0, 0, 0};
  if (!degenerate) {
    const double Sxx = C[0], Sxy = C[1], Sxz = C[2], Syx = C[3], Syy = C[4], Syz = C[5], Szx = C[6], Szy = C[7], Szz = C[8];
    double A[4][4] = {{Sxx + Syy + Szz, Syz - Szy, Szx - Sxz, Sxy - Syx},
                      {Syz - Szy, Sxx - Syy - Szz, Sxy + Syx, Szx + Sxz},
                      {Szx - Sxz, Sxy + Syx, -Sxx + Syy - Szz, Syz + Szy},
                      {Sxy - Syx, Szx + Sxz, Syz + Szy, -Sxx - Syy + Szz}};
    double V[4][4] = {{1, 0, 0, 0}, {0, 1, 0, 0}, {0, 0, 1, 0}, {0, 0, 0, 1}};
    for (int sweep = 0; sweep < PA_SWEEPS; ++sweep) {
#pragma unroll
      for (int pq = 0; pq < 6; ++pq) {
        const int p = pq < 3 ? 0 : (pq < 5 ? 1 : 2), q = pq < 3 ? pq + 1 : (pq < 5 ? pq - 1 : 3);
        const double apq = A[p][q];
        if (apq == 0.0) continue;
        const double th = (A[q][q] - A[p][p]) / (2.0 * apq);
        const double at = fabs(th);     // th^2 would overflow beyond 1e154; there t = 1/(2 th) to working precision
        const double t = (th >= 0.0 ? 1.0 : -1.0) * (at > 1e150 ? 0.5 / at : 1.0 / (at + sqrt(fma(th, th, 1.0))));
        const double c = rsqrt(fma(t, t, 1.0)), s = t * c;   // |t| <= 1
#pragma unroll
        for (int k = 0; k < 4; ++k) {   // A <- A J (columns p, q)
          const double akp = A[k][p], akq = A[k][q];
          A[k][p] = c * akp - s * akq; A[k][q] = s * akp + c * akq;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {   // A <- J^T A (rows p, q)
          const double apk = A[p][k], aqk = A[q][k];
          A[p][k] = c * apk - s * aqk; A[q][k] = s * apk + c * aqk;
        }
#pragma unroll
        for (int k = 0; k < 4; ++k) {
          const double vkp = V[k][p], vkq = V[k][q];
          V[k][p] = c * vkp - s * vkq; V[k][q] = s * vkp + c * vkq;
        }
      }
    }
    double qv[4] = {V[0][0], V[1][0], V[2][0], V[3][0]}, lmax = A[0][0];   // eigenvector of the largest eigenvalue
#pragma unroll
    for (int m = 1; m < 4; ++m)
      if (A[m][m] > lmax) {
        lmax = A[m][m];
#pragma unroll
        for (int k = 0; k < 4; ++k) qv[k] = V[k][m];
      }
    const double qn = 1.0 / sqrt(qv[0] * qv[0] + qv[1] * qv[1] + qv[2] * qv[2] + qv[3] * qv[3]);
    const double w = qv[0] * qn, x = qv[1] * qn, y = qv[2] * qn, z = qv[3] * qn;
    const double R[9] = {w * w + x * x - y * y - z * z, 2 * (x * y - w * z), 2 * (x * z + w * y),
                         2 * (x * y + w * z), w * w - x * x + y * y - z * z, 2 * (y * z - w * x),
                         2 * (x * z - w * y), 2 * (y * z + w * x), w * w - x * x - y * y + z * z};
    const double sc = lmax / var;   // the largest eigenvalue of Horn's matrix is trace(R C) at the optimum
#pragma unroll
    for (int k = 0; k < 9; ++k) sR[k] = (float)(sc * R[k]);
  }

  // pass 2: residuals in centred coordinates (p^_i - q_i = s R X_i - Y_i), root-relative errors, aligned points
  const float mpf[3] = {(float)ma[0], (float)ma[1], (float)ma[2]}, mqf[3] = {(float)mb[0], (float)mb[1], (float)mb[2]};
  float rp[3], rq[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    rp[k] = a.root_pred ? __ldg(a.root_pred + (size_t)b * 3 + k) : p0[k];
    rq[k] = a.root_gt ? __ldg(a.root_gt + (size_t)b * 3 + k) : q0[k];
  }
  float* al = a.aligned ? a.aligned + (size_t)b * N * 3 : nullptr;
  double pa_acc = 0.0, ra_acc = 0.0;
  for (int i = lane; i < N; i += 32) {
    float p[3], q[3], X[3], Y[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      p[k] = __ldg(P + 3 * i + k); q[k] = __ldg(Q + 3 * i + k);
      X[k] = (p[k] - p0[k]) - mpf[k]; Y[k] = (q[k] - q0[k]) - mqf[k];
    }
    float d2 = 0.f, e2 = 0.f;
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float u = fmaf(sR[3 * k], X[0], fmaf(sR[3 * k + 1], X[1], sR[3 * k + 2] * X[2]));
      const float d = u - Y[k], e = (p[k] - rp[k]) - (q[k] - rq[k]);
      d2 = fmaf(d, d, d2); e2 = fmaf(e, e, e2);
      if (al) al[3 * i + k] = degenerate ? __int_as_float(0x7fc00000) : (u + mqf[k]) + q0[k];
    }
    pa_acc += (double)sqrtf(d2);
    ra_acc += (double)sqrtf(e2);
  }
  pa_acc = warp_sum_d(pa_acc);
  ra_acc = warp_sum_d(ra_acc);
  if (lane == 0) {
    const bool valid = a.hv ? __ldg(a.hv + b) != 0.0f : true;
    const float pa = (float)(pa_acc * inv_n), ra = (float)(ra_acc * inv_n), nan = __int_as_float(0x7fc00000);
    if (a.per_hand) {
      a.per_hand[(size_t)b * 2 + 0] = (valid && !degenerate) ? pa : nan;
      a.per_hand[(size_t)b * 2 + 1] = valid ? ra : nan;
    }
    float* o = partial + (size_t)b * KS;
    const bool use_pa = valid && !degenerate;
    o[0] = use_pa ? pa : 0.f; o[1] = use_pa ? 1.f : 0.f; o[2] = valid ? ra : 0.f; o[3] = valid ? 1.f : 0.f;
    o[4] = (valid && degenerate) ? 1.f : 0.f; o[5] = 0.f; o[6] = 0.f; o[7] = 0.f;
  }
}

// GT-side glue of process_data_light (src/callbacks/process/process_arctic.py:42-65), one hand side:
//   Tr0 = mean_j (j3d_full - joints_cano);  v3d_cam = vertices_cano + Tr0;  cam_t = j3d_full[:,0] - joints_cano[:,0];
//   cam_t_wp = perspective_to_weak_perspective_torch(cam_t, (K00+K11)/2, img_res)   (common/camera.py:10-29)
// One CTA of 128 threads per hand: warp 0 reduces the 21 joint offsets, all threads then stream the 778 vertices.
__global__ void __launch_bounds__(128) gt_process_kernel(const float* __restrict__ joints, const float* __restrict__ verts,
                                                         const float* __restrict__ j3d_full, const float* __restrict__ K, int B, float img_res,
                                                         float* __restrict__ v3d_cam, float* __restrict__ cam_t, float* __restrict__ cam_t_wp) {
  __shared__ float tr[3];
  const int b = blockIdx.x;
  if (threadIdx.x < 32) {
    const int j = threadIdx.x;
    float d[3] = {0.f, 0.f, 0.f};
    if (j < NOJ) {
      const size_t o = ((size_t)b * NOJ + j) * 3;
#pragma unroll
      for (int k = 0; k < 3; ++k) d[k] = __ldg(j3d_full + o + k) - __ldg(joints + o + k);
    }
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      const float root = __shfl_sync(0xffffffffu, d[k], 0);
      const float m = warp_sum(d[k]) / (float)NOJ;
      if (j == 0) {
        tr[k] = m;
        if (cam_t) cam_t[(size_t)b * 3 + k] = root;
        if (cam_t_wp && k == 2) {
          const float f = __fdiv_rn(__fadd_rn(__ldg(K + (size_t)b * 9 + 0), __ldg(K + (size_t)b * 9 + 4)), 2.0f);
          cam_t_wp[(size_t)b * 3 + 0] = __fdiv_rn(2.0f * f, __fadd_rn(__fmul_rn(img_res, root), 1e-9f));
        }
        if (cam_t_wp && k < 2) cam_t_wp[(size_t)b * 3 + 1 + k] = root;
      }
    }
  }
  __syncthreads();
  if (v3d_cam) {
    const float t0 = tr[0], t1 = tr[1], t2 = tr[2];
    const float* vi = verts + (size_t)b * HB_NUM_VERTS * 3;
    float* vo = v3d_cam + (size_t)b * HB_NUM_VERTS * 3;
    for (int e = threadIdx.x; e < HB_NUM_VERTS * 3; e += 128) {
      const int k = e % 3;
      vo[e] = __ldg(vi + e) + (k == 0 ? t0 : (k == 1 ? t1 : t2));
    }
  }
}

// KPE features of a crop box (src/datasets/hands_light_dataset.py:259-279) and their sinusoidal encodings
// (src/models/hands_light/model.py:444-460), batched.  Angles are computed in float64 like numpy and cast to fp32:
//   center_angle (2)  = atan2(c - K[.,2], K[.,.]) for the box centre,  corner_angle (8) for the corners
//   (x0,y0), (x0,y1), (x1,y0), (x1,y1);  enc[l][c][0/1] = sin / cos(2^l * angle[c]),  l < L.
__global__ void kpe_kernel(const int32_t* __restrict__ bbox, const float* __restrict__ K, int n, int L, float* __restrict__ center_angle,
                           float* __restrict__ corner_angle, float* __restrict__ center_enc, float* __restrict__ corner_enc) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n) return;
  const double x0 = bbox[(size_t)q * 4 + 0], y0 = bbox[(size_t)q * 4 + 1], x1 = bbox[(size_t)q * 4 + 2], y1 = bbox[(size_t)q * 4 + 3];
  const double fx = K[(size_t)q * 9 + 0], fy = K[(size_t)q * 9 + 4], cx = K[(size_t)q * 9 + 2], cy = K[(size_t)q * 9 + 5];
  float ang[10];
  ang[0] = (float)atan2((x0 + x1) / 2.0 - cx, fx);
  ang[1] = (float)atan2((y0 + y1) / 2.0 - cy, fy);
  const double xs[4] = {x0, x0, x1, x1}, ys[4] = {y0, y1, y0, y1};
#pragma unroll
  for (int c = 0; c < 4; ++c) { ang[2 + 2 * c] = (float)atan2(xs[c] - cx, fx); ang[3 + 2 * c] = (float)atan2(ys[c] - cy, fy); }
  if (center_angle) { center_angle[(size_t)q * 2 + 0] = ang[0]; center_angle[(size_t)q * 2 + 1] = ang[1]; }
  if (corner_angle) {
#pragma unroll
    for (int c = 0; c < 8; ++c) corner_angle[(size_t)q * 8 + c] = ang[2 + c];
  }
  float freq = 1.0f;
  for (int l = 0; l < L; ++l, freq *= 2.0f) {
    if (center_enc) {
#pragma unroll
      for (int c = 0; c < 2; ++c) {
        const float a = __fmul_rn(freq, ang[c]);
        center_enc[((size_t)q * L + l) * 4 + c * 2 + 0] = sinf(a); center_enc[((size_t)q * L + l) * 4 + c * 2 + 1] = cosf(a);
      }
    }
    if (corner_enc) {
#pragma unroll
      for (int c = 0; c < 8; ++c) {
        const float a = __fmul_rn(freq, ang[2 + c]);
        corner_enc[((size_t)q * L + l) * 16 + c * 2 + 0] = sinf(a); corner_enc[((size_t)q * L + l) * 16 + c * 2 + 1] = cosf(a);
      }
    }
  }
}

// ---- masked vector MSE terms: cam_t.wp (+ .init), relative translation l-r, pose and beta regressions ------------------
// src/callbacks/loss/loss_arctic_sf.py:52-69,94-129,146-158 with src/utils/loss_modules.py:99-113 (vector_loss, MSE,
// return_mean=False, dist * is_valid[..., None]; an all-invalid batch gives zeros -- the same numbers), gated per sample
// by meta_info['is_*_loss'], reduced with .mean() over B*D elements.
//   d[b][e] = (pred[b][e] - pred_minus[b][e]) - (gt[b][e] - gt_minus[b][e])          (the `_minus` operands are optional)
//   sum     = sum_b valid[b] * valid2[b] * gate[b] * ( sum_e d^2  +  sum_e (pred2[b][e] - gt[b][e] + gt_minus)^2 if pred2 )
// One warp per sample; partial[b] then the fixed-order single-block reduction: bit-reproducible.
struct VecArgs {
  const float* pred; const float* pred_minus; const float* gt; const float* gt_minus; const float* pred2;
  const float* valid; const float* valid2; const float* gate; int B; int D;
};

__device__ __forceinline__ float vec_mask(const VecArgs& a, int b) {
  float m = 1.0f;
  if (a.valid) m *= __ldg(a.valid + b);
  if (a.valid2) m *= __ldg(a.valid2 + b);
  if (a.gate) m *= __ldg(a.gate + b);
  return m;
}

__global__ void __launch_bounds__(128) vec_loss_fwd_kernel(VecArgs a, float* __restrict__ partial) {
  const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= a.B) return;
  float acc = 0.f;
  for (int e = lane; e < a.D; e += 32) {
    const size_t o = (size_t)b * a.D + e;
    const float t = __ldg(a.gt + o) - (a.gt_minus ? __ldg(a.gt_minus + o) : 0.f);
    const float d = (__ldg(a.pred + o) - (a.pred_minus ? __ldg(a.pred_minus + o) : 0.f)) - t;
    acc = fmaf(d, d, acc);
    if (a.pred2) { const float d2 = __ldg(a.pred2 + o) - t; acc = fmaf(d2, d2, acc); }
  }
  acc = warp_sum(acc);
  if (lane == 0) partial[b] = acc * vec_mask(a, b);
}

__global__ void __launch_bounds__(1024) vec_reduce_kernel(const float* __restrict__ partial, int B, float* __restrict__ sum) {
  __shared__ float sh[1024];
  float acc = 0.f;
  for (int b = threadIdx.x; b < B; b += 1024) acc += partial[b];
  sh[threadIdx.x] = acc;
  __syncthreads();
  for (int m = 512; m > 0; m >>= 1) {
    if (threadIdx.x < m) sh[threadIdx.x] += sh[threadIdx.x + m];
    __syncthreads();
  }
  if (threadIdx.x == 0) sum[0] = sh[0];
}

__global__ void __launch_bounds__(128) vec_loss_bwd_kernel(VecArgs a, const float* __restrict__ g_loss, float* __restrict__ g_pred,
                                                           float* __restrict__ g_pred_minus, float* __restrict__ g_pred2) {
  const int b = blockIdx.x * 4 + (threadIdx.x >> 5), lane = threadIdx.x & 31;
  if (b >= a.B) return;
  const float k = 2.0f * vec_mask(a, b) * __ldg(g_loss) / ((float)a.B * (float)a.D);   // loss = sum / (B*D)
  for (int e = lane; e < a.D; e += 32) {
    const size_t o = (size_t)b * a.D + e;
    const float t = __ldg(a.gt + o) - (a.gt_minus ? __ldg(a.gt_minus + o) : 0.f);
    const float d = (__ldg(a.pred + o) - (a.pred_minus ? __ldg(a.pred_minus + o) : 0.f)) - t;
    if (g_pred) g_pred[o] = k * d;
    if (g_pred_minus) g_pred_minus[o] = -k * d;
    if (g_pred2) g_pred2[o] = a.pred2 ? k * (__ldg(a.pred2 + o) - t) : 0.f;
  }
}

// pytorch3d axis_angle_to_matrix as the reference applies it to the GT pose (loss_arctic_sf.py:48-49) =
// quaternion_to_matrix(axis_angle_to_quaternion(aa)) (common/rot.py:754-784, 86-115)
__global__ void aa_to_matrix_kernel(const float* __restrict__ aa, int N, float* __restrict__ R) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  const float x = aa[(size_t)n * 3], y = aa[(size_t)n * 3 + 1], z = aa[(size_t)n * 3 + 2];
  const float ang = sqrtf(x * x + y * y + z * z);
  const float half = ang * 0.5f;
  const float eps = 1e-6f;
  const float soa = fabsf(ang) < eps ? 0.5f - (ang * ang) / 48.0f : sinf(half) / ang;
  const float r = cosf(half), i = x * soa, j = y * soa, k = z * soa;
  const float two_s = 2.0f / (r * r + i * i + j * j + k * k);
  float* o = R + (size_t)n * 9;
  o[0] = 1.f - two_s * (j * j + k * k); o[1] = two_s * (i * j - k * r);       o[2] = two_s * (i * k + j * r);
  o[3] = two_s * (i * j + k * r);       o[4] = 1.f - two_s * (i * i + k * k); o[5] = two_s * (j * k - i * r);
  o[6] = two_s * (i * k - j * r);       o[7] = two_s * (j * k + i * r);       o[8] = 1.f - two_s * (i * i + j * j);
}

}  // namespace hb

using namespace hb;

extern "C" int hb_vec_loss_fwd(const float* pred, const float* pred_minus, const float* gt, const float* gt_minus, const float* pred2,
                               const float* valid, const float* valid2, const float* gate, int B, int D, float* partial, float* sum, void* stream) {
  if (B < 0 || D <= 0 || !sum || (B > 0 && (!pred || !gt || !partial))) { set_error("hb_vec_loss_fwd: bad argument"); return HB_E_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  VecArgs a{pred, pred_minus, gt, gt_minus, pred2, valid, valid2, gate, B, D};
  if (B > 0) {
    vec_loss_fwd_kernel<<<(B + 3) / 4, 128, 0, st>>>(a, partial);
    g_launches++;
    int rc = check_launch("vec_loss_fwd_kernel");
    if (rc) return rc;
  }
  vec_reduce_kernel<<<1, 1024, 0, st>>>(partial, B, sum);
  g_launches++;
  return check_launch("vec_reduce_kernel");
}

extern "C" int hb_vec_loss_bwd(const float* pred, const float* pred_minus, const float* gt, const float* gt_minus, const float* pred2,
                               const float* valid, const float* valid2, const float* gate, int B, int D, const float* g_loss,
                               float* g_pred, float* g_pred_minus, float* g_pred2, void* stream) {
  if (B < 0 || D <= 0 || (B > 0 && (!pred || !gt || !g_loss))) { set_error("hb_vec_loss_bwd: bad argument"); return HB_E_ARG; }
  if (B == 0) return 0;
  VecArgs a{pred, pred_minus, gt, gt_minus, pred2, valid, valid2, gate, B, D};
  vec_loss_bwd_kernel<<<(B + 3) / 4, 128, 0, (cudaStream_t)stream>>>(a, g_loss, g_pred, g_pred_minus, g_pred2);
  g_launches++;
  return check_launch("vec_loss_bwd_kernel");
}

extern "C" int hb_axis_angle_to_matrix(const float* aa, int N, float* R, void* stream) {
  if (N < 0 || (N > 0 && (!aa || !R))) { set_error("hb_axis_angle_to_matrix: bad argument"); return HB_E_ARG; }
  if (N == 0) return 0;
  aa_to_matrix_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(aa, N, R);
  g_launches++;
  return check_launch("aa_to_matrix_kernel");
}



static int kp_check(const char* what, const float* j3d, const float* j2d, const float* gt3, const float* gt2, const float* jv, int B) {
  if (B < 0 || (B > 0 && (!j3d || !j2d || !gt3 || !gt2 || !jv))) { set_error("%s: bad argument", what); return HB_E_ARG; }
  return 0;
}

extern "C" int hb_kp_loss_fwd(const float* j3d_cam, const float* j2d_norm, const float* gt_j3d_cam, const float* gt_j2d_norm,
                              const float* joints_valid, const float* hand_valid, const float* gate_j3d, const float* gate_j2d, int B,
                              float img_res, float* partial, float* sums, void* stream) {
  int rc = kp_check("hb_kp_loss_fwd", j3d_cam, j2d_norm, gt_j3d_cam, gt_j2d_norm, joints_valid, B);
  if (rc) return rc;
  if (!sums || (B > 0 && !partial)) { set_error("hb_kp_loss_fwd: NULL output"); return HB_E_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  KpArgs a{j3d_cam, j2d_norm, gt_j3d_cam, gt_j2d_norm, joints_valid, hand_valid, gate_j3d, gate_j2d, B, img_res};
  if (B > 0) {
    kp_loss_fwd_kernel<<<(B + 3) / 4, 128, 0, st>>>(a, partial);
    g_launches++;
    rc = check_launch("kp_loss_fwd_kernel");
    if (rc) return rc;
  }
  kp_reduce_kernel<<<1, 1024, 0, st>>>(partial, B, sums);
  g_launches++;
  return check_launch("kp_reduce_kernel");
}

extern "C" int hb_kp_loss_bwd(const float* j3d_cam, const float* j2d_norm, const float* gt_j3d_cam, const float* gt_j2d_norm,
                              const float* joints_valid, const float* gate_j3d, const float* gate_j2d, int B, const float* g_loss_kp3d,
                              const float* g_loss_kp2d, float* g_j3d_cam, float* g_j2d_norm, void* stream) {
  int rc = kp_check("hb_kp_loss_bwd", j3d_cam, j2d_norm, gt_j3d_cam, gt_j2d_norm, joints_valid, B);
  if (rc) return rc;
  if (B == 0) return 0;
  KpArgs a{j3d_cam, j2d_norm, gt_j3d_cam, gt_j2d_norm, joints_valid, nullptr, gate_j3d, gate_j2d, B, 0.f};
  kp_loss_bwd_kernel<<<(B + 3) / 4, 128, 0, (cudaStream_t)stream>>>(a, g_loss_kp3d, g_loss_kp2d, g_j3d_cam, g_j2d_norm);
  g_launches++;
  return check_launch("kp_loss_bwd_kernel");
}

extern "C" int hb_mrrpe(const float* j3d_cam_r, const float* j3d_cam_l, const float* gt_j3d_cam_r, const float* gt_j3d_cam_l,
                        const float* valid, int B, float* partial, float* sums, void* stream) {
  if (B < 0 || !sums || (B > 0 && (!j3d_cam_r || !j3d_cam_l || !gt_j3d_cam_r || !gt_j3d_cam_l || !partial))) { set_error("hb_mrrpe: bad argument"); return HB_E_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  if (B > 0) {
    mrrpe_kernel<<<(B + 127) / 128, 128, 0, st>>>(j3d_cam_r, j3d_cam_l, gt_j3d_cam_r, gt_j3d_cam_l, valid, B, partial);
    g_launches++;
    int rc = check_launch("mrrpe_kernel");
    if (rc) return rc;
  }
  kp_reduce_kernel<<<1, 1024, 0, st>>>(partial, B, sums);
  g_launches++;
  return check_launch("kp_reduce_kernel");
}

extern "C" int hb_procrustes_metrics(const float* pred, const float* gt, int B, int N, const float* root_pred, const float* root_gt,
                                     const float* hand_valid, float* per_hand, float* aligned, float* partial, float* sums, void* stream) {
  if (B < 0 || !sums || (B > 0 && (!pred || !gt || !partial || N < 1))) { set_error("hb_procrustes_metrics: bad argument"); return HB_E_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  if (B > 0) {
    ProcArgs a{pred, gt, root_pred, root_gt, hand_valid, B, N, per_hand, aligned};
    procrustes_kernel<<<(B + 3) / 4, 128, 0, st>>>(a, partial);
    g_launches++;
    int rc = check_launch("procrustes_kernel");
    if (rc) return rc;
  }
  kp_reduce_kernel<<<1, 1024, 0, st>>>(partial, B, sums);
  g_launches++;
  return check_launch("kp_reduce_kernel");
}

extern "C" int hb_gt_process(const float* joints3d, const float* vertices, const float* j3d_full, const float* K, int B, float img_res,
                             float* v3d_cam, float* cam_t, float* cam_t_wp, void* stream) {
  if (B < 0 || (B > 0 && (!joints3d || !j3d_full || (v3d_cam && !vertices) || (cam_t_wp && !K)))) { set_error("hb_gt_process: bad argument"); return HB_E_ARG; }
  if (B == 0) return 0;
  gt_process_kernel<<<B, 128, 0, (cudaStream_t)stream>>>(joints3d, vertices, j3d_full, K, B, img_res, v3d_cam, cam_t, cam_t_wp);
  g_launches++;
  return check_launch("gt_process_kernel");
}

extern "C" int hb_kpe_features(const int32_t* bbox, const float* K, int n, int n_freq, float* center_angle, float* corner_angle,
                               float* center_enc, float* corner_enc, void* stream) {
  if (n < 0 || n_freq < 0 || n_freq > 30 || (n > 0 && (!bbox || !K))) { set_error("hb_kpe_features: bad argument"); return HB_E_ARG; }
  if (n == 0) return 0;
  kpe_kernel<<<(n + 127) / 128, 128, 0, (cudaStream_t)stream>>>(bbox, K, n, n_freq, center_angle, corner_angle, center_enc, corner_enc);
  g_launches++;
  return check_launch("kpe_kernel");
}
