// MANO layer + head, forward and backward (sm_100a).
//
// Two kernel families:
//   * pose kernels  : one thread per (hand, joint), 16-lane shuffle groups walk the kinematic tree.
//                     log map (rot.py:118-193) -> Rodrigues -> folded joint regression -> chain ->
//                     skinning transforms A, the blendshape feature row as TF32 hi/lo slabs, the 16 posed joints
//                     with camera translation and 2D projection (mano_head.py:42-51).
//   * blendshapes   : v_posed = v_template + [posedirs; shapedirs^T]^T F on tcgen05, 3xTF32 (K3+K5, mano_tc.cu).
//   * skin kernels  : one thread per vertex, HBF hands per CTA, 5 vertex slices.
//                     T_v = sum_j W[v,j] A_j ; x = T_v [v_posed;1]          (K7)
//                     finger-tip joints + projection (K8, K11), coalesced stores through smem.
//                     Backward recomputes T_v, reduces dA over vertices in smem and writes dL/dv_posed as TF32 hi/lo
//                     slabs; the feature gradient is their contraction with the basis on tcgen05 (mano_tc.cu).
// Workspace layout (floats), G = ceil(B/HBF), G128 = ceil(B/128).  The forward's regions are a prefix of the backward's,
// so a backward-sized workspace holds what the forward wrote where hb_mano_head_bwd_reuse() looks for it.
//   A   [G][HBF][AS]          16 x (3x4) transforms
//   OFF [G][HBF][8]           t1 (transl or 0), t2 (cam_t or 0), pad
//   fh, fl [G128][19][1024]   feature rows, TF32 hi / lo parts in UMMA slab order
//   vp  [G128*128][2400]      v_posed, coordinate-major per hand
//   backward only:
//   gA  [NSLICE][G][HBF][AS], gO [NSLICE][G][HBF][8]   per-slice partials
//   gvh, gvl [G128][300][1024]                         dL/dv_posed, TF32 hi / lo parts in UMMA slab order
//   gfeat [G_MAXSPLIT][G128*128][160]                  split-K partials of the feature gradient
#include "hb_common.cuh"
#include "pose_math.cuh"

namespace hb {

__host__ __device__ inline size_t ws_groups(int B) { return (size_t)(B + HBF - 1) / HBF; }
__host__ __device__ inline size_t ws_g128(int B) { return (size_t)(B + 127) / 128; }
__host__ __device__ inline size_t ws_A(int B) { (void)B; return 0; }
__host__ __device__ inline size_t ws_OFF(int B) { return ws_A(B) + ws_groups(B) * HBF * AS; }
__host__ __device__ inline size_t ws_fh(int B) { return ws_OFF(B) + ws_groups(B) * HBF * 8; }
__host__ __device__ inline size_t ws_fl(int B) { return ws_fh(B) + ws_g128(B) * 19 * 1024; }
__host__ __device__ inline size_t ws_vp(int B) { return ws_fl(B) + ws_g128(B) * 19 * 1024; }
__host__ __device__ inline size_t ws_fwd_end(int B) { return ws_vp(B) + ws_g128(B) * 128 * 2400; }
__host__ __device__ inline size_t ws_gA(int B) { return ws_fwd_end(B); }
__host__ __device__ inline size_t ws_gO(int B) { return ws_gA(B) + (size_t)NSLICE * ws_groups(B) * HBF * AS; }
__host__ __device__ inline size_t ws_gvh(int B) { return ws_gO(B) + (size_t)NSLICE * ws_groups(B) * HBF * 8; }
__host__ __device__ inline size_t ws_gvl(int B) { return ws_gvh(B) + ws_g128(B) * 300 * 1024; }
__host__ __device__ inline size_t ws_gfeat(int B) { return ws_gvl(B) + ws_g128(B) * 300 * 1024; }
__host__ __device__ inline size_t ws_gfeat_part(int B) { return ws_g128(B) * 128 * 160; }
__host__ __device__ inline size_t ws_bwd_end(int B) { return ws_gfeat(B) + (size_t)G_MAXSPLIT * ws_gfeat_part(B); }

// -------------------------------------------------------------------------------------------
// per-(hand, joint) forward state
// -------------------------------------------------------------------------------------------
struct JointState {
  float M[9];      // input rotation (after pre_rot), rotmat mode only
  float Min[9];    // raw input rotation (before pre_rot), joint 0 only
  Rot6dCtx r6;     // 6D input modes only
  LogMapCtx lm;
  float r[3];      // full_pose = aa + pose_mean
  RodCtx rod;
  float R[9];      // local rotation
  float J[3];      // rest joint
  float rel[3];    // J - J_parent
  float Rwp[9];    // parent's world rotation
  float Rw[9];     // world rotation
  float t[3];      // world translation == posed joint
  float camt[3];
  float t1[3];
};

struct PoseArgs {
  const float* pose; int fmt; const float* pre_rot; const float* betas;   // fmt: 0 axis-angle, 1 rotmat, 2+L 6D layout L
  const float* cam; const float* K; const float* transl; int B; float img_res; float min_s;
  float* fh; float* fl;   // feature slabs (hi / lo TF32 parts) in the workspace
};

__device__ __forceinline__ float shfl16(float v, int src) { return __shfl_sync(0xffffffffu, v, src, 16); }

__device__ __forceinline__ void pose_forward(const ManoConst& c, const PoseArgs& a, int b, int i, JointState& s) {
  float aa[3];
  if (a.fmt) {
    if (a.fmt == 1) {
      const float* m = a.pose + ((size_t)b * NJ + i) * 9;
#pragma unroll
      for (int k = 0; k < 9; ++k) s.M[k] = __ldg(m + k);
    } else {
      float x6[6];
#pragma unroll
      for (int k = 0; k < 6; ++k) x6[k] = __ldg(a.pose + ((size_t)b * NJ + i) * 6 + k);
      rot6d_fwd(x6, a.fmt - 2, s.M, s.r6);
    }
    if (i == 0 && a.pre_rot) {
      float P[9];
#pragma unroll
      for (int k = 0; k < 9; ++k) { P[k] = __ldg(a.pre_rot + (size_t)b * 9 + k); s.Min[k] = s.M[k]; }
      float T[9];
      mat3_mul(P, s.Min, T);
#pragma unroll
      for (int k = 0; k < 9; ++k) s.M[k] = T[k];
    }
    logmap_fwd(s.M, aa, s.lm);
  } else {
#pragma unroll
    for (int k = 0; k < 3; ++k) aa[k] = __ldg(a.pose + (size_t)b * 48 + i * 3 + k);
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) s.r[k] = __fadd_rn(aa[k], __ldg(c.pose_mean + i * 3 + k));
  rodrigues_fwd(s.r, s.R, s.rod);
  // folded joint regression J = Jt + Jsd . beta
  float beta[NB];
#pragma unroll
  for (int l = 0; l < NB; ++l) beta[l] = __ldg(a.betas + (size_t)b * NB + l);
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float acc = __ldg(c.Jt + i * 3 + k);
#pragma unroll
    for (int l = 0; l < NB; ++l) acc = fmaf(__ldg(c.Jsd + (i * 3 + k) * NB + l), beta[l], acc);
    s.J[k] = acc;
  }
  // kinematic chain over the tree levels
  const int parent = i == 0 ? 0 : c.parents[i];
  const int level = c.level[i];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    const float jp = shfl16(s.J[k], parent);
    s.rel[k] = i == 0 ? s.J[k] : s.J[k] - jp;
    s.t[k] = s.J[k];
  }
#pragma unroll
  for (int k = 0; k < 9; ++k) { s.Rw[k] = s.R[k]; s.Rwp[k] = (k % 4 == 0) ? 1.f : 0.f; }
  for (int round = 1; round <= c.depth; ++round) {
    float pR[9], pt[3];
#pragma unroll
    for (int k = 0; k < 9; ++k) pR[k] = shfl16(s.Rw[k], parent);
#pragma unroll
    for (int k = 0; k < 3; ++k) pt[k] = shfl16(s.t[k], parent);
    if (level == round) {
#pragma unroll
      for (int k = 0; k < 9; ++k) s.Rwp[k] = pR[k];
      mat3_mul(pR, s.R, s.Rw);
      float rt[3];
      mat3_vec(pR, s.rel, rt);
#pragma unroll
      for (int k = 0; k < 3; ++k) s.t[k] = rt[k] + pt[k];
    }
  }
  // camera translation (camera.py:462-474 with f = (K00+K11)/2, mano_head.py:42)
  s.camt[0] = s.camt[1] = s.camt[2] = 0.f;
  if (a.cam) {
    const float f = __fdiv_rn(__fadd_rn(__ldg(a.K + (size_t)b * 9 + 0), __ldg(a.K + (size_t)b * 9 + 4)), 2.0f);
    s.camt[0] = __ldg(a.cam + (size_t)b * 3 + 1);
    s.camt[1] = __ldg(a.cam + (size_t)b * 3 + 2);
    s.camt[2] = cam_tz(__ldg(a.cam + (size_t)b * 3 + 0), f, a.img_res, a.min_s);
  }
#pragma unroll
  for (int k = 0; k < 3; ++k) s.t1[k] = a.transl ? __ldg(a.transl + (size_t)b * 3 + k) : 0.f;
}

__global__ void __launch_bounds__(128) mano_pose_fwd_kernel(ManoConst c, PoseArgs a, float* __restrict__ ws,
                                                            float* __restrict__ joints3d, float* __restrict__ j3d_cam,
                                                            float* __restrict__ j2d, float* __restrict__ cam_t_out) {
  const int i = threadIdx.x & 15;
  const int braw = blockIdx.x * 8 + (threadIdx.x >> 4);
  const bool live = braw < a.B;
  const int b = live ? braw : a.B - 1;
  JointState s;
  pose_forward(c, a, b, i, s);
  if (!live) return;
  const size_t g = b / HBF, h = b % HBF;
  float* A = ws + ws_A(a.B) + (g * HBF + h) * AS + i * 12;
  {
    // feature row F = [R_1 - I, ..., R_15 - I, betas, 0 pad] in UMMA slab order: [group128][k-step][k-half][row-group][row][4]
    // (mano_tc.cu)
    const size_t gb = (size_t)(b / 128) * 19 * 1024;
    const int hl = b % 128;
    const int rowoff = (hl >> 3) * 32 + (hl & 7) * 4;
    const int p0 = i > 0 ? (i - 1) * 9 : NPF, np = i > 0 ? 9 : FS - NPF;
    for (int k = 0; k < np; ++k) {
      const int pidx = p0 + k;
      float val;
      if (i > 0) val = s.R[k] - ((k % 4 == 0) ? 1.f : 0.f);
      else val = pidx < NP ? __ldg(a.betas + (size_t)b * NB + (pidx - NPF)) : 0.f;
      const float hi = tf32_round(val), lo = tf32_round(val - hi);
      const size_t o = gb + (size_t)(pidx >> 3) * 1024 + ((pidx >> 2) & 1) * 512 + rowoff + (pidx & 3);
      a.fh[o] = hi; a.fl[o] = lo;
    }
  }
  if (i == 0) {
    float* off = ws + ws_OFF(a.B) + (g * HBF + h) * 8;
#pragma unroll
    for (int k = 0; k < 3; ++k) { off[k] = s.t1[k]; off[3 + k] = s.camt[k]; }
    off[6] = off[7] = 0.f;
    if (cam_t_out) {
#pragma unroll
      for (int k = 0; k < 3; ++k) cam_t_out[(size_t)b * 3 + k] = s.camt[k];
    }
  }
  // A_i = [Rw | t - Rw J]
  float rj[3];
  mat3_vec(s.Rw, s.J, rj);
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    A[r * 4 + 0] = s.Rw[r * 3 + 0]; A[r * 4 + 1] = s.Rw[r * 3 + 1]; A[r * 4 + 2] = s.Rw[r * 3 + 2];
    A[r * 4 + 3] = s.t[r] - rj[r];
  }
  float jw[3], jc[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) { jw[k] = s.t[k] + s.t1[k]; jc[k] = jw[k] + s.camt[k]; }
  const size_t jo = ((size_t)b * NOJ + i);
  if (joints3d) { joints3d[jo * 3 + 0] = jw[0]; joints3d[jo * 3 + 1] = jw[1]; joints3d[jo * 3 + 2] = jw[2]; }
  if (j3d_cam) { j3d_cam[jo * 3 + 0] = jc[0]; j3d_cam[jo * 3 + 1] = jc[1]; j3d_cam[jo * 3 + 2] = jc[2]; }
  if (j2d) {
    float Km[9], uv[2];
#pragma unroll
    for (int k = 0; k < 9; ++k) Km[k] = __ldg(a.K + (size_t)b * 9 + k);
    project_fwd(Km, jc, a.img_res, uv);
    j2d[jo * 2 + 0] = uv[0]; j2d[jo * 2 + 1] = uv[1];
  }
}

// -------------------------------------------------------------------------------------------
// skinning kernels
// -------------------------------------------------------------------------------------------
constexpr int XS = VPB * 3 + 2;  // per-hand stride of the vertex staging tile (482: even, and 2 mod 32)

__device__ __forceinline__ int tip_slot(const ManoConst& c, int v) {
  int t = -1;
#pragma unroll
  for (int k = 0; k < 5; ++k) if (c.tips[k] == v) t = k;
  return t;
}

// T (3x4, row-major 12) = sum_j w[j] * A[j].  Packed f32x2 FMAs (sm_100 FFMA2: two IEEE fp32 FMAs per issue slot; each lane is
// exactly fmaf(w[j], A[j][k], T[k]), so the result is bit-identical to the scalar form): 6 instead of 12 FMA issues per joint.
__device__ __forceinline__ void blend_transforms(const float* __restrict__ Ah, const float (&w)[NJ], float (&T)[12]) {
  float2 t[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) t[k] = make_float2(0.f, 0.f);
  const float4* a4 = reinterpret_cast<const float4*>(Ah);
#pragma unroll
  for (int j = 0; j < NJ; ++j) {
    const float4 r0 = a4[j * 3 + 0], r1 = a4[j * 3 + 1], r2 = a4[j * 3 + 2];
    const float2 ww = make_float2(w[j], w[j]);
    t[0] = __ffma2_rn(ww, make_float2(r0.x, r0.y), t[0]); t[1] = __ffma2_rn(ww, make_float2(r0.z, r0.w), t[1]);
    t[2] = __ffma2_rn(ww, make_float2(r1.x, r1.y), t[2]); t[3] = __ffma2_rn(ww, make_float2(r1.z, r1.w), t[3]);
    t[4] = __ffma2_rn(ww, make_float2(r2.x, r2.y), t[4]); t[5] = __ffma2_rn(ww, make_float2(r2.z, r2.w), t[5]);
  }
#pragma unroll
  for (int k = 0; k < 6; ++k) { T[2 * k] = t[k].x; T[2 * k + 1] = t[k].y; }
}

struct SkinFwdOut { float* vertices; float* v3d; float* joints3d; float* j3d_cam; float* j2d; };

__global__ void __launch_bounds__(VPB, 5) mano_skin_fwd_kernel(ManoConst c, const float* __restrict__ ws, const float* __restrict__ Kmat,
                                                                int B, float img_res, SkinFwdOut o, const float* __restrict__ vp) {
  extern __shared__ __align__(16) float smem[];
  float* As = smem;                                // [HBF][AS]
  float* Os = As + HBF * AS;                       // [HBF][8]
  float* Xs = Os + HBF * 8;                        // [HBF][XS]
  const int tid = threadIdx.x;
  const int g = blockIdx.x, slice = blockIdx.y;
  const int v = slice * VPB + tid;
  const int b0 = g * HBF;
  {
    const float4* srcA = reinterpret_cast<const float4*>(ws + ws_A(B) + (size_t)g * HBF * AS);
    const float4* srcO = reinterpret_cast<const float4*>(ws + ws_OFF(B) + (size_t)g * HBF * 8);
    // (only the transforms of this CTA's share of the group's hands)
    const int a0 = (int)blockIdx.z * (HBF / (int)gridDim.z) * AS / 4, a1 = a0 + (HBF / (int)gridDim.z) * AS / 4;
    for (int idx = a0 + tid; idx < a1; idx += VPB) reinterpret_cast<float4*>(As)[idx] = srcA[idx];
    for (int idx = tid; idx < HBF * 8 / 4; idx += VPB) reinterpret_cast<float4*>(Os)[idx] = srcO[idx];
  }
  __syncthreads();
  // v_posed comes from the tensor-core kernel: [hand][k][800] coordinate-major, coalesced over vertices
#pragma unroll 4
  for (int h = (int)blockIdx.z * (HBF / (int)gridDim.z); h < ((int)blockIdx.z + 1) * (HBF / (int)gridDim.z); ++h) {
    const int b = min(b0 + h, B - 1);
    const float* src = vp + (size_t)b * (3 * VP) + v;
    Xs[h * XS + 3 * tid + 0] = __ldg(src); Xs[h * XS + 3 * tid + 1] = __ldg(src + VP); Xs[h * XS + 3 * tid + 2] = __ldg(src + 2 * VP);
  }
  float w[NJ];
#pragma unroll
  for (int j = 0; j < NJ; ++j) w[j] = __ldg(c.Wt + j * VP + v);
  const int tip = v < NV ? tip_slot(c, v) : -1;
  // small batches: the group's 16 hands are split over gridDim.z CTAs (more CTAs in flight, shorter serial chain)
  const int hz0 = (int)blockIdx.z * (HBF / (int)gridDim.z);
  const int nh = min(hz0 + HBF / (int)gridDim.z, B - b0);
  for (int h = hz0; h < nh; ++h) {
    float T[12];
    blend_transforms(As + h * AS, w, T);
    float* xs = Xs + h * XS + 3 * tid;
    const float px = xs[0], py = xs[1], pz = xs[2];
    const float x = fmaf(T[0], px, fmaf(T[1], py, fmaf(T[2], pz, T[3])));
    const float y = fmaf(T[4], px, fmaf(T[5], py, fmaf(T[6], pz, T[7])));
    const float z = fmaf(T[8], px, fmaf(T[9], py, fmaf(T[10], pz, T[11])));
    xs[0] = x; xs[1] = y; xs[2] = z;
    if (tip >= 0) {
      const int b = b0 + h;
      const float* of = Os + h * 8;
      const float jw[3] = {x + of[0], y + of[1], z + of[2]};
      const float jc[3] = {jw[0] + of[3], jw[1] + of[4], jw[2] + of[5]};
      const size_t jo = (size_t)b * NOJ + NJ + tip;
      if (o.joints3d) { o.joints3d[jo * 3 + 0] = jw[0]; o.joints3d[jo * 3 + 1] = jw[1]; o.joints3d[jo * 3 + 2] = jw[2]; }
      if (o.j3d_cam) { o.j3d_cam[jo * 3 + 0] = jc[0]; o.j3d_cam[jo * 3 + 1] = jc[1]; o.j3d_cam[jo * 3 + 2] = jc[2]; }
      if (o.j2d) {
        float Km[9], uv[2];
#pragma unroll
        for (int k = 0; k < 9; ++k) Km[k] = __ldg(Kmat + (size_t)b * 9 + k);
        project_fwd(Km, jc, img_res, uv);
        o.j2d[jo * 2 + 0] = uv[0]; o.j2d[jo * 2 + 1] = uv[1];
      }
    }
  }
  __syncthreads();
  // coalesced float2 stores: this slice owns floats [slice*480, slice*480 + nvalid) of each hand's 2334
  const int nvalid = min(VPB, NV - slice * VPB) * 3;
  for (int h = hz0; h < nh; ++h) {
    const float* of = Os + h * 8;
    const size_t base = (size_t)(b0 + h) * (NV * 3) + (size_t)slice * VPB * 3;
    for (int e = tid * 2; e < nvalid; e += VPB * 2) {
      const float2 val = *reinterpret_cast<const float2*>(Xs + h * XS + e);
      const int k0 = e % 3, k1 = (e + 1) % 3;
      float2 vw;
      vw.x = val.x + of[k0]; vw.y = val.y + of[k1];
      if (o.vertices) *reinterpret_cast<float2*>(o.vertices + base + e) = vw;
      if (o.v3d) {
        float2 vc;
        vc.x = vw.x + of[3 + k0]; vc.y = vw.y + of[3 + k1];
        *reinterpret_cast<float2*>(o.v3d + base + e) = vc;
      }
    }
  }
}

// ---- backward ----------------------------------------------------------------------------------
struct SkinBwdIn { const float* g_vertices; const float* g_v3d; const float* g_joints3d; const float* g_j3d_cam; const float* g_j2d; };

constexpr int HSUB = 8;           // hands per reduction pass of the backward kernel

__global__ void __launch_bounds__(VPB, 5) mano_skin_bwd_kernel(ManoConst c, float* __restrict__ ws, const float* __restrict__ Kmat,
                                                                int B, float img_res, SkinBwdIn gi, const float* __restrict__ vp,
                                                                float* __restrict__ gvh, float* __restrict__ gvl) {
  extern __shared__ __align__(16) float smem[];
  float* As = smem;                                    // [HBF][AS]
  float* Os = As + HBF * AS;                           // [HBF][8]
  float* Vs = Os + HBF * 8;                            // [HSUB][XS]   v_posed
  float* Gv = Vs + HSUB * XS;                          // [HSUB][XS]   dL/dvertex
  float* Og = Gv + HSUB * XS;                          // [HSUB][8]    per-hand sums of g_vertices / g_v3d (+ tip joints)
  float* Ogw = Og + HSUB * 8;                          // [VPB/32][HSUB][8] the same per warp (summed in warp order: deterministic)
  const int tid = threadIdx.x;
  const int g = blockIdx.x, slice = blockIdx.y;
  const int v = slice * VPB + tid;
  const int b0 = g * HBF;
  const size_t G = ws_groups(B);
  {
    const float4* srcA = reinterpret_cast<const float4*>(ws + ws_A(B) + (size_t)g * HBF * AS);
    const float4* srcO = reinterpret_cast<const float4*>(ws + ws_OFF(B) + (size_t)g * HBF * 8);
    // (only the transforms of this CTA's share of the group's hands)
    const int a0 = gridDim.z > 1 ? (int)blockIdx.z * HSUB * AS / 4 : 0, a1 = gridDim.z > 1 ? a0 + HSUB * AS / 4 : HBF * AS / 4;
    for (int idx = a0 + tid; idx < a1; idx += VPB) reinterpret_cast<float4*>(As)[idx] = srcA[idx];
    for (int idx = tid; idx < HBF * 8 / 4; idx += VPB) reinterpret_cast<float4*>(Os)[idx] = srcO[idx];
  }
  __syncthreads();
  float w[NJ];
#pragma unroll
  for (int j = 0; j < NJ; ++j) w[j] = __ldg(c.Wt + j * VP + v);
  const bool vlive = v < NV;
  const int tip = vlive ? tip_slot(c, v) : -1;
  const int lane = tid & 31;

#pragma unroll
  for (int sub = 0; sub < HBF / HSUB; ++sub) {
    // small batches: the group's passes are split over gridDim.z CTAs (block-uniform; the loop stays unrolled)
    if (gridDim.z > 1 && sub != (int)blockIdx.z) continue;
#pragma unroll
    for (int hh = 0; hh < HSUB; ++hh) {
      // v_posed from the tensor-core kernel: [hand][k][800], coalesced over vertices
      const int b = min(b0 + sub * HSUB + hh, B - 1);
      const float* src = vp + (size_t)b * (3 * VP) + v;
      Vs[hh * XS + 3 * tid + 0] = __ldg(src); Vs[hh * XS + 3 * tid + 1] = __ldg(src + VP); Vs[hh * XS + 3 * tid + 2] = __ldg(src + 2 * VP);
    }
    __syncthreads();
    // ---- phase L: per vertex, per hand: T_v, upstream vertex gradient, g_p = R_v^T gV
    for (int hh = 0; hh < HSUB; ++hh) {
      const int h = sub * HSUB + hh;
      const int b = b0 + h;
      float gv[3] = {0.f, 0.f, 0.f};
      float s1[3] = {0.f, 0.f, 0.f}, s2[3] = {0.f, 0.f, 0.f};  // sums feeding g_transl / g_cam_t
      float gp[3] = {0.f, 0.f, 0.f};
      if (b < B && vlive) {
        float T[12];
        blend_transforms(As + h * AS, w, T);
        const size_t vo = (size_t)b * (NV * 3) + (size_t)v * 3;
        if (gi.g_vertices) {
#pragma unroll
          for (int k = 0; k < 3; ++k) { const float t = __ldg(gi.g_vertices + vo + k); gv[k] += t; s1[k] += t; }
        }
        if (gi.g_v3d) {
#pragma unroll
          for (int k = 0; k < 3; ++k) { const float t = __ldg(gi.g_v3d + vo + k); gv[k] += t; s2[k] += t; }
        }
        if (tip >= 0) {
          const size_t jo = (size_t)b * NOJ + NJ + tip;
          if (gi.g_joints3d) {
#pragma unroll
            for (int k = 0; k < 3; ++k) { const float t = __ldg(gi.g_joints3d + jo * 3 + k); gv[k] += t; s1[k] += t; }
          }
          float gjc[3] = {0.f, 0.f, 0.f};
          if (gi.g_j3d_cam) {
#pragma unroll
            for (int k = 0; k < 3; ++k) gjc[k] = __ldg(gi.g_j3d_cam + jo * 3 + k);
          }
          if (gi.g_j2d) {
            const float* xs = Vs + hh * XS + 3 * tid;
            const float px = xs[0], py = xs[1], pz = xs[2];
            const float* of = Os + h * 8;
            float X[3];
            X[0] = fmaf(T[0], px, fmaf(T[1], py, fmaf(T[2], pz, T[3]))) + of[0] + of[3];
            X[1] = fmaf(T[4], px, fmaf(T[5], py, fmaf(T[6], pz, T[7]))) + of[1] + of[4];
            X[2] = fmaf(T[8], px, fmaf(T[9], py, fmaf(T[10], pz, T[11]))) + of[2] + of[5];
            float Km[9], guv[2], gX[3];
#pragma unroll
            for (int k = 0; k < 9; ++k) Km[k] = __ldg(Kmat + (size_t)b * 9 + k);
            guv[0] = __ldg(gi.g_j2d + jo * 2 + 0); guv[1] = __ldg(gi.g_j2d + jo * 2 + 1);
            project_bwd(Km, X, img_res, guv, gX);
#pragma unroll
            for (int k = 0; k < 3; ++k) gjc[k] += gX[k];
          }
#pragma unroll
          for (int k = 0; k < 3; ++k) { gv[k] += gjc[k]; s2[k] += gjc[k]; }
        }
        gp[0] = T[0] * gv[0] + T[4] * gv[1] + T[8] * gv[2];
        gp[1] = T[1] * gv[0] + T[5] * gv[1] + T[9] * gv[2];
        gp[2] = T[2] * gv[0] + T[6] * gv[1] + T[10] * gv[2];
      }
      Gv[hh * XS + 3 * tid + 0] = gv[0]; Gv[hh * XS + 3 * tid + 1] = gv[1]; Gv[hh * XS + 3 * tid + 2] = gv[2];
      {
        // dL/dv_posed goes to the tensor-core reduction (mano_gfeat_tc_kernel) as TF32 hi/lo UMMA slabs:
        // [group128][k-step = c'/8][k-half][row-group][row][4], c' = k*800 + v
        const int hl = b % 128;
        const size_t gb = (size_t)(b / 128) * 300 * 1024 + (size_t)(hl >> 3) * 32 + (hl & 7) * 4;
#pragma unroll
        for (int k = 0; k < 3; ++k) {
          const int cp = k * VP + v;
          const size_t o = gb + (size_t)(cp >> 3) * 1024 + ((cp >> 2) & 1) * 512 + (cp & 3);
          const float hi = tf32_round(gp[k]);
          gvh[o] = hi; gvl[o] = tf32_round(gp[k] - hi);
        }
      }
      // per-hand sums: warp shuffle tree, one slot per warp; the slots are added in warp order after the barrier (no float
      // atomics: g_cam / g_transl do not depend on the order the warps arrive in)
#pragma unroll
      for (int k = 0; k < 3; ++k) {
        float a1 = s1[k], a2 = s2[k];
#pragma unroll
        for (int m = 16; m > 0; m >>= 1) { a1 += __shfl_xor_sync(0xffffffffu, a1, m); a2 += __shfl_xor_sync(0xffffffffu, a2, m); }
        if (lane == 0) { Ogw[((tid >> 5) * HSUB + hh) * 8 + k] = a1; Ogw[((tid >> 5) * HSUB + hh) * 8 + 3 + k] = a2; }
      }
    }
    __syncthreads();
    if (tid < HSUB * 8 && (tid & 7) < 6) {
      float t = 0.f;
#pragma unroll
      for (int wdx = 0; wdx < VPB / 32; ++wdx) t += Ogw[wdx * HSUB * 8 + tid];
      Og[tid] = t;
    } else if (tid < HSUB * 8) Og[tid] = 0.f;
    // ---- phase A: gA[h][j][r][cc] = sum_v W[v][j] gV[v][r] * [v_posed;1][cc]     thread = (hand, joint)
    if (tid < HSUB * NJ) {
      const int hh = tid & (HSUB - 1), j = tid / HSUB;
      // packed f32x2 FMAs: (ga[2m], ga[2m+1]) += g_r * (p_a, p_b) with the homogeneous 1 as the fourth coordinate
      // (fmaf(g, 1, ga) == ga + g exactly, so the sums equal the scalar form bit for bit)
      float2 ga2[6];
#pragma unroll
      for (int k = 0; k < 6; ++k) ga2[k] = make_float2(0.f, 0.f);
      const float* gvp = Gv + hh * XS;
      const float* vpp = Vs + hh * XS;
      const float* wv = c.Wv + (size_t)(slice * VPB) * NJ + j;
#pragma unroll 4
      for (int vv = 0; vv < VPB; ++vv) {
        const float wj = __ldg(wv + vv * NJ);
        const float g0 = wj * gvp[3 * vv + 0], g1 = wj * gvp[3 * vv + 1], g2 = wj * gvp[3 * vv + 2];
        const float2 p01 = make_float2(vpp[3 * vv + 0], vpp[3 * vv + 1]), p2w = make_float2(vpp[3 * vv + 2], 1.0f);
        ga2[0] = __ffma2_rn(make_float2(g0, g0), p01, ga2[0]); ga2[1] = __ffma2_rn(make_float2(g0, g0), p2w, ga2[1]);
        ga2[2] = __ffma2_rn(make_float2(g1, g1), p01, ga2[2]); ga2[3] = __ffma2_rn(make_float2(g1, g1), p2w, ga2[3]);
        ga2[4] = __ffma2_rn(make_float2(g2, g2), p01, ga2[4]); ga2[5] = __ffma2_rn(make_float2(g2, g2), p2w, ga2[5]);
      }
      float ga[12];
#pragma unroll
      for (int k = 0; k < 6; ++k) { ga[2 * k] = ga2[k].x; ga[2 * k + 1] = ga2[k].y; }
      const int h = sub * HSUB + hh;
      float* dst = ws + ws_gA(B) + (((size_t)slice * G + g) * HBF + h) * AS + j * 12;
#pragma unroll
      for (int k = 0; k < 12; ++k) dst[k] = ga[k];
    }
    if (tid < HSUB * 8) {   // written by this same thread above
      const int hh = tid >> 3, k = tid & 7;
      const int h = sub * HSUB + hh;
      ws[ws_gO(B) + (((size_t)slice * G + g) * HBF + h) * 8 + k] = Og[hh * 8 + k];
    }
    __syncthreads();
  }
}

// ---- pose backward: chain^T, Rodrigues^T, log-map^T --------------------------------------------
struct PoseBwdArgs {
  const float* g_joints3d; const float* g_j3d_cam; const float* g_j2d; const float* g_cam_t;
  float* g_pose; float* g_betas; float* g_cam; float* g_transl; float* g_pre_rot;
};

__global__ void __launch_bounds__(128, 4) mano_pose_bwd_kernel(ManoConst c, PoseArgs a, const float* __restrict__ ws, PoseBwdArgs o,
                                                            const float* __restrict__ gFt, int gf_parts, size_t gf_stride) {
  const int i = threadIdx.x & 15;
  const int braw = blockIdx.x * 8 + (threadIdx.x >> 4);
  const bool live = braw < a.B;
  const int b = live ? braw : a.B - 1;
  JointState s;
  pose_forward(c, a, b, i, s);
  const size_t G = ws_groups(a.B), g = b / HBF, h = b % HBF;
  // sum the slice partials (fixed order -> deterministic)
  float gA[12];
#pragma unroll
  for (int k = 0; k < 12; ++k) gA[k] = 0.f;
  float gFr[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) gFr[k] = 0.f;
  float gbeta[NB];
#pragma unroll
  for (int l = 0; l < NB; ++l) gbeta[l] = 0.f;
  float gO[6] = {0.f, 0.f, 0.f, 0.f, 0.f, 0.f};
  for (int sl = 0; sl < NSLICE; ++sl) {
    const size_t row = ((size_t)sl * G + g) * HBF + h;
    const float* pa = ws + ws_gA(a.B) + row * AS + i * 12;
#pragma unroll
    for (int k = 0; k < 12; ++k) gA[k] += pa[k];
    if (i == 0) {
      const float* po = ws + ws_gO(a.B) + row * 8;
#pragma unroll
      for (int k = 0; k < 6; ++k) gO[k] += po[k];
    }
  }
  // feature gradient reduced over all vertices by the tensor-core kernel: split-K partials [part][hand][160], added in order
  for (int part = 0; part < gf_parts; ++part) {
    const float* pf = gFt + (size_t)part * gf_stride + (size_t)b * 160;
    if (i > 0) {
#pragma unroll
      for (int k = 0; k < 9; ++k) gFr[k] += __ldg(pf + (i - 1) * 9 + k);
    } else {
#pragma unroll
      for (int l = 0; l < NB; ++l) gbeta[l] += __ldg(pf + NPF + l);
    }
  }
  // gradient arriving at this posed joint: joints3d = t + t1 ; j3d_cam = joints3d + cam_t ; j2d = proj(j3d_cam)
  float gj1[3] = {0.f, 0.f, 0.f}, gj2[3] = {0.f, 0.f, 0.f};
  {
    const size_t jo = (size_t)b * NOJ + i;
    if (o.g_joints3d) {
#pragma unroll
      for (int k = 0; k < 3; ++k) gj1[k] = __ldg(o.g_joints3d + jo * 3 + k);
    }
    if (o.g_j3d_cam) {
#pragma unroll
      for (int k = 0; k < 3; ++k) gj2[k] = __ldg(o.g_j3d_cam + jo * 3 + k);
    }
    if (o.g_j2d) {
      float Km[9], X[3], guv[2], gX[3];
#pragma unroll
      for (int k = 0; k < 9; ++k) Km[k] = __ldg(a.K + (size_t)b * 9 + k);
#pragma unroll
      for (int k = 0; k < 3; ++k) X[k] = s.t[k] + s.t1[k] + s.camt[k];
      guv[0] = __ldg(o.g_j2d + jo * 2 + 0); guv[1] = __ldg(o.g_j2d + jo * 2 + 1);
      project_bwd(Km, X, a.img_res, guv, gX);
#pragma unroll
      for (int k = 0; k < 3; ++k) gj2[k] += gX[k];
    }
  }
  // A_i = [Rw | t - Rw J]
  float gRw[9], gt[3], gJ[3];
#pragma unroll
  for (int r = 0; r < 3; ++r) {
    const float gat = gA[r * 4 + 3];
#pragma unroll
    for (int cc = 0; cc < 3; ++cc) gRw[r * 3 + cc] = gA[r * 4 + cc] - gat * s.J[cc];
    gt[r] = gat + gj1[r] + gj2[r];
  }
  {
    const float gat[3] = {gA[3], gA[7], gA[11]};
    float tmp[3];
    matT3_vec(s.Rw, gat, tmp);
#pragma unroll
    for (int k = 0; k < 3; ++k) gJ[k] = -tmp[k];
  }
  // reverse tree walk: deepest level first; parents gather from their children
  const int level = c.level[i];
  float gR[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) gR[k] = 0.f;
  for (int round = c.depth; round >= 1; --round) {
    float send[15];
    if (level == round) {
      // Rw = Rwp R ; t = Rwp rel + tp
      matT3_mul(s.Rwp, gRw, gR);                 // g_R(local) = Rwp^T gRw
      float t1m[9];
      mat3_mulT(gRw, s.R, t1m);                  // gRw R^T
#pragma unroll
      for (int r = 0; r < 3; ++r)
#pragma unroll
        for (int cc = 0; cc < 3; ++cc) send[r * 3 + cc] = t1m[r * 3 + cc] + gt[r] * s.rel[cc];
      float grel[3];
      matT3_vec(s.Rwp, gt, grel);
#pragma unroll
      for (int k = 0; k < 3; ++k) { send[9 + k] = gt[k]; send[12 + k] = grel[k]; gJ[k] += grel[k]; }
    } else {
#pragma unroll
      for (int k = 0; k < 15; ++k) send[k] = 0.f;
    }
#pragma unroll
    for (int cs = 0; cs < 5; ++cs) {
      const int ch = c.child[i][cs];
      const int src = ch < 0 ? i : ch;
      const bool take = ch >= 0 && c.level[src] == round;
#pragma unroll
      for (int k = 0; k < 15; ++k) {
        const float val = shfl16(send[k], src);
        if (take) {
          if (k < 9) gRw[k] += val;
          else if (k < 12) gt[k - 9] += val;
          else gJ[k - 12] -= val;
        }
      }
    }
  }
  if (level == 0) {
#pragma unroll
    for (int k = 0; k < 9; ++k) gR[k] = gRw[k];
#pragma unroll
    for (int k = 0; k < 3; ++k) gJ[k] += gt[k];
  }
  // pose-corrective blendshape path: F[(i-1)*9+k] = R[k] - I
#pragma unroll
  for (int k = 0; k < 9; ++k) gR[k] += gFr[k];
  float g_r[3];
  rodrigues_bwd(s.r, s.rod, gR, g_r);
  // betas: J = Jt + Jsd beta  (+ the shape-blendshape rows already in gbeta on lane 0)
#pragma unroll
  for (int l = 0; l < NB; ++l) {
    float acc = gbeta[l];
#pragma unroll
    for (int k = 0; k < 3; ++k) acc = fmaf(__ldg(c.Jsd + (i * 3 + k) * NB + l), gJ[k], acc);
#pragma unroll
    for (int m = 8; m > 0; m >>= 1) acc += __shfl_xor_sync(0xffffffffu, acc, m, 16);
    gbeta[l] = acc;
  }
  // camera / translation sums over the 16 chain joints (tips and vertices arrive through gO)
  float sj1[3], sj2[3];
#pragma unroll
  for (int k = 0; k < 3; ++k) {
    float a1 = gj1[k], a2 = gj2[k];
#pragma unroll
    for (int m = 8; m > 0; m >>= 1) { a1 += __shfl_xor_sync(0xffffffffu, a1, m, 16); a2 += __shfl_xor_sync(0xffffffffu, a2, m, 16); }
    sj1[k] = a1; sj2[k] = a2;
  }
  if (!live) return;
  if (a.fmt) {
    float gM[9];
    logmap_bwd(s.lm, g_r, gM);
    if (i == 0 && a.pre_rot) {
      // M = P Min : g_Min = P^T gM ; g_P = gM Min^T
      float P[9], gMin[9];
#pragma unroll
      for (int k = 0; k < 9; ++k) P[k] = __ldg(a.pre_rot + (size_t)b * 9 + k);
      matT3_mul(P, gM, gMin);
      if (o.g_pre_rot) {
        float gP[9];
        mat3_mulT(gM, s.Min, gP);
#pragma unroll
        for (int k = 0; k < 9; ++k) o.g_pre_rot[(size_t)b * 9 + k] = gP[k];
      }
#pragma unroll
      for (int k = 0; k < 9; ++k) gM[k] = gMin[k];
    }
    if (a.fmt == 1) {
#pragma unroll
      for (int k = 0; k < 9; ++k) o.g_pose[((size_t)b * NJ + i) * 9 + k] = gM[k];
    } else {
      float g6[6];
      rot6d_bwd(s.r6, a.fmt - 2, gM, g6);
#pragma unroll
      for (int k = 0; k < 6; ++k) o.g_pose[((size_t)b * NJ + i) * 6 + k] = g6[k];
    }
  } else {
#pragma unroll
    for (int k = 0; k < 3; ++k) o.g_pose[(size_t)b * 48 + i * 3 + k] = g_r[k];
  }
  if (i == 0) {
#pragma unroll
    for (int l = 0; l < NB; ++l) o.g_betas[(size_t)b * NB + l] = gbeta[l];
    float gt2[3], gt1[3];
#pragma unroll
    for (int k = 0; k < 3; ++k) {
      gt2[k] = sj2[k] + gO[3 + k] + (o.g_cam_t ? __ldg(o.g_cam_t + (size_t)b * 3 + k) : 0.f);
      gt1[k] = sj1[k] + gO[k] + sj2[k] + gO[3 + k];
    }
    if (o.g_transl) {
#pragma unroll
      for (int k = 0; k < 3; ++k) o.g_transl[(size_t)b * 3 + k] = gt1[k];
    }
    if (o.g_cam && a.cam) {
      const float f = __fdiv_rn(__fadd_rn(__ldg(a.K + (size_t)b * 9 + 0), __ldg(a.K + (size_t)b * 9 + 4)), 2.0f);
      const float sc = __ldg(a.cam + (size_t)b * 3 + 0);
      o.g_cam[(size_t)b * 3 + 0] = gt2[2] * cam_tz_grad_s(sc, f, a.img_res, a.min_s);
      o.g_cam[(size_t)b * 3 + 1] = gt2[0];
      o.g_cam[(size_t)b * 3 + 2] = gt2[1];
    }
  }
}

// ---- small free-function kernels ------------------------------------------------------------------
__global__ void logmap_fwd_kernel(const float* __restrict__ R, int N, float* __restrict__ aa) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float m[9], out[3];
#pragma unroll
  for (int k = 0; k < 9; ++k) m[k] = __ldg(R + (size_t)n * 9 + k);
  LogMapCtx ctx;
  logmap_fwd(m, out, ctx);
  aa[(size_t)n * 3 + 0] = out[0]; aa[(size_t)n * 3 + 1] = out[1]; aa[(size_t)n * 3 + 2] = out[2];
}
__global__ void logmap_bwd_kernel(const float* __restrict__ R, const float* __restrict__ g_aa, int N, float* __restrict__ g_R) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float m[9], out[3], ga[3], gm[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) m[k] = __ldg(R + (size_t)n * 9 + k);
#pragma unroll
  for (int k = 0; k < 3; ++k) ga[k] = __ldg(g_aa + (size_t)n * 3 + k);
  LogMapCtx ctx;
  logmap_fwd(m, out, ctx);
  logmap_bwd(ctx, ga, gm);
#pragma unroll
  for (int k = 0; k < 9; ++k) g_R[(size_t)n * 9 + k] = gm[k];
}
__global__ void rot6d_fwd_kernel(const float* __restrict__ x6, int N, int layout, float* __restrict__ R) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float x[6], m[9];
#pragma unroll
  for (int k = 0; k < 6; ++k) x[k] = __ldg(x6 + (size_t)n * 6 + k);
  Rot6dCtx ctx;
  rot6d_fwd(x, layout, m, ctx);
#pragma unroll
  for (int k = 0; k < 9; ++k) R[(size_t)n * 9 + k] = m[k];
}
__global__ void rot6d_bwd_kernel(const float* __restrict__ x6, const float* __restrict__ g_R, int N, int layout, float* __restrict__ g_x6) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float x[6], m[9], gm[9], gx[6];
#pragma unroll
  for (int k = 0; k < 6; ++k) x[k] = __ldg(x6 + (size_t)n * 6 + k);
#pragma unroll
  for (int k = 0; k < 9; ++k) gm[k] = __ldg(g_R + (size_t)n * 9 + k);
  Rot6dCtx ctx;
  rot6d_fwd(x, layout, m, ctx);
  rot6d_bwd(ctx, layout, gm, gx);
#pragma unroll
  for (int k = 0; k < 6; ++k) g_x6[(size_t)n * 6 + k] = gx[k];
}
__global__ void project_fwd_kernel(const float* __restrict__ K, const float* __restrict__ pts, int B, int N, float img_res, float* __restrict__ out) {
  const size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= (size_t)B * N) return;
  const size_t b = n / N;
  float Km[9], X[3], uv[2];
#pragma unroll
  for (int k = 0; k < 9; ++k) Km[k] = __ldg(K + b * 9 + k);
#pragma unroll
  for (int k = 0; k < 3; ++k) X[k] = __ldg(pts + n * 3 + k);
  project_fwd(Km, X, img_res, uv);
  out[n * 2 + 0] = uv[0]; out[n * 2 + 1] = uv[1];
}
__global__ void project_bwd_kernel(const float* __restrict__ K, const float* __restrict__ pts, const float* __restrict__ g_out, int B, int N, float img_res, float* __restrict__ g_pts) {
  const size_t n = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= (size_t)B * N) return;
  const size_t b = n / N;
  float Km[9], X[3], guv[2], gX[3];
#pragma unroll
  for (int k = 0; k < 9; ++k) Km[k] = __ldg(K + b * 9 + k);
#pragma unroll
  for (int k = 0; k < 3; ++k) X[k] = __ldg(pts + n * 3 + k);
  guv[0] = __ldg(g_out + n * 2 + 0); guv[1] = __ldg(g_out + n * 2 + 1);
  project_bwd(Km, X, img_res, guv, gX);
  g_pts[n * 3 + 0] = gX[0]; g_pts[n * 3 + 1] = gX[1]; g_pts[n * 3 + 2] = gX[2];
}
__global__ void weak_to_persp_kernel(const float* __restrict__ cam, const float* __restrict__ focal, const float* __restrict__ g_cam_t, int B,
                                     float img_res, float min_s, float* __restrict__ out, int backward) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  const float s = cam[b * 3 + 0], f = focal[b];
  if (!backward) {
    out[b * 3 + 0] = cam[b * 3 + 1]; out[b * 3 + 1] = cam[b * 3 + 2]; out[b * 3 + 2] = cam_tz(s, f, img_res, min_s);
  } else {
    out[b * 3 + 0] = g_cam_t[b * 3 + 2] * cam_tz_grad_s(s, f, img_res, min_s);
    out[b * 3 + 1] = g_cam_t[b * 3 + 0]; out[b * 3 + 2] = g_cam_t[b * 3 + 1];
  }
}
__global__ void persp_to_weak_kernel(const float* __restrict__ cam_t, const float* __restrict__ focal, int B, float img_res, float* __restrict__ out) {
  const int b = blockIdx.x * blockDim.x + threadIdx.x;
  if (b >= B) return;
  out[b * 3 + 0] = __fdiv_rn(2.0f * focal[b], __fadd_rn(__fmul_rn(img_res, cam_t[b * 3 + 2]), 1e-9f));
  out[b * 3 + 1] = cam_t[b * 3 + 0]; out[b * 3 + 2] = cam_t[b * 3 + 1];
}
__global__ void rot_apply_kernel(const float* __restrict__ R, const float* __restrict__ M, int N, int transpose_R, float* __restrict__ out) {
  const int n = blockIdx.x * blockDim.x + threadIdx.x;
  if (n >= N) return;
  float r[9], m[9], o[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) { r[k] = __ldg(R + (size_t)n * 9 + k); m[k] = __ldg(M + (size_t)n * 9 + k); }
  if (transpose_R) matT3_mul(r, m, o); else mat3_mul(r, m, o);
#pragma unroll
  for (int k = 0; k < 9; ++k) out[(size_t)n * 9 + k] = o[k];
}

}  // namespace hb

// =================================================================================================
// C ABI
// =================================================================================================
using namespace hb;

extern "C" size_t hb_mano_workspace_bytes(int B, int backward) {
  if (B <= 0) return 0;
  return sizeof(float) * (backward ? ws_bwd_end(B) : ws_fwd_end(B));
}

static int check_common(const hb_mano* h, const float* pose, const float* betas, const float* cam, const float* K, int B,
                        void* workspace, size_t wbytes, int backward) {
  if (!h || !pose || !betas || B < 0 || (B > 0 && !workspace)) { set_error("hb_mano_head: NULL argument or negative batch"); return HB_E_ARG; }
  if ((cam == nullptr) != (K == nullptr)) { set_error("hb_mano_head: cam and K must be given together"); return HB_E_ARG; }
  if (wbytes < hb_mano_workspace_bytes(B, backward)) { set_error("hb_mano_head: workspace too small (%zu < %zu)", wbytes, hb_mano_workspace_bytes(B, backward)); return HB_E_WORKSPACE; }
  if (!aligned8(workspace) || (reinterpret_cast<uintptr_t>(workspace) & 15u)) { set_error("hb_mano_head: workspace must be 16-byte aligned"); return HB_E_ALIGN; }
  return 0;
}

// CTAs per (16-hand group, vertex slice) of the skinning kernels: the group's hands are split over two CTAs (shorter serial
// chain per CTA, twice the CTAs in flight).  Measured fwd+bwd of one side, 1 vs 2: 1024 hands 162 -> 145 us, 2048 221 -> 207,
// 4096 344 -> 337, 8192 626 -> 614.
constexpr unsigned kSkinHsplit = 2;

static const size_t kSkinFwdSmem = sizeof(float) * (HBF * AS + HBF * 8 + HBF * XS);
static const size_t kSkinBwdSmem = sizeof(float) * (HBF * AS + HBF * 8 + 2 * HSUB * XS + HSUB * 8 + (VPB / 32) * HSUB * 8);

extern "C" int hb_mano_head_fwd(const hb_mano* h, const float* pose, int pose_format, const float* pre_rot, const float* betas,
                                const float* cam, const float* K, const float* transl, int B, float img_res, float min_s,
                                float* vertices, float* v3d_cam, float* joints3d, float* j3d_cam, float* j2d_norm, float* cam_t,
                                void* workspace, size_t workspace_bytes, void* stream) {
  int rc = check_common(h, pose, betas, cam, K, B, workspace, workspace_bytes, 0);
  if (rc) return rc;
  if (B == 0) return 0;
  if (!cam && (v3d_cam || j3d_cam || j2d_norm || cam_t)) { set_error("hb_mano_head_fwd: camera outputs requested without cam/K"); return HB_E_ARG; }
  if (pose_format < 0 || pose_format > HB_POSE_ROT6D + HB_ROT6D_COLS_PAIRED) { set_error("hb_mano_head_fwd: unknown pose_format %d", pose_format); return HB_E_ARG; }
  if (pre_rot && !pose_format) { set_error("hb_mano_head_fwd: pre_rot needs rotation-matrix or 6D pose input"); return HB_E_ARG; }
  if ((vertices && !aligned8(vertices)) || (v3d_cam && !aligned8(v3d_cam))) { set_error("hb_mano_head_fwd: vertex outputs must be 8-byte aligned"); return HB_E_ALIGN; }
  cudaStream_t st = (cudaStream_t)stream;
  float* ws = (float*)workspace;
  float* fh = ws + ws_fh(B);
  float* fl = ws + ws_fl(B);
  float* vpo = ws + ws_vp(B);
  PoseArgs a{pose, pose_format, pre_rot, betas, cam, K, transl, B, img_res, min_s, fh, fl};
  mano_pose_fwd_kernel<<<(B + 7) / 8, 128, 0, st>>>(h->c, a, ws, joints3d, j3d_cam, j2d_norm, cam_t);
  g_launches++;
  rc = check_launch("mano_pose_fwd_kernel");
  if (rc) return rc;
  rc = launch_blend_tc(fh, fl, h->c.Bhi, h->c.Blo, h->c.Vt, B, vpo, st);
  if (rc) return rc;
  SkinFwdOut o{vertices, v3d_cam, joints3d, j3d_cam, j2d_norm};
  dim3 grid((unsigned)ws_groups(B), NSLICE, kSkinHsplit);
  HB_CUDA(cudaFuncSetAttribute(mano_skin_fwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSkinFwdSmem));
  mano_skin_fwd_kernel<<<grid, VPB, kSkinFwdSmem, st>>>(h->c, ws, K, B, img_res, o, vpo);
  g_launches++;
  return check_launch("mano_skin_fwd_kernel");
}

static int mano_head_bwd_impl(const hb_mano* h, const float* pose, int pose_format, const float* pre_rot, const float* betas,
                              const float* cam, const float* K, const float* transl, int B, float img_res, float min_s,
                              const float* g_vertices, const float* g_v3d_cam, const float* g_joints3d, const float* g_j3d_cam,
                              const float* g_j2d_norm, const float* g_cam_t, float* g_pose, float* g_betas, float* g_cam,
                              float* g_transl, float* g_pre_rot, void* workspace, size_t workspace_bytes, void* stream, bool reuse) {
  int rc = check_common(h, pose, betas, cam, K, B, workspace, workspace_bytes, 1);
  if (rc) return rc;
  if (B == 0) return 0;
  if (!g_pose || !g_betas) { set_error("hb_mano_head_bwd: g_pose and g_betas are required"); return HB_E_ARG; }
  if (!cam && (g_v3d_cam || g_j3d_cam || g_j2d_norm || g_cam_t)) { set_error("hb_mano_head_bwd: camera gradients given without cam/K"); return HB_E_ARG; }
  if (pose_format < 0 || pose_format > HB_POSE_ROT6D + HB_ROT6D_COLS_PAIRED) { set_error("hb_mano_head_bwd: unknown pose_format %d", pose_format); return HB_E_ARG; }
  if (pre_rot && !pose_format) { set_error("hb_mano_head_bwd: pre_rot needs rotation-matrix or 6D pose input"); return HB_E_ARG; }
  cudaStream_t st = (cudaStream_t)stream;
  float* ws = (float*)workspace;
  float* fh = ws + ws_fh(B);
  float* fl = ws + ws_fl(B);
  float* vpo = ws + ws_vp(B);
  float* gvh = ws + ws_gvh(B);
  float* gvl = ws + ws_gvl(B);
  float* gft = ws + ws_gfeat(B);
  PoseArgs a{pose, pose_format, pre_rot, betas, cam, K, transl, B, img_res, min_s, fh, fl};
  if (!reuse) {
    mano_pose_fwd_kernel<<<(B + 7) / 8, 128, 0, st>>>(h->c, a, ws, nullptr, nullptr, nullptr, nullptr);
    g_launches++;
    rc = check_launch("mano_pose_fwd_kernel");
    if (rc) return rc;
    rc = launch_blend_tc(fh, fl, h->c.Bhi, h->c.Blo, h->c.Vt, B, vpo, st);
    if (rc) return rc;
  }
  SkinBwdIn gi{g_vertices, g_v3d_cam, g_joints3d, g_j3d_cam, g_j2d_norm};
  dim3 grid((unsigned)ws_groups(B), NSLICE, kSkinHsplit);
  HB_CUDA(cudaFuncSetAttribute(mano_skin_bwd_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSkinBwdSmem));
  mano_skin_bwd_kernel<<<grid, VPB, kSkinBwdSmem, st>>>(h->c, ws, K, B, img_res, gi, vpo, gvh, gvl);
  g_launches++;
  rc = check_launch("mano_skin_bwd_kernel");
  if (rc) return rc;
  rc = launch_gfeat_tc(gvh, gvl, h->c.Ph, h->c.Pl, B, gft, st);
  if (rc) return rc;
  PoseBwdArgs o{g_joints3d, g_j3d_cam, g_j2d_norm, g_cam_t, g_pose, g_betas, g_cam, g_transl, g_pre_rot};
  mano_pose_bwd_kernel<<<(B + 7) / 8, 128, 0, st>>>(h->c, a, ws, o, gft, gfeat_nsplit(B), ws_gfeat_part(B));
  g_launches++;
  return check_launch("mano_pose_bwd_kernel");
}

extern "C" int hb_mano_head_bwd(const hb_mano* h, const float* pose, int pose_format, const float* pre_rot, const float* betas,
                                const float* cam, const float* K, const float* transl, int B, float img_res, float min_s,
                                const float* g_vertices, const float* g_v3d_cam, const float* g_joints3d, const float* g_j3d_cam,
                                const float* g_j2d_norm, const float* g_cam_t, float* g_pose, float* g_betas, float* g_cam,
                                float* g_transl, float* g_pre_rot, void* workspace, size_t workspace_bytes, void* stream) {
  return mano_head_bwd_impl(h, pose, pose_format, pre_rot, betas, cam, K, transl, B, img_res, min_s, g_vertices, g_v3d_cam, g_joints3d, g_j3d_cam,
                            g_j2d_norm, g_cam_t, g_pose, g_betas, g_cam, g_transl, g_pre_rot, workspace, workspace_bytes, stream, false);
}

extern "C" int hb_mano_head_bwd_reuse(const hb_mano* h, const float* pose, int pose_format, const float* pre_rot, const float* betas,
                                      const float* cam, const float* K, const float* transl, int B, float img_res, float min_s,
                                      const float* g_vertices, const float* g_v3d_cam, const float* g_joints3d, const float* g_j3d_cam,
                                      const float* g_j2d_norm, const float* g_cam_t, float* g_pose, float* g_betas, float* g_cam,
                                      float* g_transl, float* g_pre_rot, void* workspace, size_t workspace_bytes, void* stream) {
  return mano_head_bwd_impl(h, pose, pose_format, pre_rot, betas, cam, K, transl, B, img_res, min_s, g_vertices, g_v3d_cam, g_joints3d, g_j3d_cam,
                            g_j2d_norm, g_cam_t, g_pose, g_betas, g_cam, g_transl, g_pre_rot, workspace, workspace_bytes, stream, true);
}

extern "C" int hb_rot6d_to_rotmat_fwd(const float* x6, int N, int layout, float* R, void* stream) {
  if (N < 0 || layout < 0 || layout > HB_ROT6D_COLS_PAIRED || (N > 0 && (!x6 || !R))) { set_error("hb_rot6d_to_rotmat_fwd: bad argument"); return HB_E_ARG; }
  if (N == 0) return 0;
  rot6d_fwd_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(x6, N, layout, R);
  g_launches++;
  return check_launch("rot6d_fwd_kernel");
}
extern "C" int hb_rot6d_to_rotmat_bwd(const float* x6, const float* g_R, int N, int layout, float* g_x6, void* stream) {
  if (N < 0 || layout < 0 || layout > HB_ROT6D_COLS_PAIRED || (N > 0 && (!x6 || !g_R || !g_x6))) { set_error("hb_rot6d_to_rotmat_bwd: bad argument"); return HB_E_ARG; }
  if (N == 0) return 0;
  rot6d_bwd_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(x6, g_R, N, layout, g_x6);
  g_launches++;
  return check_launch("rot6d_bwd_kernel");
}
extern "C" int hb_matrix_to_axis_angle_fwd(const float* R, int N, float* aa, void* stream) {
  if (N < 0 || (N > 0 && (!R || !aa))) { set_error("hb_matrix_to_axis_angle_fwd: bad argument"); return HB_E_ARG; }
  if (N == 0) return 0;
  logmap_fwd_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(R, N, aa);
  g_launches++;
  return check_launch("logmap_fwd_kernel");
}
extern "C" int hb_matrix_to_axis_angle_bwd(const float* R, const float* g_aa, int N, float* g_R, void* stream) {
  if (N < 0 || (N > 0 && (!R || !g_aa || !g_R))) { set_error("hb_matrix_to_axis_angle_bwd: bad argument"); return HB_E_ARG; }
  if (N == 0) return 0;
  logmap_bwd_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(R, g_aa, N, g_R);
  g_launches++;
  return check_launch("logmap_bwd_kernel");
}
extern "C" int hb_project2d_fwd(const float* K, const float* pts, int B, int N, float img_res, float* out, void* stream) {
  if (B < 0 || N < 0 || ((size_t)B * N > 0 && (!K || !pts || !out))) { set_error("hb_project2d_fwd: bad argument"); return HB_E_ARG; }
  const size_t n = (size_t)B * N;
  if (n == 0) return 0;
  project_fwd_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(K, pts, B, N, img_res, out);
  g_launches++;
  return check_launch("project_fwd_kernel");
}
extern "C" int hb_project2d_bwd(const float* K, const float* pts, const float* g_out, int B, int N, float img_res, float* g_pts, void* stream) {
  if (B < 0 || N < 0 || ((size_t)B * N > 0 && (!K || !pts || !g_out || !g_pts))) { set_error("hb_project2d_bwd: bad argument"); return HB_E_ARG; }
  const size_t n = (size_t)B * N;
  if (n == 0) return 0;
  project_bwd_kernel<<<(unsigned)((n + 127) / 128), 128, 0, (cudaStream_t)stream>>>(K, pts, g_out, B, N, img_res, g_pts);
  g_launches++;
  return check_launch("project_bwd_kernel");
}
extern "C" int hb_weak_to_persp_fwd(const float* cam, const float* focal, int B, float img_res, float min_s, float* cam_t, void* stream) {
  if (B < 0 || (B > 0 && (!cam || !focal || !cam_t))) { set_error("hb_weak_to_persp_fwd: bad argument"); return HB_E_ARG; }
  if (B == 0) return 0;
  weak_to_persp_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(cam, focal, nullptr, B, img_res, min_s, cam_t, 0);
  g_launches++;
  return check_launch("weak_to_persp_kernel");
}
extern "C" int hb_weak_to_persp_bwd(const float* cam, const float* focal, const float* g_cam_t, int B, float img_res, float min_s, float* g_cam, void* stream) {
  if (B < 0 || (B > 0 && (!cam || !focal || !g_cam_t || !g_cam))) { set_error("hb_weak_to_persp_bwd: bad argument"); return HB_E_ARG; }
  if (B == 0) return 0;
  weak_to_persp_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(cam, focal, g_cam_t, B, img_res, min_s, g_cam, 1);
  g_launches++;
  return check_launch("weak_to_persp_kernel");
}
extern "C" int hb_persp_to_weak_fwd(const float* cam_t, const float* focal, int B, float img_res, float* cam_wp, void* stream) {
  if (B < 0 || (B > 0 && (!cam_t || !focal || !cam_wp))) { set_error("hb_persp_to_weak_fwd: bad argument"); return HB_E_ARG; }
  if (B == 0) return 0;
  persp_to_weak_kernel<<<(B + 127) / 128, 128, 0, (cudaStream_t)stream>>>(cam_t, focal, B, img_res, cam_wp);
  g_launches++;
  return check_launch("persp_to_weak_kernel");
}
extern "C" int hb_rot_apply(const float* R, const float* M, int N, int transpose_R, float* out, void* stream) {
  if (N < 0 || (N > 0 && (!R || !M || !out))) { set_error("hb_rot_apply: bad argument"); return HB_E_ARG; }
  if (N == 0) return 0;
  rot_apply_kernel<<<(N + 127) / 128, 128, 0, (cudaStream_t)stream>>>(R, M, N, transpose_R, out);
  g_launches++;
  return check_launch("rot_apply_kernel");
}
