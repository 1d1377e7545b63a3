// Shared definitions for libhands_b200.so (sm_100a only).
#pragma once
#include <cuda_runtime.h>
#include <stdint.h>
#include <atomic>
#include "../../include/hands_b200.h"

namespace hb {

constexpr int NV = HB_NUM_VERTS;   // 778 vertices
constexpr int NJ = HB_NUM_JOINTS;  // 16 kinematic joints
constexpr int NOJ = HB_NUM_OUT_JOINTS;  // 21 output joints (16 + 5 finger tips)
constexpr int NB = HB_NUM_BETAS;   // 10 shape coefficients
constexpr int NPF = 135;           // pose-feature length (15 joints x 9)
constexpr int NP = NPF + NB;       // 145 rows of the stacked blendshape basis [posedirs; shapedirs^T]
constexpr int FS = 152;            // feature row stride (NP padded to a multiple of 8)
constexpr int AS = 192;            // 16 joints x (3x4) skinning transforms per hand

// Vertex-slice geometry of the skinning kernels: 5 CTAs x 160 threads cover 778 (800 padded) vertices.
constexpr int VPB = 160;
constexpr int NSLICE = 5;
constexpr int VP = VPB * NSLICE;   // 800
constexpr int HBF = 16;            // hands per skinning group (the A / OFF workspace regions are laid out by it)

// MANO constants, device-resident, re-laid-out for coalesced access (built by hb_mano_create).
struct ManoConst {
  const float* Vt;    // [3][VP]       v_template transposed
  const float* Wt;    // [16][VP]      lbs_weights transposed
  const float* Wv;    // [VP][16]      lbs_weights, vertex-major, zero-padded
  const float* Jt;    // [16][3]       J_regressor @ v_template           (fp64 fold)
  const float* Jsd;   // [16][3][10]   J_regressor @ shapedirs            (fp64 fold)
  const float* pose_mean;  // [48]
  const float* Bhi;   // [10 tiles][19 k-steps][240 x 8] TF32 high parts of the stacked basis, UMMA slab order (mano_tc.cu)
  const float* Blo;   // same, low parts
  const float* Ph;    // [300 k-steps][160 x 8] TF32 high parts of the basis for the backward reduction over vertex coordinates
  const float* Pl;    // same, low parts
  int parents[NJ];
  int level[NJ];       // depth of each joint in the kinematic tree (root = 0)
  int child[NJ][5];    // child joints, -1 padded
  int depth;           // max level
  int tips[5];
};

extern std::atomic<uint64_t> g_launches;
void set_error(const char* fmt, ...);
int check_launch(const char* what);

#define HB_CUDA(call)                                                     \
  do {                                                                    \
    cudaError_t _e = (call);                                              \
    if (_e != cudaSuccess) {                                              \
      hb::set_error("%s failed: %s", #call, cudaGetErrorString(_e));      \
      return (int)_e;                                                     \
    }                                                                     \
  } while (0)

// TF32 split used by the tensor-core path: hi = x rounded to 10 mantissa bits, lo = (x - hi) rounded likewise
__host__ __device__ inline float tf32_round(float x) {
  union { float f; uint32_t u; } c;
  c.f = x;
  c.u = (c.u + 0x1000u) & 0xFFFFE000u;
  return c.f;
}

size_t tc_smem_bytes();
int launch_blend_tc(const float* Fhi, const float* Flo, const float* Bhi, const float* Blo, const float* vt, int B, float* vp, cudaStream_t st);
constexpr int G_MAXSPLIT = 4;   // split-K parts of the backward feature contraction (partials [part][B128][160] in the workspace)
int gfeat_nsplit(int B);
int launch_gfeat_tc(const float* gvh, const float* gvl, const float* Ph, const float* Pl, int B, float* gF, cudaStream_t st);

static inline bool aligned8(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 7u) == 0; }

}  // namespace hb

struct hb_mano {
  hb::ManoConst c;
  int device;
  void* blob;  // one device allocation holding every array above
};
