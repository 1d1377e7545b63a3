// Library plumbing: error string, launch counter, MANO constant upload.
#include <cstdarg>
#include <cstdio>
#include <cstring>
#include <vector>
#include "hb_common.cuh"

namespace hb {

std::atomic<uint64_t> g_launches{0};
static thread_local char g_err[512] = "";

void set_error(const char* fmt, ...) {
  va_list ap;
  va_start(ap, fmt);
  vsnprintf(g_err, sizeof(g_err), fmt, ap);
  va_end(ap);
}

int check_launch(const char* what) {
  cudaError_t e = cudaGetLastError();
  if (e != cudaSuccess) {
    set_error("%s launch failed: %s", what, cudaGetErrorString(e));
    return (int)e;
  }
  return 0;
}

}  // namespace hb

using namespace hb;

extern "C" const char* hb_last_error_string(void) { return g_err; }
extern "C" int hb_version(void) { return HB_VERSION; }
extern "C" uint64_t hb_launch_count(void) { return g_launches.load(); }

extern "C" int hb_mano_create(const float* v_template, const float* shapedirs, const float* posedirs, const float* J_regressor,
                              const float* lbs_weights, const int32_t* parents, const float* pose_mean, const int32_t* tip_ids,
                              int device, hb_mano** out) {
  if (!v_template || !shapedirs || !posedirs || !J_regressor || !lbs_weights || !parents || !pose_mean || !tip_ids || !out) {
    set_error("hb_mano_create: NULL argument");
    return HB_E_ARG;
  }
  // kinematic tree: parents must precede children; at most 5 children per joint
  ManoConst c;
  memset(&c, 0, sizeof(c));
  for (int i = 0; i < NJ; ++i)
    for (int k = 0; k < 5; ++k) c.child[i][k] = -1;
  int nchild[NJ] = {0};
  c.depth = 0;
  for (int i = 0; i < NJ; ++i) {
    c.parents[i] = parents[i];
    if (i == 0) { c.level[0] = 0; continue; }
    const int p = parents[i];
    if (p < 0 || p >= i) { set_error("hb_mano_create: parents[%d]=%d must be in [0,%d)", i, p, i); return HB_E_ARG; }
    if (nchild[p] >= 5) { set_error("hb_mano_create: joint %d has more than 5 children", p); return HB_E_UNSUPPORTED; }
    c.child[p][nchild[p]++] = i;
    c.level[i] = c.level[p] + 1;
    if (c.level[i] > c.depth) c.depth = c.level[i];
  }
  for (int k = 0; k < 5; ++k) {
    if (tip_ids[k] < 0 || tip_ids[k] >= NV) { set_error("hb_mano_create: tip id %d out of range", tip_ids[k]); return HB_E_ARG; }
    c.tips[k] = tip_ids[k];
  }
  // host-side re-layout
  const size_t nVt = (size_t)3 * VP, nWt = (size_t)NJ * VP, nWv = (size_t)VP * NJ;
  const size_t nJt = NJ * 3, nJsd = NJ * 3 * NB, nPm = 48;
  const size_t nB = (size_t)10 * 19 * 240 * 8;   // tensor-core operand slabs
  const size_t nPs = (size_t)300 * 160 * 8;
  size_t off = 0;
  auto take = [&](size_t n) { size_t o = off; off += (n + 3) / 4 * 4; return o; };  // keep 16-byte alignment
  const size_t oVt = take(nVt), oWt = take(nWt), oWv = take(nWv), oJt = take(nJt), oJsd = take(nJsd), oPm = take(nPm), oBh = take(nB), oBl = take(nB), oPh = take(nPs), oPl = take(nPs);
  std::vector<float> hostbuf(off, 0.0f);
  float* Vt = hostbuf.data() + oVt;
  float* Wt = hostbuf.data() + oWt; float* Wv = hostbuf.data() + oWv; float* Jt = hostbuf.data() + oJt;
  float* Jsd = hostbuf.data() + oJsd; float* Pm = hostbuf.data() + oPm;
  for (int v = 0; v < NV; ++v) {
    for (int k = 0; k < 3; ++k) Vt[(size_t)k * VP + v] = v_template[v * 3 + k];
    for (int j = 0; j < NJ; ++j) { Wt[(size_t)j * VP + v] = lbs_weights[v * NJ + j]; Wv[(size_t)v * NJ + j] = lbs_weights[v * NJ + j]; }
  }
  for (int j = 0; j < NJ; ++j)
    for (int k = 0; k < 3; ++k) {
      double acc = 0.0;
      for (int v = 0; v < NV; ++v) acc += (double)J_regressor[(size_t)j * NV + v] * (double)v_template[v * 3 + k];
      Jt[j * 3 + k] = (float)acc;
      for (int l = 0; l < NB; ++l) {
        double a2 = 0.0;
        for (int v = 0; v < NV; ++v) a2 += (double)J_regressor[(size_t)j * NV + v] * (double)shapedirs[((size_t)v * 3 + k) * NB + l];
        Jsd[(j * 3 + k) * NB + l] = (float)a2;
      }
    }
  for (int k = 0; k < 48; ++k) Pm[k] = pose_mean[k];
  // stacked blendshape basis [posedirs; shapedirs^T]: row p < NP, coordinate k of vertex v < NV
  auto basis = [&](int p, int k, int v) {
    return p < NPF ? posedirs[(size_t)p * (NV * 3) + 3 * v + k] : shapedirs[((size_t)v * 3 + k) * NB + (p - NPF)];
  };
  // tensor-core B operand: column c' = k*800 + v (coordinate-major), tile = c'/240, UMMA K-major no-swizzle slabs
  // [tile][k-step][k-half][row-group][row][4]; split into TF32 hi/lo parts
  {
    float* Bh = hostbuf.data() + oBh;
    float* Bl = hostbuf.data() + oBl;
    for (int tile = 0; tile < 10; ++tile)
      for (int ks = 0; ks < 19; ++ks)
        for (int n = 0; n < 240; ++n)
          for (int kk = 0; kk < 8; ++kk) {
            const int cp = tile * 240 + n, pidx = ks * 8 + kk;
            const int k = cp / VP, v = cp % VP;
            const float val = (pidx < NP && v < NV) ? basis(pidx, k, v) : 0.0f;
            const float hi = tf32_round(val), lo = tf32_round(val - hi);
            const size_t o = ((size_t)tile * 19 + ks) * 1920 + (size_t)(kk >> 2) * 960 + (n >> 3) * 32 + (n & 7) * 4 + (kk & 3);
            Bh[o] = hi; Bl[o] = lo;
          }
    // backward reduction operand: rows = features p (160, zero above 144), K = c' (2400), slabs [k-step][k-half][row-group][row][4]
    float* Ph = hostbuf.data() + oPh;
    float* Pl = hostbuf.data() + oPl;
    for (int ks = 0; ks < 300; ++ks)
      for (int pidx = 0; pidx < 160; ++pidx)
        for (int kk = 0; kk < 8; ++kk) {
          const int cp = ks * 8 + kk;
          const int k = cp / VP, v = cp % VP;
          const float val = (pidx < NP && v < NV) ? basis(pidx, k, v) : 0.0f;
          const float hi = tf32_round(val), lo = tf32_round(val - hi);
          const size_t o = (size_t)ks * 1280 + (size_t)(kk >> 2) * 640 + (pidx >> 3) * 32 + (pidx & 7) * 4 + (kk & 3);
          Ph[o] = hi; Pl[o] = lo;
        }
  }

  int prev = -1;
  HB_CUDA(cudaGetDevice(&prev));
  HB_CUDA(cudaSetDevice(device));
  void* blob = nullptr;
  cudaError_t e = cudaMalloc(&blob, off * sizeof(float));
  if (e == cudaSuccess) e = cudaMemcpy(blob, hostbuf.data(), off * sizeof(float), cudaMemcpyHostToDevice);
  cudaSetDevice(prev);
  if (e != cudaSuccess) {
    if (blob) cudaFree(blob);
    set_error("hb_mano_create: device upload failed: %s", cudaGetErrorString(e));
    return (int)e;
  }
  const float* d = (const float*)blob;
  c.Vt = d + oVt; c.Wt = d + oWt; c.Wv = d + oWv; c.Jt = d + oJt; c.Jsd = d + oJsd; c.pose_mean = d + oPm; c.Bhi = d + oBh; c.Blo = d + oBl; c.Ph = d + oPh; c.Pl = d + oPl;
  hb_mano* hm = new hb_mano;
  hm->c = c; hm->device = device; hm->blob = blob;
  *out = hm;
  return 0;
}

extern "C" int hb_mano_destroy(hb_mano* h) {
  if (!h) return 0;
  int prev = -1;
  cudaGetDevice(&prev);
  cudaSetDevice(h->device);
  cudaFree(h->blob);
  cudaSetDevice(prev);
  delete h;
  return 0;
}
