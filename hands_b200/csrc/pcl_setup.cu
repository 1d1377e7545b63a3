// Perspective Crop Layer, step 1: the float64 homography (hands_light_dataset.py:357-386, 425-454).
// Compiled with -fmad=false so the device evaluates the same un-fused float64 operations as the
// reference's numpy code on the host (the result is cast to fp32; a fused multiply-add in float64 can
// flip the last fp32 bit of P or R).
#include "hb_common.cuh"

namespace hb {

constexpr int PF = HB_PCL_PARAM_FLOATS;

// ---- 3x3 helpers in float64 -------------------------------------------------------------------
__host__ __device__ inline void inv3(const double* m, double* o) {
  const double a = m[0], b = m[1], c = m[2], d = m[3], e = m[4], f = m[5], g = m[6], h = m[7], i = m[8];
  const double A = e * i - f * h, Bc = -(d * i - f * g), Cc = d * h - e * g;
  const double det = a * A + b * Bc + c * Cc;
  const double id = 1.0 / det;
  o[0] = A * id; o[1] = -(b * i - c * h) * id; o[2] = (b * f - c * e) * id;
  o[3] = Bc * id; o[4] = (a * i - c * g) * id; o[5] = -(a * f - c * d) * id;
  o[6] = Cc * id; o[7] = -(a * h - b * g) * id; o[8] = (a * e - b * d) * id;
}
__host__ __device__ inline void mul3(const double* a, const double* b, double* o) {
  for (int r = 0; r < 3; ++r)
    for (int c = 0; c < 3; ++c) o[r * 3 + c] = a[r * 3 + 0] * b[c] + a[r * 3 + 1] * b[3 + c] + a[r * 3 + 2] * b[6 + c];
}

// hands_light_dataset.py:357-386, 425-454 for one crop, float64.  Returns s.
__host__ __device__ inline int pcl_homography64(const int32_t* bb, const float* Kf, int img_res, double* P, double* Rv) {
  double K[9], Ki[9];
  for (int k = 0; k < 9; ++k) K[k] = (double)Kf[k];
  inv3(K, Ki);
  const double cx = (double)(bb[0] + bb[2]) / 2.0, cy = (double)(bb[1] + bb[3]) / 2.0;
  const int w = bb[2] - bb[0], h = bb[3] - bb[1];
  int s = w > h ? w : h;
  if (s <= 0) s = img_res;   // empty box -> whole image (hands_light_dataset.py:450-454); an inverted box (the reference raises in
                             // linspace; the Python wrapper rejects it) is treated the same so the kernels stay in bounds
  const double p0 = Ki[0] * cx + Ki[1] * cy + Ki[2], p1 = Ki[3] * cx + Ki[4] * cy + Ki[5], p2 = Ki[6] * cx + Ki[7] * cy + Ki[8];
  const double x = p0, y = p1;
  const double n1x = sqrt(1.0 + x * x), d1x = 1.0 / n1x;
  const double d1xy = 1.0 / sqrt(1.0 + x * x + y * y);
  const double d1xy1x = 1.0 / sqrt((1.0 + x * x + y * y) * (1.0 + x * x));
  Rv[0] = d1x;      Rv[1] = -x * y * d1xy1x; Rv[2] = x * d1xy;
  Rv[3] = 0.0 * x;  Rv[4] = n1x * d1xy;      Rv[5] = y * d1xy;
  Rv[6] = -x * d1x; Rv[7] = -y * d1xy1x;     Rv[8] = 1.0 * d1xy;
  const double plen = sqrt(p0 * p0 + p1 * p1 + p2 * p2);
  const double sx = 1.0 / sqrt(p0 * p0 + p2 * p2);
  const double sy = sqrt(p0 * p0 + 1.0) / sqrt(p0 * p0 + p1 * p1 + 1.0);
  double Kv[9] = {0, 0, 0.5, 0, 0, 0.5, 0, 0, 1.0};
  Kv[0] = plen * K[0] / ((double)s * sx);
  Kv[4] = plen * K[4] / ((double)s * sy);
  double Kvi[9], T[9];
  inv3(Kv, Kvi);
  mul3(Rv, Kvi, T);
  mul3(K, T, P);
  return s;
}

__global__ void pcl_setup_kernel(const int32_t* __restrict__ bbox, const float* __restrict__ K, int n, int img_res,
                                 float* __restrict__ params, float* __restrict__ Rout) {
  const int q = blockIdx.x * blockDim.x + threadIdx.x;
  if (q >= n) return;
  double P[9], Rv[9];
  int32_t bb[4];
  float Kf[9];
#pragma unroll
  for (int k = 0; k < 4; ++k) bb[k] = bbox[(size_t)q * 4 + k];
#pragma unroll
  for (int k = 0; k < 9; ++k) Kf[k] = K[(size_t)q * 9 + k];
  const int s = pcl_homography64(bb, Kf, img_res, P, Rv);
  float* rec = params + (size_t)q * PF;
  double Pf[9], Pi[9];
#pragma unroll
  for (int k = 0; k < 9; ++k) { rec[k] = (float)P[k]; Pf[k] = (double)rec[k]; }
  inv3(Pf, Pi);
#pragma unroll
  for (int k = 0; k < 9; ++k) rec[9 + k] = (float)Pi[k];
  rec[18] = __int_as_float(s);
  rec[19] = img_res > 1 ? __fdiv_rn((float)(s - 1), (float)(img_res - 1)) : 0.0f;
  rec[20] = s > 1 ? __fdiv_rn(1.0f, (float)(s - 1)) : 0.0f;
  rec[21] = __int_as_float(0);
  // source-pixel bounding box of the crop's bilinear footprint (corners of the unit square under P; a
  // homography maps the square to a convex quad, so the corner box bounds it) -- used to cull source tiles
  int fx0 = 0, fx1 = img_res - 1, fy0 = 0, fy1 = img_res - 1;
  {
    double xmin = 1e30, xmax = -1e30, ymin = 1e30, ymax = -1e30;
    bool ok = true;
    for (int cy = 0; cy < 2; ++cy)
      for (int cx = 0; cx < 2; ++cx) {
        const double X = Pf[0] * cx + Pf[1] * cy + Pf[2], Y = Pf[3] * cx + Pf[4] * cy + Pf[5], Z = Pf[6] * cx + Pf[7] * cy + Pf[8];
        if (!(Z > 1e-9)) { ok = false; continue; }
        const double ix = X / Z - 0.5, iy = Y / Z - 0.5;
        xmin = fmin(xmin, ix); xmax = fmax(xmax, ix); ymin = fmin(ymin, iy); ymax = fmax(ymax, iy);
      }
    if (ok) {
      xmin = fmax(xmin - 1.5, -4.0); ymin = fmax(ymin - 1.5, -4.0);
      xmax = fmin(xmax + 2.5, (double)img_res + 4.0); ymax = fmin(ymax + 2.5, (double)img_res + 4.0);
      fx0 = (int)floor(xmin); fx1 = (int)ceil(xmax); fy0 = (int)floor(ymin); fy1 = (int)ceil(ymax);
    }
  }
  rec[22] = __int_as_float(fx0); rec[23] = __int_as_float(fx1); rec[24] = __int_as_float(fy0); rec[25] = __int_as_float(fy1);
#pragma unroll
  for (int k = 26; k < PF; ++k) rec[k] = 0.0f;
  if (Rout) {
#pragma unroll
    for (int k = 0; k < 9; ++k) Rout[(size_t)q * 9 + k] = (float)Rv[k];
  }
}

}  // namespace hb

using namespace hb;

extern "C" int hb_pcl_setup(const int32_t* bbox, const float* K, int n_crops, int img_res, float* params, float* R_virt2orig, void* stream) {
  if (n_crops < 0 || img_res <= 0 || (n_crops > 0 && (!bbox || !K || !params))) { set_error("hb_pcl_setup: bad argument"); return HB_E_ARG; }
  if (n_crops == 0) return 0;
  pcl_setup_kernel<<<(n_crops + 127) / 128, 128, 0, (cudaStream_t)stream>>>(bbox, K, n_crops, img_res, params, R_virt2orig);
  g_launches++;
  return check_launch("pcl_setup_kernel");
}

extern "C" int hb_pcl_homography_host(const int32_t* bbox_host, const float* K_host, int img_res, float* P_host, float* R_host, int32_t* s_host) {
  if (!bbox_host || !K_host || !P_host || !R_host || !s_host || img_res <= 0) { set_error("hb_pcl_homography_host: bad argument"); return HB_E_ARG; }
  double P[9], Rv[9];
  *s_host = pcl_homography64(bbox_host, K_host, img_res, P, Rv);
  for (int k = 0; k < 9; ++k) { P_host[k] = (float)P[k]; R_host[k] = (float)Rv[k]; }
  return 0;
}

