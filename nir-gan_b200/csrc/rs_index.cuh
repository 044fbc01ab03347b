// The six indices of RemoteSensingIndices (utils/remote_sensing_indices.py:84-319) at one pixel, shared by the fused
// pixel losses and index maps of elementwise.cu and the index bands of the whole-scene blend (scene.cu), so that every
// kernel evaluates the same expressions.  t: target NIR, p: predicted NIR; R, G, Bl: the pixel's red, green, blue.
#pragma once

namespace ng {

struct RsPix {
  float it, ip, dip;     // index of the target, of the prediction, d(index of the prediction)/dpred
};
__device__ __forceinline__ RsPix rs_ndvi(float t, float p, float band, float eps) {
  const float dp = p + band + eps;
  return {(t - band) / (t + band + eps), (p - band) / dp, (2.f * band + eps) / (dp * dp)};
}
__device__ __forceinline__ RsPix rs_gndvi(float t, float p, float R, float G) {
  // (n - G) / (ndvi(n) + G) with ndvi(n) = (n - R) / (n + R), no epsilon (remote_sensing_indices.py:169-176)
  const float ndt = (t - R) / (t + R), ndp = (p - R) / (p + R);
  const float dnd = 2.f * R / ((p + R) * (p + R));
  const float den = ndp + G;
  return {(t - G) / (ndt + G), (p - G) / den, (den - (p - G) * dnd) / (den * den)};
}
__device__ __forceinline__ RsPix rs_savi(float t, float p, float R) {
  const float dp = p + R + 0.5f;
  return {1.5f * (t - R) / (t + R + 0.5f), 1.5f * (p - R) / dp, 1.5f * (2.f * R + 0.5f) / (dp * dp)};
}
__device__ __forceinline__ RsPix rs_msavi(float t, float p, float R) {
  const float st = sqrtf((2.f * t + 1.f) * (2.f * t + 1.f) - 8.f * (t - R));
  const float sp = sqrtf((2.f * p + 1.f) * (2.f * p + 1.f) - 8.f * (p - R));
  return {(2.f * t + 1.f - st) / 2.f, (2.f * p + 1.f - sp) / 2.f, 1.f - (2.f * p - 1.f) / sp};
}
__device__ __forceinline__ RsPix rs_evi(float t, float p, float R, float Bl, float eps) {
  const float k = (R - 7.5f) * (Bl + 1.f);
  const float dt = (t + 6.f) * k + eps, dp = (p + 6.f) * k + eps;
  return {2.5f * ((t - R) / dt), 2.5f * ((p - R) / dp), 2.5f * (k * (6.f + R) + eps) / (dp * dp)};
}

}  // namespace ng
