// Word augmentation for handwriting-recognition training (the recogniser's input: NHWC with C = 1, fp32, h = 32).
// Nothing in the reference: this is the classic HTR augmentation of the paper's HTR experiments (random affine warp of each
// word plus thin / thick strokes), as a kernel that draws no random numbers -- the caller passes them (sg_random), so a
// launch is deterministic, capturable in a CUDA graph and testable with chosen parameters.
//
// Row b of u [n, 7] (U[-1, 1)) maps linearly to the word's parameters:
//   theta = u0 * rot_deg (degrees), k = u1 * shear (x += k * y), sx = 1 + u2 * scale, sy = 1 + u3 * scale,
//   tx = u4 * translate_px, ty = u5 * translate_px, morphology: 3x3 grey minimum if u6 < -1 + 2 p_morph, 3x3 grey maximum if
//   u6 > 1 - 2 p_morph, none otherwise.
// Forward map about the word's centre c = (W_b / 2, h / 2):  dst = c + t + Rot(theta) Shear(k) Scale(sx, sy) (src - c).
// Output pixel (x, y), x < W_b, samples src bilinearly at the inverse map, coordinates clamped to [0, W_b - 1] x [0, h - 1]
// (border replicate: word images have background at their border, so no background value or ink polarity is assumed);
// the optional min / max runs over the warped image's 3x3 neighbourhood inside the word.  Columns >= W_b are copied bit for
// bit, so a ragged batch stays ragged.  With all ranges zero the output equals the input bit for bit.
#include <math.h>

#include "common.cuh"

#define AUG_THREADS 256

struct aug_map {
  float m00, m01, m10, m11;    // inverse of Rot(theta) Shear(k) Scale(sx, sy)
  float tx, ty;
  int morph;                   // -1 minimum, +1 maximum, 0 none
};

__device__ __forceinline__ aug_map aug_params(const float* __restrict__ u, float rot_turns, float shear, float scale, float translate_px,
                                              float p_morph) {
  aug_map p;
  float s, a;
  sincospif(__ldg(u + 0) * rot_turns, &s, &a);      // theta in half turns: exact argument reduction, no local-memory slow path
  const float k = __ldg(u + 1) * shear;
  const float sx = 1.f + __ldg(u + 2) * scale, sy = 1.f + __ldg(u + 3) * scale;
  // Scale^-1 Shear^-1 Rot^-1 = diag(1/sx, 1/sy) [[1, -k], [0, 1]] [[a, s], [-s, a]]
  p.m00 = (a + k * s) / sx;
  p.m01 = (s - k * a) / sx;
  p.m10 = -s / sy;
  p.m11 = a / sy;
  p.tx = __ldg(u + 4) * translate_px;
  p.ty = __ldg(u + 5) * translate_px;
  const float u6 = __ldg(u + 6);
  p.morph = u6 < -1.f + 2.f * p_morph ? -1 : (u6 > 1.f - 2.f * p_morph ? 1 : 0);
  return p;
}

// the warped word at output pixel (x, y) of a word of wb columns: bilinear, border replicate.  Identity parameters give
// exactly (x, y) with zero fractions, i.e. the source pixel itself.
__device__ __forceinline__ float aug_warp(const float* __restrict__ img, int w, int h, int wb, float cx, float cy, const aug_map& p,
                                          int x, int y) {
  const float dx = ((float)x - cx) - p.tx, dy = ((float)y - cy) - p.ty;
  float sx = cx + (p.m00 * dx + p.m01 * dy);
  float sy = cy + (p.m10 * dx + p.m11 * dy);
  sx = fminf(fmaxf(sx, 0.f), (float)(wb - 1));
  sy = fminf(fmaxf(sy, 0.f), (float)(h - 1));
  const float fx = floorf(sx), fy = floorf(sy);
  const int x0 = (int)fx, y0 = (int)fy;
  const int x1 = min(x0 + 1, wb - 1), y1 = min(y0 + 1, h - 1);
  const float ax = sx - fx, ay = sy - fy;
  const float* r0 = img + (long long)y0 * w;
  const float* r1 = img + (long long)y1 * w;
  const float p00 = __ldg(r0 + x0), p01 = __ldg(r0 + x1), p10 = __ldg(r1 + x0), p11 = __ldg(r1 + x1);
  const float top = p00 + ax * (p01 - p00);
  const float bot = p10 + ax * (p11 - p10);
  return top + ay * (bot - top);
}

// one thread per output pixel; a sample's parameters are recomputed per thread (a few dozen instructions against a
// bilinear gather: the kernel is bound by memory and the gathers, not by this arithmetic)
__global__ void __launch_bounds__(AUG_THREADS) k_word_augment(const float* __restrict__ src, float* __restrict__ dst, int n, int h, int w,
                                                              const int* __restrict__ widths, const float* __restrict__ u, float rot_turns,
                                                              float shear, float scale, float translate_px, float p_morph) {
  const long long hw = (long long)h * w, total = (long long)n * hw;
  for (long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int b = (int)(i / hw);
    const int r = (int)(i - (long long)b * hw);
    const int y = r / w, x = r - y * w;
    const int wb = widths ? __ldg(widths + b) : w;
    if (wb < 1 || wb > w) {                   // a width the host could not check (device memory): never a plausible image
      dst[i] = __int_as_float(0x7fffffff);
      continue;
    }
    if (x >= wb) {                            // right of the word: untouched
      dst[i] = __ldg(src + i);
      continue;
    }
    const aug_map p = aug_params(u + 7LL * b, rot_turns, shear, scale, translate_px, p_morph);
    const float* img = src + (long long)b * hw;
    const float cx = 0.5f * (float)wb, cy = 0.5f * (float)h;
    float v = aug_warp(img, w, h, wb, cx, cy, p, x, y);
    if (p.morph != 0) {
      // neighbours outside the word are left out (equivalent to replicating its border)
      for (int yy = max(y - 1, 0); yy <= min(y + 1, h - 1); ++yy)
        for (int xx = max(x - 1, 0); xx <= min(x + 1, wb - 1); ++xx) {
          if (xx == x && yy == y) continue;
          const float q = aug_warp(img, w, h, wb, cx, cy, p, xx, yy);
          v = p.morph < 0 ? fminf(v, q) : fmaxf(v, q);
        }
    }
    dst[i] = v;
  }
}

static bool aug_range_ok(float v) { return isfinite(v) && v >= 0.f; }

extern "C" int sg_word_augment(sg_ctx* ctx, const float* src, float* dst, int n, int h, int w, const int* widths, const float* u,
                               float rot_deg, float shear, float scale, float translate_px, float p_morph) {
  SG_REQUIRE(ctx, "sg_word_augment: NULL context");
  SG_REQUIRE(n >= 0, "sg_word_augment: n = %d < 0", n);
  SG_REQUIRE(h == 32, "sg_word_augment: h = %d; word images have 32 rows", h);
  SG_REQUIRE(w >= 1, "sg_word_augment: w = %d < 1", w);
  SG_REQUIRE(aug_range_ok(rot_deg) && aug_range_ok(shear) && aug_range_ok(translate_px),
             "sg_word_augment: ranges must be finite and >= 0 (rotation %g, shear %g, translate %g)", rot_deg, shear, translate_px);
  SG_REQUIRE(aug_range_ok(scale) && scale < 1.f, "sg_word_augment: scale %g outside [0, 1)", scale);
  SG_REQUIRE(isfinite(p_morph) && p_morph >= 0.f && p_morph <= 0.5f, "sg_word_augment: p_morph %g outside [0, 0.5]", p_morph);
  if (n == 0) return SG_OK;
  SG_REQUIRE(src && dst && u, "sg_word_augment: NULL src, dst or u");
  const long long total = (long long)n * h * w;
  const char *s0 = (const char*)src, *s1 = (const char*)(src + total), *d0 = (const char*)dst, *d1 = (const char*)(dst + total);
  SG_REQUIRE(d1 <= s0 || s1 <= d0, "sg_word_augment: dst overlaps src (the warp reads neighbours: it runs out of place)");
  const float rot_turns = (float)((double)rot_deg / 180.0);
  long long blocks = (total + AUG_THREADS - 1) / AUG_THREADS;
  const long long cap = (long long)ctx->num_sms * 16;
  if (blocks > cap) blocks = cap;
  sg_launch(ctx, k_word_augment, (unsigned int)blocks, AUG_THREADS, 0, src, dst, n, h, w, widths, u, rot_turns, shear, scale,
            translate_px, p_morph);
  SG_POST_LAUNCH(ctx);
  return SG_OK;
}
