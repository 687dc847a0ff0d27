// a3: camera-ray generation + stratified coarse samples  (keras_nerf/data/rays.py:69-130)
// HBM-write-bound: 24 + 4*N bytes per ray out (+ 4*N in when the uniforms are supplied).
// Random ray batches over all training views (knerf_generate_ray_batch): the same per-ray arithmetic, plus the target
// rgb, 24 + 4*N + 12 bytes out and one scattered 16-byte read per ray.
// Forward-facing scenes (knerf_generate_rays_ndc, knerf_generate_ray_batch_ndc): the same kernels instantiated with
// NDC = true map each world ray into normalized device coordinates (ndc_map) and scale its depths; same traffic.
#include "common.cuh"

namespace knerf {

struct Pose {
  float r[3][3];
  float t[3];
};

// rays.py:89-109: unit direction of pixel (x, y) under `pose` -- no pixel-centre offset; cam = (xc, -yc, -1).
// Shared by rays_kernel and ray_batch_kernel: the same pixel gives the same bits in both.
__device__ __forceinline__ void camera_direction(const Pose& pose, uint32_t x, uint32_t y, float Wf, float Hf,
                                                 float focal, float (&out)[3]) {
  const float xc = __fdiv_rn(__fsub_rn((float)x, Wf * 0.5f), focal);
  const float yc = __fdiv_rn(__fsub_rn((float)y, Hf * 0.5f), focal);
  float dir[3];
#pragma unroll
  for (int i = 0; i < 3; ++i) {
    // rays.py:103-107: broadcast multiply then reduce_sum over j = 0,1,2 (products rounded separately)
    const float p0 = __fmul_rn(xc, pose.r[i][0]);
    const float p1 = __fmul_rn(-yc, pose.r[i][1]);
    const float p2 = __fmul_rn(-1.0f, pose.r[i][2]);
    dir[i] = __fadd_rn(__fadd_rn(p0, p1), p2);
  }
  const float nrm = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(dir[0], dir[0]), __fmul_rn(dir[1], dir[1])),
                                         __fmul_rn(dir[2], dir[2])));
#pragma unroll
  for (int i = 0; i < 3; ++i) out[i] = __fdiv_rn(dir[i], nrm);   // rays.py:108-109
}

// Stratified coarse depths of one warp's rays [base, base + n) (rays.py:116-127): the warp walks their n * N samples
// in units of VEC (4 = one 16-byte store), consecutive lanes on consecutive addresses of t.  Sample k of ray r uses
// u[r * N + k], or Philox(seed) at that counter.
struct Strata {
  float near_, far_, delta, interval, half_iv;
  int N;
  __device__ __forceinline__ Strata(float near_in, float far_in, int n) : near_(near_in), far_(far_in), N(n) {
    delta = __fdiv_rn(__fsub_rn(far_, near_), (float)(N - 1));   // tf.linspace step
    interval = __fdiv_rn(__fsub_rn(far_, near_), (float)N);       // rays.py:120 (N, not N-1)
    half_iv = interval * 0.5f;
  }
};

// NDC: sample k of ray r is written as scale[r] * s_k (scale = the warp's 32 NDC direction norms, in shared memory).
template <int VEC, bool NDC = false>
__device__ __forceinline__ void stream_samples(const Strata& s, uint32_t base, uint32_t n, uint32_t lane,
                                               const float* __restrict__ u, uint64_t seed, float* __restrict__ t,
                                               const float* scale = nullptr) {
  const int N = s.N;
  const uint32_t per_ray = (uint32_t)(N / VEC);
  const uint32_t units = n * per_ray;
  for (uint32_t unit = lane; unit < units; unit += 32) {
    const uint32_t r = unit / per_ray;
    const int s0 = (int)(unit - r * per_ray) * VEC;
    const int64_t ray = (int64_t)base + r;
    float uu[VEC];
    const int64_t e0 = ray * N + s0;
    if (u != nullptr) {
      if (VEC == 4) {
        const float4 v = ld_stream4(reinterpret_cast<const float4*>(u + e0));
        uu[0] = v.x; uu[1 % VEC] = v.y; uu[2 % VEC] = v.z; uu[3 % VEC] = v.w;
      } else {
        uu[0] = ld_stream(u + e0);
      }
    } else {
      if (VEC == 4) {
        uint32_t rr[4];
        philox4x32(seed, (uint64_t)e0 >> 2, rr);   // e0 % 4 == 0
#pragma unroll
        for (int k = 0; k < VEC; ++k) uu[k] = u01(rr[k]);
      } else {
        uu[0] = philox_uniform(seed, (uint64_t)e0);
      }
    }
    float out[VEC];
#pragma unroll
    for (int k = 0; k < VEC; ++k) {
      const int i = s0 + k;
      // tf.linspace: exact end points, start + delta*i in between (rays.py:116-117)
      float lin = __fadd_rn(s.near_, __fmul_rn(s.delta, (float)i));
      if (i == N - 1) lin = s.far_;
      if (i == 0) lin = s.near_;
      const float noise = __fsub_rn(__fmul_rn(uu[k], s.interval), s.half_iv);   // rays.py:122-123
      out[k] = fminf(fmaxf(__fadd_rn(lin, noise), s.near_), s.far_);            // rays.py:126-127
    }
    if (NDC) {
      const float sc = scale[r];
#pragma unroll
      for (int k = 0; k < VEC; ++k) out[k] = __fmul_rn(sc, out[k]);
    }
    if (VEC == 4) {
      *reinterpret_cast<float4*>(t + e0) = make_float4(out[0], out[1 % VEC], out[2 % VEC], out[3 % VEC]);
    } else {
      t[e0] = out[0];
    }
  }
}

// Vanilla NeRF's ndc_rays(H, W, focal, near = 1, o, w) for a ray of origin o and direction w (w_z < 0): shift o to the
// plane z = -1, o' = o + tau*w with tau = -(1 + o_z)/w_z, then
//   o_ndc = (sx*o'_x/o'_z, sy*o'_y/o'_z, 1 + 2/o'_z),  d_ndc = (sx*(w_x/w_z - o'_x/o'_z), sy*(w_y/w_z - o'_y/o'_z), -2/o'_z)
// with sx = -2f/W, sy = -2f/H.  Writes o_ndc and d_ndc/|d_ndc| and returns |d_ndc|.  Every operation is rounded on its
// own (no contraction) in this order; tests/test_gpu_llff.py restates it in NumPy fp32 bit for bit.
struct NdcMap {
  float sx, sy;
  __device__ __forceinline__ NdcMap(float focal, float Wf, float Hf) {
    sx = __fdiv_rn(-2.0f * focal, Wf);
    sy = __fdiv_rn(-2.0f * focal, Hf);
  }
  __device__ __forceinline__ float operator()(const float (&o)[3], const float (&w)[3], float (&o_ndc)[3],
                                              float (&d_ndc)[3]) const {
    const float tau = __fdiv_rn(-__fadd_rn(1.0f, o[2]), w[2]);
    float op[3];
#pragma unroll
    for (int i = 0; i < 3; ++i) op[i] = __fadd_rn(o[i], __fmul_rn(tau, w[i]));
    const float rx = __fdiv_rn(op[0], op[2]), ry = __fdiv_rn(op[1], op[2]);
    const float q = __fdiv_rn(2.0f, op[2]);
    o_ndc[0] = __fmul_rn(sx, rx);
    o_ndc[1] = __fmul_rn(sy, ry);
    o_ndc[2] = __fadd_rn(1.0f, q);
    float dn[3];
    dn[0] = __fmul_rn(sx, __fsub_rn(__fdiv_rn(w[0], w[2]), rx));
    dn[1] = __fmul_rn(sy, __fsub_rn(__fdiv_rn(w[1], w[2]), ry));
    dn[2] = -q;
    const float nrm = __fsqrt_rn(__fadd_rn(__fadd_rn(__fmul_rn(dn[0], dn[0]), __fmul_rn(dn[1], dn[1])),
                                           __fmul_rn(dn[2], dn[2])));
#pragma unroll
    for (int i = 0; i < 3; ++i) d_ndc[i] = __fdiv_rn(dn[i], nrm);
    return nrm;
  }
};

// One warp per 32 consecutive rays.  Phase 1: lane l computes origin and direction of ray base + l (every lane busy:
// the two divisions, the normalisation and its three divisions cost the warp one pass per 32 rays instead of one per
// ray).  Phase 2: stream_samples.  Index arithmetic is 32-bit.
// NDC (near_ = 0, far_ = 1): phase 1 writes the NDC ray and keeps |d_ndc| in the warp's slot of shared memory, which
// phase 2 reads for the depth scale (no shuffles in its divergent loop).
template <int VEC, bool NDC>
__global__ void __launch_bounds__(256) rays_kernel(Pose pose, int H, int W, float focal, float near_,
                                                   float far_, int N, const float* __restrict__ u,
                                                   uint64_t seed, float* __restrict__ o,
                                                   float* __restrict__ d, float* __restrict__ t) {
  const uint32_t n_rays = (uint32_t)H * (uint32_t)W;
  const float Wf = (float)W, Hf = (float)H;
  const Strata strata(near_, far_, N);
  __shared__ float ndc_norm[NDC ? 256 : 1];
  const NdcMap ndc(focal, Wf, Hf);
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t base = warp * 32; base < n_rays; base += n_warps * 32) {
    const uint32_t ray = base + lane;
    if (ray < n_rays) {
      const uint32_t y = ray / (uint32_t)W, x = ray - y * (uint32_t)W;
      float dir[3];
      camera_direction(pose, x, y, Wf, Hf, focal, dir);
      if constexpr (NDC) {
        float on[3], dn[3];
        ndc_norm[threadIdx.x] = ndc(pose.t, dir, on, dn);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          d[(size_t)ray * 3 + i] = dn[i];
          o[(size_t)ray * 3 + i] = on[i];
        }
      } else {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          d[(size_t)ray * 3 + i] = dir[i];
          o[(size_t)ray * 3 + i] = pose.t[i];                // rays.py:112-113
        }
      }
    }
    if constexpr (NDC) {
      __syncwarp();
      stream_samples<VEC, true>(strata, base, min(32u, n_rays - base), lane, u, seed, t,
                                ndc_norm + (threadIdx.x & ~31u));
      __syncwarp();                                          // the slot is rewritten by the next pass
    } else {
      stream_samples<VEC>(strata, base, min(32u, n_rays - base), lane, u, seed, t);
    }
  }
}

// ---- random ray batches over all training views (knerf_generate_ray_batch) --------------------------------------
// Epoch permutation of [0, P): a balanced Feistel network on b bits (b the smallest even width >= 2 with 2^b >= P),
// 4 rounds, cycle-walked until the value is < P.  Round function: the splitmix64 finaliser of (half ^ round key),
// round key r = mix64(mix64(perm_seed) ^ (epoch * G + C)) + r * G.  tests/ray_batch_oracle.py restates it.
__host__ __device__ __forceinline__ uint64_t mix64(uint64_t z) {
  z ^= z >> 30; z *= 0xBF58476D1CE4E5B9ull;
  z ^= z >> 27; z *= 0x94D049BB133111EBull;
  return z ^ (z >> 31);
}

constexpr uint64_t kGolden64 = 0x9E3779B97F4A7C15ull;
constexpr int kFeistelRounds = 4;

struct EpochPerm {
  uint64_t P, key;
  uint32_t half;   // bits per Feistel half
  uint64_t mask;
  __device__ __forceinline__ uint64_t round_trip(uint64_t v) const {
    uint64_t L = v >> half, R = v & mask;
#pragma unroll
    for (int r = 0; r < kFeistelRounds; ++r) {
      const uint64_t F = mix64(R ^ (key + (uint64_t)r * kGolden64)) & mask;
      const uint64_t nl = R;
      R = L ^ F;
      L = nl;
    }
    return (L << half) | R;
  }
  __device__ __forceinline__ uint64_t operator()(uint64_t i) const {   // i < P
    uint64_t v = round_trip(i);
    while (v >= P) v = round_trip(v);   // cycle walk: ends, the cycle through i returns below P
    return v;
  }
};

// One warp per 32 consecutive batch rays.  Phase 1: lane l finds the pixel of ray base + l, reads its pose and its
// rgb (one scattered 16-byte load when C == 4) and writes o, d, target (and pixel).  Phase 2: stream_samples with
// batch-local counters, exactly as rays_kernel (NDC as there).
template <int VEC, bool NDC>
__global__ void __launch_bounds__(256) ray_batch_kernel(const float* __restrict__ images, int H, int W, int C,
                                                        bool rgba16, const float* __restrict__ c2w, float focal,
                                                        float near_, float far_, int N, EpochPerm perm,
                                                        int64_t first, uint32_t n_rays, const float* __restrict__ u,
                                                        uint64_t seed, float* __restrict__ o, float* __restrict__ d,
                                                        float* __restrict__ t, float* __restrict__ target,
                                                        int64_t* __restrict__ pixel) {
  const uint64_t HW = (uint64_t)H * (uint64_t)W;
  const float Wf = (float)W, Hf = (float)H;
  const Strata strata(near_, far_, N);
  __shared__ float ndc_norm[NDC ? 256 : 1];
  const NdcMap ndc(focal, Wf, Hf);
  const uint32_t lane = threadIdx.x & 31;
  const uint32_t warp = (blockIdx.x * blockDim.x + threadIdx.x) >> 5, n_warps = (gridDim.x * blockDim.x) >> 5;
  for (uint32_t base = warp * 32; base < n_rays; base += n_warps * 32) {
    const uint32_t ray = base + lane;
    if (ray < n_rays) {
      const uint64_t p = perm((uint64_t)first + ray);
      const uint64_t img = p / HW;
      const uint32_t in_img = (uint32_t)(p - img * HW);
      const uint32_t y = in_img / (uint32_t)W, x = in_img - y * (uint32_t)W;
      const float* m = c2w + img * 16;
      Pose pose;
#pragma unroll
      for (int i = 0; i < 3; ++i) {
#pragma unroll
        for (int j = 0; j < 3; ++j) pose.r[i][j] = __ldg(m + i * 4 + j);
        pose.t[i] = __ldg(m + i * 4 + 3);
      }
      float dir[3];
      camera_direction(pose, x, y, Wf, Hf, focal, dir);
      const float* px = images + p * (uint64_t)C;
      float rgb[3];
      if (rgba16) {
        const float4 v = __ldg(reinterpret_cast<const float4*>(px));
        rgb[0] = v.x; rgb[1] = v.y; rgb[2] = v.z;
      } else {
#pragma unroll
        for (int i = 0; i < 3; ++i) rgb[i] = __ldg(px + i);
      }
      if constexpr (NDC) {
        float on[3], dn[3];
        ndc_norm[threadIdx.x] = ndc(pose.t, dir, on, dn);
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          d[(size_t)ray * 3 + i] = dn[i];
          o[(size_t)ray * 3 + i] = on[i];
          target[(size_t)ray * 3 + i] = rgb[i];
        }
      } else {
#pragma unroll
        for (int i = 0; i < 3; ++i) {
          d[(size_t)ray * 3 + i] = dir[i];
          o[(size_t)ray * 3 + i] = pose.t[i];
          target[(size_t)ray * 3 + i] = rgb[i];
        }
      }
      if (pixel != nullptr) pixel[ray] = (int64_t)p;
    }
    if constexpr (NDC) {
      __syncwarp();
      stream_samples<VEC, true>(strata, base, min(32u, n_rays - base), lane, u, seed, t,
                                ndc_norm + (threadIdx.x & ~31u));
      __syncwarp();
    } else {
      stream_samples<VEC>(strata, base, min(32u, n_rays - base), lane, u, seed, t);
    }
  }
}

__global__ void __launch_bounds__(256) uniform_kernel(float* __restrict__ out, int64_t n, uint64_t seed,
                                                      uint64_t offset) {
  const int64_t n4 = (n + 3) / 4;
  for (int64_t g = blockIdx.x * (int64_t)blockDim.x + threadIdx.x; g < n4;
       g += (int64_t)gridDim.x * blockDim.x) {
    uint32_t r[4];
    philox4x32(seed, offset + (uint64_t)g, r);
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const int64_t e = g * 4 + k;
      if (e < n) out[e] = u01(r[k]);
    }
  }
}

}  // namespace knerf

using namespace knerf;

namespace {

// The argument checks and launch of knerf_generate_rays and knerf_generate_rays_ndc (`fn` names the entry point in the
// messages); the NDC instantiation stratifies [0, 1] and scales each ray's depths by |d_ndc| in the kernel.
template <bool NDC>
int launch_rays(const char* fn, const float* c2w_host, int H, int W, float focal, float near_, float far_,
                int n_samples, const float* u, uint64_t seed, float* o, float* d, float* t, void* stream) {
  KN_CHECK_ARG(c2w_host && o && d && t, "%s: null pointer", fn);
  KN_CHECK_ARG(H > 0 && W > 0 && n_samples > 0 && focal > 0.f, "%s: bad shape H=%d W=%d N=%d focal=%g", fn, H, W,
               n_samples, (double)focal);
  Pose p;
  for (int i = 0; i < 3; ++i) {
    for (int j = 0; j < 3; ++j) p.r[i][j] = c2w_host[i * 4 + j];   // rays.py:99
    p.t[i] = c2w_host[i * 4 + 3];                                  // rays.py:100
  }
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = (n_samples % 4 == 0) && ((reinterpret_cast<uintptr_t>(t) & 15) == 0) &&
                   (u == nullptr || (reinterpret_cast<uintptr_t>(u) & 15) == 0);
  KN_CHECK_ARG((int64_t)H * W < (int64_t)1 << 31 && (int64_t)n_samples * 32 < (int64_t)1 << 31,
               "%s: image too large (%d x %d)", fn, H, W);
  const int grid = (int)std::min<int64_t>(cdiv((int64_t)H * W, 256), (int64_t)kNumSMs * 16);
  if (vec)
    rays_kernel<4, NDC><<<grid, 256, 0, st>>>(p, H, W, focal, near_, far_, n_samples, u, seed, o, d, t);
  else
    rays_kernel<1, NDC><<<grid, 256, 0, st>>>(p, H, W, focal, near_, far_, n_samples, u, seed, o, d, t);
  KN_LAUNCH_CHECK();
  return KNERF_OK;
}

template <bool NDC>
int launch_ray_batch(const char* fn, const float* images, int n_img, int H, int W, int C, const float* c2w,
                     float focal, float near_, float far_, int n_samples, uint64_t perm_seed, uint64_t epoch,
                     int64_t first, int64_t R, const float* u, uint64_t seed, float* o, float* d, float* t,
                     float* target, int64_t* pixel, void* stream) {
  KN_CHECK_ARG(images && c2w && o && d && t && target, "%s: null pointer", fn);
  KN_CHECK_ARG(n_img > 0 && H > 0 && W > 0 && n_samples > 0 && focal > 0.f,
               "%s: bad shape n_img=%d H=%d W=%d N=%d focal=%g", fn, n_img, H, W, n_samples, (double)focal);
  KN_CHECK_ARG(C >= 3, "%s: C=%d channels, need >= 3", fn, C);
  KN_CHECK_ARG((int64_t)H * W < (int64_t)1 << 31 && (int64_t)n_samples * 32 < (int64_t)1 << 31,
               "%s: image too large (%d x %d)", fn, H, W);
  const int64_t P = (int64_t)n_img * H * W;
  KN_CHECK_ARG(first >= 0 && R >= 0 && first <= P - R, "%s: window [%lld, %lld + %lld) outside [0, %lld)", fn,
               (long long)first, (long long)first, (long long)R, (long long)P);
  KN_CHECK_ARG(R < (int64_t)1 << 31, "%s: R=%lld rays per call, need < 2^31", fn, (long long)R);
  if (R == 0) return KNERF_OK;
  EpochPerm perm;
  perm.P = (uint64_t)P;
  perm.key = mix64(mix64(perm_seed) ^ (epoch * kGolden64 + 0xD1B54A32D192ED03ull));
  int bits = 2;
  while (bits < 62 && ((uint64_t)1 << bits) < (uint64_t)P) bits += 2;
  perm.half = (uint32_t)(bits / 2);
  perm.mask = ((uint64_t)1 << perm.half) - 1;
  cudaStream_t st = (cudaStream_t)stream;
  const bool vec = (n_samples % 4 == 0) && ((reinterpret_cast<uintptr_t>(t) & 15) == 0) &&
                   (u == nullptr || (reinterpret_cast<uintptr_t>(u) & 15) == 0);
  const bool rgba16 = C == 4 && (reinterpret_cast<uintptr_t>(images) & 15) == 0;
  const int grid = (int)std::min<int64_t>(cdiv(R, 256), (int64_t)kNumSMs * 16);
  if (vec)
    ray_batch_kernel<4, NDC><<<grid, 256, 0, st>>>(images, H, W, C, rgba16, c2w, focal, near_, far_, n_samples,
                                                   perm, first, (uint32_t)R, u, seed, o, d, t, target, pixel);
  else
    ray_batch_kernel<1, NDC><<<grid, 256, 0, st>>>(images, H, W, C, rgba16, c2w, focal, near_, far_, n_samples,
                                                   perm, first, (uint32_t)R, u, seed, o, d, t, target, pixel);
  KN_LAUNCH_CHECK();
  return KNERF_OK;
}

}  // namespace

extern "C" int knerf_generate_rays(const float* c2w_host, int H, int W, float focal, float near_,
                                   float far_, int n_samples, const float* u, uint64_t seed, float* o,
                                   float* d, float* t, void* stream) {
  return launch_rays<false>("knerf_generate_rays", c2w_host, H, W, focal, near_, far_, n_samples, u, seed, o, d, t,
                            stream);
}

extern "C" int knerf_generate_rays_ndc(const float* c2w_host, int H, int W, float focal, int n_samples,
                                       const float* u, uint64_t seed, float* o, float* d, float* t, void* stream) {
  return launch_rays<true>("knerf_generate_rays_ndc", c2w_host, H, W, focal, 0.0f, 1.0f, n_samples, u, seed, o, d,
                           t, stream);
}

extern "C" int knerf_generate_ray_batch(const float* images, int n_img, int H, int W, int C, const float* c2w,
                                        float focal, float near_, float far_, int n_samples, uint64_t perm_seed,
                                        uint64_t epoch, int64_t first, int64_t R, const float* u, uint64_t seed,
                                        float* o, float* d, float* t, float* target, int64_t* pixel, void* stream) {
  return launch_ray_batch<false>("knerf_generate_ray_batch", images, n_img, H, W, C, c2w, focal, near_, far_,
                                 n_samples, perm_seed, epoch, first, R, u, seed, o, d, t, target, pixel, stream);
}

extern "C" int knerf_generate_ray_batch_ndc(const float* images, int n_img, int H, int W, int C, const float* c2w,
                                            float focal, int n_samples, uint64_t perm_seed, uint64_t epoch,
                                            int64_t first, int64_t R, const float* u, uint64_t seed, float* o,
                                            float* d, float* t, float* target, int64_t* pixel, void* stream) {
  return launch_ray_batch<true>("knerf_generate_ray_batch_ndc", images, n_img, H, W, C, c2w, focal, 0.0f, 1.0f,
                                n_samples, perm_seed, epoch, first, R, u, seed, o, d, t, target, pixel, stream);
}

extern "C" int knerf_uniform(float* out, int64_t n, uint64_t seed, uint64_t offset, void* stream) {
  KN_CHECK_ARG(out && n >= 0, "knerf_uniform: bad arguments");
  if (n == 0) return KNERF_OK;
  const int grid = (int)std::min<int64_t>(cdiv(cdiv(n, 4), 256), (int64_t)kNumSMs * 16);
  uniform_kernel<<<grid, 256, 0, (cudaStream_t)stream>>>(out, n, seed, offset);
  KN_LAUNCH_CHECK();
  return KNERF_OK;
}
