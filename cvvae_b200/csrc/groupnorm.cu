// GroupNorm(32) statistics + fused normalise/affine/SiLU, and the token LayerNorm of the temporal
// attention.  HBM-bound kernels: 128-bit loads/stores, ~8 CTAs per SM, statistics reduced thread (fp32) -> block
// (shared 64-bit fixed-point atomics) -> device (global 64-bit fixed-point atomics; order-independent, reproducible).
//
// Replaces Normalize()+nonlinearity (reference models/vae_models.py:187-195,392-401), nn.GroupNorm+nn.SiLU
// of models/vae_blocks3d_sd3.py, and norm_t (models/vae_models.py:571).  One rounding to 16 bit at the
// end instead of the reference's three (GN out, sigmoid, product).
#include "common.cuh"

namespace cvvae {

struct GnView {
  const void* x;
  void* y;
  int T, H, W, C;
  long long xs_b, xs_t, xs_h, xs_w;
  long long ys_b, ys_t, ys_h, ys_w;
  int x_dense, y_dense;  // pixel stride == C and rows/frames contiguous within a sample-unit
  int per_frame;
  long long pix_per_unit;   // T*H*W, or H*W when per_frame
  long long pix_per_block;
  int groups;
};

__device__ __forceinline__ long long gn_offset(long long pix, int unit_t, int per_frame, int H, int W, long long s_t,
                                               long long s_h, long long s_w, int dense, int C) {
  // pix indexes positions inside one statistics unit (a sample, or a frame when per_frame)
  if (dense) return (per_frame ? unit_t * s_t : 0) + pix * C;
  const int w = static_cast<int>(pix % W);
  const long long r = pix / W;
  const int h = static_cast<int>(r % H);
  const int t = per_frame ? unit_t : static_cast<int>(r / H);
  return t * s_t + h * s_h + w * s_w;
}

template <int DT>
__global__ void __launch_bounds__(256) gn_stats_kernel(const GnView v, unsigned long long* __restrict__ stats) {
  using E = Elem<DT>;
  __shared__ unsigned long long s_sum[64];
  __shared__ unsigned long long s_sq[64];
  const int unit = blockIdx.y;  // b or b*T+t
  const int b = v.per_frame ? unit / v.T : unit;
  const int ut = v.per_frame ? unit % v.T : 0;
  const int vecs = v.C >> 3;          // 16-byte vectors per position
  const int lanes = 256 / vecs;       // positions per sweep
  const int vec = threadIdx.x % vecs;
  const int pl = threadIdx.x / vecs;
  const int cpg = v.C / v.groups;
  if (threadIdx.x < 64) {
    s_sum[threadIdx.x] = 0ull;
    s_sq[threadIdx.x] = 0ull;
  }
  __syncthreads();
  const long long p0 = static_cast<long long>(blockIdx.x) * v.pix_per_block;
  long long p1 = p0 + v.pix_per_block;
  if (p1 > v.pix_per_unit) p1 = v.pix_per_unit;
  const typename E::T* xb = reinterpret_cast<const typename E::T*>(v.x) + b * v.xs_b;
  float s[8], q[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) s[j] = q[j] = 0.f;
  if (pl < lanes) {
    // 4 independent 128-bit loads in flight per thread (HBM latency x bandwidth needs ~35 KB in flight per SM)
    constexpr int U = 4;
    long long p = p0 + pl;
    for (; p + static_cast<long long>(U - 1) * lanes < p1; p += static_cast<long long>(U) * lanes) {
      uint4 u[U];
#pragma unroll
      for (int i = 0; i < U; ++i) {
        const long long off = gn_offset(p + static_cast<long long>(i) * lanes, ut, v.per_frame, v.H, v.W, v.xs_t, v.xs_h,
                                        v.xs_w, v.x_dense, v.C);
        u[i] = __ldg(reinterpret_cast<const uint4*>(xb + off + vec * 8));
      }
#pragma unroll
      for (int i = 0; i < U; ++i) {
        const uint32_t uw[4] = {u[i].x, u[i].y, u[i].z, u[i].w};
#pragma unroll
        for (int j = 0; j < 4; ++j) {
          const float2 f = E::to_f2(uw[j]);
          s[2 * j] += f.x;
          q[2 * j] = fmaf(f.x, f.x, q[2 * j]);
          s[2 * j + 1] += f.y;
          q[2 * j + 1] = fmaf(f.y, f.y, q[2 * j + 1]);
        }
      }
    }
    for (; p < p1; p += lanes) {
      const long long off = gn_offset(p, ut, v.per_frame, v.H, v.W, v.xs_t, v.xs_h, v.xs_w, v.x_dense, v.C);
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(xb + off + vec * 8));
      const uint32_t uw[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 f = E::to_f2(uw[j]);
        s[2 * j] += f.x;
        q[2 * j] = fmaf(f.x, f.x, q[2 * j]);
        s[2 * j + 1] += f.y;
        q[2 * j + 1] = fmaf(f.y, f.y, q[2 * j + 1]);
      }
    }
    // fold the 8 channels of this thread into their group(s)
    if (cpg >= 8) {
      float ts = 0.f, tq = 0.f;
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        ts += s[j];
        tq += q[j];
      }
      const int g = (vec * 8) / cpg;
      atomicAdd(&s_sum[g], gn_fix(ts, kGnSumScale));
      atomicAdd(&s_sq[g], gn_fix(tq, kGnSqScale));
    } else {
      for (int j0 = 0; j0 < 8; j0 += cpg) {
        float ts = 0.f, tq = 0.f;
        for (int j = j0; j < j0 + cpg; ++j) {
          ts += s[j];
          tq += q[j];
        }
        const int g = (vec * 8 + j0) / cpg;
        atomicAdd(&s_sum[g], gn_fix(ts, kGnSumScale));
        atomicAdd(&s_sq[g], gn_fix(tq, kGnSqScale));
      }
    }
  }
  __syncthreads();
  if (threadIdx.x < v.groups) {
    unsigned long long* o = stats + (static_cast<long long>(unit) * v.groups + threadIdx.x) * 2;
    atomicAdd(o, s_sum[threadIdx.x]);
    atomicAdd(o + 1, s_sq[threadIdx.x]);
  }
}

__device__ __forceinline__ uint4 ld_stream(const void* p) {
  uint4 r;
  asm volatile("ld.global.nc.L1::no_allocate.v4.u32 {%0,%1,%2,%3}, [%4];"
               : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
  return r;
}
__device__ __forceinline__ void st_stream(void* p, const uint4& v) {
  asm volatile("st.global.cs.v4.u32 [%0], {%1,%2,%3,%4};" ::"l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

template <int DT, int U, int HINT>
__global__ void __launch_bounds__(256) gn_apply_kernel(const GnView v, const long long* __restrict__ stats,
                                                       const float* __restrict__ gamma, const float* __restrict__ beta,
                                                       float eps, int silu) {
  using E = Elem<DT>;
  extern __shared__ float s_ab[];  // [C] scale, [C] shift
  float* s_a = s_ab;
  float* s_b = s_ab + v.C;
  const int unit = blockIdx.y;
  const int b = v.per_frame ? unit / v.T : unit;
  const int ut = v.per_frame ? unit % v.T : 0;
  const int cpg = v.C / v.groups;
  const double cnt = static_cast<double>(v.pix_per_unit) * cpg;
  for (int c = threadIdx.x; c < v.C; c += blockDim.x) {
    const int g = c / cpg;
    const double sum = static_cast<double>(stats[(static_cast<long long>(unit) * v.groups + g) * 2]) / kGnSumScale;
    const double sq = static_cast<double>(stats[(static_cast<long long>(unit) * v.groups + g) * 2 + 1]) / kGnSqScale;
    const double mean = sum / cnt;
    double var = sq / cnt - mean * mean;
    if (var < 0.0) var = 0.0;
    const float rstd = static_cast<float>(1.0 / sqrt(var + static_cast<double>(eps)));
    const float a = rstd * gamma[c];
    s_a[c] = a;
    s_b[c] = beta[c] - static_cast<float>(mean) * a;
  }
  __syncthreads();
  const int vecs = v.C >> 3;
  const int lanes = 256 / vecs;
  const int vec = threadIdx.x % vecs;
  const int pl = threadIdx.x / vecs;
  if (pl >= lanes) return;
  float a[8], sh[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) {
    a[j] = s_a[vec * 8 + j];
    sh[j] = s_b[vec * 8 + j];
  }
  const long long p0 = static_cast<long long>(blockIdx.x) * v.pix_per_block;
  long long p1 = p0 + v.pix_per_block;
  if (p1 > v.pix_per_unit) p1 = v.pix_per_unit;
  const typename E::T* xb = reinterpret_cast<const typename E::T*>(v.x) + b * v.xs_b;
  typename E::T* yb = reinterpret_cast<typename E::T*>(v.y) + b * v.ys_b;
  auto transform = [&](const uint4& u) {
    const uint32_t uw[4] = {u.x, u.y, u.z, u.w};
    uint32_t ow[4];
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const float2 f = E::to_f2(uw[j]);
      float r0 = fmaf(f.x, a[2 * j], sh[2 * j]);
      float r1 = fmaf(f.y, a[2 * j + 1], sh[2 * j + 1]);
      if (silu) {
        r0 = silu_f(r0);
        r1 = silu_f(r1);
      }
      ow[j] = E::pack2(r0, r1);
    }
    return make_uint4(ow[0], ow[1], ow[2], ow[3]);
  };
  long long p = p0 + pl;   // U independent 128-bit loads in flight per thread
  for (; p + static_cast<long long>(U - 1) * lanes < p1; p += static_cast<long long>(U) * lanes) {
    uint4 u[U];
    long long yo[U];
#pragma unroll
    for (int i = 0; i < U; ++i) {
      const long long pp = p + static_cast<long long>(i) * lanes;
      const long long xo = gn_offset(pp, ut, v.per_frame, v.H, v.W, v.xs_t, v.xs_h, v.xs_w, v.x_dense, v.C);
      yo[i] = gn_offset(pp, ut, v.per_frame, v.H, v.W, v.ys_t, v.ys_h, v.ys_w, v.y_dense, v.C);
      u[i] = HINT ? ld_stream(xb + xo + vec * 8) : __ldg(reinterpret_cast<const uint4*>(xb + xo + vec * 8));
    }
#pragma unroll
    for (int i = 0; i < U; ++i) {
      if (HINT) st_stream(yb + yo[i] + vec * 8, transform(u[i]));
      else *reinterpret_cast<uint4*>(yb + yo[i] + vec * 8) = transform(u[i]);
    }
  }
  for (; p < p1; p += lanes) {
    const long long xo = gn_offset(p, ut, v.per_frame, v.H, v.W, v.xs_t, v.xs_h, v.xs_w, v.x_dense, v.C);
    const long long yo = gn_offset(p, ut, v.per_frame, v.H, v.W, v.ys_t, v.ys_h, v.ys_w, v.y_dense, v.C);
    *reinterpret_cast<uint4*>(yb + yo + vec * 8) = transform(__ldg(reinterpret_cast<const uint4*>(xb + xo + vec * 8)));
  }
}

static int fill_view(GnView& v, const cvvae_tensor5* x, const cvvae_tensor5* y, int groups, int per_frame) {
  CVVAE_CHECK_ARG(x->s_c == 1 && x->C % 8 == 0, "groupnorm: needs channels-last input with C %% 8 == 0 (C=%d s_c=%lld)", x->C,
                  (long long)x->s_c);
  const int vecs = x->C / 8;
  CVVAE_CHECK_ARG(vecs <= 256 && (256 % vecs) == 0, "groupnorm: C/8 = %d must divide 256", vecs);
  CVVAE_CHECK_ARG(groups > 0 && groups <= 64 && x->C % groups == 0, "groupnorm: bad group count %d for C=%d", groups, x->C);
  const int cpg = x->C / groups;
  CVVAE_CHECK_ARG(cpg >= 8 ? (cpg % 8 == 0) : (8 % cpg == 0), "groupnorm: channels per group %d unsupported", cpg);
  CVVAE_CHECK_ARG((x->s_w % 8 == 0) && (x->s_h % 8 == 0) && (x->s_t % 8 == 0) && (x->s_b % 8 == 0) &&
                      reinterpret_cast<uintptr_t>(x->ptr) % 16 == 0,
                  "groupnorm: input not 16-byte aligned");
  v.x = x->ptr;
  v.T = x->T; v.H = x->H; v.W = x->W; v.C = x->C;
  v.xs_b = x->s_b; v.xs_t = x->s_t; v.xs_h = x->s_h; v.xs_w = x->s_w;
  v.x_dense = (x->s_w == x->C) && (x->s_h == 1ll * x->W * x->C) && (per_frame || x->s_t == 1ll * x->H * x->W * x->C);
  v.per_frame = per_frame ? 1 : 0;
  v.groups = groups;
  v.pix_per_unit = per_frame ? 1ll * x->H * x->W : 1ll * x->T * x->H * x->W;
  if (y) {
    CVVAE_CHECK_ARG(y->s_c == 1 && y->C == x->C && y->B == x->B && y->T == x->T && y->H == x->H && y->W == x->W,
                    "groupnorm: output shape mismatch");
    CVVAE_CHECK_ARG((y->s_w % 8 == 0) && (y->s_h % 8 == 0) && (y->s_t % 8 == 0) && (y->s_b % 8 == 0) &&
                        reinterpret_cast<uintptr_t>(y->ptr) % 16 == 0,
                    "groupnorm: output not 16-byte aligned");
    v.y = y->ptr;
    v.ys_b = y->s_b; v.ys_t = y->s_t; v.ys_h = y->s_h; v.ys_w = y->s_w;
    v.y_dense = (y->s_w == y->C) && (y->s_h == 1ll * y->W * y->C) && (per_frame || y->s_t == 1ll * y->H * y->W * y->C);
  }
  return CVVAE_OK;
}

static void pick_grid(GnView& v, int units, dim3& grid) {
  // Positions per CTA depend on the per-unit extent ONLY (not on the batch size, not on the SM count of the device): the
  // fp32 per-thread partial sums of gn_stats_kernel group the same way whether a clip runs alone, in a tile batch or on
  // another GPU, so tile batching and sharding stay bit-identical at any size.  ~1184 CTAs per unit (8 per SM of a
  // 148-SM part), at least 256 positions each.
  constexpr long long kBlocksPerUnit = 1184;
  long long ppb = (v.pix_per_unit + kBlocksPerUnit - 1) / kBlocksPerUnit;
  if (ppb < 256) ppb = 256;
  v.pix_per_block = ppb;
  grid = dim3(static_cast<unsigned>((v.pix_per_unit + ppb - 1) / ppb), static_cast<unsigned>(units));
}

// --------------------------------------------------------------------------- LayerNorm over C per token
template <int DT>
__global__ void __launch_bounds__(256) layernorm_kernel(const GnView v, long long tokens, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, float eps, int B) {
  using E = Elem<DT>;
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const long long tok = static_cast<long long>(blockIdx.x) * 8 + warp;
  if (tok >= tokens) return;
  const long long per_b = 1ll * v.T * v.H * v.W;
  const int b = static_cast<int>(tok / per_b);
  const long long pix = tok % per_b;
  const long long xo = b * v.xs_b + gn_offset(pix, 0, 0, v.H, v.W, v.xs_t, v.xs_h, v.xs_w, v.x_dense, v.C);
  const long long yo = b * v.ys_b + gn_offset(pix, 0, 0, v.H, v.W, v.ys_t, v.ys_h, v.ys_w, v.y_dense, v.C);
  const typename E::T* xp = reinterpret_cast<const typename E::T*>(v.x) + xo;
  typename E::T* yp = reinterpret_cast<typename E::T*>(v.y) + yo;
  const int vecs = v.C >> 3;
  constexpr int MAXV = 4;  // C <= 1024
  float f[MAXV][8];
  float sum = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int vi = lane + i * 32;
    if (vi < vecs) {
      const uint4 u = __ldg(reinterpret_cast<const uint4*>(xp + vi * 8));
      const uint32_t uw[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const float2 t2 = E::to_f2(uw[j]);
        f[i][2 * j] = t2.x;
        f[i][2 * j + 1] = t2.y;
        sum += t2.x + t2.y;
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, o);
  const float mean = sum / v.C;
  float sq = 0.f;
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int vi = lane + i * 32;
    if (vi < vecs) {
#pragma unroll
      for (int j = 0; j < 8; ++j) {
        const float d = f[i][j] - mean;
        sq = fmaf(d, d, sq);
      }
    }
  }
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) sq += __shfl_xor_sync(0xffffffffu, sq, o);
  const float rstd = rsqrtf(sq / v.C + eps);
#pragma unroll
  for (int i = 0; i < MAXV; ++i) {
    const int vi = lane + i * 32;
    if (vi < vecs) {
      uint32_t ow[4];
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        const int c = vi * 8 + 2 * j;
        const float r0 = (f[i][2 * j] - mean) * rstd * __ldg(gamma + c) + __ldg(beta + c);
        const float r1 = (f[i][2 * j + 1] - mean) * rstd * __ldg(gamma + c + 1) + __ldg(beta + c + 1);
        ow[j] = E::pack2(r0, r1);
      }
      *reinterpret_cast<uint4*>(yp + vi * 8) = make_uint4(ow[0], ow[1], ow[2], ow[3]);
    }
  }
}

}  // namespace cvvae

using namespace cvvae;

namespace cvvae {
int gn_stats_run(const cvvae_tensor5* x, int32_t groups, int32_t per_frame, int64_t* stats, int32_t dtype,
                 cudaStream_t stream, bool zero_first);
}

extern "C" int cvvae_groupnorm_stats(const cvvae_tensor5* x, int32_t groups, int32_t per_frame, int64_t* stats,
                                     int32_t dtype, void* stream_) {
  CVVAE_CHECK_ARG(tensor_ok(x) && stats, "cvvae_groupnorm_stats: null argument");
  return cvvae::gn_stats_run(x, groups, per_frame, stats, dtype, static_cast<cudaStream_t>(stream_), true);
}

int cvvae::gn_stats_run(const cvvae_tensor5* x, int32_t groups, int32_t per_frame, int64_t* stats, int32_t dtype,
                        cudaStream_t stream, bool zero_first) {
  GnView v{};
  int rc = fill_view(v, x, nullptr, groups, per_frame);
  if (rc) return rc;
  const int units = per_frame ? x->B * x->T : x->B;
  if (zero_first) CVVAE_CUDA(cudaMemsetAsync(stats, 0, sizeof(double) * 2 * groups * units, stream));
  dim3 grid;
  pick_grid(v, units, grid);
  CVVAE_DISPATCH_DTYPE(dtype, { gn_stats_kernel<DT><<<grid, 256, 0, stream>>>(v, reinterpret_cast<unsigned long long*>(stats)); });
  CVVAE_LAUNCH_CHECK();
  return CVVAE_OK;
}

extern "C" int cvvae_groupnorm_apply(const cvvae_tensor5* x, const cvvae_tensor5* y, int32_t groups, int32_t per_frame,
                                     const int64_t* stats, const float* gamma, const float* beta, float eps, int32_t silu,
                                     int32_t dtype, void* stream_) {
  CVVAE_CHECK_ARG(tensor_ok(x) && tensor_ok(y) && stats && gamma && beta, "cvvae_groupnorm_apply: null argument");
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  GnView v{};
  int rc = fill_view(v, x, y, groups, per_frame);
  if (rc) return rc;
  const int units = per_frame ? x->B * x->T : x->B;
  dim3 grid;
  pick_grid(v, units, grid);
  const size_t smem = sizeof(float) * 2 * x->C;
  const long long* st = reinterpret_cast<const long long*>(stats);
  // 4 loads in flight per thread + streaming (no-allocate / evict-first) accesses: 5.7 TB/s on 1.4 GB tensors, 87 % of the
  // measured copy bandwidth (U = 8 or fewer CTAs per SM measured slower, plain ld/st 4 % slower)
  CVVAE_DISPATCH_DTYPE(dtype, { gn_apply_kernel<DT, 4, 1><<<grid, 256, smem, stream>>>(v, st, gamma, beta, eps, silu); });
  CVVAE_LAUNCH_CHECK();
  return CVVAE_OK;
}

extern "C" int cvvae_layernorm(const cvvae_tensor5* x, const cvvae_tensor5* y, const float* gamma, const float* beta,
                               float eps, int32_t dtype, void* stream_) {
  CVVAE_CHECK_ARG(tensor_ok(x) && tensor_ok(y) && gamma && beta, "cvvae_layernorm: null argument");
  CVVAE_CHECK_ARG(x->C <= 1024, "cvvae_layernorm: C=%d > 1024 unsupported", x->C);
  cudaStream_t stream = static_cast<cudaStream_t>(stream_);
  GnView v{};
  int rc = fill_view(v, x, y, 1, 0);
  if (rc) return rc;
  const long long tokens = 1ll * x->B * x->T * x->H * x->W;
  const long long blocks = (tokens + 7) / 8;
  CVVAE_CHECK_ARG(blocks < (1ll << 31), "cvvae_layernorm: too many tokens");
  CVVAE_DISPATCH_DTYPE(dtype, {
    layernorm_kernel<DT><<<static_cast<unsigned>(blocks), 256, 0, stream>>>(v, tokens, gamma, beta, eps, x->B);
  });
  CVVAE_LAUNCH_CHECK();
  return CVVAE_OK;
}
