// Training tier (SURVEY §8(f) #1): value_and_grad of the photometric loss of
// training.py:171-212 (mean squared error of the coarse and the fine rgb,
// training.py:173) through NerfModel.__call__, in fp32.
//
// Unlike the fused forward kernels this path is layer-wise: the forward pass keeps a
// TAPE in HBM (every Dense layer's output, the encoded inputs, the sample points) and
// the backward pass walks it in reverse.  All kernels are hand-written fp32 SIMT:
//   * sgemm_kernel: one tiled GEMM template for the three shapes of a Dense layer
//       forward   Y  = act([X | IN] W + b)
//       backward  dX = dZ W^T         (dZ = dY * act'(Y), formed while loading)
//                 dW = [X | IN]^T dZ  (reduction over the rows: split + atomicAdd)
//   * colsum_kernel (bias gradients), encode / se3 / raw-activation kernels and their
//     adjoints, the adjoint of volumetric_rendering, embedding scatter-add, Adam.
// 180 GB of HBM holds the tape of a whole gpu_fullhd training batch (~31 GB); the
// caller may still process a batch in ray chunks (gradients accumulate).
// z_fine is a constant of the fine level (lax.stop_gradient, model_utils.py:211).
#pragma once
#include "common.cuh"
#include "nfb_handle.h"
#include "ray_kernels.cuh"

namespace nfb {
namespace train {

constexpr int kTile = 64;      // C tile (kTile x kTile), 256 threads, 4 x 4 per thread
constexpr int kBK = 16;

// activation derivative expressed through the OUTPUT y = act(z) (every registered
// activation is invertible enough for that: configs.py:27-32).
__device__ __forceinline__ float act_grad_from_output(float y, int act) {
  switch (act) {
    case kRelu: return y > 0.f ? 1.f : 0.f;
    case kElu: return y > 0.f ? 1.f : y + 1.f;
    case kLeakyRelu: return y >= 0.f ? 1.f : 0.01f;
    case kTanh: return 1.f - y * y;
    case kSigmoid: return y * (1.f - y);
    case kSoftplus: return 1.f - expf(-y);          // sigmoid(z) with y = log(1 + e^z)
    default: return 1.f;
  }
}

// ---------------------------------------------------------------------------
// One GEMM template.  C(m, n) (+)= sum_k A(m, k) * B(k, n) with element functors:
// slow address arithmetic, fast inner product (shared-memory tiles, 4x4 register
// tile).  gridDim.z splits the reduction (kSplitAtomic: results are atomicAdd-ed).
// ---------------------------------------------------------------------------
struct GemmShape { long long M; int N; long long K; };

template <class FA, class FB, class FC>
__global__ void __launch_bounds__(256)
sgemm_kernel(GemmShape sh, FA fa, FB fb, FC fc, long long k_per_split) {
  __shared__ float As[kBK][kTile + 4];
  __shared__ float Bs[kBK][kTile + 4];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const long long m0 = (long long)blockIdx.x * kTile;
  const int n0 = blockIdx.y * kTile;
  const long long k_begin = (long long)blockIdx.z * k_per_split;
  const long long k_end = min(sh.K, k_begin + k_per_split);
  float acc[4][4];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) acc[i][j] = 0.f;
  for (long long k0 = k_begin; k0 < k_end; k0 += kBK) {
    // A tile: kTile rows x kBK; B tile: kBK x kTile  (4 elements per thread each)
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int idx = tid + e * 256;
      {
        const int mm = idx / kBK, kk = idx % kBK;       // consecutive threads walk k: row-major A coalesces
        const long long m = m0 + mm, k = k0 + kk;
        As[kk][mm] = (m < sh.M && k < k_end) ? fa(m, k) : 0.f;
      }
      {
        const int kk = idx / kTile, nn = idx % kTile;   // consecutive threads walk n
        const long long k = k0 + kk;
        const int n = n0 + nn;
        Bs[kk][nn] = (k < k_end && n < sh.N) ? fb(k, n) : 0.f;
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < kBK; ++kk) {
      const float4 a4 = *reinterpret_cast<const float4*>(&As[kk][ty * 4]);
      const float4 b4 = *reinterpret_cast<const float4*>(&Bs[kk][tx * 4]);
      const float a[4] = {a4.x, a4.y, a4.z, a4.w}, b[4] = {b4.x, b4.y, b4.z, b4.w};
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const long long m = m0 + ty * 4 + i;
      const int n = n0 + tx * 4 + j;
      if (m < sh.M && n < sh.N) fc(m, n, acc[i][j]);
    }
}

// The same GEMM with a 128 x 128 C tile, an 8 x 8 register tile per thread (two 4 x 4 quadrant pairs, so that
// every shared-memory read is a 16-byte vector and the A reads are warp broadcasts), k-steps of 8 and a register
// prefetch of the next k-step's operands under the arithmetic of the current one (one __syncthreads per step).
// 64 FMAs per 4 LDS.128 instead of 16 per 2: the layer-wise training tier is GEMM-bound (3 x the forward FLOPs
// per step), and this template runs it about twice as fast as sgemm_kernel.
// kAKFast / kBNFast: which index of the element functor is contiguous in memory (k for a row-major A, n for a
// row-major B) - the loader walks that index with consecutive threads.
constexpr int kT2 = 128, kBK2 = 8, kPad2 = 4;
template <bool kAKFast, bool kBNFast, class FA, class FB, class FC>
__global__ void __launch_bounds__(256, 2)
sgemm128_kernel(GemmShape sh, FA fa, FB fb, FC fc, long long k_per_split) {
  __shared__ __align__(16) float As[2][kBK2][kT2 + kPad2];
  __shared__ __align__(16) float Bs[2][kBK2][kT2 + kPad2];
  const int tid = threadIdx.x;
  const int tx = tid & 15, ty = tid >> 4;
  const long long m0 = (long long)blockIdx.x * kT2;
  const int n0 = blockIdx.y * kT2;
  const long long k_begin = (long long)blockIdx.z * k_per_split;
  const long long k_end = min(sh.K, k_begin + k_per_split);
  float acc[8][8];
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) acc[i][j] = 0.f;
  float ra[4], rb[4];
  auto fetch = [&](long long k0) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int idx = tid + e * 256;
      {
        const int mm = kAKFast ? idx / kBK2 : idx % kT2, kk = kAKFast ? idx % kBK2 : idx / kT2;
        const long long m = m0 + mm, k = k0 + kk;
        ra[e] = (m < sh.M && k < k_end) ? fa(m, k) : 0.f;
      }
      {
        const int kk = kBNFast ? idx / kT2 : idx % kBK2, nn = kBNFast ? idx % kT2 : idx / kBK2;
        const long long k = k0 + kk;
        const int n = n0 + nn;
        rb[e] = (k < k_end && n < sh.N) ? fb(k, n) : 0.f;
      }
    }
  };
  auto stash = [&](int buf) {
#pragma unroll
    for (int e = 0; e < 4; ++e) {
      const int idx = tid + e * 256;
      As[buf][kAKFast ? idx % kBK2 : idx / kT2][kAKFast ? idx / kBK2 : idx % kT2] = ra[e];
      Bs[buf][kBNFast ? idx / kT2 : idx % kBK2][kBNFast ? idx % kT2 : idx / kBK2] = rb[e];
    }
  };
  int buf = 0;
  if (k_begin < k_end) {
    fetch(k_begin);
    stash(0);
  }
  __syncthreads();
  for (long long k0 = k_begin; k0 < k_end; k0 += kBK2) {
    const bool more = k0 + kBK2 < k_end;
    if (more) fetch(k0 + kBK2);                       // global loads in flight under the FMAs below
#pragma unroll
    for (int kk = 0; kk < kBK2; ++kk) {
      const float4 a0 = *reinterpret_cast<const float4*>(&As[buf][kk][ty * 4]);
      const float4 a1 = *reinterpret_cast<const float4*>(&As[buf][kk][64 + ty * 4]);
      const float4 b0 = *reinterpret_cast<const float4*>(&Bs[buf][kk][tx * 4]);
      const float4 b1 = *reinterpret_cast<const float4*>(&Bs[buf][kk][64 + tx * 4]);
      const float a[8] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y, a1.z, a1.w};
      const float b[8] = {b0.x, b0.y, b0.z, b0.w, b1.x, b1.y, b1.z, b1.w};
#pragma unroll
      for (int i = 0; i < 8; ++i)
#pragma unroll
        for (int j = 0; j < 8; ++j) acc[i][j] = fmaf(a[i], b[j], acc[i][j]);
    }
    if (more) {
      stash(buf ^ 1);                                 // the other buffer: its last readers passed the previous barrier
      __syncthreads();
      buf ^= 1;
    }
  }
#pragma unroll
  for (int i = 0; i < 8; ++i)
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      const long long m = m0 + (i < 4 ? ty * 4 + i : 64 + ty * 4 + (i - 4));
      const int n = n0 + (j < 4 ? tx * 4 + j : 64 + tx * 4 + (j - 4));
      if (m < sh.M && n < sh.N) fc(m, n, acc[i][j]);
    }
}

// [X (rows x k_x, ld ldx) | IN (rows x k_in, ld ldin, column offset folded into the pointer)]
struct ConcatA {
  const float* x; int ldx, k_x; const float* in; int ldin;
  __device__ float operator()(long long m, long long k) const {
    return k < k_x ? x[m * ldx + k] : in[m * ldin + (k - k_x)];
  }
};
struct ConcatAT {                  // transposed view for dW: A^T(k, row)
  ConcatA a;
  __device__ float operator()(long long k, long long m) const { return a(m, k); }
};
struct WeightB {                   // W (K x npad) row-major
  const float* w; int ld;
  __device__ float operator()(long long k, int n) const { return w[k * ld + n]; }
};
struct WeightBT {                  // W^T: (n, k) -> W[k][n]; "k" of the GEMM is the layer's n
  const float* w; int ld;
  __device__ float operator()(long long n, int k) const { return w[(long long)k * ld + n]; }
};
struct DZ {                        // dZ(m, n) = dY(m, n) * act'(Y(m, n))
  const float* dy; const float* y; int ld; int act;
  __device__ float operator()(long long m, long long n) const {
    return dy[m * ld + n] * act_grad_from_output(y[m * ld + n], act);
  }
};
struct DZB {                       // same as a B operand (k = row)
  DZ z;
  __device__ float operator()(long long m, int n) const { return z(m, n); }
};
struct StoreBiasAct {
  float* y; int ld; const float* bias; int act;
  __device__ void operator()(long long m, int n, float v) const { y[m * ld + n] = apply_act(v + bias[n], act); }
};
struct AccumSplit {                // dX / dIN: += into the producer's gradient buffer(s)
  float* dx; int ldx, k_x; float* din; int ldin;
  __device__ void operator()(long long m, int k, float v) const {
    if (k < k_x) dx[m * ldx + k] += v;
    else din[m * ldin + (k - k_x)] += v;
  }
};
struct AtomicAdd {
  float* c; int ld;
  __device__ void operator()(long long m, int n, float v) const { atomicAdd(c + m * ld + n, v); }
};

// db[n] += sum_m dZ(m, n)
__global__ void colsum_kernel(DZ z, long long rows, int n, float* __restrict__ db) {
  const int col = blockIdx.x * 32 + (threadIdx.x & 31);
  const int lane_row = threadIdx.x >> 5;              // 8 row lanes
  float s = 0.f;
  if (col < n)
    for (long long m = (long long)blockIdx.y * 8 + lane_row; m < rows; m += (long long)gridDim.y * 8) s += z(m, col);
  __shared__ float red[8][33];
  red[lane_row][threadIdx.x & 31] = s;
  __syncthreads();
  if (lane_row == 0 && col < n) {
    float t = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) t += red[i][threadIdx.x & 31];
    atomicAdd(db + col, t);
  }
}

// ---------------------------------------------------------------------------
// Encoded inputs (R3 / R6) and their adjoints.
// ---------------------------------------------------------------------------
struct EncodeArgs {
  const float* origins; const float* directions; const float* z;   // rays / (B,S) z; z null = free points
  const float* pts_in;        // (rows,3) points to encode instead of o + z d (the warped points), or null
  const float* cond;          // (B, cond_stride)
  const float* window;        // (F) or null
  float* pts_out;             // (rows,3) the encoded point (tape), or null
  float* in;                  // (rows, ld)
  int F, ld, S, cond_stride, cond_off, n_cond;     // cond[cond_off .. +n_cond) follows the encoding
  long long rows;
};
__global__ void encode_kernel(const EncodeArgs a) {
  const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= a.rows) return;
  const long long ray = m / a.S;
  float x[3];
  if (a.pts_in) {
#pragma unroll
    for (int c = 0; c < 3; ++c) x[c] = a.pts_in[m * 3 + c];
  } else {
    const float z = a.z ? a.z[m] : 0.f;
#pragma unroll
    for (int c = 0; c < 3; ++c) x[c] = a.origins[ray * 3 + c] + z * a.directions[ray * 3 + c];
  }
  if (a.pts_out) {
#pragma unroll
    for (int c = 0; c < 3; ++c) a.pts_out[m * 3 + c] = x[c];
  }
  float* o = a.in + m * a.ld;
#pragma unroll
  for (int c = 0; c < 3; ++c) o[c] = x[c];
  const int nf = 6 * a.F;
  for (int f = 0; f < nf; ++f) {
    float v = posenc_feature(x, f);
    if (a.window) v = a.window[f / 6] * v;
    o[3 + f] = v;
  }
  const float* c = a.cond + ray * a.cond_stride + a.cond_off;
  for (int q = 0; q < a.n_cond; ++q) o[3 + nf + q] = c[q];
  for (int q = 3 + nf + a.n_cond; q < a.ld; ++q) o[q] = 0.f;
}

// dIN -> dx (rows,3) (+= when accumulate) and per-ray dcond (atomicAdd over the ray's samples).
struct EncodeBwdArgs {
  const float* pts;           // (rows,3) the point that was encoded
  const float* window; const float* din; int F, ld, S, cond_stride, cond_off, n_cond;
  float* dpts;                // (rows,3) or null
  float* dcond;               // (B, cond_stride) or null
  long long rows;
};
__global__ void encode_bwd_kernel(const EncodeBwdArgs a) {
  const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= a.rows) return;
  const float* g = a.din + m * a.ld;
  if (a.dpts) {
    float x[3], dx[3];
#pragma unroll
    for (int c = 0; c < 3; ++c) { x[c] = a.pts[m * 3 + c]; dx[c] = g[c]; }
    for (int f = 0; f < a.F; ++f) {
      const float w = a.window ? a.window[f] : 1.f;
      const float s = exp2f((float)f);
#pragma unroll
      for (int c = 0; c < 3; ++c) {
        const float ang = x[c] * s;
        // d/dx sin(s x) = s cos(s x);  d/dx sin(s x + hp) = s cos(s x + hp)
        dx[c] = fmaf(g[3 + f * 6 + c] * w * s, cosf(ang), dx[c]);
        dx[c] = fmaf(g[3 + f * 6 + 3 + c] * w * s, cosf(ang + kHalfPiF), dx[c]);
      }
    }
#pragma unroll
    for (int c = 0; c < 3; ++c) a.dpts[m * 3 + c] = dx[c];
  }
  if (a.dcond) {
    const long long ray = m / a.S;
    for (int q = 0; q < a.n_cond; ++q) {
      const float v = g[3 + 6 * a.F + q];
      if (v != 0.f) atomicAdd(a.dcond + ray * a.cond_stride + a.cond_off + q, v);
    }
  }
}

// ---------------------------------------------------------------------------
// Warp tail (R5) and its adjoint by forward-mode duals (9 or 15 directions: the
// head outputs w, v, (pivot), (translation) and the point).
// ---------------------------------------------------------------------------
struct WarpTailArgs {
  const float* head; int ld;  // (rows, ld): [w v (p) (t)] or the translation (3)
  const float* pts;           // (rows,3)
  float* warped;              // (rows,3)
  int warp_type, pivot, trans;
  long long rows;
};
__global__ void warp_tail_kernel(const WarpTailArgs a) {
  const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= a.rows) return;
  const float* h = a.head + m * a.ld;
  float x[3] = {a.pts[m * 3], a.pts[m * 3 + 1], a.pts[m * 3 + 2]}, y[3];
  if (a.warp_type == 2) {
    float wv[12];
#pragma unroll
    for (int q = 0; q < 12; ++q) wv[q] = h[q];
    se3_apply(wv, x, y, a.pivot ? wv + 6 : nullptr, a.trans ? wv + (a.pivot ? 9 : 6) : nullptr);
  } else {
#pragma unroll
    for (int c = 0; c < 3; ++c) y[c] = x[c] + h[c];
  }
#pragma unroll
  for (int c = 0; c < 3; ++c) a.warped[m * 3 + c] = y[c];
}

// Forward-mode dual number with N tangent directions.
template <int N>
struct Dual {
  float v; float d[N];
};
template <int N> __device__ __forceinline__ Dual<N> dconst(float v) {
  Dual<N> r; r.v = v;
#pragma unroll
  for (int i = 0; i < N; ++i) r.d[i] = 0.f;
  return r;
}
template <int N> __device__ __forceinline__ Dual<N> operator+(const Dual<N>& a, const Dual<N>& b) {
  Dual<N> r; r.v = a.v + b.v;
#pragma unroll
  for (int i = 0; i < N; ++i) r.d[i] = a.d[i] + b.d[i];
  return r;
}
template <int N> __device__ __forceinline__ Dual<N> operator-(const Dual<N>& a, const Dual<N>& b) {
  Dual<N> r; r.v = a.v - b.v;
#pragma unroll
  for (int i = 0; i < N; ++i) r.d[i] = a.d[i] - b.d[i];
  return r;
}
template <int N> __device__ __forceinline__ Dual<N> operator*(const Dual<N>& a, const Dual<N>& b) {
  Dual<N> r; r.v = a.v * b.v;
#pragma unroll
  for (int i = 0; i < N; ++i) r.d[i] = a.d[i] * b.v + a.v * b.d[i];
  return r;
}
template <int N> __device__ __forceinline__ Dual<N> operator/(const Dual<N>& a, const Dual<N>& b) {
  Dual<N> r; r.v = a.v / b.v;
  const float inv = 1.f / b.v;
#pragma unroll
  for (int i = 0; i < N; ++i) r.d[i] = (a.d[i] - r.v * b.d[i]) * inv;
  return r;
}
template <int N> __device__ __forceinline__ Dual<N> dsqrt(const Dual<N>& a) {
  Dual<N> r; r.v = sqrtf(a.v);
  const float k = 0.5f / r.v;
#pragma unroll
  for (int i = 0; i < N; ++i) r.d[i] = a.d[i] * k;
  return r;
}
template <int N> __device__ __forceinline__ Dual<N> dsin(const Dual<N>& a) {
  Dual<N> r; r.v = sinf(a.v);
  const float c = cosf(a.v);
#pragma unroll
  for (int i = 0; i < N; ++i) r.d[i] = a.d[i] * c;
  return r;
}
template <int N> __device__ __forceinline__ Dual<N> dcos(const Dual<N>& a) {
  Dual<N> r; r.v = cosf(a.v);
  const float s = -sinf(a.v);
#pragma unroll
  for (int i = 0; i < N; ++i) r.d[i] = a.d[i] * s;
  return r;
}

// SE3Field.warp tail (warping.py:330-352) on duals; in[0..5] = w, v, in[6..8] = pivot,
// in[9..11] = translation, x = point (all seeded by the caller).
template <int N>
__device__ void se3_dual(const Dual<N>* in, const Dual<N>* x_in, bool pivot, bool trans, Dual<N>* out) {
  using D = Dual<N>;
  D theta = dsqrt(in[0] * in[0] + in[1] * in[1] + in[2] * in[2]);
  D w[3] = {in[0] / theta, in[1] / theta, in[2] / theta};
  D v[3] = {in[3] / theta, in[4] / theta, in[5] / theta};
  D x[3] = {x_in[0], x_in[1], x_in[2]};
  const D* pv = in + 6;
  const D* tr = in + (pivot ? 9 : 6);
  if (pivot) for (int c = 0; c < 3; ++c) x[c] = x[c] + pv[c];
  D zero = dconst<N>(0.f), one = dconst<N>(1.f);
  D W[3][3] = {{zero, zero - w[2], w[1]}, {w[2], zero, zero - w[0]}, {zero - w[1], w[0], zero}};
  D W2[3][3];
  for (int i = 0; i < 3; ++i)
    for (int j = 0; j < 3; ++j) W2[i][j] = W[i][0] * W[0][j] + W[i][1] * W[1][j] + W[i][2] * W[2][j];
  D s = dsin(theta), c = dcos(theta);
  D omc = one - c, tms = theta - s;
  for (int i = 0; i < 3; ++i) {
    D rx = zero, p = zero;
    for (int j = 0; j < 3; ++j) {
      D eye = (i == j) ? one : zero;
      D R = eye + s * W[i][j] + omc * W2[i][j];
      D M = theta * eye + omc * W[i][j] + tms * W2[i][j];
      rx = rx + R * x[j];
      p = p + M * v[j];
    }
    out[i] = rx + p;
    if (pivot) out[i] = out[i] - pv[i];
    if (trans) out[i] = out[i] + tr[i];
  }
}

struct WarpTailBwdArgs {
  const float* head; int ld; const float* pts; const float* dwarped;   // (rows,3)
  float* dhead;               // (rows, ld): += the gradient of the head outputs
  int warp_type, pivot, trans;
  long long rows;
};
__global__ void warp_tail_bwd_kernel(const WarpTailBwdArgs a) {
  const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= a.rows) return;
  const float g[3] = {a.dwarped[m * 3], a.dwarped[m * 3 + 1], a.dwarped[m * 3 + 2]};
  float* dh = a.dhead + m * a.ld;
  if (a.warp_type != 2) {
#pragma unroll
    for (int c = 0; c < 3; ++c) dh[c] += g[c];       // warped = x + t
    return;
  }
  // d(warped)/d(head) by forward mode: one direction per head output (the points carry
  // no parameter upstream: x = o + z d with z a constant).
  constexpr int N = 12;
  const int nh = 6 + (a.pivot ? 3 : 0) + (a.trans ? 3 : 0);
  Dual<N> in[12], x[3], out[3];
  for (int q = 0; q < 12; ++q) {
    in[q] = dconst<N>(q < nh ? a.head[m * a.ld + q] : 0.f);
    if (q < nh) in[q].d[q] = 1.f;
  }
  for (int c = 0; c < 3; ++c) x[c] = dconst<N>(a.pts[m * 3 + c]);
  se3_dual<N>(in, x, a.pivot != 0, a.trans != 0, out);
  for (int q = 0; q < nh; ++q) dh[q] += g[0] * out[0].d[q] + g[1] * out[1].d[q] + g[2] * out[2].d[q];
}

// ---------------------------------------------------------------------------
// R8: raw -> (sigmoid(rgb), sigma_act(alpha)); R9 adjoint + the photometric loss.
// ---------------------------------------------------------------------------
__global__ void raw_to_samples_kernel(const float* __restrict__ rgb_raw, int ld_rgb,
                                      const float* __restrict__ alpha_raw, int ld_a, int sigma_act,
                                      float4* __restrict__ samples, long long rows) {
  const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= rows) return;
  float4 o;
  o.x = sigmoidf(rgb_raw[m * ld_rgb]); o.y = sigmoidf(rgb_raw[m * ld_rgb + 1]); o.z = sigmoidf(rgb_raw[m * ld_rgb + 2]);
  o.w = apply_act(alpha_raw[m * ld_a], sigma_act);
  samples[m] = o;
}

// One warp per ray: loss = mean((rgb - target)^2) over the LOCAL batch (training.py:173),
// d(loss)/d(raw) through volumetric_rendering (model_utils.py:104-126).
struct CompositeBwdArgs {
  const float4* samples; const float* z; const float* directions;   // forward results
  const float* out;           // (B,6) forward rgb...
  const float* target;        // (B,3)
  const float* rgb_raw; int ld_rgb; const float* alpha_raw; int ld_a;
  float* d_rgb_raw; float* d_alpha_raw;     // same layouts: = (not +=)
  float* loss;                // += this level's loss (scalar)
  float scale;                // 1 / (batch_rays * 3)
  int num_rays, S, white_bg, sample_at_infinity, sigma_act;
};
__global__ void composite_bwd_kernel(const CompositeBwdArgs a) {
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int ray = blockIdx.x * kRaysPerBlock + warp;
  if (ray >= a.num_rays) return;
  extern __shared__ float sh[];
  const int S = a.S;
  float* gw = sh + warp * 4 * S;       // d loss / d w_i
  float* suf = gw + S;                 // sum_{k>i} gw_k w_k
  float* al = suf + S;                 // alpha_i
  float* tr = al + S;                  // T_i
  float g[3];
  float l = 0.f;
#pragma unroll
  for (int c = 0; c < 3; ++c) {
    const float diff = a.out[ray * 6 + c] - a.target[ray * 3 + c];
    g[c] = 2.f * diff * a.scale;
    l += diff * diff * a.scale;
  }
  if (lane == 0) atomicAdd(a.loss, l);
  const float dx = a.directions[ray * 3], dy = a.directions[ray * 3 + 1], dz = a.directions[ray * 3 + 2];
  const float dnorm = sqrtf(dx * dx + dy * dy + dz * dz);
  const float last = a.sample_at_infinity ? 1e10f : 1e-19f;
  const float gsum = g[0] + g[1] + g[2];
  for (int i = lane; i < S; i += 32) {
    const size_t m = (size_t)ray * S + i;
    const float4 c = a.samples[m];
    // rgb = sum w c (+ (1 - sum w) on a white background, model_utils.py:121-122)
    float v = g[0] * c.x + g[1] * c.y + g[2] * c.z;
    if (a.white_bg) v -= gsum;
    gw[i] = v;
    float dist = (i + 1 < S) ? (a.z[m + 1] - a.z[m]) : last;
    al[i] = -expm1f(-c.w * (dist * dnorm));
  }
  __syncwarp();
  if (lane == 0) {
    // w_i = alpha_i T_i, T_i = prod_{j<i} (1 - alpha_j + eps)  (model_utils.py:108-114):
    // dL/dalpha_i = gw_i T_i - (sum_{k>i} gw_k w_k) / (1 - alpha_i + eps)
    float t = 1.f;
    for (int i = 0; i < S; ++i) { tr[i] = t; t = t * (1.0f - al[i] + 1e-10f); }
    float acc = 0.f;
    for (int i = S - 1; i >= 0; --i) { suf[i] = acc; acc += gw[i] * (al[i] * tr[i]); }
  }
  __syncwarp();
  for (int i = lane; i < S; i += 32) {
    const size_t m = (size_t)ray * S + i;
    const float4 c = a.samples[m];
    float dist = (i + 1 < S) ? (a.z[m + 1] - a.z[m]) : last;
    dist = dist * dnorm;
    const float dalpha = gw[i] * tr[i] - suf[i] / (1.0f - al[i] + 1e-10f);
    const float dsigma = dalpha * dist * expf(-c.w * dist);      // alpha = 1 - exp(-sigma dist)
    const float raw = a.alpha_raw[m * a.ld_a];
    float dact;                                                    // sigma = act(raw)
    if (a.sigma_act == kSoftplus) dact = 1.f / (1.f + expf(-raw));
    else if (a.sigma_act == kRelu) dact = raw > 0.f ? 1.f : 0.f;
    else dact = act_grad_from_output(c.w, a.sigma_act);
    a.d_alpha_raw[m * a.ld_a] = dsigma * dact;
    const float w = al[i] * tr[i];
    // rgb_i = sigmoid(raw): d/draw = c (1 - c)
    a.d_rgb_raw[m * a.ld_rgb + 0] = g[0] * w * c.x * (1.f - c.x);
    a.d_rgb_raw[m * a.ld_rgb + 1] = g[1] * w * c.y * (1.f - c.y);
    a.d_rgb_raw[m * a.ld_rgb + 2] = g[2] * w * c.z * (1.f - c.z);
  }
}

// ---------------------------------------------------------------------------
// Embedding gradients: dcond (B, stride) -> table rows (glo.py:41-53), per the layout
// ray_cond_kernel wrote: [warp glo (G) | trunk (A) | alpha (A) | rgb: viewdirs, (A), camera].
// ---------------------------------------------------------------------------
struct CondBwdArgs {
  const float* dcond; int stride, num_rays;
  const unsigned* warp_id; const unsigned* app_id; const unsigned* cam_id;
  float* d_warp_table; float* d_app_table; float* d_cam_table;
  int n_warp, n_app, n_cam, G, A, C, Fv, use_viewdirs, use_app, use_cam, use_trunk_c, use_alpha_c;
  // The warp block [0, G) is a GLO row for 'glo' (scale 1) and 'blend' (scale 1 - time_alpha,
  // warping.py:132-133).  'time' has no GLO table (warp_glo = 0): its warp_id may hold float timestamps.
  int warp_glo; float warp_scale;
};
__global__ void cond_bwd_kernel(const CondBwdArgs a) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= (long long)a.num_rays * a.stride) return;
  const int ray = (int)(idx / a.stride);
  int q = (int)(idx - (long long)ray * a.stride);
  const float v = a.dcond[idx];
  if (v == 0.f) return;
  auto app = [&](int j) {
    unsigned id = a.app_id ? a.app_id[ray] : 0u;
    id = min(id, (unsigned)(a.n_app - 1));
    atomicAdd(a.d_app_table + (size_t)id * a.A + j, v);
  };
  if (q < a.G) {
    if (!a.warp_glo) return;
    unsigned id = a.warp_id ? a.warp_id[ray] : 0u;
    id = min(id, (unsigned)(a.n_warp - 1));
    atomicAdd(a.d_warp_table + (size_t)id * a.G + q, a.warp_scale * v);
    return;
  }
  q -= a.G;
  const int tc = (a.use_app && a.use_trunk_c) ? a.A : 0;
  if (q < tc) { app(q); return; }
  q -= tc;
  const int ac = (a.use_app && a.use_alpha_c) ? a.A : 0;
  if (q < ac) { app(q); return; }
  q -= ac;
  const int dv = a.use_viewdirs ? 3 + 6 * a.Fv : 0;
  if (q < dv) return;                                   // view directions carry no parameter
  q -= dv;
  if (q < ac) { app(q); return; }
  q -= ac;
  if (a.use_cam && q < a.C) {
    unsigned id = a.cam_id ? a.cam_id[ray] : 0u;
    id = min(id, (unsigned)(a.n_cam - 1));
    atomicAdd(a.d_cam_table + (size_t)id * a.C + q, v);
  }
}

// ---------------------------------------------------------------------------
// TimeEncoder backward, first stage: per condition vector, the encoder's input row (the input
// stage of time_embed_kernel, same arithmetic) and the seed dZ of its output layer,
// seed_scale * dcond[:, 0:G] (1 for 'time', time_alpha for 'blend': warping.py:132-133).  The
// layers themselves go through the training GEMMs (net_forward / net_backward).
// ---------------------------------------------------------------------------
struct TimeTapeArgs {
  const float* time_f;        // (rows) metadata['time'], or null
  const unsigned* time_id;    // (rows) ids read as timestamps, float(id), or null
  int F;                      // metadata_encoder_num_freqs
  float window[20];           // cosine_easing_window(F, alpha) as run_cond builds it
  const float* dcond; int cond_stride, G; float seed_scale;
  float* in; int ld_in;       // (rows, ld_in): [t, w_f sin(2^f t), w_f sin(2^f t + pi/2)]_f
  float* seed; int ld_seed;   // (rows, ld_seed); the padding columns stay as they are (zero)
  long long rows;
};
__global__ void time_tape_kernel(const __grid_constant__ TimeTapeArgs a) {
  const long long m = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (m >= a.rows) return;
  const float t = a.time_f ? a.time_f[m] : (float)a.time_id[m];
  float* o = a.in + m * a.ld_in;
  o[0] = t;
  for (int k = 1; k < 1 + 2 * a.F; ++k) {
    const int f = (k - 1) >> 1;
    float ang = t * exp2f((float)f);
    if ((k - 1) & 1) ang = ang + kHalfPiF;
    o[k] = a.window[f] * sinf(ang);
  }
  const float* g = a.dcond + m * a.cond_stride;
  for (int q = 0; q < a.G; ++q) a.seed[m * a.ld_seed + q] = a.seed_scale * g[q];
}

// packed (K x ld, column offset) gradient -> the caller's dense (rows x cols) tensor (+=).
__global__ void unpack_grad_kernel(const float* __restrict__ packed, float* __restrict__ dst, long long rows,
                                   long long cols, int ld, int c_off) {
  const long long idx = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (idx >= rows * cols) return;
  const long long r = idx / cols, c = idx - r * cols;
  dst[idx] += packed[r * ld + c_off + c];
}

// flax.optim.Adam (beta1 0.9, beta2 0.999, eps 1e-8, no weight decay): one fused pass.
__global__ void adam_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                            float* __restrict__ v, long long n, float lr, float b1, float b2, float eps,
                            float bc1, float bc2) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= n) return;
  const float gi = g[i];
  const float mi = b1 * m[i] + (1.f - b1) * gi;
  const float vi = b2 * v[i] + (1.f - b2) * gi * gi;
  m[i] = mi; v[i] = vi;
  const float mhat = mi / bc1, vhat = vi / bc2;
  p[i] = p[i] - lr * mhat / (sqrtf(vhat) + eps);
}

}  // namespace train
}  // namespace nfb
