// SIMT kernels (see kernels.cuh).  Reference semantics cited per kernel.
#include <cstdlib>

#include "kernels.cuh"
#include "tc_gemm.cuh"

namespace ddnm {

static constexpr int MAX_C = 2048;  // widest concat in either UNet

bool pdl_enabled() {
  static const bool on = [] {
    const char* v = std::getenv("DDNM_PDL");
    return !(v && v[0] == '0');
  }();
  return on;
}

__device__ __forceinline__ float swishf(float x) { return x / (1.0f + expf(-x)); }
// x * sigmoid(x) on the special-function unit: 2^(-x log2 e) by ex2.approx, the quotient by rcp.approx (relative error ~2e-7, two
// orders below the fp16 split that follows it).  The GroupNorm pass is within ~1.4x of being issue-bound with the library expf and
// the IEEE division (~20 instructions per element); this form is 5.
__device__ __forceinline__ float swishf_fast(float x) {
  float e;
  asm("ex2.approx.ftz.f32 %0, %1;" : "=f"(e) : "f"(x * -1.4426950408889634f));
  return __fdividef(x, 1.0f + e);
}

// ---------------------------------------------------------------------------------------------------------------
// Per-channel sums for GroupNorm (torch.nn.GroupNorm(32, C): models.py:32-33 / nn.py:17-19) of a tensor that was NOT
// produced by the tensor-core kernel (whose epilogue accumulates them itself).  One CTA = one image x one pixel chunk;
// every thread owns 4 fixed channels (float4 loads along the contiguous NHWC channel axis) and adds its partial sums to the
// per-(image, channel) 128-bit fixed-point accumulators (StatAcc).
// ---------------------------------------------------------------------------------------------------------------
__global__ void gn_stats_kernel(const float* __restrict__ x, int HW, int C, int ld, int pix_per_cta,
                                StatAcc* __restrict__ stats, int st_ld) {
  pdl_prologue();
  const int n = blockIdx.y;
  const int C4 = C >> 2;
  const int rows = blockDim.x / C4;
  const int c4 = threadIdx.x % C4;
  const int prow = threadIdx.x / C4;
  const int p0 = blockIdx.x * pix_per_cta;
  const int p1 = min(HW, p0 + pix_per_cta);
  float s[4] = {0, 0, 0, 0}, q[4] = {0, 0, 0, 0};
  if (prow < rows) {
    const float* base = x + (long long)n * HW * ld + c4 * 4;
    const size_t step = (size_t)rows * ld;
    int p = p0 + prow;
    const float* ptr = base + (size_t)p * ld;
    // 4 independent 16-byte loads in flight per thread (the compiler does not unroll this loop on its own)
    for (; p + 3 * rows < p1; p += 4 * rows, ptr += 4 * step) {
      const float4 v0 = __ldg(reinterpret_cast<const float4*>(ptr));
      const float4 v1 = __ldg(reinterpret_cast<const float4*>(ptr + step));
      const float4 v2 = __ldg(reinterpret_cast<const float4*>(ptr + 2 * step));
      const float4 v3 = __ldg(reinterpret_cast<const float4*>(ptr + 3 * step));
      s[0] += (v0.x + v1.x) + (v2.x + v3.x); q[0] += (v0.x * v0.x + v1.x * v1.x) + (v2.x * v2.x + v3.x * v3.x);
      s[1] += (v0.y + v1.y) + (v2.y + v3.y); q[1] += (v0.y * v0.y + v1.y * v1.y) + (v2.y * v2.y + v3.y * v3.y);
      s[2] += (v0.z + v1.z) + (v2.z + v3.z); q[2] += (v0.z * v0.z + v1.z * v1.z) + (v2.z * v2.z + v3.z * v3.z);
      s[3] += (v0.w + v1.w) + (v2.w + v3.w); q[3] += (v0.w * v0.w + v1.w * v1.w) + (v2.w * v2.w + v3.w * v3.w);
    }
    for (; p < p1; p += rows, ptr += step) {
      const float4 v = __ldg(reinterpret_cast<const float4*>(ptr));
      s[0] += v.x; q[0] += v.x * v.x;
      s[1] += v.y; q[1] += v.y * v.y;
      s[2] += v.z; q[2] += v.z * v.z;
      s[3] += v.w; q[3] += v.w * v.w;
    }
    // every thread's partial sums (a fixed set of pixels, summed in a fixed order) go straight into the order-independent
    // fixed-point accumulators: no floating-point atomics anywhere, so the statistics are bit-reproducible
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      StatAcc* d = stats + ((size_t)n * st_ld + c4 * 4 + j) * 2;
      stat_add(d, s[j]);
      stat_add(d + 1, q[j]);
    }
  }
}

void gn_stats(const View& x, cudaStream_t st) {
  DDNM_CHECK(x.C % 4 == 0 && x.C <= MAX_C && x.ld % 4 == 0 && x.st != nullptr, "gn_stats: unsupported channel count / no stats slot");
  const int C4 = x.C / 4;
  const int rows = std::max(1, 256 / C4);
  const int threads = C4 * rows;
  const int HW = x.H * x.W;
  long long want = cdivll((long long)HW * x.N, 592);
  int ppc = (int)std::max<long long>(rows * 4, cdivll(want, rows) * rows);
  dim3 grid(cdiv(HW, ppc), x.N);
  launch_pdl(gn_stats_kernel, grid, dim3(threads), 0, st, 1, (const float*)x.p, HW, x.C, x.ld, ppc, x.st, x.st_ld);
  CUDA_CHECK(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------------------------
// Normalise (+ SiLU) and split to fp16 hi/lo.  Produces the A operand of the tensor-core convolution, i.e. fuses
//   h = nonlinearity(norm(x))            models.py:117-118,124-125   (x * sigmoid(x), GN eps 1e-6)
//   (nearest x2 upsampling needs no copy: the consumer convolution runs as 4 parity phases on this low-res split)
//   F.pad(x, (0,1,0,1)) + stride 2       models.py:67-71   (SPLIT_S2D: parity phases; pad = TMA zero fill)
// Each thread converts 8 channels of one pixel: 2 x float4 in, 16 B out per plane.
// ---------------------------------------------------------------------------------------------------------------
template <bool F32OUT>
__global__ void gn_apply_kernel(const float* __restrict__ x, int H, int W, int C, int ld, int N, int groups,
                                const StatAcc* __restrict__ stats, int st_ld, const float* __restrict__ gamma,
                                const float* __restrict__ beta, float eps, int silu, int mode, int pix_per_cta,
                                __half* __restrict__ hi, __half* __restrict__ lo, float* __restrict__ out32,
                                const float* __restrict__ ss, int ss_ld, __half* __restrict__ raw_hi,
                                __half* __restrict__ raw_lo) {
  pdl_prologue();
  // dynamic smem: [2*C] doubles (the image's per-channel sums, staged with ONE independent load per channel) then sc[C], sh[C].
  // (Summing a group's sums straight from global memory made every thread walk a chain of 2*cpg dependent-issue loads,
  // ~10-16 us of latency in front of every CTA's first pixel.)
  extern __shared__ double gn_smem[];
  double* sd = gn_smem;
  float* sc = reinterpret_cast<float*>(gn_smem + 2 * (size_t)C);
  float* sh = sc + C;
  const int n = blockIdx.y;
  const int HW = H * W;
  if (stats) {
    const int cpg = C / groups;
    const double cnt = (double)HW * cpg;
    const StatAcc* gsrc = stats + (size_t)n * st_ld * 2;
    for (int c = threadIdx.x; c < 2 * C; c += blockDim.x) sd[c] = stat_value(gsrc[c]);
    __syncthreads();
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      const int g0 = (c / cpg) * cpg;   // the group's channels are adjacent
      double s1 = 0, s2 = 0;
      for (int j = 0; j < cpg; ++j) {
        s1 += sd[2 * (g0 + j)];
        s2 += sd[2 * (g0 + j) + 1];
      }
      const double mean = s1 / cnt;
      double var = s2 / cnt - mean * mean;
      var = var < 0 ? 0 : var;
      const float rstd = (float)(1.0 / sqrt(var + (double)eps));
      float a = rstd * gamma[c];
      float b = beta[c] - (float)mean * a;
      if (ss) {  // h = norm(h) * (1 + scale) + shift
        const float one_plus = 1.0f + ss[(size_t)n * ss_ld + c];
        a *= one_plus;
        b = fmaf(b, one_plus, ss[(size_t)n * ss_ld + C + c]);
      }
      sc[c] = a;
      sh[c] = b;
    }
  } else {
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      sc[c] = 1.f;
      sh[c] = 0.f;
    }
  }
  __syncthreads();
  const int C8 = C >> 3;
  const int rows = blockDim.x / C8;
  const int c8 = threadIdx.x % C8, prow = threadIdx.x / C8;
  if (prow >= rows) return;
  const int c = c8 * 8;
  float a8[8], b8[8];
#pragma unroll
  for (int j = 0; j < 8; ++j) { a8[j] = sc[c + j]; b8[j] = sh[c + j]; }
  const int p0 = blockIdx.x * pix_per_cta;
  if (mode == SPLIT_AVG2) {
    // output pixel = mean of the 2x2 block of ACTIVATED inputs (avg_pool2d after norm + SiLU)
    const int Wo = W >> 1, HWo = (H >> 1) * Wo;
    const int q1 = min(HWo, p0 + pix_per_cta);
    for (int q = p0 + prow; q < q1; q += rows) {
      const int oy = q / Wo, ox = q - oy * Wo;
      float acc[8] = {0, 0, 0, 0, 0, 0, 0, 0};
#pragma unroll
      for (int d = 0; d < 4; ++d) {
        const float* sp = x + ((size_t)n * HW + (size_t)(2 * oy + (d >> 1)) * W + 2 * ox + (d & 1)) * ld + c;
        const float4 a = __ldg(reinterpret_cast<const float4*>(sp));
        const float4 b = __ldg(reinterpret_cast<const float4*>(sp + 4));
        float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
#pragma unroll
        for (int j = 0; j < 8; ++j) {
          v[j] = fmaf(v[j], a8[j], b8[j]);
          if (silu) v[j] = swishf_fast(v[j]);
          acc[j] += v[j];
        }
      }
      __align__(16) __half h8[8];
      __align__(16) __half l8[8];
#pragma unroll
      for (int j = 0; j < 8; ++j) split_f16(acc[j] * 0.25f, h8[j], l8[j]);
      const size_t o = ((size_t)n * HWo + q) * C + c;
      *reinterpret_cast<uint4*>(hi + o) = *reinterpret_cast<const uint4*>(h8);
      *reinterpret_cast<uint4*>(lo + o) = *reinterpret_cast<const uint4*>(l8);
    }
    return;
  }
  const int p1 = min(HW, p0 + pix_per_cta);
  const float* src = x + ((size_t)n * HW + p0 + prow) * ld + c;
  const size_t step = (size_t)rows * ld;
  // software-pipelined: the next pixel's 32 bytes are already in flight while this one is converted and stored
  float4 a = make_float4(0.f, 0.f, 0.f, 0.f), b = a;
  if (p0 + prow < p1) {
    a = __ldg(reinterpret_cast<const float4*>(src));
    b = __ldg(reinterpret_cast<const float4*>(src + 4));
  }
  for (int p = p0 + prow; p < p1; p += rows, src += step) {
    float v[8] = {a.x, a.y, a.z, a.w, b.x, b.y, b.z, b.w};
    if (p + rows < p1) {
      a = __ldg(reinterpret_cast<const float4*>(src + step));
      b = __ldg(reinterpret_cast<const float4*>(src + step + 4));
    }
    if (!F32OUT && raw_hi) {  // second output: the un-normalised tensor (input of the 1x1 shortcut convolution)
      uint4 rh, rl;
      split2_f16(v[0], v[1], rh.x, rl.x);
      split2_f16(v[2], v[3], rh.y, rl.y);
      split2_f16(v[4], v[5], rh.z, rl.z);
      split2_f16(v[6], v[7], rh.w, rl.w);
      const size_t o = ((size_t)n * HW + p) * C + c;
      *reinterpret_cast<uint4*>(raw_hi + o) = rh;
      *reinterpret_cast<uint4*>(raw_lo + o) = rl;
    }
#pragma unroll
    for (int j = 0; j < 8; ++j) {
      v[j] = fmaf(v[j], a8[j], b8[j]);
      if (silu) v[j] = swishf_fast(v[j]);
    }
    if (F32OUT) {
      float* d = out32 + ((size_t)n * HW + p) * C + c;
      *reinterpret_cast<float4*>(d) = make_float4(v[0], v[1], v[2], v[3]);
      *reinterpret_cast<float4*>(d + 4) = make_float4(v[4], v[5], v[6], v[7]);
    } else {
      uint4 hv, lv;   // two values per conversion instruction (same roundings as split_f16)
      split2_f16(v[0], v[1], hv.x, lv.x);
      split2_f16(v[2], v[3], hv.y, lv.y);
      split2_f16(v[4], v[5], hv.z, lv.z);
      split2_f16(v[6], v[7], hv.w, lv.w);
      if (mode == SPLIT_SAME) {
        const size_t o = ((size_t)n * HW + p) * C + c;
        *reinterpret_cast<uint4*>(hi + o) = hv;
        *reinterpret_cast<uint4*>(lo + o) = lv;
      } else {
        const int y = p / W, xx = p - y * W;
        {  // SPLIT_S2D
          const int ph = (y & 1) * 2 + (xx & 1);
          const int Hh = H >> 1, Wh = W >> 1;
          const size_t o = ((((size_t)ph * N + n) * Hh + (y >> 1)) * Wh + (xx >> 1)) * C + c;
          *reinterpret_cast<uint4*>(hi + o) = hv;
          *reinterpret_cast<uint4*>(lo + o) = lv;
        }
      }
    }
  }
}

static void gn_apply_launch(const View& x, int groups, bool normalise, const float* gamma, const float* beta, float eps,
                            bool silu, int mode, __half* hi, __half* lo, float* out32, cudaStream_t st, const float* ss, int ss_ld,
                            __half* raw_hi = nullptr, __half* raw_lo = nullptr) {
  if (raw_hi) DDNM_CHECK(mode == SPLIT_SAME && raw_lo && !out32, "raw side output only with the plain split");
  DDNM_CHECK(x.C % 8 == 0 && x.C <= MAX_C && x.ld % 4 == 0, "gn_apply: unsupported channel count");
  if (mode == SPLIT_S2D || mode == SPLIT_AVG2) DDNM_CHECK(x.H % 2 == 0 && x.W % 2 == 0, "space-to-depth / avg-pool need even dims");
  const StatAcc* stats = normalise ? x.st : nullptr;
  if (normalise) DDNM_CHECK(x.st != nullptr && x.C % groups == 0, "normalisation needs the tensor's per-channel sums (View::st)");
  if (ss) DDNM_CHECK(normalise, "scale-shift needs a normalisation");
  const int HW = mode == SPLIT_AVG2 ? x.H * x.W / 4 : x.H * x.W;   // pixels the grid iterates over
  const int C8 = x.C / 8;
  const int rows = std::max(1, 256 / C8);
  const int threads = C8 * rows;
  long long want = cdivll((long long)HW * x.N, 148 * 8);
  int ppc = (int)std::max<long long>(rows, cdivll(want, rows) * rows);
  dim3 grid(cdiv(HW, ppc), x.N);
  const size_t smem = (size_t)x.C * 24;   // 2 doubles + 2 floats per channel (<= 48 KiB at MAX_C)
  if (out32)
    launch_pdl(gn_apply_kernel<true>, grid, dim3(threads), smem, st, 1, (const float*)x.p, x.H, x.W, x.C, x.ld, x.N, groups, stats, x.st_ld, gamma,
               beta, eps, (int)silu, mode, ppc, (__half*)nullptr, (__half*)nullptr, out32, ss, ss_ld, (__half*)nullptr, (__half*)nullptr);
  else
    launch_pdl(gn_apply_kernel<false>, grid, dim3(threads), smem, st, 1, (const float*)x.p, x.H, x.W, x.C, x.ld, x.N, groups, stats, x.st_ld, gamma,
               beta, eps, (int)silu, mode, ppc, hi, lo, (float*)nullptr, ss, ss_ld, raw_hi, raw_lo);
  CUDA_CHECK(cudaGetLastError());
}

void gn_apply_split(const View& x, int groups, bool normalise, const float* gamma, const float* beta, float eps,
                    bool silu, int mode, __half* hi, __half* lo, cudaStream_t s, const float* ss, int ss_ld, __half* raw_hi,
                    __half* raw_lo) {
  gn_apply_launch(x, groups, normalise, gamma, beta, eps, silu, mode, hi, lo, nullptr, s, ss, ss_ld, raw_hi, raw_lo);
}
void gn_apply_f32(const View& x, int groups, const float* gamma, const float* beta, float eps, bool silu, float* out,
                  cudaStream_t s) {
  gn_apply_launch(x, groups, true, gamma, beta, eps, silu, SPLIT_SAME, nullptr, nullptr, out, s, nullptr, 0);
}

// ---------------------------------------------------------------------------------------------------------------
// Stem: conv_in = Conv2d(3, ch, 3, padding=1) (models.py:228-232, 311) on the caller's NCHW tensor, NHWC result.
// Lane <-> 4 output channels (weights live in registers), warp walks over pixels; output rows are written as
// full 512-byte segments.  blockIdx.z selects a 128-channel slab of Cout.
// ---------------------------------------------------------------------------------------------------------------
template <int CIN>
__global__ void __launch_bounds__(256) conv_small_cin_kernel(const float* __restrict__ x, const float* __restrict__ w,
                                                             const float* __restrict__ bias, float* __restrict__ out,
                                                             int H, int W, int Cout, int ld, StatAcc* __restrict__ stats, int st_ld) {
  pdl_prologue();
  constexpr int KT = CIN * 9;
  constexpr int TW = 64, TH = 8;  // output tile per CTA: one warp per row
  __shared__ float tile[CIN][TH + 2][TW + 2];
  __shared__ float red[TH][128][2];   // per-row channel sums of the tile (GroupNorm statistics of the output, when asked for)
  const int slabs = (Cout + 127) / 128;
  const int n = blockIdx.z / slabs;
  const int slab = blockIdx.z % slabs;
  const int y0 = blockIdx.y * TH;
  const int x0 = blockIdx.x * TW;
  for (int i = threadIdx.x; i < CIN * (TH + 2) * (TW + 2); i += blockDim.x) {
    const int xx = i % (TW + 2), r = (i / (TW + 2)) % (TH + 2), c = i / ((TH + 2) * (TW + 2));
    const int gy = y0 + r - 1, gx = x0 + xx - 1;
    tile[c][r][xx] = (gy >= 0 && gy < H && gx >= 0 && gx < W) ? __ldg(&x[(((size_t)n * CIN + c) * H + gy) * W + gx]) : 0.f;
  }
  const int lane = threadIdx.x & 31, warp = threadIdx.x >> 5;
  const int co = slab * 128 + lane * 4;
  const bool active = co < Cout;
  float wr[KT][4];
  float b4[4] = {0, 0, 0, 0};
  if (active) {
#pragma unroll
    for (int k = 0; k < KT; ++k)
#pragma unroll
      for (int j = 0; j < 4; ++j) wr[k][j] = __ldg(&w[(size_t)(co + j) * KT + k]);  // OIHW: k = ci*9 + ky*3 + kx
#pragma unroll
    for (int j = 0; j < 4; ++j) b4[j] = __ldg(&bias[co + j]);
  }
  __syncthreads();
  const int y = y0 + warp;
  float s4[4] = {0.f, 0.f, 0.f, 0.f}, q4[4] = {0.f, 0.f, 0.f, 0.f};
  float* orow = out + (((size_t)n * H + y) * W + x0) * ld + co;
  // two pixels per iteration: the 3 x 4 window of each input channel is read once (LDS.64 pairs) for 2 x 27 x 4 FMAs, and the two
  // accumulator sets give the FMA pipe independent work while the next window loads
  for (int px = 0; active && y < H && px < TW && x0 + px < W; px += 2) {
    float acc0[4] = {b4[0], b4[1], b4[2], b4[3]};
    float acc1[4] = {b4[0], b4[1], b4[2], b4[3]};
#pragma unroll
    for (int c = 0; c < CIN; ++c)
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const float2 v01 = *reinterpret_cast<const float2*>(&tile[c][warp + r][px]);
        const float2 v23 = *reinterpret_cast<const float2*>(&tile[c][warp + r][px + 2]);
        const float v[4] = {v01.x, v01.y, v23.x, v23.y};
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          const int k = c * 9 + r * 3 + d;
#pragma unroll
          for (int j = 0; j < 4; ++j) {
            acc0[j] = fmaf(v[d], wr[k][j], acc0[j]);
            acc1[j] = fmaf(v[d + 1], wr[k][j], acc1[j]);
          }
        }
      }
    *reinterpret_cast<float4*>(orow + (size_t)px * ld) = make_float4(acc0[0], acc0[1], acc0[2], acc0[3]);
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      s4[j] += acc0[j];
      q4[j] = fmaf(acc0[j], acc0[j], q4[j]);
    }
    if (x0 + px + 1 < W) {
      *reinterpret_cast<float4*>(orow + (size_t)(px + 1) * ld) = make_float4(acc1[0], acc1[1], acc1[2], acc1[3]);
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        s4[j] += acc1[j];
        q4[j] = fmaf(acc1[j], acc1[j], q4[j]);
      }
    }
  }
  if (stats == nullptr) return;
  // the tile's per-channel sums: rows (warps) combined in a fixed order, then one order-independent fixed-point add per statistic
#pragma unroll
  for (int j = 0; j < 4; ++j) {
    red[warp][lane * 4 + j][0] = s4[j];
    red[warp][lane * 4 + j][1] = q4[j];
  }
  __syncthreads();
  const int c = threadIdx.x & 127, which = threadIdx.x >> 7;
  if (slab * 128 + c < Cout) {
    float t = 0.f;
#pragma unroll
    for (int r = 0; r < TH; ++r) t += red[r][c][which];
    stat_add(stats + ((size_t)n * st_ld + slab * 128 + c) * 2 + which, t);
  }
}

void conv3x3_small_cin(const float* x, int Cin, const float* w, const float* bias, const View& out, cudaStream_t st) {
  DDNM_CHECK(Cin == 3, "stem convolution expects 3 input channels");
  DDNM_CHECK(out.C % 4 == 0, "stem Cout % 4");
  dim3 grid(cdiv(out.W, 64), cdiv(out.H, 8), out.N * cdiv(out.C, 128));
  // the GroupNorm sums of the output come out of the same pass when the view carries accumulators
  launch_pdl(conv_small_cin_kernel<3>, grid, dim3(256), 0, st, 1, x, w, bias, out.p, out.H, out.W, out.C, out.ld, out.st, out.st_ld);
  CUDA_CHECK(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------------------------
// Network head in one kernel: h = conv_out(nonlinearity(norm_out(h)))  (models.py:338-340; unet.py:613-617 `out`), NCHW result.
// Cout is 3 (or 6 with learned sigma): on the tensor cores the N tile has to be padded to 64 columns and the kernel is paced by
// streaming the A operand (0.6 ms + a 0.2 ms GroupNorm pass + the NCHW copy at 256x256, B = 16).  Here the fp32 activation is read
// ONCE: a CTA stages an (8 + 2) x (128 + 2) halo tile of 16 channels at a time in shared memory with the GroupNorm affine and SiLU
// applied on the way in (zero outside the image: the convolution's padding), each thread owns 4 consecutive pixels x COP output
// channels and per (channel, tap row) reads 6 activations + 3 broadcast weight vectors for 12 * Cout exact fp32 FMAs.
// ---------------------------------------------------------------------------------------------------------------
constexpr int HD_TW = 128, HD_TH = 8, HD_CH = 16, HD_PITCH = 132, HD_PLANE = (HD_TH + 2) * HD_PITCH + 4;
template <int COP>
__global__ void __launch_bounds__(256) head_conv_kernel(const float* __restrict__ x, int H, int W, int C, int ld, int groups,
                                                        const StatAcc* __restrict__ stats, int st_ld, const float* __restrict__ gamma,
                                                        const float* __restrict__ beta, float eps, const float* __restrict__ w,
                                                        const float* __restrict__ bias, int Cout, float* __restrict__ out) {
  pdl_prologue();
  extern __shared__ float hd_smem[];
  float* act = hd_smem;                           // [HD_CH][HD_PLANE]
  float* wsm = act + HD_CH * HD_PLANE;            // [HD_CH][3][3][COP]
  float* sc = wsm + HD_CH * 9 * COP;              // [C] scale, [C] shift
  float* sh = sc + C;
  const int n = blockIdx.z, y0 = blockIdx.y * HD_TH, x0 = blockIdx.x * HD_TW;
  {
    // per-(image, channel) GroupNorm affine from the producer's sums (same arithmetic as gn_apply_kernel)
    const int cpg = C / groups;
    const double cnt = (double)H * W * cpg;
    const StatAcc* gsrc = stats + (size_t)n * st_ld * 2;
    for (int c = threadIdx.x; c < C; c += blockDim.x) {
      const int g0 = (c / cpg) * cpg;
      double s1 = 0, s2 = 0;
      for (int j = 0; j < cpg; ++j) {
        s1 += stat_value(gsrc[2 * (g0 + j)]);
        s2 += stat_value(gsrc[2 * (g0 + j) + 1]);
      }
      const double mean = s1 / cnt;
      double var = s2 / cnt - mean * mean;
      var = var < 0 ? 0 : var;
      const float rstd = (float)(1.0 / sqrt(var + (double)eps));
      const float a = rstd * gamma[c];
      sc[c] = a;
      sh[c] = beta[c] - (float)mean * a;
    }
  }
  const int ty = threadIdx.x >> 5, tx4 = (threadIdx.x & 31) * 4;   // 8 rows x 32 groups of 4 pixels
  float acc[4][COP];
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int co = 0; co < COP; ++co) acc[i][co] = 0.f;
  for (int c0 = 0; c0 < C; c0 += HD_CH) {
    __syncthreads();   // previous chunk consumed (first pass: the coefficient table is complete)
    // ---- stage the chunk: activations (normalised, activated, zero-padded) and weights
    // thread <-> (4-channel group q, tile column): its 10 rows are 10 independent 16-byte loads in flight, then their conversion
    // (one load per iteration exposed ~160 memory latencies per CTA: 0.83 ms for the kernel); addresses advance by a row pitch,
    // the 8 GroupNorm coefficients of the thread's channels are read once per chunk
    {
      const int q = threadIdx.x & 3;
      const int c = c0 + 4 * q;
      const float a0 = sc[c], a1 = sc[c + 1], a2 = sc[c + 2], a3 = sc[c + 3];
      const float b0 = sh[c], b1 = sh[c + 1], b2 = sh[c + 2], b3 = sh[c + 3];
#pragma unroll 1
      for (int col = threadIdx.x >> 2; col < HD_TW + 2; col += 64) {
        const int gx = x0 + col - 1;
        const bool xin = gx >= 0 && gx < W;
        const float* src = x + (((size_t)n * H + (y0 - 1)) * W + gx) * ld + c;   // row y0 - 1 (dereferenced only when inside)
        float4 v[HD_TH + 2];
#pragma unroll
        for (int r = 0; r < HD_TH + 2; ++r) {
          const int gy = y0 + r - 1;
          v[r] = make_float4(0.f, 0.f, 0.f, 0.f);
          if (xin && gy >= 0 && gy < H) v[r] = __ldg(reinterpret_cast<const float4*>(src + (size_t)r * W * ld));
        }
        float* d = act + (4 * q) * HD_PLANE + col;
#pragma unroll
        for (int r = 0; r < HD_TH + 2; ++r) {
          const int gy = y0 + r - 1;
          float4 t = v[r];
          if (xin && gy >= 0 && gy < H) {   // outside the image the ACTIVATED value is zero (the convolution's padding)
            t.x = swishf_fast(fmaf(t.x, a0, b0));
            t.y = swishf_fast(fmaf(t.y, a1, b1));
            t.z = swishf_fast(fmaf(t.z, a2, b2));
            t.w = swishf_fast(fmaf(t.w, a3, b3));
          }
          d[r * HD_PITCH] = t.x;
          d[r * HD_PITCH + HD_PLANE] = t.y;
          d[r * HD_PITCH + 2 * HD_PLANE] = t.z;
          d[r * HD_PITCH + 3 * HD_PLANE] = t.w;
        }
      }
    }
    for (int i = threadIdx.x; i < HD_CH * 9 * COP; i += blockDim.x) {
      const int co = i % COP, t = (i / COP) % 9, ch = i / (9 * COP);
      wsm[i] = co < Cout ? __ldg(&w[((size_t)co * C + c0 + ch) * 9 + t]) : 0.f;   // OIHW
    }
    __syncthreads();
    // ---- 4 pixels x COP channels per thread
#pragma unroll 2
    for (int ch = 0; ch < HD_CH; ++ch) {
#pragma unroll
      for (int r = 0; r < 3; ++r) {
        const float* ap = act + ch * HD_PLANE + (ty + r) * HD_PITCH + tx4;
        const float4 a0 = *reinterpret_cast<const float4*>(ap);
        const float2 a1 = *reinterpret_cast<const float2*>(ap + 4);
        const float a[6] = {a0.x, a0.y, a0.z, a0.w, a1.x, a1.y};
        const float* wp = wsm + (ch * 9 + r * 3) * COP;
#pragma unroll
        for (int d = 0; d < 3; ++d) {
          float wv[COP];   // one broadcast 16-byte read per 4 output channels (scalar reads made the loop LDS-bound)
#pragma unroll
          for (int c4 = 0; c4 < COP / 4; ++c4) {
            const float4 t = *reinterpret_cast<const float4*>(wp + d * COP + 4 * c4);
            wv[4 * c4 + 0] = t.x; wv[4 * c4 + 1] = t.y; wv[4 * c4 + 2] = t.z; wv[4 * c4 + 3] = t.w;
          }
#pragma unroll
          for (int co = 0; co < COP; ++co)
#pragma unroll
            for (int i = 0; i < 4; ++i) acc[i][co] = fmaf(a[i + d], wv[co], acc[i][co]);
        }
      }
    }
  }
  const int y = y0 + ty, xx = x0 + tx4;
  if (y < H && xx < W) {
#pragma unroll
    for (int co = 0; co < COP; ++co) {
      if (co < Cout) {
        const float b = bias[co];
        float* o = out + (((size_t)n * Cout + co) * H + y) * W + xx;
        if (xx + 3 < W && (W & 3) == 0) {
          *reinterpret_cast<float4*>(o) = make_float4(acc[0][co] + b, acc[1][co] + b, acc[2][co] + b, acc[3][co] + b);
        } else {
          for (int i = 0; i < 4 && xx + i < W; ++i) o[i] = acc[i][co] + b;
        }
      }
    }
  }
}

bool head_conv_supported(const View& h, int Cout) { return h.C % HD_CH == 0 && h.C <= 1024 && Cout >= 1 && Cout <= 8 && h.ld % 4 == 0; }

void head_conv(const View& h, int groups, const float* gamma, const float* beta, float eps, const float* w, const float* bias, int Cout,
               float* out_nchw, cudaStream_t st) {
  DDNM_CHECK(head_conv_supported(h, Cout) && h.st != nullptr && h.C % groups == 0, "head convolution: unsupported shape");
  const int cop = Cout <= 4 ? 4 : 8;
  const size_t smem = ((size_t)HD_CH * HD_PLANE + (size_t)HD_CH * 9 * cop + 2 * (size_t)h.C) * sizeof(float);
  dim3 grid(cdiv(h.W, HD_TW), cdiv(h.H, HD_TH), h.N);
  static bool attr4[64] = {}, attr8[64] = {};
  if (cop == 4) {
    if (first_use_on_device(attr4)) CUDA_CHECK(cudaFuncSetAttribute(head_conv_kernel<4>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    launch_pdl(head_conv_kernel<4>, grid, dim3(256), smem, st, 1, (const float*)h.p, h.H, h.W, h.C, h.ld, groups, (const StatAcc*)h.st, h.st_ld, gamma,
               beta, eps, w, bias, Cout, out_nchw);
  } else {
    if (first_use_on_device(attr8)) CUDA_CHECK(cudaFuncSetAttribute(head_conv_kernel<8>, cudaFuncAttributeMaxDynamicSharedMemorySize, 100 * 1024));
    launch_pdl(head_conv_kernel<8>, grid, dim3(256), smem, st, 1, (const float*)h.p, h.H, h.W, h.C, h.ld, groups, (const StatAcc*)h.st, h.st_ld, gamma,
               beta, eps, w, bias, Cout, out_nchw);
  }
  CUDA_CHECK(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------------------------
// Second half of a split-K convolution (tc_gemm.cu, TcParams::split_k): out = sum of the S partial results in a fixed order
// + per-(image, channel) add + residual, and the GroupNorm sums of the result.  One CTA per (image, few pixels), thread <-> 4 channels.
// ---------------------------------------------------------------------------------------------------------------
__global__ void __launch_bounds__(256) splitk_reduce_kernel(const float* __restrict__ part, int S, long long stride, int HW, int C,
                                                            float* __restrict__ out, int ld, const float* __restrict__ chanadd, int ca_ld,
                                                            const float* __restrict__ residual, int ldr, StatAcc* __restrict__ stats,
                                                            int st_ld, int ppc) {
  pdl_prologue();
  const int n = blockIdx.y, p0 = blockIdx.x * ppc, p1 = min(HW, p0 + ppc);
  for (int c4 = threadIdx.x; c4 < (C >> 2); c4 += blockDim.x) {
    const int c = c4 * 4;
    const float4 ca = chanadd ? __ldg(reinterpret_cast<const float4*>(chanadd + (size_t)n * ca_ld + c)) : make_float4(0.f, 0.f, 0.f, 0.f);
    float s4[4] = {0.f, 0.f, 0.f, 0.f}, q4[4] = {0.f, 0.f, 0.f, 0.f};
    for (int p = p0; p < p1; ++p) {
      const size_t pix = (size_t)n * HW + p;
      float4 a = *reinterpret_cast<const float4*>(part + pix * C + c);
      for (int k = 1; k < S; ++k) {
        const float4 b = *reinterpret_cast<const float4*>(part + (size_t)k * stride + pix * C + c);
        a.x += b.x; a.y += b.y; a.z += b.z; a.w += b.w;
      }
      a.x += ca.x; a.y += ca.y; a.z += ca.z; a.w += ca.w;
      if (residual) {
        const float4 r = *reinterpret_cast<const float4*>(residual + pix * ldr + c);
        a.x += r.x; a.y += r.y; a.z += r.z; a.w += r.w;
      }
      *reinterpret_cast<float4*>(out + pix * ld + c) = a;
      s4[0] += a.x; s4[1] += a.y; s4[2] += a.z; s4[3] += a.w;
      q4[0] = fmaf(a.x, a.x, q4[0]); q4[1] = fmaf(a.y, a.y, q4[1]); q4[2] = fmaf(a.z, a.z, q4[2]); q4[3] = fmaf(a.w, a.w, q4[3]);
    }
    if (stats) {
#pragma unroll
      for (int j = 0; j < 4; ++j) {
        StatAcc* d = stats + ((size_t)n * st_ld + c + j) * 2;
        stat_add(d, s4[j]);
        stat_add(d + 1, q4[j]);
      }
    }
  }
}
void splitk_reduce(const float* part, int S, long long stride, const View& out, const float* chanadd, int ca_ld, const float* residual,
                   int ldr, cudaStream_t st) {
  DDNM_CHECK(out.C % 4 == 0 && out.ld % 4 == 0 && S >= 2, "split-K reduce: unsupported shape");
  const int HW = out.H * out.W;
  // a CTA reduces 2048 values of one image (ppc pixels x C channels): the fp32 grouping of the GroupNorm sums then depends on the
  // layer's shape only, so a row's result is the same in an engine of any batch size (a ragged last batch rides on a bigger engine)
  const int ppc = std::max(1, 2048 / out.C);
  dim3 grid(cdiv(HW, ppc), out.N);
  launch_pdl(splitk_reduce_kernel, grid, dim3(std::min(256, out.C / 4)), 0, st, 1, part, S, stride, HW, out.C, out.p, out.ld, chanadd, ca_ld, residual,
             ldr, out.st, out.st_ld, ppc);
  CUDA_CHECK(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------------------------
// Timestep MLP pieces (models.py:6-24, 305-308, 121).  One warp per output element.
// ---------------------------------------------------------------------------------------------------------------
// The activations (N x K, act_in applied once) are staged in shared memory; each warp then produces LIN_OPW output features,
// reading each weight row exactly once with 16-byte loads and reusing it for every image of the batch.
constexpr int LIN_NB = 16;    // images per accumulator pass
constexpr int LIN_OPW = 2;    // output features per warp (8 left a 512-feature layer with 8 CTAs: 40-50 us of pure latency each)
constexpr int LIN_WREG = 8;   // float4 weight registers per lane loaded ahead (K <= 1024 in one go)
__global__ void __launch_bounds__(256) linear_kernel(const float* __restrict__ in, int N, int K, const float* __restrict__ W,
                                                     const float* __restrict__ bias, int O, float* __restrict__ out, int ldo,
                                                     int act_in, int act_out) {
  extern __shared__ float lin_in[];
  for (int i = threadIdx.x; i < N * K; i += 256) {
    float v = in[i];
    if (act_in) v = swishf(v);
    lin_in[i] = v;
  }
  __syncthreads();
  const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
  const int o0 = (blockIdx.x * 8 + warp) * LIN_OPW;
  const int K4 = K >> 2;
  for (int oo = 0; oo < LIN_OPW; ++oo) {
    const int o = o0 + oo;
    if (o >= O) return;
    const float4* w4 = reinterpret_cast<const float4*>(W + (long long)o * K);
    for (int n0 = 0; n0 < N; n0 += LIN_NB) {
      float acc[LIN_NB];
#pragma unroll
      for (int j = 0; j < LIN_NB; ++j) acc[j] = 0.f;
      // the whole weight row first (independent loads, one latency), then the products
      for (int kbase = 0; kbase < K4; kbase += 32 * LIN_WREG) {
        float4 wv[LIN_WREG];
#pragma unroll
        for (int i = 0; i < LIN_WREG; ++i) {
          const int k4 = kbase + lane + 32 * i;
          wv[i] = k4 < K4 ? __ldg(w4 + k4) : make_float4(0.f, 0.f, 0.f, 0.f);
        }
#pragma unroll
        for (int i = 0; i < LIN_WREG; ++i) {
          const int k4 = kbase + lane + 32 * i;
          if (k4 < K4) {
#pragma unroll
            for (int j = 0; j < LIN_NB; ++j) {
              if (n0 + j < N) {
                const float4 v = reinterpret_cast<const float4*>(lin_in + (long long)(n0 + j) * K)[k4];
                acc[j] = fmaf(v.x, wv[i].x, fmaf(v.y, wv[i].y, fmaf(v.z, wv[i].z, fmaf(v.w, wv[i].w, acc[j]))));
              }
            }
          }
        }
      }
#pragma unroll
      for (int j = 0; j < LIN_NB; ++j) {
        float a = acc[j];
#pragma unroll
        for (int s = 16; s > 0; s >>= 1) a += __shfl_xor_sync(0xffffffffu, a, s);
        if (lane == 0 && n0 + j < N) {
          float r = a + (bias ? bias[o] : 0.f);
          if (act_out) r = swishf(r);
          out[(long long)(n0 + j) * ldo + o] = r;
        }
      }
    }
  }
}
void linear(const float* in, int N, int K, const float* W, const float* bias, int O, float* out, int ldo, int act_in,
            int act_out, cudaStream_t st) {
  DDNM_CHECK(K % 4 == 0, "linear: K must be a multiple of 4");
  static bool attr[64] = {};
  constexpr int kMaxSmem = 160 * 1024;
  if (first_use_on_device(attr)) CUDA_CHECK(cudaFuncSetAttribute(linear_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, kMaxSmem));
  const int rows_max = std::max(1, kMaxSmem / (K * 4));
  for (int n0 = 0; n0 < N; n0 += rows_max) {     // batches whose activations exceed the staging buffer go in row chunks
    const int n = std::min(rows_max, N - n0);
    linear_kernel<<<cdiv(O, 8 * LIN_OPW), 256, (size_t)n * K * 4, st>>>(in + (long long)n0 * K, n, K, W, bias, O,
                                                                         out + (long long)n0 * ldo, ldo, act_in, act_out);
  }
  CUDA_CHECK(cudaGetLastError());
}

__global__ void add_label_swish_kernel(float* __restrict__ v, const float* __restrict__ table, const int* __restrict__ labels, int N,
                                       int D, int num_classes) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  if (i >= N * D) return;
  const int n = i / D, d = i - n * D;
  const int y = labels[n];
  if (y < 0 || y >= num_classes) {
    if (d == 0) printf("ddnm_b200: class label %d of image %d is outside [0, %d)\n", y, n, num_classes);
    __trap();
  }
  v[i] = swishf(v[i] + table[(size_t)y * D + d]);
}
void add_label_swish(float* v, const float* table, const int* labels, int N, int D, int num_classes, cudaStream_t st) {
  add_label_swish_kernel<<<cdiv(N * D, 256), 256, 0, st>>>(v, table, labels, N, D, num_classes);
  CUDA_CHECK(cudaGetLastError());
}

__global__ void sinusoid_kernel(const float* __restrict__ t, int N, const float* __restrict__ freq, int dim, int sin_first,
                                float* __restrict__ emb) {
  const int i = blockIdx.x * blockDim.x + threadIdx.x;
  const int half = dim / 2;
  if (i >= N * half) return;
  const int n = i / half, k = i % half;
  const float a = t[n] * freq[k];
  const float s = sinf(a), c = cosf(a);
  emb[(long long)n * dim + k] = sin_first ? s : c;
  emb[(long long)n * dim + half + k] = sin_first ? c : s;
}
void sinusoid(const float* t, int N, const float* freq, int dim, bool sin_first, float* emb, cudaStream_t st) {
  sinusoid_kernel<<<cdiv(N * (dim / 2), 128), 128, 0, st>>>(t, N, freq, dim, sin_first ? 1 : 0, emb);
  CUDA_CHECK(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------------------------
// Batched fp32 GEMM, 64x64x16 tiles, 4x4 per thread (torch.bmm in AttnBlock, models.py:177,185).
// ---------------------------------------------------------------------------------------------------------------
template <bool BT>
__global__ void __launch_bounds__(256) sgemm_kernel(int M, int N, int K, float alpha, const float* __restrict__ A, int lda,
                                                    long long sa, long long sa2, const float* __restrict__ B, int ldb,
                                                    long long sb, long long sb2, float* __restrict__ C, int ldc, long long sc,
                                                    long long sc2, int inner_n) {
  pdl_prologue();
  constexpr int SK = 32;   // k depth of a shared-memory tile
  __shared__ float As[SK][64 + 4], Bs[SK][64 + 4];
  const int bo = blockIdx.z / inner_n, bi = blockIdx.z % inner_n;
  A += bo * sa + bi * sa2; B += bo * sb + bi * sb2; C += bo * sc + bi * sc2;
  const int m0 = blockIdx.y * 64, n0 = blockIdx.x * 64;
  const int tx = threadIdx.x % 16, ty = threadIdx.x / 16;
  float acc[4][4] = {};
  for (int k0 = 0; k0 < K; k0 += SK) {
    for (int i = threadIdx.x; i < 64 * SK; i += 256) {
      const int kk = i % SK, mm = i / SK;
      As[kk][mm] = (m0 + mm < M && k0 + kk < K) ? A[(long long)(m0 + mm) * lda + k0 + kk] : 0.f;
    }
    if (BT) {
      for (int i = threadIdx.x; i < 64 * SK; i += 256) {
        const int kk = i % SK, nn = i / SK;
        Bs[kk][nn] = (n0 + nn < N && k0 + kk < K) ? B[(long long)(n0 + nn) * ldb + k0 + kk] : 0.f;
      }
    } else {
      for (int i = threadIdx.x; i < 64 * SK; i += 256) {
        const int nn = i % 64, kk = i / 64;
        Bs[kk][nn] = (n0 + nn < N && k0 + kk < K) ? B[(long long)(k0 + kk) * ldb + n0 + nn] : 0.f;
      }
    }
    __syncthreads();
#pragma unroll
    for (int kk = 0; kk < SK; ++kk) {
      float a[4], bb[4];
#pragma unroll
      for (int i = 0; i < 4; ++i) a[i] = As[kk][ty * 4 + i];
#pragma unroll
      for (int j = 0; j < 4; ++j) bb[j] = Bs[kk][tx * 4 + j];
#pragma unroll
      for (int i = 0; i < 4; ++i)
#pragma unroll
        for (int j = 0; j < 4; ++j) acc[i][j] = fmaf(a[i], bb[j], acc[i][j]);
    }
    __syncthreads();
  }
#pragma unroll
  for (int i = 0; i < 4; ++i)
#pragma unroll
    for (int j = 0; j < 4; ++j) {
      const int m = m0 + ty * 4 + i, n = n0 + tx * 4 + j;
      if (m < M && n < N) C[(long long)m * ldc + n] = alpha * acc[i][j];
    }
}
void sgemm_batched(bool bt, int outer_n, int inner_n, int M, int N, int K, float alpha, const float* A, int lda, long long sa,
                   long long sa2, const float* B, int ldb, long long sb, long long sb2, float* C, int ldc, long long sc,
                   long long sc2, cudaStream_t st) {
  dim3 grid(cdiv(N, 64), cdiv(M, 64), outer_n * inner_n);
  DDNM_CHECK(grid.z <= 65535, "too many GEMM batches for one launch");
  if (bt)
    launch_pdl(sgemm_kernel<true>, grid, dim3(256), 0, st, 1, M, N, K, alpha, A, lda, sa, sa2, B, ldb, sb, sb2, C, ldc, sc, sc2, inner_n);
  else
    launch_pdl(sgemm_kernel<false>, grid, dim3(256), 0, st, 1, M, N, K, alpha, A, lda, sa, sa2, B, ldb, sb, sb2, C, ldc, sc, sc2, inner_n);
  CUDA_CHECK(cudaGetLastError());
}

// softmax over the last dim, one warp per row (F.softmax(w_, dim=2), models.py:179)
__global__ void softmax_kernel(float* __restrict__ x, long long rows, int cols) {
  pdl_prologue();
  const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  float* r = x + row * cols;
  float m = -INFINITY;
  for (int i = lane; i < cols; i += 32) m = fmaxf(m, r[i]);
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, s));
  float sum = 0.f;
  for (int i = lane; i < cols; i += 32) {
    const float e = expf(r[i] - m);
    r[i] = e;
    sum += e;
  }
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, s);
  const float inv = 1.0f / sum;
  for (int i = lane; i < cols; i += 32) r[i] *= inv;
}
// softmax over the last dim with the probabilities emitted as fp16 (hi, lo) planes — the A operand of the P.V GEMM
__global__ void softmax_split_kernel(const float* __restrict__ x, long long rows, int cols, __half* __restrict__ hi,
                                     __half* __restrict__ lo) {
  pdl_prologue();
  const long long row = ((long long)blockIdx.x * blockDim.x + threadIdx.x) >> 5;
  const int lane = threadIdx.x & 31;
  if (row >= rows) return;
  const float* r = x + row * cols;
  float m = -INFINITY;
  for (int i = lane; i < cols; i += 32) m = fmaxf(m, r[i]);
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) m = fmaxf(m, __shfl_xor_sync(0xffffffffu, m, s));
  float sum = 0.f;
  for (int i = lane; i < cols; i += 32) sum += expf(r[i] - m);
#pragma unroll
  for (int s = 16; s > 0; s >>= 1) sum += __shfl_xor_sync(0xffffffffu, sum, s);
  const float inv = 1.0f / sum;
  for (int i = lane * 2; i < cols; i += 64) {
    __half h0, l0, h1, l1;
    split_f16(expf(r[i] - m) * inv, h0, l0);
    split_f16(expf(r[i + 1] - m) * inv, h1, l1);
    *reinterpret_cast<__half2*>(hi + row * cols + i) = __halves2half2(h0, h1);
    *reinterpret_cast<__half2*>(lo + row * cols + i) = __halves2half2(l0, l1);
  }
}
void softmax_split(const float* x, long long rows, int cols, __half* hi, __half* lo, cudaStream_t st) {
  DDNM_CHECK(cols % 2 == 0, "softmax_split: even row length");
  launch_pdl(softmax_split_kernel, dim3((unsigned)cdivll(rows * 32, 256)), dim3(256), 0, st, 1, x, rows, cols, hi, lo);
  CUDA_CHECK(cudaGetLastError());
}

// V^T planes for the P.V GEMM: src[(img*T + t)*ld + head*head_stride + off + c] -> dst[((img*heads + head)*ch + c)*T + t]
__global__ void transpose_split_kernel(const float* __restrict__ src, int ld, int head_stride, int off, int T, int heads, int ch,
                                       __half* __restrict__ hi, __half* __restrict__ lo) {
  pdl_prologue();
  __shared__ float tile[32][33];
  const int img = blockIdx.z / heads, head = blockIdx.z % heads;
  const int t0 = blockIdx.x * 32, c0 = blockIdx.y * 32;
  const int tx = threadIdx.x & 31, ty = threadIdx.x >> 5;  // 32 x 8
  for (int j = ty; j < 32; j += 8) {
    const int t = t0 + j, c = c0 + tx;
    tile[j][tx] = (t < T && c < ch) ? src[((size_t)img * T + t) * ld + (size_t)head * head_stride + off + c] : 0.f;
  }
  __syncthreads();
  for (int j = ty; j < 32; j += 8) {
    const int c = c0 + j, t = t0 + tx;
    if (c < ch && t < T) {
      __half h, l;
      split_f16(tile[tx][j], h, l);
      const size_t o = (((size_t)img * heads + head) * ch + c) * T + t;
      hi[o] = h;
      lo[o] = l;
    }
  }
}
void transpose_split(const float* src, int ld, int head_stride, int off, int images, int T, int heads, int ch, __half* hi,
                     __half* lo, cudaStream_t st) {
  dim3 grid(cdiv(T, 32), cdiv(ch, 32), images * heads);
  launch_pdl(transpose_split_kernel, grid, dim3(256), 0, st, 1, src, ld, head_stride, off, T, heads, ch, hi, lo);
  CUDA_CHECK(cudaGetLastError());
}

void softmax_rows(float* x, long long rows, int cols, cudaStream_t st) {
  launch_pdl(softmax_kernel, dim3((unsigned)cdivll(rows * 32, 256)), dim3(256), 0, st, 1, x, rows, cols);
  CUDA_CHECK(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------------------------
// weight preparation (once per model load)
// ---------------------------------------------------------------------------------------------------------------
__global__ void split_weight_kernel(const float* __restrict__ w, int Cout, int Cin, int taps, __half* __restrict__ hi,
                                    __half* __restrict__ lo, int ktot, int koff) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)Cout * Cin * taps;
  if (i >= total) return;
  const int ci = (int)(i % Cin);
  const int tap = (int)((i / Cin) % taps);
  const int co = (int)(i / ((long long)Cin * taps));
  const float v = w[((long long)co * Cin + ci) * taps + tap];
  __half h, l;
  split_f16(v, h, l);
  const long long o = (long long)co * ktot + koff + (long long)tap * Cin + ci;
  hi[o] = h;
  lo[o] = l;
}
// Phase weights of conv3x3(nearest_upsample_x2(.)): output parity (py, px) sees a 2x2 stencil on the low-res input whose
// taps are sums of the 3x3 taps that land on the same source pixel (rows: py=0 -> {0},{1,2}; py=1 -> {0,1},{2}; same for columns).
// dst[((py*2+px)*Cout + co)*4*Cin + (dy*2+dx)*Cin + ci]
__global__ void presum_up2_kernel(const float* __restrict__ w, int Cout, int Cin, __half* __restrict__ hi, __half* __restrict__ lo) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long per_phase = (long long)Cout * 4 * Cin;
  if (i >= 4 * per_phase) return;
  const int ci = (int)(i % Cin);
  const int tap = (int)((i / Cin) % 4);
  const int co = (int)((i / (4LL * Cin)) % Cout);
  const int ph = (int)(i / per_phase);
  const int py = ph >> 1, px = ph & 1, dy = tap >> 1, dx = tap & 1;
  const int r0 = py == 0 ? (dy == 0 ? 0 : 1) : (dy == 0 ? 0 : 2), r1 = py == 0 ? (dy == 0 ? 0 : 2) : (dy == 0 ? 1 : 2);
  const int c0 = px == 0 ? (dx == 0 ? 0 : 1) : (dx == 0 ? 0 : 2), c1 = px == 0 ? (dx == 0 ? 0 : 2) : (dx == 0 ? 1 : 2);
  const float* wp = w + ((long long)co * Cin + ci) * 9;
  float acc = 0.f;
  for (int r = r0; r <= r1; ++r)
    for (int c = c0; c <= c1; ++c) acc += wp[r * 3 + c];
  __half h, l;
  split_f16(acc, h, l);
  hi[i] = h;
  lo[i] = l;
}
void presum_up2_weights(const float* w_oihw, int Cout, int Cin, __half* hi, __half* lo, cudaStream_t st) {
  const long long total = 4LL * Cout * 4 * Cin;
  presum_up2_kernel<<<(int)cdivll(total, 256), 256, 0, st>>>(w_oihw, Cout, Cin, hi, lo);
  CUDA_CHECK(cudaGetLastError());
}

void split_conv_weight(const float* w, int Cout, int Cin, int taps, __half* hi, __half* lo, int ktot, int koff, cudaStream_t st) {
  const long long total = (long long)Cout * Cin * taps;
  split_weight_kernel<<<(int)cdivll(total, 256), 256, 0, st>>>(w, Cout, Cin, taps, hi, lo, ktot, koff);
  CUDA_CHECK(cudaGetLastError());
}

// ---------------------------------------------------------------------------------------------------------------
// Direct convolution, one thread per output element (validation only).
// ---------------------------------------------------------------------------------------------------------------
__global__ void conv_direct_kernel(const float* __restrict__ x, int xH, int xW, int Cin, int xld, const float* __restrict__ w,
                                   const float* __restrict__ bias, int mode, int up2, float* __restrict__ out, int N, int H,
                                   int W, int Cout, int old) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)N * H * W * Cout;
  if (i >= total) return;
  const int co = (int)(i % Cout);
  const long long pix = i / Cout;
  const int ox = (int)(pix % W), oy = (int)((pix / W) % H), n = (int)(pix / ((long long)W * H));
  const int taps = mode == TAPS_1X1 ? 1 : 9;
  const int inH = up2 ? 2 * xH : xH, inW = up2 ? 2 * xW : xW;  // logical (post-upsample) input size
  float acc = bias ? bias[co] : 0.f;
  for (int tap = 0; tap < taps; ++tap) {
    int iy, ix;
    if (mode == TAPS_1X1) { iy = oy; ix = ox; }
    else if (mode == TAPS_3X3) { iy = oy + tap / 3 - 1; ix = ox + tap % 3 - 1; }
    else { iy = 2 * oy + tap / 3; ix = 2 * ox + tap % 3; }
    if (iy < 0 || iy >= inH || ix < 0 || ix >= inW) continue;
    if (up2) { iy >>= 1; ix >>= 1; }
    const float* xp = x + (((long long)n * xH + iy) * xW + ix) * xld;
    const float* wp = w + (long long)co * Cin * taps + tap;
    for (int ci = 0; ci < Cin; ++ci) acc = fmaf(xp[ci], wp[(long long)ci * taps], acc);
  }
  out[pix * old + co] = acc;
}
void conv_direct_ref(const View& x, const float* w, const float* bias, int mode, bool up2, const View& out, cudaStream_t st) {
  const long long total = out.pixels() * out.C;
  conv_direct_kernel<<<(int)cdivll(total, 256), 256, 0, st>>>(x.p, x.H, x.W, x.C, x.ld, w, bias, mode, up2 ? 1 : 0, out.p, out.N,
                                                             out.H, out.W, out.C, out.ld);
  CUDA_CHECK(cudaGetLastError());
}

__global__ void nchw_to_nhwc_kernel(const float* __restrict__ s, int N, int C, int H, int W, float* __restrict__ d, int ld) {
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)N * C * H * W;
  if (i >= total) return;
  const int c = (int)(i % C);
  const long long pix = i / C;
  const long long hw = pix % ((long long)H * W);
  const int n = (int)(pix / ((long long)H * W));
  d[pix * ld + c] = s[((long long)n * C + c) * H * W + hw];
}
void nchw_to_nhwc(const float* src, int N, int C, int H, int W, const View& dst, cudaStream_t st) {
  const long long total = (long long)N * C * H * W;
  nchw_to_nhwc_kernel<<<(int)cdivll(total, 256), 256, 0, st>>>(src, N, C, H, W, dst.p, dst.ld);
  CUDA_CHECK(cudaGetLastError());
}
__global__ void nhwc_to_nchw_kernel(const float* __restrict__ s, int N, int C, int H, int W, int ld, float* __restrict__ d) {
  pdl_prologue();
  const long long i = (long long)blockIdx.x * blockDim.x + threadIdx.x;
  const long long total = (long long)N * C * H * W;
  if (i >= total) return;
  const long long hw = i % ((long long)H * W);
  const int c = (int)((i / ((long long)H * W)) % C);
  const int n = (int)(i / ((long long)H * W * C));
  d[i] = s[((long long)n * H * W + hw) * ld + c];
}
void nhwc_to_nchw(const View& src, float* dst, cudaStream_t st) {
  const long long total = src.pixels() * src.C;
  launch_pdl(nhwc_to_nchw_kernel, dim3((unsigned)cdivll(total, 256)), dim3(256), 0, st, 1, (const float*)src.p, src.N, src.C, src.H, src.W, src.ld, dst);
  CUDA_CHECK(cudaGetLastError());
}

}  // namespace ddnm
