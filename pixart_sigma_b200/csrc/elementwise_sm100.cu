// HBM-bound helper kernels of the block: LayerNorm + adaLN-single modulate, KV token compression.
// One warp per token row, 128-bit loads/stores, fp32 statistics (two-pass over registers: mean, then variance).
#include "host_common.cuh"
#include "ptx.cuh"

#ifndef PXA_LN_CTAS_PER_SM
#define PXA_LN_CTAS_PER_SM 2
#endif

namespace pxa {

PXA_DEVICE float warp_sum(float v) {
#pragma unroll
  for (int o = 16; o > 0; o >>= 1) v += __shfl_xor_sync(0xffffffffu, v, o);
  return v;
}

// ------------------------------------------------------------------------------------------------- LN + modulate
// C = 32 lanes * kVec * 4 elements (1152 -> kVec = 9). Each lane owns kVec float4 groups, group g at column
// (g*32 + lane)*4, so every warp-level access is a contiguous 512 B (fp32) / 256 B (bf16) segment.
// Grid-stride over the rows with the NEXT row's loads issued before the current row is reduced: a warp always has one full row
// (4.6 KB fp32) in flight, and the grid is a fixed number of CTAs per SM instead of M / 8 short-lived ones (round 2: the
// one-row-per-warp launch ran at 4.4 TB/s).
template <int kVec, typename XT>
PXA_DEVICE void ln_load_row(const XT* __restrict__ xr, int lane, float4 (&v)[kVec]) {
#pragma unroll
  for (int g = 0; g < kVec; ++g) {
    const int col = (g * 32 + lane) * 4;
    if constexpr (sizeof(XT) == 4) {
      v[g] = *reinterpret_cast<const float4*>(xr + col);
    } else {
      uint2 u = *reinterpret_cast<const uint2*>(xr + col);
      v[g] = make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
    }
  }
}

template <int kVec, typename XT>
__global__ void __launch_bounds__(256, 2) ln_modulate_kernel(const XT* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                                             const float* __restrict__ shift,
                                                             const float* __restrict__ scale, long long mod_bs,
                                                             int rows_per_batch, int M, int ldx, float eps, int reverse) {
  constexpr int C = kVec * 128;
  const int lane = threadIdx.x & 31;
  const int stride = gridDim.x * 8;
  int r = blockIdx.x * 8 + (threadIdx.x >> 5);
  if (r >= M) return;
  float4 v[kVec], nxt[kVec];
  ln_load_row<kVec, XT>(x + (size_t)(reverse ? M - 1 - r : r) * ldx, lane, v);
  for (; r < M; r += stride) {
    const int row = reverse ? M - 1 - r : r;
    const bool more = r + stride < M;
    if (more) ln_load_row<kVec, XT>(x + (size_t)(reverse ? M - 1 - (r + stride) : r + stride) * ldx, lane, nxt);
    float s = 0.f;
#pragma unroll
    for (int g = 0; g < kVec; ++g) s += (v[g].x + v[g].y) + (v[g].z + v[g].w);
    const float mean = warp_sum(s) * (1.0f / C);
    float ss = 0.f;
#pragma unroll
    for (int g = 0; g < kVec; ++g) {
      const float a = v[g].x - mean, b = v[g].y - mean, c = v[g].z - mean, d = v[g].w - mean;
      ss += (a * a + b * b) + (c * c + d * d);
    }
    const float rstd = rsqrtf(warp_sum(ss) * (1.0f / C) + eps);
    const int bidx = row / rows_per_batch;
    const float* sh = shift + (size_t)bidx * mod_bs;
    const float* sc = scale + (size_t)bidx * mod_bs;
    __nv_bfloat16* orow = out + (size_t)row * C;
#pragma unroll
    for (int g = 0; g < kVec; ++g) {
      const int col = (g * 32 + lane) * 4;
      const float4 a = __ldg(reinterpret_cast<const float4*>(sc + col));
      const float4 b = __ldg(reinterpret_cast<const float4*>(sh + col));
      const float y0 = fmaf((v[g].x - mean) * rstd, 1.0f + a.x, b.x);
      const float y1 = fmaf((v[g].y - mean) * rstd, 1.0f + a.y, b.y);
      const float y2 = fmaf((v[g].z - mean) * rstd, 1.0f + a.z, b.z);
      const float y3 = fmaf((v[g].w - mean) * rstd, 1.0f + a.w, b.w);
      *reinterpret_cast<uint2*>(orow + col) = make_uint2(pack_bf16x2(y0, y1), pack_bf16x2(y2, y3));
    }
    if (more) {
#pragma unroll
      for (int g = 0; g < kVec; ++g) v[g] = nxt[g];
    }
  }
}

// ------------------------------------------------------------------------------------------------- KV compress
// Depthwise 2x2 stride-2 conv + bias, then LayerNorm(affine) over channels; one warp per OUTPUT token, blockIdx.y
// selects K (0) or V (1). Reads 4 input rows (bf16), writes one row.
template <int kVec>
__global__ void __launch_bounds__(256) kv_compress_kernel(const __nv_bfloat16* __restrict__ k_in,
                                                          const __nv_bfloat16* __restrict__ v_in,
                                                          __nv_bfloat16* __restrict__ k_out,
                                                          __nv_bfloat16* __restrict__ v_out,
                                                          const __nv_bfloat16* __restrict__ conv_w,
                                                          const __nv_bfloat16* __restrict__ conv_b,
                                                          const __nv_bfloat16* __restrict__ ln_w,
                                                          const __nv_bfloat16* __restrict__ ln_b, int B, int H, int W,
                                                          int ld_in, float eps) {
  constexpr int C = kVec * 128;
  const int Ho = H >> 1, Wo = W >> 1;
  const int orow = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (orow >= B * Ho * Wo) return;
  const __nv_bfloat16* in = blockIdx.y == 0 ? k_in : v_in;
  __nv_bfloat16* out = blockIdx.y == 0 ? k_out : v_out;
  const int b = orow / (Ho * Wo);
  const int p = orow % (Ho * Wo);
  const int py = p / Wo, px = p % Wo;
  const __nv_bfloat16* base = in + ((size_t)b * H * W + (size_t)(2 * py) * W + 2 * px) * ld_in;
  float4 acc[kVec];
#pragma unroll
  for (int g = 0; g < kVec; ++g) {
    const int col = (g * 32 + lane) * 4;
    // conv weight [C,1,2,2]: channel c taps at conv_w[c*4 + dy*2 + dx]; 4 channels = 16 bf16 = 2 x 16 B
    const uint4 w01 = __ldg(reinterpret_cast<const uint4*>(conv_w + col * 4));
    const uint4 w23 = __ldg(reinterpret_cast<const uint4*>(conv_w + col * 4 + 8));
    const uint2 bb = __ldg(reinterpret_cast<const uint2*>(conv_b + col));
    float4 a = make_float4(bf16_lo(bb.x), bf16_hi(bb.x), bf16_lo(bb.y), bf16_hi(bb.y));
    const float wt[4][4] = {{bf16_lo(w01.x), bf16_hi(w01.x), bf16_lo(w01.y), bf16_hi(w01.y)},
                            {bf16_lo(w01.z), bf16_hi(w01.z), bf16_lo(w01.w), bf16_hi(w01.w)},
                            {bf16_lo(w23.x), bf16_hi(w23.x), bf16_lo(w23.y), bf16_hi(w23.y)},
                            {bf16_lo(w23.z), bf16_hi(w23.z), bf16_lo(w23.w), bf16_hi(w23.w)}};
#pragma unroll
    for (int t = 0; t < 4; ++t) {  // tap t = dy*2 + dx
      const uint2 u = *reinterpret_cast<const uint2*>(base + ((size_t)(t >> 1) * W + (t & 1)) * ld_in + col);
      a.x = fmaf(wt[0][t], bf16_lo(u.x), a.x);
      a.y = fmaf(wt[1][t], bf16_hi(u.x), a.y);
      a.z = fmaf(wt[2][t], bf16_lo(u.y), a.z);
      a.w = fmaf(wt[3][t], bf16_hi(u.y), a.w);
    }
    acc[g] = a;   // kept in fp32 through the LayerNorm (more precise than the reference's bf16 conv output)
  }
  float s = 0.f;
#pragma unroll
  for (int g = 0; g < kVec; ++g) s += (acc[g].x + acc[g].y) + (acc[g].z + acc[g].w);
  const float mean = warp_sum(s) * (1.0f / C);
  float ss = 0.f;
#pragma unroll
  for (int g = 0; g < kVec; ++g) {
    const float a = acc[g].x - mean, b2 = acc[g].y - mean, c = acc[g].z - mean, d = acc[g].w - mean;
    ss += (a * a + b2 * b2) + (c * c + d * d);
  }
  const float rstd = rsqrtf(warp_sum(ss) * (1.0f / C) + eps);
  __nv_bfloat16* orowp = out + (size_t)orow * C;
#pragma unroll
  for (int g = 0; g < kVec; ++g) {
    const int col = (g * 32 + lane) * 4;
    const uint2 gw = __ldg(reinterpret_cast<const uint2*>(ln_w + col));
    const uint2 gb = __ldg(reinterpret_cast<const uint2*>(ln_b + col));
    const float y0 = fmaf((acc[g].x - mean) * rstd, bf16_lo(gw.x), bf16_lo(gb.x));
    const float y1 = fmaf((acc[g].y - mean) * rstd, bf16_hi(gw.x), bf16_hi(gb.x));
    const float y2 = fmaf((acc[g].z - mean) * rstd, bf16_lo(gw.y), bf16_lo(gb.y));
    const float y3 = fmaf((acc[g].w - mean) * rstd, bf16_hi(gw.y), bf16_hi(gb.y));
    *reinterpret_cast<uint2*>(orowp + col) = make_uint2(pack_bf16x2(y0, y1), pack_bf16x2(y2, y3));
  }
}

}  // namespace pxa

extern "C" int pxa_ln_modulate(const PxaLnModArgs* args, void* stream) {
  using namespace pxa;
  if (!args) return fail(PXA_ERR_ARG, "null args");
  const PxaLnModArgs& a = *args;
  if (!a.x || !a.out || !a.shift || !a.scale) return fail(PXA_ERR_ARG, "null pointer");
  if (a.C != 1152) return fail(PXA_ERR_ARG, "pxa_ln_modulate is specialised for C=1152 (got %d)", a.C);
  if (a.M <= 0 || a.rows_per_batch <= 0) return fail(PXA_ERR_ARG, "bad M / rows_per_batch");
  if ((a.ldx & 3) || (a.mod_batch_stride & 3)) return fail(PXA_ERR_ALIGN, "ldx / mod_batch_stride must be multiples of 4");
  if ((reinterpret_cast<uintptr_t>(a.x) | reinterpret_cast<uintptr_t>(a.out) | reinterpret_cast<uintptr_t>(a.shift) |
       reinterpret_cast<uintptr_t>(a.scale)) & 15)
    return fail(PXA_ERR_ALIGN, "pointers must be 16-byte aligned");
  PXA_REQUIRE_SM100();
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  int grid = (a.M + 7) / 8;
  const int resident = device_info().sms * PXA_LN_CTAS_PER_SM;               // grid-stride: a fixed number of CTAs per SM
  if (a.max_ctas > 0) { if (grid > a.max_ctas) grid = a.max_ctas; }
  else if (grid > resident) grid = resident;
  if (a.x_dtype == PXA_DTYPE_F32)
    ln_modulate_kernel<9, float><<<grid, 256, 0, s>>>(reinterpret_cast<const float*>(a.x),
                                                      reinterpret_cast<__nv_bfloat16*>(a.out), a.shift, a.scale,
                                                      a.mod_batch_stride, a.rows_per_batch, a.M, a.ldx, a.eps, a.reverse_rows);
  else
    ln_modulate_kernel<9, __nv_bfloat16><<<grid, 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(a.x),
                                                              reinterpret_cast<__nv_bfloat16*>(a.out), a.shift,
                                                              a.scale, a.mod_batch_stride, a.rows_per_batch, a.M,
                                                              a.ldx, a.eps, a.reverse_rows);
  launch_counter()++;
  PXA_CHECK_CUDA(cudaGetLastError());
  return PXA_OK;
}

extern "C" int pxa_kv_compress_conv2_ln(const PxaKvCompressArgs* args, void* stream) {
  using namespace pxa;
  if (!args) return fail(PXA_ERR_ARG, "null args");
  const PxaKvCompressArgs& a = *args;
  if (!a.k_in || !a.v_in || !a.k_out || !a.v_out || !a.conv_w || !a.conv_b || !a.ln_w || !a.ln_b)
    return fail(PXA_ERR_ARG, "null pointer");
  if (a.C != 1152) return fail(PXA_ERR_ARG, "specialised for C=1152 (got %d)", a.C);
  if (a.B <= 0 || a.H < 2 || a.W < 2) return fail(PXA_ERR_ARG, "bad B/H/W");
  if (a.ld_in & 7) return fail(PXA_ERR_ALIGN, "ld_in must be a multiple of 8");
  if ((reinterpret_cast<uintptr_t>(a.k_in) | reinterpret_cast<uintptr_t>(a.v_in) | reinterpret_cast<uintptr_t>(a.k_out) |
       reinterpret_cast<uintptr_t>(a.v_out) | reinterpret_cast<uintptr_t>(a.conv_w) |
       reinterpret_cast<uintptr_t>(a.conv_b) | reinterpret_cast<uintptr_t>(a.ln_w) | reinterpret_cast<uintptr_t>(a.ln_b)) & 15)
    return fail(PXA_ERR_ALIGN, "pointers must be 16-byte aligned");
  PXA_REQUIRE_SM100();
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const int rows = a.B * (a.H / 2) * (a.W / 2);
  dim3 grid((rows + 7) / 8, 2);
  kv_compress_kernel<9><<<grid, 256, 0, s>>>(
      reinterpret_cast<const __nv_bfloat16*>(a.k_in), reinterpret_cast<const __nv_bfloat16*>(a.v_in),
      reinterpret_cast<__nv_bfloat16*>(a.k_out), reinterpret_cast<__nv_bfloat16*>(a.v_out),
      reinterpret_cast<const __nv_bfloat16*>(a.conv_w), reinterpret_cast<const __nv_bfloat16*>(a.conv_b),
      reinterpret_cast<const __nv_bfloat16*>(a.ln_w), reinterpret_cast<const __nv_bfloat16*>(a.ln_b), a.B, a.H, a.W,
      a.ld_in, a.eps);
  launch_counter()++;
  PXA_CHECK_CUDA(cudaGetLastError());
  return PXA_OK;
}

namespace pxa {

// ------------------------------------------------------------------------------------------------- DPM-Solver++ step
// One thread per 4 consecutive latent elements (hw % 4 == 0): CFG combine + data prediction + multistep update.
template <typename OT>
__global__ void __launch_bounds__(256) dpm_step_kernel(const OT* __restrict__ mo, float* __restrict__ x,
                                                       float* __restrict__ x0_prev, long long obs, int n, int hw,
                                                       float cfg, float sigma_s, float inv_alpha_s, float a, float b,
                                                       float c) {
  const int per_img = hw;                                    // 4 channels * hw elements / 4 per thread
  const long long total = (long long)n * per_img;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int img = (int)(i / per_img);
    const int e = (int)(i - (long long)img * per_img) * 4;   // element offset inside the image's [4, hw] block
    const OT* pu = mo + (size_t)img * obs + e;               // channel ch at ch*hw + p == contiguous [4, hw] prefix
    const OT* pc = mo + (size_t)(img + n) * obs + e;
    float eu[4], ec[4];
    if constexpr (sizeof(OT) == 4) {
      const float4 u = *reinterpret_cast<const float4*>(pu), v = *reinterpret_cast<const float4*>(pc);
      eu[0] = u.x; eu[1] = u.y; eu[2] = u.z; eu[3] = u.w;
      ec[0] = v.x; ec[1] = v.y; ec[2] = v.z; ec[3] = v.w;
    } else {
      const uint2 u = *reinterpret_cast<const uint2*>(pu), v = *reinterpret_cast<const uint2*>(pc);
      eu[0] = bf16_lo(u.x); eu[1] = bf16_hi(u.x); eu[2] = bf16_lo(u.y); eu[3] = bf16_hi(u.y);
      ec[0] = bf16_lo(v.x); ec[1] = bf16_hi(v.x); ec[2] = bf16_lo(v.y); ec[3] = bf16_hi(v.y);
    }
    const size_t off = (size_t)img * 4 * hw + e;
    const float4 xv = *reinterpret_cast<const float4*>(x + off);
    float4 pv = make_float4(0.f, 0.f, 0.f, 0.f);
    if (c != 0.f) pv = *reinterpret_cast<const float4*>(x0_prev + off);
    const float xs[4] = {xv.x, xv.y, xv.z, xv.w};
    const float ps[4] = {pv.x, pv.y, pv.z, pv.w};
    float xn[4], x0[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float eps = eu[k] + cfg * (ec[k] - eu[k]);
      x0[k] = (xs[k] - sigma_s * eps) * inv_alpha_s;
      xn[k] = a * xs[k] - b * x0[k] - c * (x0[k] - ps[k]);
    }
    *reinterpret_cast<float4*>(x + off) = make_float4(xn[0], xn[1], xn[2], xn[3]);
    *reinterpret_cast<float4*>(x0_prev + off) = make_float4(x0[0], x0[1], x0[2], x0[3]);
  }
}

}  // namespace pxa

extern "C" int pxa_dpm_solver_pp_step(const PxaDpmStepArgs* args, void* stream) {
  using namespace pxa;
  if (!args) return fail(PXA_ERR_ARG, "null args");
  const PxaDpmStepArgs& a = *args;
  if (!a.model_out || !a.x || !a.x0_prev) return fail(PXA_ERR_ARG, "null pointer");
  if (a.n <= 0 || a.hw <= 0 || (a.hw & 3)) return fail(PXA_ERR_ARG, "n > 0 and hw a positive multiple of 4 required (n=%d hw=%d)", a.n, a.hw);
  if (a.out_batch_stride < 4LL * a.hw) return fail(PXA_ERR_ARG, "out_batch_stride smaller than 4*hw");
  const int esz = a.out_dtype == PXA_DTYPE_F32 ? 4 : 2;
  if (a.out_dtype != PXA_DTYPE_F32 && a.out_dtype != PXA_DTYPE_BF16) return fail(PXA_ERR_ARG, "out_dtype must be PXA_DTYPE_F32 or PXA_DTYPE_BF16");
  if ((reinterpret_cast<uintptr_t>(a.model_out) & (4 * esz - 1)) || ((a.out_batch_stride * esz) & (4 * esz - 1)) ||
      ((reinterpret_cast<uintptr_t>(a.x) | reinterpret_cast<uintptr_t>(a.x0_prev)) & 15))
    return fail(PXA_ERR_ALIGN, "model_out / x / x0_prev must be aligned to 4 elements");
  PXA_REQUIRE_SM100();
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const long long total = (long long)a.n * a.hw;
  int grid = (int)((total + 255) / 256);
  const int cap = device_info().sms * 8;
  if (grid > cap) grid = cap;
  if (a.out_dtype == PXA_DTYPE_F32)
    dpm_step_kernel<float><<<grid, 256, 0, s>>>(reinterpret_cast<const float*>(a.model_out), a.x, a.x0_prev, a.out_batch_stride,
                                                a.n, a.hw, a.cfg_scale, a.sigma_s, a.inv_alpha_s, a.a, a.b, a.c);
  else
    dpm_step_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(a.model_out), a.x, a.x0_prev,
                                                        a.out_batch_stride, a.n, a.hw, a.cfg_scale, a.sigma_s, a.inv_alpha_s,
                                                        a.a, a.b, a.c);
  launch_counter()++;
  PXA_CHECK_CUDA(cudaGetLastError());
  return PXA_OK;
}

namespace pxa {

// ------------------------------------------------------------------------------------------------- SA-Solver step
// One thread per 4 consecutive latent elements (hw % 4 == 0): CFG combine + data prediction + corrector + next predictor.
// Explicitly rounded operations (no FMA contraction) so the pass reproduces the reference's sequence of float32 tensor ops.
struct SaStepScalars {
  float cfg, sigma, inv_alpha, cA, c0, c1, cN, pA, p0, p1, pN;
};

PXA_DEVICE float4 ld4(const float* p) { return *reinterpret_cast<const float4*>(p); }

template <typename OT>
PXA_DEVICE void ld_out4(const OT* p, float (&v)[4]) {
  if constexpr (sizeof(OT) == 4) {
    const float4 u = *reinterpret_cast<const float4*>(p);
    v[0] = u.x; v[1] = u.y; v[2] = u.z; v[3] = u.w;
  } else {
    const uint2 u = *reinterpret_cast<const uint2*>(p);
    v[0] = bf16_lo(u.x); v[1] = bf16_hi(u.x); v[2] = bf16_lo(u.y); v[3] = bf16_hi(u.y);
  }
}

// a * x + (b * y + c * z) + d * w, each product and sum rounded
PXA_DEVICE float pc_update(float a, float x, float b, float y, float c, float z, float d, float w) {
  return __fadd_rn(__fadd_rn(__fmul_rn(a, x), __fadd_rn(__fmul_rn(b, y), __fmul_rn(c, z))), __fmul_rn(d, w));
}

template <typename OT>
__global__ void __launch_bounds__(256) sa_step_kernel(const OT* __restrict__ mo, float* __restrict__ x,
                                                      float* __restrict__ xp, float* __restrict__ x0_prev,
                                                      const float* __restrict__ noise, const float* __restrict__ noise_next,
                                                      long long obs, int n, int hw, int cond_off, int has_corr,
                                                      SaStepScalars s) {
  const long long total = (long long)n * hw;                // 4 channels * hw elements / 4 per thread, per image
  const bool read_prev = has_corr || s.p1 != 0.f;
  for (long long i = blockIdx.x * (long long)blockDim.x + threadIdx.x; i < total; i += (long long)gridDim.x * blockDim.x) {
    const int img = (int)(i / hw);
    const int e = (int)(i - (long long)img * hw) * 4;        // element offset inside the image's [4, hw] block
    float ec[4], eps[4];
    ld_out4(mo + (size_t)(img + cond_off) * obs + e, ec);
    if (cond_off) {
      float eu[4];
      ld_out4(mo + (size_t)img * obs + e, eu);
#pragma unroll
      for (int k = 0; k < 4; ++k) eps[k] = __fadd_rn(eu[k], __fmul_rn(s.cfg, __fsub_rn(ec[k], eu[k])));
    } else {
#pragma unroll
      for (int k = 0; k < 4; ++k) eps[k] = ec[k];
    }
    const size_t off = (size_t)img * 4 * hw + e;
    const float4 pv4 = ld4(xp + off), nn4 = ld4(noise_next + off);
    float4 xv4 = pv4, nv4 = make_float4(0.f, 0.f, 0.f, 0.f), qv4 = nv4;
    if (has_corr) { xv4 = ld4(x + off); nv4 = ld4(noise + off); }
    if (read_prev) qv4 = ld4(x0_prev + off);
    const float p[4] = {pv4.x, pv4.y, pv4.z, pv4.w}, nn[4] = {nn4.x, nn4.y, nn4.z, nn4.w};
    const float xs[4] = {xv4.x, xv4.y, xv4.z, xv4.w}, nz[4] = {nv4.x, nv4.y, nv4.z, nv4.w};
    const float q[4] = {qv4.x, qv4.y, qv4.z, qv4.w};
    float x0[4], xc[4], xn[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      x0[k] = __fmul_rn(__fsub_rn(p[k], __fmul_rn(s.sigma, eps[k])), s.inv_alpha);
      xc[k] = has_corr ? pc_update(s.cA, xs[k], s.c0, x0[k], s.c1, q[k], s.cN, nz[k]) : p[k];
      xn[k] = pc_update(s.pA, xc[k], s.p0, x0[k], s.p1, q[k], s.pN, nn[k]);
    }
    *reinterpret_cast<float4*>(x + off) = make_float4(xc[0], xc[1], xc[2], xc[3]);
    *reinterpret_cast<float4*>(xp + off) = make_float4(xn[0], xn[1], xn[2], xn[3]);
    *reinterpret_cast<float4*>(x0_prev + off) = make_float4(x0[0], x0[1], x0[2], x0[3]);
  }
}

}  // namespace pxa

extern "C" int pxa_sa_solver_step(const PxaSaStepArgs* args, void* stream) {
  using namespace pxa;
  if (!args) return fail(PXA_ERR_ARG, "null args");
  const PxaSaStepArgs& a = *args;
  if (!a.model_out || !a.x || !a.x_pred || !a.x0_prev || !a.noise || !a.noise_next) return fail(PXA_ERR_ARG, "null pointer");
  if (a.n <= 0 || a.hw <= 0 || (a.hw & 3)) return fail(PXA_ERR_ARG, "n > 0 and hw a positive multiple of 4 required (n=%d hw=%d)", a.n, a.hw);
  if (a.cond_row_offset != 0 && a.cond_row_offset != a.n) return fail(PXA_ERR_ARG, "cond_row_offset must be 0 or n");
  if (a.out_batch_stride < 4LL * a.hw) return fail(PXA_ERR_ARG, "out_batch_stride smaller than 4*hw");
  if (a.out_dtype != PXA_DTYPE_F32 && a.out_dtype != PXA_DTYPE_BF16) return fail(PXA_ERR_ARG, "out_dtype must be PXA_DTYPE_F32 or PXA_DTYPE_BF16");
  const int esz = a.out_dtype == PXA_DTYPE_F32 ? 4 : 2;
  if ((reinterpret_cast<uintptr_t>(a.model_out) & (4 * esz - 1)) || ((a.out_batch_stride * esz) & (4 * esz - 1)) ||
      ((reinterpret_cast<uintptr_t>(a.x) | reinterpret_cast<uintptr_t>(a.x_pred) | reinterpret_cast<uintptr_t>(a.x0_prev) |
        reinterpret_cast<uintptr_t>(a.noise) | reinterpret_cast<uintptr_t>(a.noise_next)) & 15))
    return fail(PXA_ERR_ALIGN, "model_out / x / x_pred / x0_prev / noise / noise_next must be aligned to 4 elements");
  PXA_REQUIRE_SM100();
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  const long long total = (long long)a.n * a.hw;
  int grid = (int)((total + 255) / 256);
  const int cap = device_info().sms * 8;
  if (grid > cap) grid = cap;
  const SaStepScalars sc{a.cfg_scale, a.sigma, a.inv_alpha, a.cA, a.c0, a.c1, a.cN, a.pA, a.p0, a.p1, a.pN};
  if (a.out_dtype == PXA_DTYPE_F32)
    sa_step_kernel<float><<<grid, 256, 0, s>>>(reinterpret_cast<const float*>(a.model_out), a.x, a.x_pred, a.x0_prev, a.noise,
                                               a.noise_next, a.out_batch_stride, a.n, a.hw, a.cond_row_offset, a.has_corr, sc);
  else
    sa_step_kernel<__nv_bfloat16><<<grid, 256, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(a.model_out), a.x, a.x_pred,
                                                       a.x0_prev, a.noise, a.noise_next, a.out_batch_stride, a.n, a.hw,
                                                       a.cond_row_offset, a.has_corr, sc);
  launch_counter()++;
  PXA_CHECK_CUDA(cudaGetLastError());
  return PXA_OK;
}

namespace pxa {

// ------------------------------------------------------------------------------------------------- fused-LN chain: first link
// a = bf16(x * mult[b]) with mult = 1 + scale, stats[row][0] = (sum x, sum x^2), stats[row][1..] = 0 (see PXA_EPI_LN_BIAS).
// One warp per row like ln_modulate: reads x once (fp32), writes a once (bf16): (4 + 2) * C bytes per row.
template <int kVec>
__global__ void __launch_bounds__(256) ln_prepare_kernel(const float* __restrict__ x, __nv_bfloat16* __restrict__ a_out,
                                                         float* __restrict__ stats, const float* __restrict__ scale,
                                                         long long mod_bs, int rows_per_batch, int M, int ldx) {
  constexpr int C = kVec * 128;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float* xr = x + (size_t)row * ldx;
  const float* sc = scale + (size_t)(row / rows_per_batch) * mod_bs;
  __nv_bfloat16* orow = a_out + (size_t)row * C;
  float s = 0.f, q = 0.f;
#pragma unroll
  for (int g = 0; g < kVec; ++g) {
    const int col = (g * 32 + lane) * 4;
    const float4 v = *reinterpret_cast<const float4*>(xr + col);
    const float4 e = __ldg(reinterpret_cast<const float4*>(sc + col));
    s += (v.x + v.y) + (v.z + v.w);
    q = fmaf(v.x, v.x, fmaf(v.y, v.y, fmaf(v.z, v.z, fmaf(v.w, v.w, q))));
    *reinterpret_cast<uint2*>(orow + col) = make_uint2(pack_bf16x2(v.x * e.x, v.y * e.y), pack_bf16x2(v.z * e.z, v.w * e.w));
  }
  s = warp_sum(s);
  q = warp_sum(q);
  if (lane < PXA_LN_STAT_PARTS)
    reinterpret_cast<float2*>(stats)[(size_t)row * PXA_LN_STAT_PARTS + lane] = lane == 0 ? make_float2(s, q) : make_float2(0.f, 0.f);
}

}  // namespace pxa

extern "C" int pxa_ln_prepare(const PxaLnPrepareArgs* args, void* stream) {
  using namespace pxa;
  if (!args) return fail(PXA_ERR_ARG, "null args");
  const PxaLnPrepareArgs& a = *args;
  if (!a.x || !a.a_out || !a.stats_out || !a.scale) return fail(PXA_ERR_ARG, "null pointer");
  if (a.M <= 0 || a.rows_per_batch <= 0) return fail(PXA_ERR_ARG, "bad M / rows_per_batch");
  if (a.C != 1152) return fail(PXA_ERR_ARG, "pxa_ln_prepare is specialised for C = 1152 (got %d)", a.C);
  if ((a.ldx & 3) || (a.mod_batch_stride & 3) ||
      ((reinterpret_cast<uintptr_t>(a.x) | reinterpret_cast<uintptr_t>(a.a_out) | reinterpret_cast<uintptr_t>(a.stats_out) |
        reinterpret_cast<uintptr_t>(a.scale)) & 15))
    return fail(PXA_ERR_ALIGN, "pointers must be 16-byte aligned, ldx / mod_batch_stride multiples of 4");
  PXA_REQUIRE_SM100();
  ln_prepare_kernel<9><<<(a.M + 7) / 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      a.x, reinterpret_cast<__nv_bfloat16*>(a.a_out), a.stats_out, a.scale, a.mod_batch_stride, a.rows_per_batch, a.M, a.ldx);
  launch_counter()++;
  PXA_CHECK_CUDA(cudaGetLastError());
  return PXA_OK;
}

namespace pxa {

// ------------------------------------------------------------------------------------------------- q / k LayerNorm (qk_norm)
// In-place LayerNorm(C = 1152, affine, fp32 statistics) on bf16 rows of stride ld: the q_norm / k_norm of
// AttentionKVCompress (PixArt_blocks.py:91-95, 133-134) applied to the q and k column slices of the qkv GEMM output.
template <int kVec>
__global__ void __launch_bounds__(256) layernorm_affine_kernel(__nv_bfloat16* __restrict__ x, const __nv_bfloat16* __restrict__ w,
                                                               const __nv_bfloat16* __restrict__ b, int M, long long ld, float eps) {
  constexpr int C = kVec * 128;
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  __nv_bfloat16* xr = x + (size_t)row * ld;
  float4 v[kVec];
  float s = 0.f;
#pragma unroll
  for (int g = 0; g < kVec; ++g) {
    const uint2 u = *reinterpret_cast<const uint2*>(xr + (g * 32 + lane) * 4);
    v[g] = make_float4(bf16_lo(u.x), bf16_hi(u.x), bf16_lo(u.y), bf16_hi(u.y));
    s += (v[g].x + v[g].y) + (v[g].z + v[g].w);
  }
  const float mean = warp_sum(s) * (1.0f / C);
  float ss = 0.f;
#pragma unroll
  for (int g = 0; g < kVec; ++g) {
    const float a0 = v[g].x - mean, a1 = v[g].y - mean, a2 = v[g].z - mean, a3 = v[g].w - mean;
    ss += (a0 * a0 + a1 * a1) + (a2 * a2 + a3 * a3);
  }
  const float rstd = rsqrtf(warp_sum(ss) * (1.0f / C) + eps);
#pragma unroll
  for (int g = 0; g < kVec; ++g) {
    const int col = (g * 32 + lane) * 4;
    const uint2 wu = __ldg(reinterpret_cast<const uint2*>(w + col));
    const uint2 bu = __ldg(reinterpret_cast<const uint2*>(b + col));
    const float y0 = fmaf((v[g].x - mean) * rstd, bf16_lo(wu.x), bf16_lo(bu.x));
    const float y1 = fmaf((v[g].y - mean) * rstd, bf16_hi(wu.x), bf16_hi(bu.x));
    const float y2 = fmaf((v[g].z - mean) * rstd, bf16_lo(wu.y), bf16_lo(bu.y));
    const float y3 = fmaf((v[g].w - mean) * rstd, bf16_hi(wu.y), bf16_hi(bu.y));
    *reinterpret_cast<uint2*>(xr + col) = make_uint2(pack_bf16x2(y0, y1), pack_bf16x2(y2, y3));
  }
}

}  // namespace pxa

extern "C" int pxa_layernorm_affine_bf16(void* x, const void* weight, const void* bias, int32_t M, int32_t C, int64_t ld,
                                         float eps, void* stream) {
  using namespace pxa;
  if (!x || !weight || !bias) return fail(PXA_ERR_ARG, "null pointer");
  if (M <= 0) return fail(PXA_ERR_ARG, "bad M");
  if (C != 1152) return fail(PXA_ERR_ARG, "pxa_layernorm_affine_bf16 is specialised for C = 1152 (got %d)", C);
  if ((ld & 3) || ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(weight) | reinterpret_cast<uintptr_t>(bias)) & 7))
    return fail(PXA_ERR_ALIGN, "x / weight / bias must be 8-byte aligned, ld a multiple of 4");
  PXA_REQUIRE_SM100();
  layernorm_affine_kernel<9><<<(M + 7) / 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      reinterpret_cast<__nv_bfloat16*>(x), reinterpret_cast<const __nv_bfloat16*>(weight),
      reinterpret_cast<const __nv_bfloat16*>(bias), M, ld, eps);
  launch_counter()++;
  PXA_CHECK_CUDA(cudaGetLastError());
  return PXA_OK;
}

namespace pxa {

// ------------------------------------------------------------------------------------------------- RMS norm (T5 encoder)
// T5LayerNorm of the T5-v1.1-XXL caption encoder (transformers `T5LayerNorm`: no mean subtraction, no bias, eps 1e-6; reference
// call site diffusion/model/t5.py:107-110 `self.model(input_ids, attention_mask)`): out[r, :] = bf16(x[r, :] * rsqrt(mean(x[r, :]^2)
// + eps) * w).  x is the fp32 residual stream.  Warp per row, two passes over the 16 KB row (the second one hits L1): HBM-bound,
// algorithmic bytes per row 4 C (read) + 2 C (write).
__global__ void __launch_bounds__(256) rmsnorm_kernel(const float* __restrict__ x, const __nv_bfloat16* __restrict__ w,
                                                      __nv_bfloat16* __restrict__ out, int M, int C, long long ldx, long long ldo,
                                                      float eps) {
  const int row = blockIdx.x * 8 + (threadIdx.x >> 5);
  const int lane = threadIdx.x & 31;
  if (row >= M) return;
  const float4* xr = reinterpret_cast<const float4*>(x + (size_t)row * ldx);
  const int nv = C >> 2;
  float ss = 0.f;
  for (int i = lane; i < nv; i += 32) {
    const float4 v = xr[i];
    ss += (v.x * v.x + v.y * v.y) + (v.z * v.z + v.w * v.w);
  }
  const float rstd = rsqrtf(warp_sum(ss) / (float)C + eps);
  __nv_bfloat16* orow = out + (size_t)row * ldo;
  for (int i = lane; i < nv; i += 32) {
    const float4 v = xr[i];
    const uint2 wu = __ldg(reinterpret_cast<const uint2*>(w + 4 * i));
    *reinterpret_cast<uint2*>(orow + 4 * i) = make_uint2(pack_bf16x2(v.x * rstd * bf16_lo(wu.x), v.y * rstd * bf16_hi(wu.x)),
                                                          pack_bf16x2(v.z * rstd * bf16_lo(wu.y), v.w * rstd * bf16_hi(wu.y)));
  }
}

}  // namespace pxa

extern "C" int pxa_rmsnorm_bf16(const float* x, const void* weight, void* out, int32_t M, int32_t C, int64_t ldx, int64_t ldo,
                                float eps, void* stream) {
  using namespace pxa;
  if (!x || !weight || !out) return fail(PXA_ERR_ARG, "null pointer");
  if (M <= 0 || C <= 0 || (C & 3)) return fail(PXA_ERR_ARG, "bad M / C (C must be a multiple of 4; got M=%d C=%d)", M, C);
  if ((ldx & 3) || (ldo & 3) || ((reinterpret_cast<uintptr_t>(x) & 15) | (reinterpret_cast<uintptr_t>(weight) & 7) |
                                  (reinterpret_cast<uintptr_t>(out) & 7)))
    return fail(PXA_ERR_ALIGN, "x must be 16-byte, weight / out 8-byte aligned; ldx, ldo multiples of 4");
  PXA_REQUIRE_SM100();
  rmsnorm_kernel<<<(M + 7) / 8, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      x, reinterpret_cast<const __nv_bfloat16*>(weight), reinterpret_cast<__nv_bfloat16*>(out), M, C, ldx, ldo, eps);
  launch_counter()++;
  PXA_CHECK_CUDA(cudaGetLastError());
  return PXA_OK;
}

namespace pxa {

// ------------------------------------------------------------------------------------------------- GroupNorm (+ SiLU), NHWC
// SDXL-VAE decoder ResnetBlock2D prologue (diffusers GroupNorm(32, eps 1e-6) -> SiLU in front of each 3x3 convolution;
// reference call site scripts/inference.py:136).  Two passes over an NHWC bf16 image: (1) per (sample, group) sum / sum of
// squares -- each thread walks pixels for a fixed 8-channel slice, CTA-level reduction in smem, one atomic per group and
// CTA; (2) y = silu((x - mean_g) rstd_g gamma_c + beta_c).  Algorithmic bytes: 2 reads + 1 write of the image (6 B/element).
constexpr int kGnThreads = 256;
constexpr int kGnMaxGroups = 64;

__global__ void __launch_bounds__(kGnThreads) gn_stats_kernel(const __nv_bfloat16* __restrict__ x, float* __restrict__ stats,
                                                              int HW, int C, int groups, int pix_per_cta) {
  __shared__ float sh[kGnMaxGroups][2];
  const int b = blockIdx.y;
  const int slices = C >> 3;                                    // 8-channel slices per pixel
  const int slice = threadIdx.x % slices, prow = threadIdx.x / slices, prows = kGnThreads / slices;
  const int cpg = C / groups;
  for (int i = threadIdx.x; i < groups * 2; i += kGnThreads) (&sh[0][0])[i] = 0.f;
  __syncthreads();
  const int p0 = blockIdx.x * pix_per_cta;
  const int p1 = min(p0 + pix_per_cta, HW);
  float s[8], q[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) s[i] = q[i] = 0.f;
  if (prow < prows) {
    const __nv_bfloat16* base = x + ((size_t)b * HW) * C + slice * 8;
#pragma unroll 4
    for (int p = p0 + prow; p < p1; p += prows) {
      const uint4 u = *reinterpret_cast<const uint4*>(base + (size_t)p * C);
      const uint32_t w[4] = {u.x, u.y, u.z, u.w};
#pragma unroll
      for (int i = 0; i < 4; ++i) {
        const float a = bf16_lo(w[i]), c = bf16_hi(w[i]);
        s[2 * i] += a; q[2 * i] = fmaf(a, a, q[2 * i]);
        s[2 * i + 1] += c; q[2 * i + 1] = fmaf(c, c, q[2 * i + 1]);
      }
    }
    // fold the 8 channels into their groups (cpg >= 8: one group; cpg = 4: two; cpg = 2 / 1: four / eight)
    const int c0 = slice * 8;
    int g_prev = c0 / cpg;
    float as = 0.f, aq = 0.f;
#pragma unroll
    for (int i = 0; i < 8; ++i) {
      const int g = (c0 + i) / cpg;
      if (g != g_prev) {
        atomicAdd(&sh[g_prev][0], as); atomicAdd(&sh[g_prev][1], aq);
        as = aq = 0.f; g_prev = g;
      }
      as += s[i]; aq += q[i];
    }
    atomicAdd(&sh[g_prev][0], as); atomicAdd(&sh[g_prev][1], aq);
  }
  __syncthreads();
  for (int i = threadIdx.x; i < groups * 2; i += kGnThreads) atomicAdd(stats + (size_t)b * groups * 2 + i, (&sh[0][0])[i]);
}

// The grid-stride is a multiple of the slices per pixel (a power of two <= 64 divides 256 x gridDim), so a thread keeps ONE
// 8-channel slice: gamma / beta are loaded once, and per pixel only the sample's (mean, rstd) of the slice's group(s) change.
template <bool kSilu>
__global__ void __launch_bounds__(kGnThreads) gn_apply_kernel(const __nv_bfloat16* __restrict__ x, __nv_bfloat16* __restrict__ out,
                                                              const float* __restrict__ stats, const __nv_bfloat16* __restrict__ gamma,
                                                              const __nv_bfloat16* __restrict__ beta, int HW, int C, int groups,
                                                              float eps, long long total_slices) {
  const int slices = C >> 3;
  const int cpg = C / groups;
  const float inv_n = 1.0f / ((float)HW * (float)cpg);
  const long long i0 = blockIdx.x * (long long)kGnThreads + threadIdx.x;
  const int slice = (int)(i0 % slices);
  const int c0 = slice * 8;
  float gm[8], bt[8];
  {
    const uint4 gu = __ldg(reinterpret_cast<const uint4*>(gamma + c0));
    const uint4 bu = __ldg(reinterpret_cast<const uint4*>(beta + c0));
    const uint32_t gw[4] = {gu.x, gu.y, gu.z, gu.w}, bw[4] = {bu.x, bu.y, bu.z, bu.w};
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      gm[2 * k] = bf16_lo(gw[k]); gm[2 * k + 1] = bf16_hi(gw[k]);
      bt[2 * k] = bf16_lo(bw[k]); bt[2 * k + 1] = bf16_hi(bw[k]);
    }
  }
  int b_prev = -1;
  float a[8], d[8];                                                // y = x * a + d  with a = rstd * gamma, d = beta - mean * a
  for (long long i = i0; i < total_slices; i += (long long)gridDim.x * kGnThreads) {
    const long long pix = i / slices;                              // b * HW + p
    const int b = (int)(pix / HW);
    if (b != b_prev) {                                             // new sample: fold its group statistics into (a, d)
      b_prev = b;
      int g_prev = -1;
      float mean = 0.f, rstd = 0.f;
#pragma unroll
      for (int k = 0; k < 8; ++k) {
        const int g = (c0 + k) / cpg;
        if (g != g_prev) {
          g_prev = g;
          const float2 st = __ldg(reinterpret_cast<const float2*>(stats) + (size_t)b * groups + g);
          mean = st.x * inv_n;
          rstd = rsqrtf(fmaxf(st.y * inv_n - mean * mean, 0.f) + eps);
        }
        a[k] = rstd * gm[k];
        d[k] = fmaf(-mean, a[k], bt[k]);
      }
    }
    const uint4 u = *reinterpret_cast<const uint4*>(x + pix * C + c0);
    const uint32_t w[4] = {u.x, u.y, u.z, u.w};
    uint32_t o[4];
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      float y0 = fmaf(bf16_lo(w[k]), a[2 * k], d[2 * k]);
      float y1 = fmaf(bf16_hi(w[k]), a[2 * k + 1], d[2 * k + 1]);
      if (kSilu) {
        y0 = __fdividef(y0, 1.0f + __expf(-y0));
        y1 = __fdividef(y1, 1.0f + __expf(-y1));
      }
      o[k] = pack_bf16x2(y0, y1);
    }
    *reinterpret_cast<uint4*>(out + pix * C + c0) = make_uint4(o[0], o[1], o[2], o[3]);
  }
}

}  // namespace pxa

extern "C" int pxa_groupnorm_silu_nhwc_bf16(const void* x, void* out, const void* gamma, const void* beta, float* stats_ws,
                                            int32_t B, int32_t HW, int32_t C, int32_t groups, float eps, int32_t silu,
                                            void* stream) {
  using namespace pxa;
  if (!x || !out || !gamma || !beta || !stats_ws) return fail(PXA_ERR_ARG, "null pointer");
  if (B <= 0 || HW <= 0 || C <= 0 || groups <= 0 || groups > kGnMaxGroups || C % groups || C % 8 || (C >> 3) > kGnThreads ||
      kGnThreads % (C >> 3))
    return fail(PXA_ERR_ARG, "bad B / HW / C / groups (C / 8 must divide %d, C %% groups == 0, groups <= %d)", kGnThreads,
                kGnMaxGroups);
  if ((reinterpret_cast<uintptr_t>(x) | reinterpret_cast<uintptr_t>(out) | reinterpret_cast<uintptr_t>(gamma) |
       reinterpret_cast<uintptr_t>(beta) | reinterpret_cast<uintptr_t>(stats_ws)) & 15)
    return fail(PXA_ERR_ALIGN, "pointers must be 16-byte aligned");
  PXA_REQUIRE_SM100();
  cudaStream_t s = reinterpret_cast<cudaStream_t>(stream);
  PXA_CHECK_CUDA(cudaMemsetAsync(stats_ws, 0, sizeof(float) * 2 * B * groups, s));
  const int sms = device_info().sms;
  int ctas_x = (4 * sms + B - 1) / B;                            // ~4 CTAs per SM over the whole batch
  int pix_per_cta = (HW + ctas_x - 1) / ctas_x;
  const int prows = kGnThreads / (C >> 3);
  if (pix_per_cta < prows) pix_per_cta = prows;
  ctas_x = (HW + pix_per_cta - 1) / pix_per_cta;
  gn_stats_kernel<<<dim3(ctas_x, B), kGnThreads, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(x), stats_ws, HW, C, groups, pix_per_cta);
  launch_counter()++;
  const long long total = (long long)B * HW * (C >> 3);
  long long blocks = (total + kGnThreads - 1) / kGnThreads;
  if (blocks > 32LL * sms) blocks = 32LL * sms;
  if (silu)
    gn_apply_kernel<true><<<(int)blocks, kGnThreads, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(x), reinterpret_cast<__nv_bfloat16*>(out),
                                                             stats_ws, reinterpret_cast<const __nv_bfloat16*>(gamma),
                                                             reinterpret_cast<const __nv_bfloat16*>(beta), HW, C, groups, eps, total);
  else
    gn_apply_kernel<false><<<(int)blocks, kGnThreads, 0, s>>>(reinterpret_cast<const __nv_bfloat16*>(x), reinterpret_cast<__nv_bfloat16*>(out),
                                                              stats_ws, reinterpret_cast<const __nv_bfloat16*>(gamma),
                                                              reinterpret_cast<const __nv_bfloat16*>(beta), HW, C, groups, eps, total);
  launch_counter()++;
  PXA_CHECK_CUDA(cudaGetLastError());
  return PXA_OK;
}

namespace pxa {

// ------------------------------------------------------------------------------------------------- AdamW on a flat bucket
// One elementwise pass over a flat fp32 (parameter, gradient, exp_avg, exp_avg_sq) bucket -- torch.optim.AdamW's update
// (decoupled weight decay, bias corrections folded into two host-computed scalars) -- optionally emitting the bf16 weight
// copy the GEMMs read.  The reference trains with AdamW(lr 2e-5, weight_decay 3e-2, eps 1e-10)
// (configs/PixArt_xl2_internal.py:48; diffusion/utils/optimizer.py:236-245 build_optimizer).  HBM-bound: 16 B read + 12 B
// (+ 2 B) written per parameter.
__global__ void __launch_bounds__(256) adamw_flat_kernel(float* __restrict__ p, const float* __restrict__ g, float* __restrict__ m,
                                                         float* __restrict__ v, __nv_bfloat16* __restrict__ shadow, long long n4,
                                                         float lr, float beta1, float beta2, float eps, float decay,
                                                         float step_size, float inv_sqrt_bc2, float grad_scale) {
  for (long long i = blockIdx.x * 256LL + threadIdx.x; i < n4; i += (long long)gridDim.x * 256) {
    float4 pv = reinterpret_cast<float4*>(p)[i];
    const float4 gv = reinterpret_cast<const float4*>(g)[i];
    float4 mv = reinterpret_cast<float4*>(m)[i];
    float4 vv = reinterpret_cast<float4*>(v)[i];
    float* pp = &pv.x; const float* gp = &gv.x; float* mp = &mv.x; float* vp = &vv.x;
#pragma unroll
    for (int k = 0; k < 4; ++k) {
      const float gk = gp[k] * grad_scale;
      mp[k] = fmaf(beta1, mp[k], (1.0f - beta1) * gk);
      vp[k] = fmaf(beta2, vp[k], (1.0f - beta2) * gk * gk);
      const float denom = sqrtf(vp[k]) * inv_sqrt_bc2 + eps;
      pp[k] = fmaf(-step_size, mp[k] / denom, pp[k] * decay);
    }
    reinterpret_cast<float4*>(p)[i] = pv;
    reinterpret_cast<float4*>(m)[i] = mv;
    reinterpret_cast<float4*>(v)[i] = vv;
    if (shadow != nullptr)
      reinterpret_cast<uint2*>(shadow)[i] = make_uint2(pack_bf16x2(pv.x, pv.y), pack_bf16x2(pv.z, pv.w));
  }
}

}  // namespace pxa

extern "C" int pxa_adamw_flat(const PxaAdamWArgs* args, void* stream) {
  using namespace pxa;
  if (!args) return fail(PXA_ERR_ARG, "null args");
  const PxaAdamWArgs& a = *args;
  if (!a.param || !a.grad || !a.exp_avg || !a.exp_avg_sq) return fail(PXA_ERR_ARG, "null pointer");
  if (a.n <= 0 || (a.n & 3)) return fail(PXA_ERR_ARG, "n must be a positive multiple of 4 (got %lld)", (long long)a.n);
  if (a.step <= 0) return fail(PXA_ERR_ARG, "step counts from 1");
  if ((reinterpret_cast<uintptr_t>(a.param) | reinterpret_cast<uintptr_t>(a.grad) | reinterpret_cast<uintptr_t>(a.exp_avg) |
       reinterpret_cast<uintptr_t>(a.exp_avg_sq)) & 15 || (reinterpret_cast<uintptr_t>(a.shadow_bf16) & 7))
    return fail(PXA_ERR_ALIGN, "param / grad / exp_avg / exp_avg_sq must be 16-byte aligned, shadow_bf16 8-byte");
  PXA_REQUIRE_SM100();
  const double bc1 = 1.0 - pow((double)a.beta1, (double)a.step), bc2 = 1.0 - pow((double)a.beta2, (double)a.step);
  const long long n4 = a.n / 4;
  long long blocks = (n4 + 255) / 256;
  const long long cap = 16LL * device_info().sms;
  if (blocks > cap) blocks = cap;
  adamw_flat_kernel<<<(int)blocks, 256, 0, reinterpret_cast<cudaStream_t>(stream)>>>(
      a.param, a.grad, a.exp_avg, a.exp_avg_sq, reinterpret_cast<__nv_bfloat16*>(a.shadow_bf16), n4, a.lr, a.beta1, a.beta2, a.eps,
      1.0f - a.lr * a.weight_decay, (float)(a.lr / bc1), (float)(1.0 / sqrt(bc2)), a.grad_scale);
  launch_counter()++;
  PXA_CHECK_CUDA(cudaGetLastError());
  return PXA_OK;
}
