// fish-diffusion hot path, B200-native: shared device/host definitions.
//
// Storage format used by every GEMM-shaped kernel on the path ("split planes"):
//   an activation tensor of logical shape [B, T, C] (channels-last) is stored as two
//   16-bit planes  planes[2][B][T][C]  with  value = hi + lo,  hi = rn16(value),
//   lo = rn16(value - hi).  In FD_F16 mode that is a 22-bit mantissa (fp32-faithful for
//   |value| < 65504), in FD_BF16 mode a 16-bit mantissa with fp32 range.  The tensor-core
//   kernel multiplies  hi*hi + lo*hi + hi*lo  with fp32 accumulation in TMEM, the SIMT twin
//   multiplies (hi+lo)*(hi+lo) in fp32 FMA.  Same bytes per element as fp32.
#pragma once
#include <cuda_runtime.h>
#include <cuda_fp16.h>
#include <cuda_bf16.h>
#include <stdint.h>

#define FD_F16 0
#define FD_BF16 1
// flag or-ed into a `prec` argument of the GEMM entry points: multiply the hi planes only (one product)
#define FD_SINGLE 0x10

#define FD_MAX_SEG 16

// epilogue kinds
#define FD_EPI_LINEAR 0
#define FD_EPI_GATE 1
#define FD_EPI_RES_SKIP 2
#define FD_EPI_MAG 3
#define FD_EPI_GATE_BWD 4

// activation kinds (linear epilogue)
#define FD_ACT_NONE 0
#define FD_ACT_RELU 1
#define FD_ACT_LRELU 2

struct FdSeg {
  int src;    // which source tensor (0/1)
  int shift;  // row (time) shift applied to the A operand: A row = t + shift (zero outside [0,T))
  int c_off;  // first channel of the source used by this segment
  int k_len;  // number of channels (K extent) of this segment; multiple of the K block
};

struct FdTapGemm {
  // ---- problem: D[b,t,n] = sum_seg sum_k src[seg.src][b, t+seg.shift, seg.c_off+k] * W[n, koff(seg)+k]
  int B, T;
  int n_total;   // output columns (rows of W)
  int k_total;   // row pitch of W: sum of seg.k_len, or more when the launch reads only the leading columns
  int num_seg;
  int prec;      // FD_F16 / FD_BF16
  int single;    // 1: one product over the hi planes (half-precision operands), 0: three split products
  FdSeg seg[FD_MAX_SEG];
  const uint16_t* src[2];   // split planes [2][B][T][src_C]
  int src_C[2];
  // element strides of the source views (row = time step, batch item, plane); the generic layout
  // [2][B][T][C] has rs = C, bs = T*C, ps = B*T*C.  Overlapping rows (rs < C) give framed views.
  long long src_rs[2], src_bs[2], src_ps[2];
  const uint16_t* w;        // split planes [2][n_total][k_total]
  float acc_scale;          // accumulators are multiplied by this (undoes power-of-two weight prescale)
  // W-operand K offsets (weight-gradient GEMMs, where "W" is a transposed activation tensor [rows][B*Tp]):
  // the K coordinate of the W operand is  koff(seg) + k0 + w_kshift + b * w_bstride_k
  int w_kshift;
  long long w_bstride_k;
  int epi;

  // ---- FD_EPI_LINEAR:  y = acc*acc_scale + bias[n] + addend[b,t,n] + res[b,t,n];  y *= post_scale
  //      if out_f32:   v = accum ? out_f32 + y : y ;  out_f32 = v   (else v = y)
  //      if out_planes: planes = split(act(v * planes_scale))
  //      rows with row_mask[b,t] != 0 produce zeros.
  const float* bias;        // [n_total] or per item [B][n_total] with bias_bstride
  int bias_bstride;
  const float* addend;      // fp32 [B,T,n_total] or null
  const float* res_f32;     // fp32 [B,T,n_total] or null
  const uint16_t* res_planes;  // split planes [2][B][T][n_total] or null
  float res_scale;          // multiplies the res_planes term (gradient chains: dx_next / sqrt(2))
  float post_scale;
  float* out_f32;           // fp32 [B,T,n_total] or null
  int out_accum;
  uint16_t* out_planes;     // split planes [2][B][T][n_total] or null
  float planes_scale;
  int act;
  float act_slope;
  const uint8_t* row_mask;  // [B,T] or null

  // ---- FD_EPI_GATE (WaveNet GEMM1): column tile of width NT holds NT/2 gate columns followed by
  //      NT/2 filter columns for residual channels [tile*NT/2, (tile+1)*NT/2).
  //      y = acc*acc_scale + gbias_full[n] - (t<dil ? gbias_lo[n] : 0) - (t+dil>=T ? gbias_hi[n] : 0) + addend[b,t,n]
  //      z = sigmoid(y_gate) * tanh(y_filter)  -> out_planes [2][B][T][C]
  //      addend (fp32 [B][T][n_total] in packed column order, or null) carries the conditioner projection when the
  //      sampler computed it once per call instead of as a K segment of every evaluation
  const float* gbias_full;  // [Bs][n_total]  (conv bias + cond bias + sum over 3 taps of W_tap.d)
  const float* gbias_lo;    // [Bs][n_total]  tap-0 (t-dil) contribution of the step vector
  const float* gbias_hi;    // [Bs][n_total]  tap-2 (t+dil) contribution
  int gbias_bstride;        // 0 => one step for the whole batch
  int dil;
  int gate_tile;            // NT (column tile the weights were packed for)

  // ---- FD_EPI_MAG (framed DFT): same column pairing as the gate epilogue (re | im per tile);
  //      out_planes[b,t,c] = split(sqrt(re^2 + im^2 + mag_eps) * mag_scale), channel count = C
  float mag_scale;
  float mag_eps;            // 1e-9 (pitch_adjustable_mel.py:85) or 0 (torchaudio Spectrogram(power=1), utils/audio.py:45)

  // ---- FD_EPI_RES_SKIP (WaveNet GEMM2): columns [0,C) residual, [C,2C) skip.
  //      x' = (x + y_res) / sqrt(2)  -> x planes updated in place
  //      skip: first_layer ? skip_f32 = y : skip_f32 += y ; last_layer: skip planes = split((skip_f32+y)*skip_scale)
  uint16_t* x_planes;       // [2][B][T][C] in/out
  uint16_t* x_out_planes;   // training: write the updated residual stream here instead of in place (or null)
  uint16_t* y_planes;       // training (GATE epilogue): pre-activations [2][B][T][2C] in packed column order (or null)
  float* skip_f32;          // [B,T,C]
  uint16_t* skip_planes;    // [2][B][T][C] (last layer only)
  float skip_scale;
  int first_layer, last_layer;
  int C;                    // residual channels

  // ---- FD_EPI_GATE_BWD (training): the accumulator is dz[b,t,c] (n_total = C columns); with the saved pre-activations
  //      y_planes [2][B][T][2C] (packed order, see FD_EPI_GATE) the epilogue writes the gradient of z = sigmoid(g) tanh(f)
  //      dy = (dz tanh(f) sg (1-sg) | dz sg (1-tanh(f)^2))  -> out_planes [2][B][T][2C] (packed order)
  //      and accumulates its column sums: cs[b][col] += cs_scale * sum_t dy,  cs_edge[0/1][b][col] += the same over the
  //      first / last `dil` steps of the item (bias gradient and rank-one step-vector term of dW1).  cs buffers are zeroed
  //      by the caller.
  float* cs;                // [B][2C] or null
  float* cs_edge;           // [2][B][2C] or null
  float cs_scale;
};

// ------------------------------------------------------------------------------------------------
// split / combine
// ------------------------------------------------------------------------------------------------
__device__ __forceinline__ void fd_split(float v, int prec, uint16_t& hi, uint16_t& lo) {
  if (prec == FD_F16) {
    v = fminf(fmaxf(v, -65504.f), 65504.f);
    __half h = __float2half_rn(v);
    __half l = __float2half_rn(v - __half2float(h));
    hi = __half_as_ushort(h);
    lo = __half_as_ushort(l);
  } else {
    __nv_bfloat16 h = __float2bfloat16_rn(v);
    __nv_bfloat16 l = __float2bfloat16_rn(v - __bfloat162float(h));
    hi = __bfloat16_as_ushort(h);
    lo = __bfloat16_as_ushort(l);
  }
}

__device__ __forceinline__ float fd_h2f(uint16_t u, int prec) {
  if (prec == FD_F16) return __half2float(__ushort_as_half(u));
  return __uint_as_float(((uint32_t)u) << 16);
}

__device__ __forceinline__ float fd_combine(uint16_t hi, uint16_t lo, int prec) {
  return fd_h2f(hi, prec) + fd_h2f(lo, prec);
}

// two neighbouring channels from their plane words (low half-word -> a, high half-word -> b)
__device__ __forceinline__ void fd_combine2(uint32_t hi2, uint32_t lo2, int prec, float& a, float& b) {
  if (prec == FD_F16) {
    const float2 h = __half22float2(*reinterpret_cast<const __half2*>(&hi2));
    const float2 l = __half22float2(*reinterpret_cast<const __half2*>(&lo2));
    a = h.x + l.x; b = h.y + l.y;
  } else {
    a = __uint_as_float(hi2 << 16) + __uint_as_float(lo2 << 16);
    b = __uint_as_float(hi2 & 0xffff0000u) + __uint_as_float(lo2 & 0xffff0000u);
  }
}

// branch-free activation of the linear epilogue: slope = 1 (none), 0 (ReLU) or the LeakyReLU slope
__device__ __forceinline__ float fd_act(float w, float slope) { return fmaf(slope, fminf(w, 0.f), fmaxf(w, 0.f)); }

// accurate-enough transcendental pieces (relative error ~1e-7; tanh.approx is 1e-3 and is NOT used)
__device__ __forceinline__ float fd_sigmoid(float x) { return __fdividef(1.f, 1.f + __expf(-x)); }
__device__ __forceinline__ float fd_tanh(float x) {
  // tanh(x) = 1 - 2/(1+exp(2x)); for tiny |x| use the odd series to keep relative accuracy
  float ax = fabsf(x);
  if (ax < 0.04f) { float x2 = x * x; return x * (1.f - x2 * (0.33333333f - 0.13333333f * x2)); }
  float e = __expf(2.f * ax);
  float r = 1.f - __fdividef(2.f, e + 1.f);
  return copysignf(r, x);
}

// ------------------------------------------------------------------------------------------------
// vector helpers: V consecutive channels (V = 4 or 8)
// ------------------------------------------------------------------------------------------------
template <int V> struct FdVec16;   // V x uint16
template <> struct FdVec16<4> { uint2 v; };
template <> struct FdVec16<8> { uint4 v; };

// two neighbouring channels at once: ONE packed, saturating conversion per plane word (F2FP.SATFINITE.*.PACK_AB)
// instead of clamp + convert + pack per element.  a -> low half-word, b -> high half-word.  Bit-identical to fd_split
// for |v| <= 65504 (f16) / all finite v (bf16).
__device__ __forceinline__ void fd_split2(float a, float b, int prec, uint32_t& hi2, uint32_t& lo2) {
  if (prec == FD_F16) {
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(hi2) : "f"(b), "f"(a));
    const float2 hf = __half22float2(*reinterpret_cast<const __half2*>(&hi2));
    asm("cvt.rn.satfinite.f16x2.f32 %0, %1, %2;" : "=r"(lo2) : "f"(b - hf.y), "f"(a - hf.x));
  } else {
    asm("cvt.rn.satfinite.bf16x2.f32 %0, %1, %2;" : "=r"(hi2) : "f"(b), "f"(a));
    const float ha = __uint_as_float(hi2 << 16), hb = __uint_as_float(hi2 & 0xffff0000u);
    asm("cvt.rn.satfinite.bf16x2.f32 %0, %1, %2;" : "=r"(lo2) : "f"(b - hb), "f"(a - ha));
  }
}

template <int V>
__device__ __forceinline__ void fd_store_planes(uint16_t* planes, size_t plane_elems, size_t off,
                                                const float (&y)[V], int prec) {
  uint32_t hi[V / 2], lo[V / 2];
#pragma unroll
  for (int i = 0; i < V / 2; ++i) fd_split2(y[2 * i], y[2 * i + 1], prec, hi[i], lo[i]);
  if (V == 4) {
    *reinterpret_cast<uint2*>(planes + off) = make_uint2(hi[0], hi[1]);
    *reinterpret_cast<uint2*>(planes + plane_elems + off) = make_uint2(lo[0], lo[1]);
  } else {
    *reinterpret_cast<uint4*>(planes + off) = make_uint4(hi[0], hi[1], hi[2 % (V / 2)], hi[3 % (V / 2)]);
    *reinterpret_cast<uint4*>(planes + plane_elems + off) = make_uint4(lo[0], lo[1], lo[2 % (V / 2)], lo[3 % (V / 2)]);
  }
}

template <int V>
__device__ __forceinline__ void fd_load_planes(const uint16_t* planes, size_t plane_elems, size_t off,
                                               float (&y)[V], int prec) {
  uint16_t hi[8], lo[8];
  if (V == 4) {
    uint2 a = *reinterpret_cast<const uint2*>(planes + off);
    uint2 b = *reinterpret_cast<const uint2*>(planes + plane_elems + off);
    hi[0] = a.x & 0xffff; hi[1] = a.x >> 16; hi[2] = a.y & 0xffff; hi[3] = a.y >> 16;
    lo[0] = b.x & 0xffff; lo[1] = b.x >> 16; lo[2] = b.y & 0xffff; lo[3] = b.y >> 16;
  } else {
    uint4 a = *reinterpret_cast<const uint4*>(planes + off);
    uint4 b = *reinterpret_cast<const uint4*>(planes + plane_elems + off);
    hi[0] = a.x & 0xffff; hi[1] = a.x >> 16; hi[2] = a.y & 0xffff; hi[3] = a.y >> 16;
    hi[4] = a.z & 0xffff; hi[5] = a.z >> 16; hi[6] = a.w & 0xffff; hi[7] = a.w >> 16;
    lo[0] = b.x & 0xffff; lo[1] = b.x >> 16; lo[2] = b.y & 0xffff; lo[3] = b.y >> 16;
    lo[4] = b.z & 0xffff; lo[5] = b.z >> 16; lo[6] = b.w & 0xffff; lo[7] = b.w >> 16;
  }
#pragma unroll
  for (int i = 0; i < V; ++i) y[i] = fd_combine(hi[i], lo[i], prec);
}

// hi plane only (single-product mode of the SIMT twin)
__device__ __forceinline__ void fd_load_hi8(const uint16_t* planes, size_t off, float (&y)[8], int prec) {
  const uint4 a = *reinterpret_cast<const uint4*>(planes + off);
  const uint32_t w[4] = {a.x, a.y, a.z, a.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    y[2 * i] = fd_h2f((uint16_t)(w[i] & 0xffff), prec);
    y[2 * i + 1] = fd_h2f((uint16_t)(w[i] >> 16), prec);
  }
}

// register-level (un)packing of 8 consecutive channels; used by the split-phase (prefetch / finish) epilogues
__device__ __forceinline__ void fd_unpack8(const uint4& a, const uint4& b, int prec, float (&y)[8]) {
  const uint32_t ha[4] = {a.x, a.y, a.z, a.w}, lb[4] = {b.x, b.y, b.z, b.w};
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    y[2 * i] = fd_combine((uint16_t)(ha[i] & 0xffff), (uint16_t)(lb[i] & 0xffff), prec);
    y[2 * i + 1] = fd_combine((uint16_t)(ha[i] >> 16), (uint16_t)(lb[i] >> 16), prec);
  }
}
__device__ __forceinline__ void fd_pack8(const float (&y)[8], int prec, uint4& a, uint4& b) {
  uint16_t hi[8], lo[8];
#pragma unroll
  for (int i = 0; i < 8; ++i) fd_split(y[i], prec, hi[i], lo[i]);
  a.x = hi[0] | ((uint32_t)hi[1] << 16); a.y = hi[2] | ((uint32_t)hi[3] << 16);
  a.z = hi[4] | ((uint32_t)hi[5] << 16); a.w = hi[6] | ((uint32_t)hi[7] << 16);
  b.x = lo[0] | ((uint32_t)lo[1] << 16); b.y = lo[2] | ((uint32_t)lo[3] << 16);
  b.z = lo[4] | ((uint32_t)lo[5] << 16); b.w = lo[6] | ((uint32_t)lo[7] << 16);
}

template <int V>
__device__ __forceinline__ void fd_load_f32(const float* p, float (&y)[V]) {
#pragma unroll
  for (int i = 0; i < V; i += 4) {
    float4 q = *reinterpret_cast<const float4*>(p + i);
    y[i] = q.x; y[i + 1] = q.y; y[i + 2] = q.z; y[i + 3] = q.w;
  }
}
template <int V>
__device__ __forceinline__ void fd_store_f32(float* p, const float (&y)[V]) {
#pragma unroll
  for (int i = 0; i < V; i += 4)
    *reinterpret_cast<float4*>(p + i) = make_float4(y[i], y[i + 1], y[i + 2], y[i + 3]);
}

// ------------------------------------------------------------------------------------------------
// Epilogues.  Each handles V consecutive output columns [n0, n0+V) of row (b,t) with raw
// accumulators acc[].  `bias*` pointers may be shared-memory or global (generic loads).
// ------------------------------------------------------------------------------------------------
template <int V, int PREC = -1>
__device__ __forceinline__ void fd_epi_linear(const FdTapGemm& p, int b, int t, int n0,
                                              const float (&acc)[V], const float* bias_tile /*[n - tile_n0] or null*/,
                                              int tile_n0) {
  const int prec = PREC < 0 ? p.prec : PREC;   // compile-time in the tensor-core kernel
  const size_t row = (size_t)b * p.T + t;
  const size_t off = row * p.n_total + n0;
  const size_t plane_elems = (size_t)p.B * p.T * p.n_total;
  float y[V];
  const bool masked = p.row_mask != nullptr && p.row_mask[row] != 0;
#pragma unroll
  for (int i = 0; i < V; ++i) y[i] = acc[i] * p.acc_scale;
  if (bias_tile != nullptr) {
#pragma unroll
    for (int i = 0; i < V; ++i) y[i] += bias_tile[n0 - tile_n0 + i];
  }
  if (p.addend != nullptr) {
    float a[V]; fd_load_f32<V>(p.addend + off, a);
#pragma unroll
    for (int i = 0; i < V; ++i) y[i] += a[i];
  }
  if (p.res_f32 != nullptr) {
    float a[V]; fd_load_f32<V>(p.res_f32 + off, a);
#pragma unroll
    for (int i = 0; i < V; ++i) y[i] += a[i];
  }
  if (p.res_planes != nullptr) {
    float a[V]; fd_load_planes<V>(p.res_planes, plane_elems, off, a, prec);
#pragma unroll
    for (int i = 0; i < V; ++i) y[i] += a[i] * p.res_scale;
  }
#pragma unroll
  for (int i = 0; i < V; ++i) y[i] *= p.post_scale;
  if (p.out_f32 != nullptr) {
    if (p.out_accum) {
      float a[V]; fd_load_f32<V>(p.out_f32 + off, a);
#pragma unroll
      for (int i = 0; i < V; ++i) y[i] += a[i];
    }
    if (masked) {
#pragma unroll
      for (int i = 0; i < V; ++i) y[i] = 0.f;
    }
    fd_store_f32<V>(p.out_f32 + off, y);
  }
  if (p.out_planes != nullptr) {
#pragma unroll
    for (int i = 0; i < V; ++i) {
      float v = y[i] * p.planes_scale;
      if (p.act == FD_ACT_RELU) v = fmaxf(v, 0.f);
      else if (p.act == FD_ACT_LRELU) v = v > 0.f ? v : v * p.act_slope;
      y[i] = masked ? 0.f : v;
    }
    fd_store_planes<V>(p.out_planes, plane_elems, off, y, prec);
  }
}

// gate epilogue: V gate accumulators + V filter accumulators for residual channels [zc0, zc0+V);
// gb_* point at the bias of the FIRST gate column of this thread's chunk, gf_* at the first filter col.
template <int V, int PREC = -1>
__device__ __forceinline__ void fd_epi_gate(const FdTapGemm& p, int b, int t, int zc0,
                                            const float (&g)[V], const float (&f)[V],
                                            const float* full_g, const float* full_f,
                                            const float* lo_g, const float* lo_f,
                                            const float* hi_g, const float* hi_f) {
  const int prec = PREC < 0 ? p.prec : PREC;   // compile-time in the tensor-core kernel
  float z[V], yg8[V], yf8[V];
  const bool e_lo = t < p.dil, e_hi = t + p.dil >= p.T;
#pragma unroll
  for (int i = 0; i < V; ++i) {
    float yg = g[i] * p.acc_scale + full_g[i];
    float yf = f[i] * p.acc_scale + full_f[i];
    if (e_lo) { yg -= lo_g[i]; yf -= lo_f[i]; }
    if (e_hi) { yg -= hi_g[i]; yf -= hi_f[i]; }
    yg8[i] = yg; yf8[i] = yf;
  }
  const int half = p.gate_tile / 2;
  const int ng = (zc0 / half) * p.gate_tile + (zc0 % half);   // packed column of the first gate channel
  const size_t yoff = ((size_t)b * p.T + t) * p.n_total;
  if (p.addend != nullptr) {
    float ag[V], af[V];
    fd_load_f32<V>(p.addend + yoff + ng, ag);
    fd_load_f32<V>(p.addend + yoff + ng + half, af);
#pragma unroll
    for (int i = 0; i < V; ++i) { yg8[i] += ag[i]; yf8[i] += af[i]; }
  }
#pragma unroll
  for (int i = 0; i < V; ++i) z[i] = fd_sigmoid(yg8[i]) * fd_tanh(yf8[i]);
  if (p.y_planes != nullptr) {   // training: keep the pre-activations (packed column order: gates | filters per tile)
    const size_t yplane = (size_t)p.B * p.T * p.n_total;
    fd_store_planes<V>(p.y_planes, yplane, yoff + ng, yg8, prec);
    fd_store_planes<V>(p.y_planes, yplane, yoff + ng + half, yf8, prec);
  }
  const size_t plane_elems = (size_t)p.B * p.T * p.C;
  const size_t off = ((size_t)b * p.T + t) * p.C + zc0;
  fd_store_planes<V>(p.out_planes, plane_elems, off, z, prec);
}

template <int V, int PREC = -1>
__device__ __forceinline__ void fd_epi_mag(const FdTapGemm& p, int b, int t, int zc0,
                                           const float (&re)[V], const float (&im)[V]) {
  const int prec = PREC < 0 ? p.prec : PREC;   // compile-time in the tensor-core kernel
  float z[V];
#pragma unroll
  for (int i = 0; i < V; ++i) {
    const float r = re[i] * p.acc_scale, q = im[i] * p.acc_scale;
    z[i] = sqrtf(r * r + q * q + p.mag_eps) * p.mag_scale;
  }
  const size_t plane_elems = (size_t)p.B * p.T * p.C;
  const size_t off = ((size_t)b * p.T + t) * p.C + zc0;
  fd_store_planes<V>(p.out_planes, plane_elems, off, z, prec);
}

// residual/skip epilogue for V consecutive packed columns [n0, n0+V) (n0 < C: residual, else skip)
template <int V, int PREC = -1>
__device__ __forceinline__ void fd_epi_res_skip(const FdTapGemm& p, int b, int t, int n0,
                                                const float (&acc)[V], const float* bias /*indexed by i*/) {
  const int prec = PREC < 0 ? p.prec : PREC;   // compile-time in the tensor-core kernel
  const size_t row = (size_t)b * p.T + t;
  const size_t plane_elems = (size_t)p.B * p.T * p.C;
  float y[V];
#pragma unroll
  for (int i = 0; i < V; ++i) y[i] = acc[i] * p.acc_scale + bias[i];
  if (n0 < p.C) {
    if (p.last_layer) return;  // the residual stream is not consumed after the last layer
    const size_t off = row * p.C + n0;
    float x[V];
    fd_load_planes<V>(p.x_planes, plane_elems, off, x, prec);
#pragma unroll
    for (int i = 0; i < V; ++i) x[i] = (x[i] + y[i]) * 0.70710678118654752440f;
    fd_store_planes<V>(p.x_out_planes != nullptr ? p.x_out_planes : p.x_planes, plane_elems, off, x, prec);
  } else {
    const size_t off = row * p.C + (n0 - p.C);
    if (!p.first_layer) {
      float s[V]; fd_load_f32<V>(p.skip_f32 + off, s);
#pragma unroll
      for (int i = 0; i < V; ++i) y[i] += s[i];
    }
    if (p.last_layer) {
#pragma unroll
      for (int i = 0; i < V; ++i) y[i] *= p.skip_scale;
      fd_store_planes<V>(p.skip_planes, plane_elems, off, y, prec);
    } else {
      fd_store_f32<V>(p.skip_f32 + off, y);
    }
  }
}

// ------------------------------------------------------------------------------------------------
// host side
// ------------------------------------------------------------------------------------------------
#ifdef __cplusplus
extern "C" {
#endif
void fd_set_error(const char* fmt, ...);
#ifdef __cplusplus
}
#endif

#define FD_CHECK_CUDA(expr)                                                                    \
  do {                                                                                         \
    cudaError_t _e = (expr);                                                                   \
    if (_e != cudaSuccess) {                                                                   \
      fd_set_error("%s:%d CUDA error %d (%s) in %s", __FILE__, __LINE__, (int)_e,              \
                   cudaGetErrorString(_e), #expr);                                             \
      return -1;                                                                               \
    }                                                                                          \
  } while (0)

#define FD_REQUIRE(cond, ...)                                                                  \
  do {                                                                                         \
    if (!(cond)) {                                                                             \
      fd_set_error(__VA_ARGS__);                                                               \
      return -2;                                                                               \
    }                                                                                          \
  } while (0)

int fd_tapgemm_simt_launch(const FdTapGemm& p, cudaStream_t stream);
int fd_tapgemm_tc_launch(const FdTapGemm& p, cudaStream_t stream);
int fd_tapgemm_tc_supported(const FdTapGemm& p);
