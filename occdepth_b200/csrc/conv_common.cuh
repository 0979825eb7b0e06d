// Device-side parameter block + shared epilogue for the implicit-GEMM convolution kernels.
#pragma once
#include "common.cuh"
#include "../../include/occdepth_b200.h"

struct ConvEpi {
  // iteration space / output mapping
  int B, OD, OH, OW;
  int omul[3], oadd[3];
  int ODf, OHf, OWf;
  int Cout;  // real output channels (stores are masked to n < Cout_store)
  int Cout_store;  // channels physically written (Cout rounded up to 8, pad written as computed zeros)
  const float* bias;
  void* out0;   // channels-last, element type T of the plan
  int out0_cstride, out0_coff;
  int act;
  int out0_exact;
  const void* res1;
  int res1_cstride, res1_coff;
  const void* res2;
  int res2_cstride, res2_coff, res2_post;
  int out1_mode;
  void* out1;
  int out1_cstride, out1_coff, out1_C;
};

__device__ __forceinline__ long long epi_pos(const ConvEpi& e, int b, int od, int oh, int ow, int oa0, int oa1,
                                             int oa2) {
  return (((long long)b * e.ODf + ((long long)od * e.omul[0] + oa0)) * e.OHf +
          ((long long)oh * e.omul[1] + oa1)) * e.OWf +
         ((long long)ow * e.omul[2] + oa2);
}
__device__ __forceinline__ long long epi_pos(const ConvEpi& e, int b, int od, int oh, int ow) {
  return epi_pos(e, b, od, oh, ow, e.oadd[0], e.oadd[1], e.oadd[2]);
}

// Epilogue arithmetic for one output position `pos` and NV consecutive channels [n0, n0+NV) held in v[] (fp32
// accumulators): v = acc + bias + res1 (+ res2); the optional second output (pre-activation value: channels-last or
// fp32 planar) is written here; on return v[] holds the out0 values act(v) (+ res2 when it is added after the
// activation).  NV is 8 or 16; n0 is a multiple of 8.  T is the activation element type.
template <typename T, int NV>
__device__ __forceinline__ void conv_epilogue_compute(const ConvEpi& e, long long pos, int b, int n0, float* v) {
#pragma unroll
  for (int g = 0; g < NV; g += 8) {
    const int n = n0 + g;
    if (n >= e.Cout_store) break;
    float* vv = v + g;
    const float4 b0 = __ldg(reinterpret_cast<const float4*>(e.bias + n));
    const float4 b1 = __ldg(reinterpret_cast<const float4*>(e.bias + n + 4));
    vv[0] += b0.x; vv[1] += b0.y; vv[2] += b0.z; vv[3] += b0.w;
    vv[4] += b1.x; vv[5] += b1.y; vv[6] += b1.z; vv[7] += b1.w;
    if (e.res1) {
      float r[8];
      Elem<T>::ld8(reinterpret_cast<const T*>(e.res1) + pos * e.res1_cstride + e.res1_coff + n, r);
#pragma unroll
      for (int i = 0; i < 8; ++i) vv[i] += r[i];
    }
    float r2[8];
    if (e.res2) {
      Elem<T>::ld8(reinterpret_cast<const T*>(e.res2) + pos * e.res2_cstride + e.res2_coff + n, r2);
      if (!e.res2_post) {
#pragma unroll
        for (int i = 0; i < 8; ++i) vv[i] += r2[i];
      }
    }
    if (e.out1_mode == OCCD_OUT1_CL) {
      Elem<T>::st8(reinterpret_cast<T*>(e.out1) + pos * e.out1_cstride + e.out1_coff + n, vv);
    } else if (e.out1_mode == OCCD_OUT1_F32_PLANAR) {
      const long long S = (long long)e.ODf * e.OHf * e.OWf;
      const long long sp = pos - (long long)b * S;
      float* o = reinterpret_cast<float*>(e.out1) + ((long long)b * e.out1_C + e.out1_coff + n) * S + sp;
#pragma unroll
      for (int i = 0; i < 8; ++i)
        if (n + i < e.Cout) o[(long long)i * S] = vv[i];
    }
    if (e.out0) {
      apply_act8<sizeof(T) == 2>(vv, e.act);
      if (e.res2 && e.res2_post) {
#pragma unroll
        for (int i = 0; i < 8; ++i) vv[i] += r2[i];
      }
    }
  }
}

// compute + direct (per-thread, 8-channel vector) global stores of out0: SIMT kernel, halo kernel
template <typename T, int NV>
__device__ __forceinline__ void conv_epilogue_row(const ConvEpi& e, int b, int od, int oh, int ow, int n0,
                                                  float* v) {
  const long long pos = epi_pos(e, b, od, oh, ow);
  conv_epilogue_compute<T, NV>(e, pos, b, n0, v);
  if (!e.out0) return;
#pragma unroll
  for (int g = 0; g < NV; g += 8) {
    const int n = n0 + g;
    if (n >= e.Cout_store) break;
    T* o0 = reinterpret_cast<T*>(e.out0) + pos * e.out0_cstride + e.out0_coff + n;
    if (e.out0_exact) Elem<T>::st8_exact(o0, v + g);
    else Elem<T>::st8(o0, v + g);
  }
}


// ---------------------------------------------------------------------------------------------------------------
// Fast path of the per-tap and halo kernels' epilogue (out0 only: no second output, no post-activation residual).  Measured
// on B200 (round 2, profiles/r02_lift_variants.txt): the row epilogue above is LATENCY bound -- 4 epilogue
// warps per scheduler walk a serial chain tcgen05.ld -> wait -> bias loads -> (residual loads) -> math -> store per
// 16 columns, at ~15 % of the SM's issue rate.  Here the chunk's bias (and residual) loads are issued BEFORE the wait
// on its TMEM load, the output / residual row pointers are formed once per tile, and the activation switch runs once
// per 16 values.
template <typename T>
struct EpiRow {
  T* out;            // out0 row of this thread: channels [n0, ...) of its output position (nullptr: nothing to store)
  const T* res;      // residual row (res1, or a post-activation res2) or nullptr
  int res_post;      // 1: the residual is added after the activation (Upsample + skip)
  const float* bias; // bias + n0
  int act, exact;
  int n_store;       // channels of this row that exist from n0 on (Cout_store - n0)
};

struct EpiPre {      // operands of one 16-column chunk, loaded ahead of the accumulator
  float4 b[4];
  float r[16];
};

template <typename T>
__device__ __forceinline__ void epi_prefetch(const EpiRow<T>& e, int c0, EpiPre& q) {
#pragma unroll
  for (int i = 0; i < 4; ++i) q.b[i] = __ldg(reinterpret_cast<const float4*>(e.bias + c0) + i);
  if (e.res) {
    if (c0 < e.n_store) Elem<T>::ld8(e.res + c0, q.r);
    if (c0 + 8 < e.n_store) Elem<T>::ld8(e.res + c0 + 8, q.r + 8);
  }
}

template <bool FAST_SILU>
__device__ __forceinline__ void apply_act16(float* v, int act) {
  if (act == ACT_NONE) return;
  if (act == ACT_RELU) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = fmaxf(v[i], 0.f);
  } else if (act == ACT_LEAKY) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = v[i] > 0.f ? v[i] : 0.01f * v[i];
  } else if (act == ACT_SILU) {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = FAST_SILU ? silu_tanh(v[i]) : __fdividef(v[i], 1.f + __expf(-v[i]));
  } else {
#pragma unroll
    for (int i = 0; i < 16; ++i) v[i] = __fdividef(1.f, 1.f + __expf(-v[i]));
  }
}

// v: accumulator values without bias; rr: this chunk's residual values (read only when e.res)
template <typename T>
__device__ __forceinline__ void epi_finish_v(const EpiRow<T>& e, int c0, float* v, const float4* qb, const float* rr) {
#pragma unroll
  for (int i = 0; i < 4; ++i) {
    v[4 * i] += qb[i].x;
    v[4 * i + 1] += qb[i].y;
    v[4 * i + 2] += qb[i].z;
    v[4 * i + 3] += qb[i].w;
  }
  if (e.res && !e.res_post) {
    if (c0 < e.n_store) {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] += rr[i];
    }
    if (c0 + 8 < e.n_store) {
#pragma unroll
      for (int i = 8; i < 16; ++i) v[i] += rr[i];
    }
  }
  apply_act16<sizeof(T) == 2>(v, e.act);
  if (e.res && e.res_post) {
    if (c0 < e.n_store) {
#pragma unroll
      for (int i = 0; i < 8; ++i) v[i] += rr[i];
    }
    if (c0 + 8 < e.n_store) {
#pragma unroll
      for (int i = 8; i < 16; ++i) v[i] += rr[i];
    }
  }
  if (e.out) {
    if (c0 < e.n_store) {
      if (e.exact) Elem<T>::st8_exact(e.out + c0, v);
      else Elem<T>::st8(e.out + c0, v);
    }
    if (c0 + 8 < e.n_store) {
      if (e.exact) Elem<T>::st8_exact(e.out + c0 + 8, v + 8);
      else Elem<T>::st8(e.out + c0 + 8, v + 8);
    }
  }
}

template <typename T>
__device__ __forceinline__ void epi_finish(const EpiRow<T>& e, int c0, const uint32_t* acc, const EpiPre& q) {
  float v[16];
#pragma unroll
  for (int i = 0; i < 16; ++i) v[i] = __uint_as_float(acc[i]);
  epi_finish_v<T>(e, c0, v, q.b, q.r);
}

// out0 only, and at most one residual: res1 (before the activation) or a post-activation res2
__device__ __forceinline__ bool epi_fast_ok(const ConvEpi& e) {
  return e.out1_mode == OCCD_OUT1_NONE && e.out0 != nullptr &&
         (e.res2 == nullptr || (e.res2_post && e.res1 == nullptr));
}

// row pointers of output position (b, od, oh, ow) + (oa0, oa1, oa2), channels from n0 on (valid == false: nothing is
// read or stored)
template <typename T>
__device__ __forceinline__ EpiRow<T> epi_row(const ConvEpi& e, bool valid, int b, int od, int oh, int ow, int n0,
                                             int oa0, int oa1, int oa2) {
  EpiRow<T> er;
  const long long pos = valid ? epi_pos(e, b, od, oh, ow, oa0, oa1, oa2) : 0;
  er.out = valid ? reinterpret_cast<T*>(e.out0) + pos * e.out0_cstride + e.out0_coff + n0 : nullptr;
  er.res = nullptr;
  er.res_post = 0;
  if (valid && e.res1) {
    er.res = reinterpret_cast<const T*>(e.res1) + pos * e.res1_cstride + e.res1_coff + n0;
  } else if (valid && e.res2) {
    er.res = reinterpret_cast<const T*>(e.res2) + pos * e.res2_cstride + e.res2_coff + n0;
    er.res_post = 1;
  }
  er.bias = e.bias + n0;
  er.act = e.act;
  er.exact = e.out0_exact;
  er.n_store = e.Cout_store - n0;
  return er;
}
template <typename T>
__device__ __forceinline__ EpiRow<T> epi_row(const ConvEpi& e, bool valid, int b, int od, int oh, int ow, int n0) {
  return epi_row<T>(e, valid, b, od, oh, ow, n0, e.oadd[0], e.oadd[1], e.oadd[2]);
}
