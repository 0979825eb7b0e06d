// Library core (error string, ABI version) + planar <-> channels-last transposes used at the module
// boundary (the reference's tensors are NCHW/NCDHW fp32; every kernel here works channels-last).
#include "common.cuh"
#include "../../include/occdepth_b200.h"
#include <string.h>

static thread_local char g_last_error[512] = "";

extern "C" void occd_set_last_error(const char* msg) {
  strncpy(g_last_error, msg ? msg : "", sizeof(g_last_error) - 1);
  g_last_error[sizeof(g_last_error) - 1] = 0;
}
extern "C" const char* occd_last_error(void) { return g_last_error; }
extern "C" int occd_abi_version(void) { return OCCD_ABI_VERSION; }

namespace {

// 32x32 smem tile transpose: in [C][S] -> out [S][cstride]
template <typename OT>
__global__ void planar_to_cl_kernel(const float* __restrict__ in, OT* __restrict__ out, int C, long long S,
                                    int cstride) {
  __shared__ float tile[32][33];
  const long long b = blockIdx.z;
  const long long s0 = (long long)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const float* inb = in + b * C * S;
  OT* outb = out + b * S * cstride;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i;
    const long long s = s0 + threadIdx.x;
    tile[i][threadIdx.x] = (c < C && s < S) ? inb[(long long)c * S + s] : 0.f;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const long long s = s0 + i;
    const int c = c0 + threadIdx.x;
    if (s < S && c < cstride) {
      const float v = tile[threadIdx.x][i];
      if constexpr (sizeof(OT) == 2) outb[s * cstride + c] = __float2bfloat16_rn(v);
      else outb[s * cstride + c] = round_tf32(v);   // OCCD_DTYPE_F32 buffers hold TF32 values (kind::tf32 operands)
    }
  }
}

template <typename IT>
__global__ void cl_to_planar_kernel(const IT* __restrict__ in, float* __restrict__ out, int C, long long S,
                                    int cstride) {
  __shared__ float tile[32][33];
  const long long b = blockIdx.z;
  const long long s0 = (long long)blockIdx.x * 32;
  const int c0 = blockIdx.y * 32;
  const IT* inb = in + b * S * cstride;
  float* outb = out + b * C * S;
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const long long s = s0 + i;
    const int c = c0 + threadIdx.x;
    float v = 0.f;
    if (s < S && c < C) {
      if constexpr (sizeof(IT) == 2) v = __bfloat162float(inb[s * cstride + c]);
      else v = inb[s * cstride + c];
    }
    tile[i][threadIdx.x] = v;
  }
  __syncthreads();
  for (int i = threadIdx.y; i < 32; i += blockDim.y) {
    const int c = c0 + i;
    const long long s = s0 + threadIdx.x;
    if (c < C && s < S) outb[(long long)c * S + s] = tile[threadIdx.x][i];
  }
}

}  // namespace

extern "C" int occd_planar_to_cl(const float* in, void* out, int out_dtype, long long B, int C, long long S,
                                 int cstride, void* stream) {
  OCCD_CHECK_ARG(in && out && B > 0 && C > 0 && S > 0 && cstride >= C, "occd_planar_to_cl: bad args");
  OCCD_CHECK_ARG(B <= 65535, "occd_planar_to_cl: batch too large");
  dim3 grid((unsigned)((S + 31) / 32), (unsigned)((cstride + 31) / 32), (unsigned)B), block(32, 8);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (out_dtype == OCCD_DTYPE_BF16)
    planar_to_cl_kernel<__nv_bfloat16><<<grid, block, 0, st>>>(in, (__nv_bfloat16*)out, C, S, cstride);
  else if (out_dtype == OCCD_DTYPE_F32)
    planar_to_cl_kernel<float><<<grid, block, 0, st>>>(in, (float*)out, C, S, cstride);
  else { occd_set_last_error("occd_planar_to_cl: dtype"); return OCCD_ERR_ARG; }
  OCCD_CHECK_LAUNCH();
  return OCCD_OK;
}

extern "C" int occd_cl_to_planar(const void* in, int in_dtype, float* out, long long B, int C, long long S,
                                 int cstride, void* stream) {
  OCCD_CHECK_ARG(in && out && B > 0 && C > 0 && S > 0 && cstride >= C, "occd_cl_to_planar: bad args");
  OCCD_CHECK_ARG(B <= 65535, "occd_cl_to_planar: batch too large");
  dim3 grid((unsigned)((S + 31) / 32), (unsigned)((C + 31) / 32), (unsigned)B), block(32, 8);
  cudaStream_t st = reinterpret_cast<cudaStream_t>(stream);
  if (in_dtype == OCCD_DTYPE_BF16)
    cl_to_planar_kernel<__nv_bfloat16><<<grid, block, 0, st>>>((const __nv_bfloat16*)in, out, C, S, cstride);
  else if (in_dtype == OCCD_DTYPE_F32)
    cl_to_planar_kernel<float><<<grid, block, 0, st>>>((const float*)in, out, C, S, cstride);
  else { occd_set_last_error("occd_cl_to_planar: dtype"); return OCCD_ERR_ARG; }
  OCCD_CHECK_LAUNCH();
  return OCCD_OK;
}
