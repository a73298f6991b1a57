// tc_host.cu — host helpers for the tensor-core kernels: tensor-map encoding through
// the driver entry point (no link-time libcuda dependency) and the abort flag.
#include "tc_common.cuh"
#include <cudaTypedefs.h>
#include <mutex>

namespace iswm {

static PFN_cuTensorMapEncodeTiled_v12000 get_encode_fn() {
  static PFN_cuTensorMapEncodeTiled_v12000 fn = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    cudaError_t e = cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres);
    if (e == cudaSuccess && qres == cudaDriverEntryPointSuccess) fn = (PFN_cuTensorMapEncodeTiled_v12000)p;
  });
  return fn;
}

static int encode_tmap(CUtensorMapDataType dtype, int esize, CUtensorMap* out, const void* base, int rank,
                       const uint64_t* dims, const uint64_t* strides_elems, const uint32_t* box) {
  auto fn = get_encode_fn();
  if (!fn) {
    set_error("cuTensorMapEncodeTiled entry point unavailable (no CUDA driver?)");
    return 3;
  }
  cuuint64_t gdim[5];
  cuuint64_t gstr[4];
  cuuint32_t bx[5], es[5];
  for (int i = 0; i < rank; i++) {
    gdim[i] = dims[i];
    bx[i] = box[i];
    es[i] = 1;
    if (i > 0) gstr[i - 1] = strides_elems[i] * esize;  // bytes
  }
  CUresult r = fn(out, dtype, (cuuint32_t)rank, const_cast<void*>(base),
                  gdim, gstr, bx, es, CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                  CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) {
    set_error("cuTensorMapEncodeTiled failed (%d): base=%p rank=%d dims=[%llu,%llu,%llu,%llu] "
              "strides=[%llu,%llu,%llu] box=[%u,%u,%u,%u]",
              (int)r, base, rank, (unsigned long long)dims[0], (unsigned long long)(rank > 1 ? dims[1] : 0),
              (unsigned long long)(rank > 2 ? dims[2] : 0), (unsigned long long)(rank > 3 ? dims[3] : 0),
              (unsigned long long)(rank > 1 ? strides_elems[1] : 0), (unsigned long long)(rank > 2 ? strides_elems[2] : 0),
              (unsigned long long)(rank > 3 ? strides_elems[3] : 0), box[0], rank > 1 ? box[1] : 0,
              rank > 2 ? box[2] : 0, rank > 3 ? box[3] : 0);
    return 3;
  }
  return 0;
}

int encode_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                     const uint64_t* strides_elems, const uint32_t* box) {
  return encode_tmap(CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, out, base, rank, dims, strides_elems, box);
}

int encode_tmap_u8(CUtensorMap* out, const void* base, int rank, const uint64_t* dims,
                   const uint64_t* strides_elems, const uint32_t* box) {
  return encode_tmap(CU_TENSOR_MAP_DATA_TYPE_UINT8, 1, out, base, rank, dims, strides_elems, box);
}

int* abort_flag_ptr() {
  static int* flag = nullptr;
  static std::once_flag once;
  std::call_once(once, [] {
    if (cudaMalloc(&flag, sizeof(int)) == cudaSuccess) cudaMemset(flag, 0, sizeof(int));
    else flag = nullptr;
  });
  return flag;
}

int read_abort_flag(int* out, bool reset) {
  int* f = abort_flag_ptr();
  if (!f) return 3;
  if (cudaMemcpy(out, f, sizeof(int), cudaMemcpyDeviceToHost) != cudaSuccess) return 3;
  if (reset && *out != 0) cudaMemset(f, 0, sizeof(int));
  return 0;
}

}  // namespace iswm

// Synchronising health check for tests: returns the abort code recorded by a timed-out
// tensor-core kernel (0 = healthy) and clears it.
extern "C" int iswm_debug_abort_code(void) {
  int v = -1;
  if (iswm::read_abort_flag(&v, true)) return -1;
  return v;
}
