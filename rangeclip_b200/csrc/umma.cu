// Host side of umma.cuh: tensor-map encoding through the driver entry point (no -lcuda link dependency).
#include "common.cuh"
#include "umma.cuh"

namespace rc {

PFN_encodeTiled get_encode_tiled() {
  static PFN_encodeTiled fn = nullptr;
  static bool tried = false;
  if (!tried) {
    tried = true;
    void* p = nullptr;
    cudaDriverEntryPointQueryResult qres;
    if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &p, cudaEnableDefault, &qres) == cudaSuccess &&
        qres == cudaDriverEntryPointSuccess)
      fn = (PFN_encodeTiled)p;
  }
  return fn;
}

int make_tmap_bf16(CUtensorMap* out, const void* base, int rank, const uint64_t* dims, const uint64_t* strides_bytes,
                   const uint32_t* box, const char* what) {
  PFN_encodeTiled enc = get_encode_tiled();
  if (!enc) return fail(RC_ERR_NO_DEVICE, "%s: cuTensorMapEncodeTiled entry point unavailable", what);
  cuuint64_t gdim[3];
  cuuint64_t gstr[2];
  cuuint32_t bx[3];
  cuuint32_t es[3] = {1, 1, 1};
  for (int i = 0; i < rank; ++i) { gdim[i] = dims[i]; bx[i] = box[i]; }
  for (int i = 0; i + 1 < rank; ++i) gstr[i] = strides_bytes[i + 1];
  const CUtensorMapSwizzle sw = (box[0] * 2 >= 128) ? CU_TENSOR_MAP_SWIZZLE_128B
                                : (box[0] * 2 == 64) ? CU_TENSOR_MAP_SWIZZLE_64B
                                                     : CU_TENSOR_MAP_SWIZZLE_32B;
  CUresult r = enc(out, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, (cuuint32_t)rank, const_cast<void*>(base), gdim, gstr, bx, es,
                   CU_TENSOR_MAP_INTERLEAVE_NONE, sw, CU_TENSOR_MAP_L2_PROMOTION_L2_128B,
                   CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
  if (r != CUDA_SUCCESS) return fail(RC_ERR_CUDA, "%s: cuTensorMapEncodeTiled failed (%d)", what, (int)r);
  return RC_OK;
}

}  // namespace rc
