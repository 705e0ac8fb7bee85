// embed_inst.cu -- the kernel instantiations of the fused path for ONE (table format, output type) pair.
//
// embed_kernels.cuh holds 46 kernel shapes per pair; compiling all six pairs in one translation unit took three minutes,
// so build.py compiles this file six times in parallel with -DSCONE_INST_QUANT=q -DSCONE_INST_OUT=o and embed.cu
// (dispatch + C ABI) calls the six entry points below.
#include "embed_kernels.cuh"

#if !defined(SCONE_INST_QUANT) || !defined(SCONE_INST_OUT)
#error "compile with -DSCONE_INST_QUANT=<SCONE_QUANT_*> -DSCONE_INST_OUT=<SCONE_OUT_BF16|SCONE_OUT_FP16>"
#endif

#define SCONE_CAT3(a, b, c) a##b##_##c
#define SCONE_INST_NAME(q, o) SCONE_CAT3(embed_launch_q, q, o)

namespace scone {

// embed_launch_q<quant>_<out>(P, params, stream, shape): SCONE_OK, an error, or kNoFit when the shape's ring cannot hold the rows
int SCONE_INST_NAME(SCONE_INST_QUANT, SCONE_INST_OUT)(int P, EmbedParams &p, cudaStream_t stream, int shape) {
    return launch_p<SCONE_INST_QUANT, SCONE_INST_OUT>(P, p, stream, shape);
}

}  // namespace scone
