// embed_inst.cu -- the kernel instantiations of the fused path for ONE (table format, output type) pair.
//
// Each pair holds the kernels embed_plan.h can plan (kShapes lists them); build.py compiles this file once per pair, in
// parallel, with -DSCONE_INST_QUANT=q -DSCONE_INST_OUT=o, and embed.cu (plan + C ABI) calls the eight entry points.
#include "embed_kernels.cuh"

#if !defined(SCONE_INST_QUANT) || !defined(SCONE_INST_OUT)
#error "compile with -DSCONE_INST_QUANT=<SCONE_QUANT_*> -DSCONE_INST_OUT=<SCONE_OUT_BF16|SCONE_OUT_FP16>"
#endif

#define SCONE_CAT3(a, b, c) a##b##_##c
#define SCONE_INST_NAME(q, o) SCONE_CAT3(embed_launch_q, q, o)

namespace scone {

// embed_launch_q<quant>_<out>(plan, params, stream): SCONE_OK or an error
int SCONE_INST_NAME(SCONE_INST_QUANT, SCONE_INST_OUT)(const EmbedPlan &pl, EmbedParams &p, cudaStream_t stream) {
    return launch_plan<SCONE_INST_QUANT, SCONE_INST_OUT>(pl, p, stream);
}

}  // namespace scone
