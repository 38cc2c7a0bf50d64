// Single translation unit of librg_b200.so: the kernels live in headers shared by the F and PnP entry points, so the
// library is built as one unit (one nvcc invocation, see build.py).
#include "ctx.cu"
#include "f_api.cu"
#include "pnp_api.cu"
#include "geom_api.cu"
#include "gs_api.cu"
#include "pnp_refine_api.cu"
#include "ba_api.cu"
#include "nccl_api.cu"
#include "p2p_api.cu"
#include "microbench.cu"
