// Translation unit of the dense_kernel instantiations that run fp64 dense Hessians: the product's solver kernels.  The
// CSR mat-vec phase is compiled out (CCQP_DENSE_ONLY): the register allocation and the schedule of the dense loop depend
// on everything inlined next to it.  Own namespace (every `ccqp::` entity of the headers becomes `ccqp_f64::`), like the
// other compilations of the same templates.
#define CCQP_DENSE_ONLY 1
#define ccqp ccqp_f64
#include "dense.cuh"
#include "kernel_build.cuh"
#undef ccqp
#include "internal.h"

const ccqp::KernelBuild ccqp::kBuildF64 = ccqp_f64::describe<ccqp::KernelBuild>("dense_f64.cu", 0);
