// Translation unit of the dense_kernel instantiations that run CSR (operator-form) Hessians.
//
// The CSR mat-vec phase is a gather: latency-bound, it wants many resident warps and few registers, the opposite of
// the dense phase (8 warps x 254 registers so that 16 256-bit loads per lane are in flight).  So the SAME solver
// programs (dense.cuh) are compiled a second time here with a different launch shape -- CCQP_CSR_THREADS threads per
// CTA (1 CTA per SM, 65536 / threads registers per thread; measured on n = 2^20, 57 entries per row, SPG, us per mat-vec:
// 256 threads 333, 512 threads 292, 1024 threads 399 -- at 64 registers the solver programs spill into the tile loop),
// the dense mat-vec loop compiled out (CCQP_CSR_ONLY) --
// inside their own namespace: every `ccqp::` entity of the headers becomes `ccqp_csr::` in this file, so the two
// compilations of the templates cannot collide.  capi.cu routes every launch of a handle that holds a CSR matrix
// through kBuildCsr; the context struct is the same plain-data struct in every namespace.
#ifndef CCQP_CSR_THREADS
#define CCQP_CSR_THREADS 512
#endif
#undef CCQP_DENSE_THREADS          // the width of the dense builds (-D, tools/sweep_gemv.py) does not apply here
#define CCQP_DENSE_THREADS CCQP_CSR_THREADS
#define CCQP_CSR_ONLY 1
#define ccqp ccqp_csr
#include "dense.cuh"
#include "kernel_build.cuh"
#undef ccqp
#include "internal.h"

const ccqp::KernelBuild ccqp::kBuildCsr = ccqp_csr::describe<ccqp::KernelBuild>("csr.cu", 2);
