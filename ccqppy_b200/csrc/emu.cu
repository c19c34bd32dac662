// Translation unit of the emulated-ranks instantiations of the dense solver kernels (dense.cuh dense_kernel_emu, fp64
// Hessians, dense and CSR phase), in their own namespace (`ccqp::` becomes `ccqp_emu::`).  Test vehicle only:
// ccqp_debug_solve_emulated().
#define CCQP_DENSE_KERNELS 0
#define CCQP_EMU_KERNELS 1
#define ccqp ccqp_emu
#include "dense.cuh"
#include "kernel_build.cuh"
#undef ccqp
#include "internal.h"

const ccqp::KernelBuild ccqp::kBuildEmu = ccqp_emu::describe<ccqp::KernelBuild>("emu.cu", 3);
