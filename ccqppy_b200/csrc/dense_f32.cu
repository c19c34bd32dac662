// Translation unit of the dense_kernel / dense_kernel_emu instantiations that run fp32-stored dense Hessians.
//
// The reference's only use of A is A.dot(v) (solvers.py:133): for a float32 A NumPy widens every entry exactly and runs
// the product in fp64.  These kernels do the same on the device -- A is streamed as fp32 (half the HBM bytes of the fp64
// kernels) and every entry is widened in a register in front of its fma -- with the fp64 loop's lane mapping, FMA chains
// and reduction order (dense.cuh dot_seg_aligned / dot_seg_generic with T = float), so a solve returns the same bits as
// the fp64 solve of the widened matrix.  The SAME solver programs (dense.cuh) are compiled a second time here, CSR phase
// compiled out, inside their own namespace (every `ccqp::` entity of the headers becomes `ccqp_f32::`), like csr.cu: the
// fp64 kernels keep their own translation unit and code (the schedule of the dense loop depends on everything inlined
// next to it).  capi.cu routes every launch of a handle that holds an fp32 matrix through kBuildF32, emulated ranks
// included (dense_kernel_emu); the context struct is the same plain-data struct in every namespace.
#define CCQP_DENSE_ONLY 1
#define CCQP_A_F32 1
#define CCQP_EMU_KERNELS 1
#define ccqp ccqp_f32
#include "dense.cuh"
#include "kernel_build.cuh"
#undef ccqp
#include "internal.h"

const ccqp::KernelBuild ccqp::kBuildF32 = ccqp_f32::describe<ccqp::KernelBuild>("dense_f32.cu", 1);
