// Drop-in replacement for the reference's include/GPUSolver.h (signatures at
// /root/reference/include/GPUSolver.h:6-10).  Same four free functions with C++
// linkage, same argument meaning, same "void, print the CUDA error, carry on"
// convention; implemented in realtimedepthdiffusion_b200/csrc/gpu_shims.cpp on top
// of the C ABI declared in include/rtdd.h.
#ifndef GPU_SOLVER_H
#define GPU_SOLVER_H

#include <cstddef>
#include <iostream>

// ref GPUSolver.h:6 / GPUSolver.cu:33-54 -- scratch planes for `levels` pyramid levels of
// floor(rows/2^l) x floor(cols/2^l); the coarsest level (levels-1) is the ungated one.
void GPUAllocateDeviceMemory(int rows, int cols, int levels);
// ref GPUSolver.h:7 / GPUSolver.cu:56-71
void GPUFreeDeviceMemory(int levels);
// ref GPUSolver.h:8 / GPUSolver.cu:264-272 -- w[d] = expf(-beta*d), d = 0..255.  Deviation: a negative, NaN or
// infinite beta is refused (error printed, previous table kept), see rtdd_load_weights.
void GPULoadWeights(float beta);
// ref GPUSolver.h:9-10 / GPUSolver.cu:274-316 -- one pyramid level, depthImage updated in
// place; all pointers are device pointers with byte pitches; beta and tolerance are accepted
// and ignored exactly as the reference ignores them.  Returns after a device sync.
void GPUMatrixFreeSolver(float *depthImage, size_t depthPitch, unsigned char *scribbleImage, size_t scribblePitch, unsigned char *grayImage,
	size_t grayPitch, int rows, int cols, float beta, int maxIterations, float tolerance, int level);

#endif
