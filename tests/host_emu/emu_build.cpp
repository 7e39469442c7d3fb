// emu_build.cpp -- TEST INFRASTRUCTURE: the dense-grid builder's content hash (csrc/ort_build.cuh: build_hash) compiled
// for the host through cuda_shim.h, so that the tests can aim grids at chosen table slots and notice when the hash
// changes.  Built on demand by tests/host_emu/emu_build.py into tests/host_emu/_build/; never part of libort_b200.so.
#include "cuda_shim.h"

// The rest of the header's device code must compile, though only build_hash runs here: inert stand-ins for the
// block-level intrinsics it uses.
#define __shared__ static
#define __launch_bounds__(n)
struct EmuDim { unsigned x, y, z; };
static const EmuDim threadIdx{ 0, 0, 0 }, blockIdx{ 0, 0, 0 }, blockDim{ 1, 1, 1 };
static inline void __syncthreads() {}
template<class T> static inline T __shfl_down_sync(unsigned, T v, int) { return v; }
template<class T> static inline T __shfl_up_sync(unsigned, T v, int) { return v; }
template<class T> static inline T atomicAdd(T* p, T v) { const T o = *p; *p += v; return o; }
static inline uint32_t atomicCAS(uint32_t* p, uint32_t cmp, uint32_t v) { const uint32_t o = *p; if (o == cmp) *p = v; return o; }
static inline uint32_t atomicMin(uint32_t* p, uint32_t v) { const uint32_t o = *p; if (v < o) *p = v; return o; }
static inline uint4 make_uint4(uint32_t x, uint32_t y, uint32_t z, uint32_t w) { return uint4{ x, y, z, w }; }

#include "../../octree_ray_tracing_b200/csrc/ort_build.cuh"

#include <cstddef>

extern "C" {

// out[i] = build_hash of the 8 words w8[8i .. 8i+7]
void emu_build_hash(const uint32_t* w8, size_t n, uint32_t* out)
{
	for (size_t i = 0; i < n; ++i)
		out[i] = ort::build_hash(w8 + 8 * i);
}

}  // extern "C"
