// Shared device/host helpers for the aecf_b200 kernels (sm_100a only).
#pragma once

// AECF_CUDA_EMU: the test-only host emulation of tests/cuda_emu (these sources compiled by g++ and run as fibers on
// the CPU, so that `-m "not gpu"` tests exercise the kernels' logic and the host code around them).  It is never
// defined in the library build; every `#ifdef AECF_CUDA_EMU` below is the emulation's stand-in for an inline-PTX
// wrapper or a launch, and the other branch is the product, token for token what it was before the split.
#ifdef AECF_CUDA_EMU
#ifdef __CUDACC__
#error "AECF_CUDA_EMU is the g++ test build of tests/cuda_emu; the library itself is never built with it"
#endif
#include "cuda_emu.h"
#else
#include <cuda_runtime.h>
#include <cuda_bf16.h>
#endif
#include <stdint.h>
#include <math.h>

#include "../../include/aecf_b200.h"

namespace aecf {

constexpr unsigned FULL_MASK = 0xffffffffu;

#define AECF_STR_(x) #x
#define AECF_STR(x) AECF_STR_(x)

// ---- host-side bookkeeping (api.cu) --------------------------------------------------
void count_launch(unsigned n = 1);
int set_cuda_error(cudaError_t err, const char* what);   // records and returns AECF_ERR_CUDA
int use_device(int device);                               // cudaSetDevice; 0 or AECF_ERR_CUDA
// Every entry point runs on the device of its descriptor and leaves the calling thread's current device as it found it
// (a caller holding tensors on several GPUs must not find torch's current device changed under it).
struct DeviceScope {
    int previous = -1, rc = AECF_OK;
    bool changed = false;
    explicit DeviceScope(int device) {
        if (cudaGetDevice(&previous) != cudaSuccess) previous = -1;
        if (previous != device) {
            rc = use_device(device);
            changed = rc == AECF_OK && previous >= 0;
        }
    }
    ~DeviceScope() { if (changed) cudaSetDevice(previous); }
    DeviceScope(const DeviceScope&) = delete;
    DeviceScope& operator=(const DeviceScope&) = delete;
};
int sm_count(int device);

// per-kernel timing (timing.cu): the current site is thread-local, set by the whole-step entry points
int  timing_begin(cudaStream_t s, int site_override = -1);   // returns a record index or -1 when disabled
void timing_end(int record, cudaStream_t s);
void note_site_gemm_kernel(const char* name);                // remembers the GEMM kernel launched from the current site
struct ScopedSite {
    int previous;
    explicit ScopedSite(int site);
    ~ScopedSite();
};
struct TimedLaunch {                                          // brackets the launches of one C-ABI call
    int record;
    cudaStream_t stream;
    explicit TimedLaunch(cudaStream_t s, int site_override = -1) : record(timing_begin(s, site_override)), stream(s) {}
    ~TimedLaunch() { if (record >= 0) timing_end(record, stream); }
};

#define AECF_CUDA_OK(call)                                              \
    do {                                                                \
        cudaError_t err__ = (call);                                     \
        if (err__ != cudaSuccess) return ::aecf::set_cuda_error(err__, #call); \
    } while (0)

// fold.cu: dWq, d_query and the packed in-projection bias gradient of a shared query, one launch; the gradients in
// grad_dtype (dtype, or fp32 next to bf16 parameters in mixed precision)
int launch_query_tail(int dtype, int grad_dtype, int D, const float* d_qp, const void* q0, const void* in_proj_weight,
                      const float* d_bias_kv, void* d_in_proj_weight, void* d_query, void* d_in_proj_bias, cudaStream_t s);

// ---- programmatic dependent launch (PDL) -----------------------------------------------------
// Every kernel of the library is launched with programmatic stream serialization and starts with
// pdl_wait(): its CTAs may be scheduled while the previous kernel of the stream is still draining
// (launch latency and per-CTA prologues -- barrier init, TMEM allocation, tensor-map prefetch --
// overlap that tail), but nothing touches global memory before the previous kernel has completed and
// flushed.
#ifdef AECF_CUDA_EMU
__device__ __forceinline__ void pdl_wait() {}

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t, Args&&... args) {
    return cuda_emu::launch(kernel, grid, block, smem, static_cast<KArgs>(args)...);
}
template <typename... KArgs, typename... Args>
inline cudaError_t launch_plain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t, Args&&... args) {
    return cuda_emu::launch(kernel, grid, block, smem, static_cast<KArgs>(args)...);
}
#else
__device__ __forceinline__ void pdl_wait() { asm volatile("griddepcontrol.wait;" ::: "memory"); }

template <typename... KArgs, typename... Args>
inline cudaError_t launch_pdl(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                              Args&&... args) {
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = grid; cfg.blockDim = block; cfg.dynamicSmemBytes = smem; cfg.stream = stream;
    cudaLaunchAttribute attr[1];
    attr[0].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[0].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr;
    cfg.numAttrs = 1;
    return cudaLaunchKernelEx(&cfg, kernel, static_cast<KArgs>(args)...);
}
// An ordinary launch (kernels that do not start with pdl_wait()).
template <typename... KArgs, typename... Args>
inline cudaError_t launch_plain(void (*kernel)(KArgs...), dim3 grid, dim3 block, size_t smem, cudaStream_t stream,
                                Args&&... args) {
    kernel<<<grid, block, smem, stream>>>(static_cast<KArgs>(args)...);
    return cudaGetLastError();
}
#endif

// Dynamic shared memory of a kernel.  The emulation points it at one host buffer (blocks run one at a time).
#ifdef AECF_CUDA_EMU
#define AECF_DYNAMIC_SMEM(type, name) type* name = reinterpret_cast<type*>(cuda_emu::dynamic_smem())
#define AECF_DYNAMIC_SMEM_ALIGNED16(type, name) type* name = reinterpret_cast<type*>(cuda_emu::dynamic_smem())
#define AECF_DYNAMIC_SMEM_ALIGNED1024(type, name) type* name = reinterpret_cast<type*>(cuda_emu::dynamic_smem())
#else
#define AECF_DYNAMIC_SMEM(type, name) extern __shared__ type name[]
#define AECF_DYNAMIC_SMEM_ALIGNED16(type, name) extern __shared__ __align__(16) type name[]
#define AECF_DYNAMIC_SMEM_ALIGNED1024(type, name) extern __shared__ __align__(1024) type name[]
#endif

inline bool aligned16(const void* p) { return (reinterpret_cast<uintptr_t>(p) & 15u) == 0; }

// ---- 16-byte vectors of the storage type ---------------------------------------------
template <typename T> struct Vec;

template <> struct Vec<float> {
    static constexpr int N = 4;
    static __device__ __forceinline__ void unpack(const uint4& r, float (&f)[4]) {
        f[0] = __uint_as_float(r.x); f[1] = __uint_as_float(r.y);
        f[2] = __uint_as_float(r.z); f[3] = __uint_as_float(r.w);
    }
    static __device__ __forceinline__ uint4 pack(const float (&f)[4]) {
        return make_uint4(__float_as_uint(f[0]), __float_as_uint(f[1]),
                          __float_as_uint(f[2]), __float_as_uint(f[3]));
    }
};

template <> struct Vec<__nv_bfloat16> {
    static constexpr int N = 8;
    static __device__ __forceinline__ void unpack(const uint4& r, float (&f)[8]) {
        const uint32_t w[4] = {r.x, r.y, r.z, r.w};
#pragma unroll
        for (int i = 0; i < 4; ++i) {
            f[2 * i] = __uint_as_float(w[i] << 16);
            f[2 * i + 1] = __uint_as_float(w[i] & 0xffff0000u);
        }
    }
    static __device__ __forceinline__ uint32_t pack2(float lo, float hi) {
#ifdef AECF_CUDA_EMU
        return cuda_emu::bf16_bits(lo) | (cuda_emu::bf16_bits(hi) << 16);
#else
        uint32_t r;   // cvt.rn.bf16x2.f32 d, a, b  puts a in the upper half
        asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
        return r;
#endif
    }
    static __device__ __forceinline__ uint4 pack(const float (&f)[8]) {
        return make_uint4(pack2(f[0], f[1]), pack2(f[2], f[3]), pack2(f[4], f[5]), pack2(f[6], f[7]));
    }
};

#ifdef AECF_CUDA_EMU
__device__ __forceinline__ uint4 ldg_stream(const void* p) { return *reinterpret_cast<const uint4*>(p); }
__device__ __forceinline__ void stg_stream(void* p, const uint4& v) { *reinterpret_cast<uint4*>(p) = v; }
// deferred like the emulation's TMA stores: the 16 bytes land when cp.async.wait_group retires their group, not before
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) { cuda_emu::cp_async_enqueue(smem_dst, gmem_src); }
__device__ __forceinline__ void cp_async_commit() { cuda_emu::cp_async_commit_group(); }
template <int N> __device__ __forceinline__ void cp_async_wait() { cuda_emu::cp_async_wait_group(N); }
#else
// Streaming 128-bit load of read-once data: read-only path, do not allocate in L1.
__device__ __forceinline__ uint4 ldg_stream(const void* p) {
    uint4 r;
    asm("ld.global.nc.L1::no_allocate.v4.u32 {%0, %1, %2, %3}, [%4];"
        : "=r"(r.x), "=r"(r.y), "=r"(r.z), "=r"(r.w) : "l"(p));
    return r;
}
#endif
__device__ __forceinline__ uint4 ldg_cached(const void* p) {
    return __ldg(reinterpret_cast<const uint4*>(p));
}
__device__ __forceinline__ void stg_vec(void* p, const uint4& v) {
    *reinterpret_cast<uint4*>(p) = v;
}
#ifndef AECF_CUDA_EMU
// Streaming store: written once, consumed by a later kernel from HBM/L2.
__device__ __forceinline__ void stg_stream(void* p, const uint4& v) {
    asm volatile("st.global.cs.v4.u32 [%0], {%1, %2, %3, %4};"
                 :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// Asynchronous 16-byte global -> shared copy (LDGSTS, bypasses L1 and the register file).
__device__ __forceinline__ void cp_async16(void* smem_dst, const void* gmem_src) {
    asm volatile("cp.async.cg.shared.global [%0], [%1], 16;"
                 :: "r"(static_cast<uint32_t>(__cvta_generic_to_shared(smem_dst))), "l"(gmem_src) : "memory");
}
__device__ __forceinline__ void cp_async_commit() { asm volatile("cp.async.commit_group;" ::: "memory"); }
template <int N> __device__ __forceinline__ void cp_async_wait() { asm volatile("cp.async.wait_group %0;" :: "n"(N) : "memory"); }
#endif

template <typename T> __device__ __forceinline__ float to_float(T v);
template <> __device__ __forceinline__ float to_float<float>(float v) { return v; }
template <> __device__ __forceinline__ float to_float<__nv_bfloat16>(__nv_bfloat16 v) { return __bfloat162float(v); }
template <typename T> __device__ __forceinline__ T from_float(float v);
template <> __device__ __forceinline__ float from_float<float>(float v) { return v; }
template <> __device__ __forceinline__ __nv_bfloat16 from_float<__nv_bfloat16>(float v) { return __float2bfloat16_rn(v); }

// ---- Philox4x32-10 (contract in include/aecf_b200.h, mirrored by oracle/philox.py) -----
__device__ __forceinline__ uint4 philox4x32_10(uint4 c, uint2 k) {
#pragma unroll
    for (int r = 0; r < 10; ++r) {
        const uint32_t hi0 = __umulhi(0xD2511F53u, c.x), lo0 = 0xD2511F53u * c.x;
        const uint32_t hi1 = __umulhi(0xCD9E8D57u, c.z), lo1 = 0xCD9E8D57u * c.z;
        c = make_uint4(hi1 ^ c.y ^ k.x, lo1, hi0 ^ c.w ^ k.y, lo0);
        if (r != 9) { k.x += 0x9E3779B9u; k.y += 0xBB67AE85u; }
    }
    return c;
}
__device__ __forceinline__ float uniform01(uint32_t x) {      // curand_uniform: (0, 1]
    return fmaf(__uint2float_rn(x), 2.3283064365386963e-10f, 1.1641532182693481e-10f);
}
constexpr uint32_t STREAM_MASK = 0u, STREAM_DROPOUT = 1u;

struct RngKey { uint32_t k0, k1, offset; unsigned long long row0; };

// The key a kernel draws with: the by-value one, or -- under CUDA-graph capture -- the (seed, offset) pair read
// from device memory at run time (aecf_pool_desc::rng_state), so that replays draw fresh numbers.
__device__ __forceinline__ RngKey effective_rng(const RngKey& by_value, const unsigned long long* state) {
    RngKey k = by_value;
    if (state != nullptr) {
        const unsigned long long seed = __ldg(state), off = __ldg(state + 1);
        k.k0 = static_cast<uint32_t>(seed); k.k1 = static_cast<uint32_t>(seed >> 32);
        k.offset = static_cast<uint32_t>(off + by_value.offset);
    }
    return k;
}

// The 4 uniforms of (row, stream, head, block) -- tokens 4*block .. 4*block+3.
__device__ __forceinline__ void draw4(const RngKey& key, unsigned long long local_row, uint32_t stream,
                                      uint32_t head, uint32_t block, float (&u)[4]) {
    const unsigned long long row = key.row0 + local_row;
    const uint4 c = make_uint4(static_cast<uint32_t>(row), static_cast<uint32_t>(row >> 32), key.offset,
                               (stream << 28) | (head << 4) | block);
    const uint4 r = philox4x32_10(c, make_uint2(key.k0, key.k1));
    u[0] = uniform01(r.x); u[1] = uniform01(r.y); u[2] = uniform01(r.z); u[3] = uniform01(r.w);
}

// Static-index select out of a small register array (keeps the array in registers).
template <int M>
__device__ __forceinline__ float select(const float (&a)[M], int i) {
    float v = a[0];
#pragma unroll
    for (int m = 1; m < M; ++m) v = (i == m) ? a[m] : v;
    return v;
}

inline int ilog2(int x) { int l = 0; while ((1 << l) < x) ++l; return l; }
inline bool is_pow2(int x) { return x > 0 && (x & (x - 1)) == 0; }

}  // namespace aecf
