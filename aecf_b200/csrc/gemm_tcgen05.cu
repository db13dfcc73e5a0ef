// bf16 GEMM on the 5th-generation tensor cores: C[m,n] = sum_k A[m,k] B[n,k] (+ bias[n]).
//
//   operands  : TMA (cp.async.bulk.tensor, 128-byte swizzle) into a 4-stage shared-memory ring;
//               K-major or MN-major in global memory -- the UMMA smem descriptor carries the major
//   math      : tcgen05.mma.cta_group::1.kind::f16, 128 x BN x 16 per instruction, issued by one
//               elected thread; fp32 accumulators live in TMEM (2 x BN columns, double buffered)
//   epilogue  : tcgen05.ld TMEM -> registers, + bias, -> bf16/fp32 -> swizzled smem -> TMA store,
//               overlapped with the next tile's main loop (persistent CTAs, one per SM)
//   split-K   : for the weight-gradient products (K = B*M rows, tiny output) each work item writes an
//               fp32 partial tile; splitk_reduce (gemm.cu) folds them in a fixed order
//
// Replaces the cuBLAS calls behind torch.nn.functional.linear at torch/nn/functional.py:5855, 6653
// and the matmuls autograd derives from them.  Descriptor bit layouts follow the PTX ISA tables as
// restated in cute/arch/mma_sm100_desc.hpp (SmemDescriptor, InstrDescriptor).
#include <cuda.h>

#include <mutex>

#include "gemm.cuh"

namespace aecf {

namespace tc {

constexpr int BM = 128;            // UMMA M (cta_group::1)
constexpr int BK = 64;             // one 128-byte swizzle atom of bf16 along K
constexpr int UMMA_K = 16;
constexpr int STAGES = 4;
constexpr int NUM_THREADS = 192;   // warp 0: TMA producer, warp 1: MMA issuer + TMEM owner, warps 2-5: epilogue
constexpr int EPI_THREADS = 128;
// (An L2 prefetch stream 12 k-blocks ahead of the ring made every projection 15-35 % SLOWER on B200 --
// profiles/r1_gemm_experiments.md -- and was removed.)
constexpr long long SPIN_LIMIT = 4000000000LL;   // ~2 s of SM clocks: trap instead of hanging the GPU

template <int BN> struct Cfg {
    static constexpr int A_BYTES = BM * BK * 2;                 // 16 KB
    static constexpr int B_BYTES = BN * BK * 2;                 // 16 / 32 KB
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int EPI_BYTES = 2 * BM * 128;              // staging: two [128 rows x 128 B] swizzled boxes
    static constexpr int ACC_STRIDE = BN > 128 ? 256 : 128;     // TMEM column stride between the two accumulators
    static constexpr int TMEM_COLS = 2 * ACC_STRIDE;            // double-buffered accumulator (a power of two)
    static constexpr int BIAS_BYTES = 2 * BN * 4;               // fp32 bias slice, double buffered by tile parity
    static constexpr int SMEM_BYTES = STAGES * STAGE_BYTES + EPI_BYTES + BIAS_BYTES + 128 /*barriers*/;
};

struct Params {
    int m, n, k;
    int tiles_m, tiles_n, groups_m, splits, kb_per_split, kb_total;   // groups_m = ceil(tiles_m / cluster size)
    int a_mn_major, b_mn_major;
    int c_is_f32;              // element type of the TMA-stored C / partial
    int has_bias, bias_is_bf16;
    const void* bias;
    int partial_rows;          // rows of one split's partial (= m) when splits > 1
    // side output (aecf_gemm_aux): columns [c_cols, n) of the product leave as fp32 into aux[row * aux_ld + j];
    // columns [0, c_cols) are the ordinary C (bias, TMA store).  Without a side output c_cols == n.
    int c_cols, aux_cols;
    long long aux_ld;
    float* aux;
};

#ifdef AECF_CUDA_EMU
#include "tcgen05_emu_wrappers.h"     // functional stand-ins for every inline-PTX wrapper below (tests/cuda_emu)
#else
// ---- raw PTX wrappers -----------------------------------------------------------------------
__device__ __forceinline__ uint32_t smem_u32(const void* p) { return static_cast<uint32_t>(__cvta_generic_to_shared(p)); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count));
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    const uint32_t addr = smem_u32(bar);
    const long long t0 = clock64();
    while (true) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(addr), "r"(parity) : "memory");
        if (done) return;
        if (clock64() - t0 > SPIN_LIMIT) __trap();          // a pipeline bug must fail, not hang the box
    }
}
__device__ __forceinline__ void fence_barrier_init() { asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory"); }
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }

__device__ __forceinline__ void tma_load_2d(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        :: "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
// Same, multicast: the box lands at the same shared-memory offset in every CTA of `mask` and completes
// bytes on the mbarrier at the same offset in each of them.
__device__ __forceinline__ void tma_load_2d_mc(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1, uint16_t mask) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes.multicast::cluster"
        " [%0], [%1, {%4, %5}], [%2], %3;"
        :: "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar)), "h"(mask), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;\n\tbarrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t cluster_ctarank() {
    uint32_t r;
    asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r));
    return r;
}
__device__ __forceinline__ void tma_store_2d(const CUtensorMap* map, const void* src, int c0, int c1) {
    asm volatile("cp.async.bulk.tensor.2d.global.shared::cta.bulk_group [%0, {%2, %3}], [%1];"
                 :: "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(src)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tma_store_commit() { asm volatile("cp.async.bulk.commit_group;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_read() { asm volatile("cp.async.bulk.wait_group.read 0;" ::: "memory"); }
__device__ __forceinline__ void tma_store_wait_all() { asm volatile("cp.async.bulk.wait_group 0;" ::: "memory"); }
__device__ __forceinline__ void prefetch_tmap(const CUtensorMap* map) {
    asm volatile("prefetch.tensormap [%0];" :: "l"(reinterpret_cast<uint64_t>(map)) : "memory");
}

__device__ __forceinline__ void umma_commit(uint64_t* bar) {     // arrives on `bar` when all prior MMAs retire
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                 :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ void umma_commit_mc(uint64_t* bar, uint16_t mask) {   // ... on `bar` in every CTA of `mask`
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 :: "r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ void umma_bf16(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :: "r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void tmem_ld_32x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0, %1, %2, %3, %4, %5, %6, %7, %8, %9, %10, %11, %12, %13, %14, %15, "
        "%16, %17, %18, %19, %20, %21, %22, %23, %24, %25, %26, %27, %28, %29, %30, %31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tmem_ld_wait() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }
// The same wait, naming the registers an earlier tcgen05.ld is still filling as read-write operands: nothing that
// consumes them can be scheduled above the wait, however far the load was issued ahead (experimental epilogues).
__device__ __forceinline__ void tmem_ld_wait_on(uint32_t (&r)[32]) {
    asm volatile("tcgen05.wait::ld.sync.aligned;"
                 : "+r"(r[0]), "+r"(r[1]), "+r"(r[2]), "+r"(r[3]), "+r"(r[4]), "+r"(r[5]), "+r"(r[6]), "+r"(r[7]),
                   "+r"(r[8]), "+r"(r[9]), "+r"(r[10]), "+r"(r[11]), "+r"(r[12]), "+r"(r[13]), "+r"(r[14]), "+r"(r[15]),
                   "+r"(r[16]), "+r"(r[17]), "+r"(r[18]), "+r"(r[19]), "+r"(r[20]), "+r"(r[21]), "+r"(r[22]), "+r"(r[23]),
                   "+r"(r[24]), "+r"(r[25]), "+r"(r[26]), "+r"(r[27]), "+r"(r[28]), "+r"(r[29]), "+r"(r[30]), "+r"(r[31])
                 :: "memory");
}
#endif  // AECF_CUDA_EMU

// Shared-memory matrix descriptor (cute::UMMA::SmemDescriptor): start address, leading/stride byte
// offsets in 16-byte units, version 1 (Blackwell), layout type 2 = SWIZZLE_128B.
__device__ __forceinline__ uint64_t make_smem_desc(uint32_t smem_addr, uint32_t lbo_bytes, uint32_t sbo_bytes) {
    uint64_t d = 0;
    d |= static_cast<uint64_t>((smem_addr >> 4) & 0x3FFF);
    d |= static_cast<uint64_t>((lbo_bytes >> 4) & 0x3FFF) << 16;
    d |= static_cast<uint64_t>((sbo_bytes >> 4) & 0x3FFF) << 32;
    d |= 1ull << 46;
    d |= 2ull << 61;
    return d;
}
// Descriptor of the 16-deep K slice `ks` of an operand tile of `rows` MN-rows in the stage buffer.
//   K-major : rows of 128 B (64 bf16 of K), 8-row groups 1024 B apart; a K slice is 32 B further in.
//   MN-major: 64-wide MN atoms, each [64 K-rows x 128 B], 8-K-row groups 1024 B apart (SBO), atoms
//             BK*128 B apart (LBO); a K slice is 16 K-rows = 2048 B further in.
__device__ __forceinline__ uint64_t operand_desc(uint32_t base, int mn_major, int ks) {
    if (!mn_major) return make_smem_desc(base + ks * (UMMA_K * 2), 0, 8 * 128);
    return make_smem_desc(base + ks * (UMMA_K * 128), BK * 128, 8 * 128);
}
// Instruction descriptor (cute::UMMA::InstrDescriptor): c=f32 [4,6)=1, a=bf16 [7,10)=1, b=bf16 [10,13)=1,
// a_major [15], b_major [16], N>>3 [17,23), M>>4 [24,29).
__device__ __forceinline__ uint32_t make_idesc(int bn, int a_mn, int b_mn) {
    return (1u << 4) | (1u << 7) | (1u << 10) | (static_cast<uint32_t>(a_mn) << 15) |
           (static_cast<uint32_t>(b_mn) << 16) | (static_cast<uint32_t>(bn >> 3) << 17) |
           (static_cast<uint32_t>(BM >> 4) << 24);
}

// ---- cta_group::2 helpers: a pair of CTAs (one cluster) works on one 256-row tile -------------------------
#ifndef AECF_CUDA_EMU
constexpr uint32_t PEER_BIT_MASK = 0xFEFFFFFFu;     // clears the CTA-rank bit of a shared::cluster address -> leader CTA
__device__ __forceinline__ void tma_load_2d_2sm(const CUtensorMap* map, uint64_t* bar, void* dst, int c0, int c1) {
    // lands in THIS CTA's shared memory, completes bytes on the LEADER CTA's barrier at the same offset
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        :: "r"(smem_u32(dst)), "l"(reinterpret_cast<uint64_t>(map)), "r"(smem_u32(bar) & PEER_BIT_MASK), "r"(c0), "r"(c1)
        : "memory");
}
__device__ __forceinline__ void umma_bf16_2sm(uint32_t tmem_d, uint64_t a_desc, uint64_t b_desc, uint32_t idesc, uint32_t acc) {
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "setp.ne.b32 p, %4, 0;\n\t"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n\t}"
        :: "r"(tmem_d), "l"(a_desc), "l"(b_desc), "r"(idesc), "r"(acc) : "memory");
}
__device__ __forceinline__ void umma_commit_2sm(uint64_t* bar, uint16_t mask) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 :: "r"(smem_u32(bar)), "h"(mask) : "memory");
}
__device__ __forceinline__ void mbar_arrive_on_cta(uint64_t* bar, uint32_t target_cta) {   // arrive on `bar` of another CTA
    asm volatile(
        "{\n\t.reg .b32 ra;\n\t"
        "mapa.shared::cluster.u32 ra, %0, %1;\n\t"
        "mbarrier.arrive.release.cluster.shared::cluster.b64 _, [ra];\n\t}"
        :: "r"(smem_u32(bar)), "r"(target_cta) : "memory");
}
__device__ __forceinline__ void mbar_wait_cluster(uint64_t* bar, uint32_t parity) {       // acquire at cluster scope
    const uint32_t addr = smem_u32(bar);
    const long long t0 = clock64();
    while (true) {
        uint32_t done;
        asm volatile(
            "{\n\t.reg .pred p;\n\t"
            "mbarrier.try_wait.parity.acquire.cluster.shared::cta.b64 p, [%1], %2;\n\t"
            "selp.u32 %0, 1, 0, p;\n\t}"
            : "=r"(done) : "r"(addr), "r"(parity) : "memory");
        if (done) return;
        if (clock64() - t0 > SPIN_LIMIT) __trap();
    }
}
#endif

// One lane of a fully active warp (the lowest).  The producer and the MMA issuer walk their loops with the WHOLE warp
// and elect inside: under `if (lane == 0)` the compiler has to emulate every uniform-datapath instruction (UTMALDG,
// UTCHMMA, UTCBAR) of the divergent region with an election loop plus vector->uniform register moves -- 38
// instructions per tcgen05.mma in r1 run 18's SASS, more issue latency than the MMA takes to execute.
#ifndef AECF_CUDA_EMU
__device__ __forceinline__ bool elect_one() {
    uint32_t pred;
    asm volatile(
        "{\n\t.reg .pred p;\n\t"
        "elect.sync _|p, 0xffffffff;\n\t"
        "selp.u32 %0, 1, 0, p;\n\t}"
        : "=r"(pred));
    return pred != 0;
}
#endif
// Advancing a shared-memory descriptor by `bytes` is an add on its 14-bit start-address field (16-byte units); every
// address stays inside the 227 KB of shared memory, so the field never carries into its neighbours.
__device__ __forceinline__ uint64_t desc_advance(uint64_t desc, uint32_t bytes) { return desc + (bytes >> 4); }
__device__ __forceinline__ uint32_t k_slice_bytes(int mn_major) { return mn_major ? UMMA_K * 128 : UMMA_K * 2; }

struct WorkItem { int m_blk, n_blk, split, kb_begin, kb_count; };

// Work items are (split, row-block group, column block); the CL CTAs of a cluster take the CL row blocks of
// a group (same column block, same k range), which is what lets them share the B tile by TMA multicast.
template <int CL>
__device__ __forceinline__ WorkItem decode(const Params& p, int item, int cta_rank) {
    WorkItem w;
    const int tiles = p.groups_m * p.tiles_n;
    w.split = item / tiles;
    const int t = item - w.split * tiles;
    const int group = t / p.tiles_n;         // n fastest: neighbouring clusters share the A row blocks in L2
    w.m_blk = group * CL + cta_rank;         // may be == tiles_m for the odd last group: loads zero-fill, stores clip
    w.n_blk = t - group * p.tiles_n;
    w.kb_begin = w.split * p.kb_per_split;
    w.kb_count = min(p.kb_per_split, p.kb_total - w.kb_begin);
    return w;
}

// Epilogue of the bf16-output path: the next 32-column group's tcgen05.ld is in flight while the current group is
// converted, and the two staging boxes alternate with `wait_group.read 1`, so neither the TMEM read latency nor the
// previous store's shared-memory read is exposed (r2 run 1, same-box A/B against the serial epilogue: the values
// product 113.0 -> 110.2 us, out_proj 38.9 -> 37.3 us, d_ctx 37.4 -> 36.4 us; the eight-warp variant was neutral and
// is gone).  fp32 output (split-K partials, fp32 C) keeps the serial rounds below.
template <int BN, int CL>
__global__ void __launch_bounds__(NUM_THREADS, 1)
gemm_tcgen05_kernel(const __grid_constant__ CUtensorMap map_a, const __grid_constant__ CUtensorMap map_b,
                    const __grid_constant__ CUtensorMap map_c, const Params p) {
    using C = Cfg<BN>;
    AECF_DYNAMIC_SMEM_ALIGNED1024(uint8_t, smem);                              // swizzle-128B tiles need 1024-byte alignment
    if (smem_u32(smem) & 1023u) __trap();
    uint8_t* stage_base = smem;
    uint8_t* epi_base = smem + STAGES * C::STAGE_BYTES;                       // 1024-aligned (stage sizes are)
    float* bias_tile = reinterpret_cast<float*>(epi_base + C::EPI_BYTES);      // [2][BN]
    uint64_t* bars = reinterpret_cast<uint64_t*>(epi_base + C::EPI_BYTES + C::BIAS_BYTES);
    uint64_t* full = bars;                        // [STAGES] TMA -> MMA
    uint64_t* empty = bars + STAGES;              // [STAGES] MMA -> TMA
    uint64_t* tmem_full = bars + 2 * STAGES;      // [2] MMA -> epilogue
    uint64_t* tmem_empty = bars + 2 * STAGES + 2; // [2] epilogue -> MMA
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * STAGES + 4);

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const int items = p.groups_m * p.tiles_n * p.splits;
    const int cta_rank = CL > 1 ? static_cast<int>(cluster_ctarank()) : 0;
    const int first_item = blockIdx.x / CL, item_stride = gridDim.x / CL;
    constexpr uint16_t kAllCtas = (1u << CL) - 1;

    if (warp == 0 && lane == 0) {
        prefetch_tmap(&map_a); prefetch_tmap(&map_b); prefetch_tmap(&map_c);
        for (int i = 0; i < STAGES; ++i) { mbar_init(&full[i], 1); mbar_init(&empty[i], CL); }   // every CTA's MMA frees a slot
        for (int i = 0; i < 2; ++i) { mbar_init(&tmem_full[i], 1); mbar_init(&tmem_empty[i], EPI_THREADS); }
        fence_barrier_init();
    }
    if (warp == 1) {                                  // one warp allocates TMEM and owns the dealloc
#ifdef AECF_CUDA_EMU
        if (lane == 0) cuda_emu::tc::tmem_alloc(tmem_slot, C::TMEM_COLS);
#else
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"(smem_u32(tmem_slot)), "r"(static_cast<uint32_t>(C::TMEM_COLS)) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
#endif
    }
    tc_fence_before();
    __syncthreads();
    if (CL > 1) cluster_sync_all();                  // peers' barriers exist before anything signals them
    tc_fence_after();
    const uint32_t tmem_base = *tmem_slot;
    pdl_wait();                                      // everything above overlapped the previous kernel's tail

    if (warp == 0) {
        // ===== TMA producer: the whole warp walks the loop, one elected lane issues (see elect_one) =====
        constexpr int PART = BN / CL;                 // this CTA's share of the B tile
        int it = 0;
        for (int item = first_item; item < items; item += item_stride) {
            const WorkItem w = decode<CL>(p, item, cta_rank);
            for (int kb = 0; kb < w.kb_count; ++kb, ++it) {
                const int s = it % STAGES;
                mbar_wait(&empty[s], ((it / STAGES) & 1) ^ 1);     // freed by the MMAs of ALL CTAs of the cluster
                if (elect_one()) {
                    uint8_t* a_dst = stage_base + s * C::STAGE_BYTES;
                    uint8_t* b_dst = a_dst + C::A_BYTES;
                    const int k0 = (w.kb_begin + kb) * BK;
                    mbar_expect_tx(&full[s], C::STAGE_BYTES);
                    if (!p.a_mn_major) {
                        tma_load_2d(&map_a, &full[s], a_dst, k0, w.m_blk * BM);
                    } else {
#pragma unroll
                        for (int a = 0; a < BM / 64; ++a)
                            tma_load_2d(&map_a, &full[s], a_dst + a * (BK * 128), w.m_blk * BM + a * 64, k0);
                    }
                    // with a cluster, this CTA fetches 1/CL of the B tile and multicasts it: every CTA's stage
                    // receives the full tile, each part read from L2 only once
                    if (!p.b_mn_major) {
                        if (CL == 1) tma_load_2d(&map_b, &full[s], b_dst + cta_rank * (PART * 128), k0, w.n_blk * BN + cta_rank * PART);
                        else tma_load_2d_mc(&map_b, &full[s], b_dst + cta_rank * (PART * 128), k0, w.n_blk * BN + cta_rank * PART, kAllCtas);
                    } else {
#pragma unroll
                        for (int a = 0; a < PART / 64; ++a) {
                            const int atom = cta_rank * (PART / 64) + a;
                            if (CL == 1) tma_load_2d(&map_b, &full[s], b_dst + atom * (BK * 128), w.n_blk * BN + atom * 64, k0);
                            else tma_load_2d_mc(&map_b, &full[s], b_dst + atom * (BK * 128), w.n_blk * BN + atom * 64, k0, kAllCtas);
                        }
                    }
                }
                __syncwarp();
            }
        }
    } else if (warp == 1) {
        // ===== MMA issuer: the whole warp walks the loop, one elected lane issues (see elect_one) =====
        const uint32_t idesc = make_idesc(BN, p.a_mn_major, p.b_mn_major);
        const uint32_t stage0 = smem_u32(stage_base);
        const uint64_t a_desc0 = operand_desc(stage0, p.a_mn_major, 0);                 // stage 0, K slice 0
        const uint64_t b_desc0 = operand_desc(stage0 + C::A_BYTES, p.b_mn_major, 0);
        const uint32_t a_ks = k_slice_bytes(p.a_mn_major), b_ks = k_slice_bytes(p.b_mn_major);
        int it = 0, tile_it = 0;
        for (int item = first_item; item < items; item += item_stride, ++tile_it) {
            const WorkItem w = decode<CL>(p, item, cta_rank);
            const int as = tile_it & 1;
            mbar_wait(&tmem_empty[as], ((tile_it >> 1) & 1) ^ 1);          // epilogue drained this accumulator
            tc_fence_after();
            const uint32_t tmem_d = tmem_base + as * C::ACC_STRIDE;
            for (int kb = 0; kb < w.kb_count; ++kb, ++it) {
                const int s = it % STAGES;
                mbar_wait(&full[s], (it / STAGES) & 1);
                tc_fence_after();
                if (elect_one()) {
                    const uint64_t a_d = desc_advance(a_desc0, s * C::STAGE_BYTES);
                    const uint64_t b_d = desc_advance(b_desc0, s * C::STAGE_BYTES);
#pragma unroll
                    for (int ks = 0; ks < BK / UMMA_K; ++ks)
                        umma_bf16(tmem_d, desc_advance(a_d, ks * a_ks), desc_advance(b_d, ks * b_ks), idesc, (kb | ks) != 0 ? 1u : 0u);
                    if (CL == 1) umma_commit(&empty[s]);                       // smem slot free once these MMAs retire
                    else umma_commit_mc(&empty[s], kAllCtas);                  // ... in every CTA that multicasts into it
                }
                __syncwarp();
            }
            if (elect_one()) umma_commit(&tmem_full[as]);                      // accumulator complete
            __syncwarp();
        }
    } else {
        // ===== epilogue: TMEM -> registers -> (+bias, convert) -> swizzled smem -> TMA store =====
        // Every epilogue warp is self-contained: it owns 32 accumulator rows (its TMEM lane quadrant), a
        // private 8 KB staging area (two [32 rows x 128 B] swizzled boxes) and issues its own TMA stores, so
        // the four warps never wait for one another -- only __syncwarp(), no block-level barrier.
        const int quad = warp & 3;                   // TMEM lane quadrant this warp may read
        const int ew = warp - 2;                     // 0..3: staging slot
        uint8_t* wbuf = epi_base + ew * (2 * 32 * 128);
        int box_it = 0;                              // bf16 output: boxes stored so far by this warp
        int tile_it = 0;
        for (int item = first_item; item < items; item += item_stride, ++tile_it) {
            const WorkItem w = decode<CL>(p, item, cta_rank);
            const int as = tile_it & 1;
            const int n0 = w.n_blk * BN, m0 = w.m_blk * BM;
            const bool tile_valid = w.m_blk < p.tiles_m;       // false only for the filler tile of an odd last group
            const bool direct = (p.splits == 1);
            mbar_wait(&tmem_full[as], (tile_it >> 1) & 1);
            tc_fence_after();
            // fp32 bias slice of this tile, in the buffer of this tile's parity.  All four warps write the same
            // values; a warp two tiles ahead would reuse this buffer, but it cannot pass the tmem_full wait
            // above before every thread has finished the tile that last used it (tmem_empty arrives after the
            // last bias read), so no reader ever sees a foreign tile's values.
            float* wbias = bias_tile + as * BN;
            if (direct && p.has_bias) {
                for (int i = lane; i < BN; i += 32) {
                    const int col = n0 + i;
                    float b = 0.f;
                    if (col < p.c_cols)
                        b = p.bias_is_bf16 ? __bfloat162float(static_cast<const __nv_bfloat16*>(p.bias)[col])
                                           : static_cast<const float*>(p.bias)[col];
                    wbias[i] = b;
                }
                __syncwarp();
            }
            const uint32_t t_row = tmem_base + as * C::ACC_STRIDE + (static_cast<uint32_t>(quad * 32) << 16);
            const int out_row0 = (direct ? 0 : w.split * p.partial_rows) + m0 + quad * 32;
            {
                if (!p.c_is_f32) {
                    // ---- pipelined bf16 epilogue: group g+1 is being read out of TMEM while group g is converted; box
                    // (g / 2) % 2 is refilled as soon as the store issued two boxes ago has read it (one may stay pending)
                    constexpr int GROUPS = BN / 32;
                    uint32_t r[2][32];
                    tmem_ld_32x32(t_row, r[0]);
#pragma unroll
                    for (int g = 0; g < GROUPS; ++g) {
                        tmem_ld_wait_on(r[g & 1]);                             // r[g & 1] has landed
                        if (g + 1 < GROUPS) tmem_ld_32x32(t_row + (g + 1) * 32, r[(g + 1) & 1]);
                        // boxes alternate ACROSS tiles too (a 192-wide tile fills three), so the box being refilled is
                        // always the one stored two commits ago
                        uint8_t* box_base = wbuf + ((box_it + (g >> 1)) & 1) * (32 * 128);
                        uint8_t* box = box_base + lane * 128;
                        if ((g & 1) == 0) {
#ifdef AECF_CUDA_EMU
                            if (lane == 0) cuda_emu::tc::store_wait_read(1);
#else
                            if (lane == 0) asm volatile("cp.async.bulk.wait_group.read 1;" ::: "memory");
#endif
                            __syncwarp();
                        }
                        float v[32];
#pragma unroll
                        for (int i = 0; i < 32; ++i) {
                            v[i] = __uint_as_float(r[g & 1][i]);
                            if (direct && p.has_bias) v[i] += wbias[g * 32 + i];
                        }
                        if (g == GROUPS - 1) {                                 // every TMEM and bias read of this tile is done
                            tc_fence_before();
                            mbar_arrive(&tmem_empty[as]);
                        }
                        if (p.aux != nullptr && n0 + g * 32 == p.c_cols) {
                            const int row = m0 + quad * 32 + lane;
                            if (tile_valid && row < p.m) {
                                float4* dst = reinterpret_cast<float4*>(p.aux + static_cast<long long>(row) * p.aux_ld);
#pragma unroll
                                for (int c = 0; c < 8; ++c)
                                    if (4 * c < p.aux_cols) dst[c] = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
                            }
                        }
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const int chunk = (g & 1) * 4 + c;
                            *reinterpret_cast<uint4*>(box + ((chunk ^ (lane & 7)) << 4)) =
                                make_uint4(Vec<__nv_bfloat16>::pack2(v[8 * c], v[8 * c + 1]),
                                           Vec<__nv_bfloat16>::pack2(v[8 * c + 2], v[8 * c + 3]),
                                           Vec<__nv_bfloat16>::pack2(v[8 * c + 4], v[8 * c + 5]),
                                           Vec<__nv_bfloat16>::pack2(v[8 * c + 6], v[8 * c + 7]));
                        }
                        if ((g & 1) == 1 || g == GROUPS - 1) {                 // a 64-column box is complete: store it
                            fence_proxy_async();
                            __syncwarp();
                            const int col0 = n0 + (g >> 1) * 64;
                            if (lane == 0) {
                                if (tile_valid && col0 < p.c_cols) tma_store_2d(&map_c, box_base, col0, out_row0);
                                tma_store_commit();                            // one group per box, stored or not
                            }
                        }
                    }
                    box_it += (GROUPS + 1) / 2;
                    continue;
                }
            }
            // the staging area holds 128 bf16 columns or 64 fp32 columns per round
            const int cols_per_round = p.c_is_f32 ? 64 : 128;
            const int rounds = (BN + cols_per_round - 1) / cols_per_round;
#pragma unroll 1
            for (int rd = 0; rd < rounds; ++rd) {
                if (lane == 0) tma_store_wait_read();                          // my previous store has left the staging area
                __syncwarp();
                const int col_in_tile = rd * cols_per_round;
                const int groups = min(cols_per_round, BN - col_in_tile) / 32;  // BN = 192: the last round is half full
#pragma unroll 1
                for (int g = 0; g < groups; ++g) {                             // 32 columns per TMEM load
                    uint32_t r[32];
                    tmem_ld_32x32(t_row + col_in_tile + g * 32, r);
                    tmem_ld_wait();
                    float v[32];
#pragma unroll
                    for (int i = 0; i < 32; ++i) {
                        v[i] = __uint_as_float(r[i]);
                        if (direct && p.has_bias) v[i] += wbias[col_in_tile + g * 32 + i];
                    }
                    if (p.aux != nullptr && n0 + col_in_tile + g * 32 == p.c_cols) {
                        // the side columns: fp32 straight from the accumulator, one row per thread (32-byte runs)
                        const int row = m0 + quad * 32 + lane;
                        if (tile_valid && row < p.m) {
                            float4* dst = reinterpret_cast<float4*>(p.aux + static_cast<long long>(row) * p.aux_ld);
#pragma unroll
                            for (int c = 0; c < 8; ++c)
                                if (4 * c < p.aux_cols) dst[c] = make_float4(v[4 * c], v[4 * c + 1], v[4 * c + 2], v[4 * c + 3]);
                        }
                    }
                    if (p.c_is_f32) {
                        // box g: [32 rows x 32 fp32 = 128 B]; 16-byte chunk c of row `lane` sits at chunk c ^ (lane & 7)
                        uint8_t* box = wbuf + g * (32 * 128) + lane * 128;
#pragma unroll
                        for (int c = 0; c < 8; ++c)
                            *reinterpret_cast<uint4*>(box + ((c ^ (lane & 7)) << 4)) =
                                make_uint4(__float_as_uint(v[4 * c]), __float_as_uint(v[4 * c + 1]),
                                           __float_as_uint(v[4 * c + 2]), __float_as_uint(v[4 * c + 3]));
                    } else {
                        // box g / 2: [32 rows x 64 bf16 = 128 B]; this load fills chunks (g % 2) * 4 .. + 3
                        uint8_t* box = wbuf + (g >> 1) * (32 * 128) + lane * 128;
#pragma unroll
                        for (int c = 0; c < 4; ++c) {
                            const int chunk = (g & 1) * 4 + c;
                            *reinterpret_cast<uint4*>(box + ((chunk ^ (lane & 7)) << 4)) =
                                make_uint4(Vec<__nv_bfloat16>::pack2(v[8 * c], v[8 * c + 1]),
                                           Vec<__nv_bfloat16>::pack2(v[8 * c + 2], v[8 * c + 3]),
                                           Vec<__nv_bfloat16>::pack2(v[8 * c + 4], v[8 * c + 5]),
                                           Vec<__nv_bfloat16>::pack2(v[8 * c + 6], v[8 * c + 7]));
                        }
                    }
                }
                if (rd == rounds - 1) {                                        // all TMEM reads of this tile done
                    tc_fence_before();
                    mbar_arrive(&tmem_empty[as]);
                }
                fence_proxy_async();                                           // smem writes -> visible to TMA
                __syncwarp();
                if (lane == 0 && tile_valid) {
                    const int col0 = n0 + col_in_tile;
                    const int box_cols = p.c_is_f32 ? 32 : 64;
#pragma unroll
                    for (int g = 0; g < 2; ++g)
                        if (col0 + g * box_cols < p.c_cols && col_in_tile + g * box_cols < BN)
                            tma_store_2d(&map_c, wbuf + g * (32 * 128), col0 + g * box_cols, out_row0);
                    tma_store_commit();
                }
            }
        }
        if (lane == 0) tma_store_wait_all();
    }

    __syncwarp();
    tc_fence_before();
    __syncthreads();
    if (CL > 1) cluster_sync_all();                  // nobody leaves while a peer may still multicast into it
    if (warp == 1) {
        tc_fence_after();
#ifndef AECF_CUDA_EMU
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;"
                     :: "r"(tmem_base), "r"(static_cast<uint32_t>(C::TMEM_COLS)) : "memory");
#endif
    }
}

// ================================================================================================
// cta_group::2 variant: the two CTAs of a cluster compute ONE 256 x 256 tile.  Each CTA stages its own
// 128 rows of A and HALF of the B tile (128 of the 256 columns), so a stage is 32 KB instead of 48 KB
// and the ring is 6 deep instead of 4 -- 5 k-blocks of load latency covered instead of 3, which is what
// the single-CTA kernel lacks (ncu: tensor pipe 59-78 % active, waiting on the ring).  The leader CTA
// issues tcgen05.mma.cta_group::2 (M = 256); each CTA's TMEM receives its own 128 accumulator rows and
// each CTA runs its own epilogue.
// ================================================================================================
constexpr int STAGES_2SM = 5;
template <int BN> struct Cfg2 {
    static constexpr int A_BYTES = BM * BK * 2;                 // 16 KB: this CTA's 128 rows
    static constexpr int B_BYTES = (BN / 2) * BK * 2;           // 16 KB: this CTA's half of the columns
    static constexpr int STAGE_BYTES = A_BYTES + B_BYTES;
    static constexpr int EPI_BUF = 2 * BM * 128;                // one staging buffer: two [128 rows x 128 B] boxes
    static constexpr int EPI_BYTES = 2 * EPI_BUF;               // double buffered: convert round r+1 while round r is stored
    static constexpr int ACC_STRIDE = BN > 128 ? 256 : 128;     // TMEM column stride between the two accumulators
    static constexpr int TMEM_COLS = 2 * ACC_STRIDE;            // a power of two (= 2 * BN for the 256-wide tiles)
    static constexpr int SMEM_BYTES = STAGES_2SM * STAGE_BYTES + EPI_BYTES + 1024 + 256;
};

#include "gemm_tcgen05_2sm.inc"

// ---- host side -------------------------------------------------------------------------------
using EncodeFn = CUresult (*)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*, const cuuint64_t*,
                              const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave, CUtensorMapSwizzle,
                              CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static EncodeFn encode_fn() {
#ifdef AECF_CUDA_EMU
    return &cuda_emu::tc::encode_tiled;
#endif
    static EncodeFn fn = nullptr;
    static std::once_flag once;
    std::call_once(once, [] {
        void* sym = nullptr;
        cudaDriverEntryPointQueryResult q;
        if (cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &sym, cudaEnableDefault, &q) == cudaSuccess &&
            q == cudaDriverEntryPointSuccess)
            fn = reinterpret_cast<EncodeFn>(sym);
    });
    return fn;
}

// 2-D row-major tensor [rows, cols] with leading dimension ld (elements); box = [box_rows, box_cols],
// box_cols * elem_bytes == 128 (one swizzle atom).
static bool make_map(CUtensorMap* map, const void* ptr, CUtensorMapDataType dt, int es, long long rows, long long cols,
                     long long ld, int box_rows, int box_cols) {
    EncodeFn fn = encode_fn();
    if (!fn) return false;
    const cuuint64_t dims[2] = {static_cast<cuuint64_t>(cols), static_cast<cuuint64_t>(rows)};
    const cuuint64_t strides[1] = {static_cast<cuuint64_t>(ld) * es};
    const cuuint32_t box[2] = {static_cast<cuuint32_t>(box_cols), static_cast<cuuint32_t>(box_rows)};
    const cuuint32_t estr[2] = {1, 1};
    return fn(map, dt, 2, const_cast<void*>(ptr), dims, strides, box, estr, CU_TENSOR_MAP_INTERLEAVE_NONE,
              CU_TENSOR_MAP_SWIZZLE_128B, CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE) ==
           CUDA_SUCCESS;
}

struct Plan { bool ok, two_sm; int bn, cluster, tiles_m, tiles_n, groups_m, splits, kb_per_split, kb_total; };

// rows of B that carry the side output: aux_cols rounded up to 16 bytes of bf16
static int aux_rows_of(int aux_cols) { return (aux_cols + 7) & ~7; }

static Plan make_plan(const aecf_gemm_desc* d, int aux_cols = 0) {
    Plan pl{};
    pl.ok = false;
    if (d->dtype_a != AECF_BF16 || d->dtype_b != AECF_BF16 || d->accumulate) return pl;
    if (d->m < 128 || d->n < 128 || d->k < 64) return pl;                 // GEMV-shaped / tiny: SIMT kernel
    if (d->m > 0x7fffffffLL || d->n > 0x7fffffffLL || d->k > 0x7fffffffLL) return pl;
    if ((d->lda * 2) % 16 != 0 || (d->ldb * 2) % 16 != 0) return pl;
    const int ces = d->dtype_c == AECF_BF16 ? 2 : 4;
    if ((d->ldc * ces) % 16 != 0) return pl;
    const long long n_total = d->n + aux_rows_of(aux_cols);
    pl.bn = d->n >= 256 ? 256 : 128;
    if (aux_cols > 0) {
        // side output: 192-wide tiles cover n + 8 with the least padding for every embed_dim of the sweep
        // (520 -> 3 tiles, 1032 -> 6, 2056 -> 11); the side columns must start a 32-column TMEM group, and the
        // 96-row halves of the B tile that the cluster multicasts exist only for a K-major B
        if (aux_cols > 32 || d->n % 32 != 0 || d->b_layout != AECF_K_MAJOR) return pl;
        pl.bn = 192;
    }
    pl.tiles_m = static_cast<int>((d->m + tc::BM - 1) / tc::BM);
    pl.tiles_n = static_cast<int>((n_total + pl.bn - 1) / pl.bn);
    pl.kb_total = static_cast<int>((d->k + tc::BK - 1) / tc::BK);
    // Pairs of CTAs (a cluster of 2) on vertically adjacent row blocks share the B tile by TMA multicast:
    // a third less L2 -> SM traffic per FLOP, which is what bounds these K = 512..1024 products.
    pl.cluster = pl.tiles_m >= 2 ? 2 : 1;
    pl.two_sm = false;        // decided below, once the k range of a work item is known
    pl.groups_m = (pl.tiles_m + pl.cluster - 1) / pl.cluster;
    const int sms = sm_count(d->device);
    const long long tiles = static_cast<long long>(pl.groups_m) * pl.cluster * pl.tiles_n;
    int splits = 1;
    if (tiles * 2 <= sms && pl.kb_total >= 16) {       // weight-gradient shape: few tiles, long reduction
        splits = static_cast<int>(sms / tiles);
        const int by_k = pl.kb_total / 8;
        if (splits > by_k) splits = by_k;
        if (splits < 1) splits = 1;
    }
    pl.kb_per_split = (pl.kb_total + splits - 1) / splits;
    pl.splits = (pl.kb_total + pl.kb_per_split - 1) / pl.kb_per_split;
    // cta_group::2 (one 256 x 256 tile per CTA pair: each CTA stages its 128 rows of A and HALF of the B tile, a third
    // fewer operand bytes delivered per FLOP, and a deeper ring).  A/B on one box with the warp-uniform issue loops
    // (profiles/r1_gemm_experiments.md, run 24): it wins from 9 k-blocks per work item on -- dX (K = 520) 109 -> 103 us,
    // [dWv ; R] 121 -> 112 us even though its 520 rows fill only 2.03 of 3 CTA pairs -- and loses on the 8-k-block
    // products (out_proj 38 -> 42 us), whose per-tile pair handshake is not amortised.
    const bool long_k = pl.kb_per_split >= 9;
    pl.two_sm = pl.cluster == 2 && pl.bn == 256 && long_k;
    if (aux_cols > 0 && pl.splits != 1) return pl;       // the side output is written by the direct epilogue only
    pl.ok = true;
    return pl;
}

}  // namespace tc

size_t gemm_tcgen05_workspace_bytes(const aecf_gemm_desc* d) {
    const tc::Plan pl = tc::make_plan(d);
    if (!pl.ok || pl.splits == 1) return 0;
    return static_cast<size_t>(pl.splits) * pl.tiles_m * tc::BM * d->n * sizeof(float);
}

int gemm_tcgen05(const aecf_gemm_desc* d, const void* A, const void* B, const void* bias, void* C, void* workspace,
                 size_t workspace_bytes, cudaStream_t s, float* aux, int aux_cols, long long aux_ld, GemmPartials* defer) {
    using namespace tc;
    if (aux == nullptr) aux_cols = 0;
    const Plan pl = make_plan(d, aux_cols);
    if (aux_cols > 0 && (!aligned16(aux) || aux_ld % 4 != 0 || aux_ld < ((aux_cols + 3) & ~3))) return AECF_ERR_UNSUPPORTED;
    const long long n_total = d->n + aux_rows_of(aux_cols);
    if (!pl.ok) return AECF_ERR_UNSUPPORTED;
    if (!aligned16(A) || !aligned16(B) || !aligned16(C)) return AECF_ERR_UNSUPPORTED;
    if (pl.splits > 1) {
        if (!workspace || workspace_bytes < gemm_tcgen05_workspace_bytes(d)) return AECF_ERR_WORKSPACE;
        if (!aligned16(workspace) || (d->n * 4) % 16 != 0) return AECF_ERR_UNSUPPORTED;
    }
    CUtensorMap map_a, map_b, map_c;
    bool ok = true;
    // A: K-major [m, k] -> box [BM rows, 64 k];  MN-major stored [k, m] -> box [64 k rows, 64 m]
    if (d->a_layout == AECF_K_MAJOR) ok &= make_map(&map_a, A, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, d->m, d->k, d->lda, BM, BK);
    else ok &= make_map(&map_a, A, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, d->k, d->m, d->lda, BK, 64);
    if (d->b_layout == AECF_K_MAJOR) ok &= make_map(&map_b, B, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, n_total, d->k, d->ldb, pl.bn / pl.cluster, BK);
    else ok &= make_map(&map_b, B, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, d->k, d->n, d->ldb, BK, 64);
    const bool partial = pl.splits > 1;
    const bool c_f32 = partial || d->dtype_c == AECF_F32;
    // store boxes: the 1SM kernel's epilogue warps each store their own 32 rows; the 2SM kernel stores 128 rows at once
    const int c_rows = pl.two_sm ? BM : 32;
    if (partial) ok &= make_map(&map_c, workspace, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, static_cast<long long>(pl.splits) * pl.tiles_m * BM, d->n, d->n, c_rows, 32);
    else if (c_f32) ok &= make_map(&map_c, C, CU_TENSOR_MAP_DATA_TYPE_FLOAT32, 4, d->m, d->n, d->ldc, c_rows, 32);
    else ok &= make_map(&map_c, C, CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, d->m, d->n, d->ldc, c_rows, 64);
    if (!ok) return AECF_ERR_UNSUPPORTED;

    Params p{};
    p.m = static_cast<int>(d->m); p.n = static_cast<int>(n_total); p.k = static_cast<int>(d->k);
    p.c_cols = static_cast<int>(d->n); p.aux = aux_cols > 0 ? aux : nullptr; p.aux_cols = aux_cols; p.aux_ld = aux_ld;
    p.tiles_m = pl.tiles_m; p.tiles_n = pl.tiles_n; p.groups_m = pl.groups_m; p.splits = pl.splits;
    p.kb_per_split = pl.kb_per_split; p.kb_total = pl.kb_total;
    p.a_mn_major = d->a_layout == AECF_MN_MAJOR; p.b_mn_major = d->b_layout == AECF_MN_MAJOR;
    p.c_is_f32 = c_f32;
    p.has_bias = bias != nullptr; p.bias_is_bf16 = d->dtype_bias == AECF_BF16; p.bias = bias;
    p.partial_rows = pl.tiles_m * BM;              // padded: a ragged last row block must not spill into the next split

    const long long items = static_cast<long long>(pl.groups_m) * pl.tiles_n * pl.splits;     // one per cluster
    const int sms = sm_count(d->device);
    long long ctas = items * pl.cluster;
    const long long cap = sms / pl.cluster * pl.cluster;
    if (ctas > cap) ctas = cap;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(static_cast<unsigned>(ctas));
    cfg.blockDim = dim3(NUM_THREADS);
    cfg.stream = s;
    cudaLaunchAttribute attr[2];
    attr[0].id = cudaLaunchAttributeClusterDimension;
    attr[0].val.clusterDim.x = pl.cluster; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
    attr[1].id = cudaLaunchAttributeProgrammaticStreamSerialization;
    attr[1].val.programmaticStreamSerializationAllowed = 1;
    cfg.attrs = attr; cfg.numAttrs = 2;
#define AECF_TC_LAUNCH(BN_, CL_)                                                                                  \
    do {                                                                                                          \
        auto kernel = gemm_tcgen05_kernel<BN_, CL_>;                                                              \
        cfg.dynamicSmemBytes = Cfg<BN_>::SMEM_BYTES;                                                              \
        AECF_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg<BN_>::SMEM_BYTES)); \
        AECF_CUDA_OK(cudaLaunchKernelEx(&cfg, kernel, map_a, map_b, map_c, p));                                   \
    } while (0)
    if (pl.two_sm) note_gemm_kernel("tcgen05 2sm bn%d splits%d", pl.bn, pl.splits);
    else note_gemm_kernel("tcgen05 1sm bn%d cluster%d splits%d", pl.bn, pl.cluster, pl.splits);
    if (pl.two_sm) {
        auto kernel = gemm_tcgen05_2sm_kernel<256>;
        cfg.dynamicSmemBytes = Cfg2<256>::SMEM_BYTES;
        AECF_CUDA_OK(cudaFuncSetAttribute(kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, Cfg2<256>::SMEM_BYTES));
        AECF_CUDA_OK(cudaLaunchKernelEx(&cfg, kernel, map_a, map_b, map_c, p));
    } else if (pl.bn == 256) { if (pl.cluster == 2) AECF_TC_LAUNCH(256, 2); else AECF_TC_LAUNCH(256, 1); }
    else if (pl.bn == 192) { if (pl.cluster == 2) AECF_TC_LAUNCH(192, 2); else AECF_TC_LAUNCH(192, 1); }
    else { if (pl.cluster == 2) AECF_TC_LAUNCH(128, 2); else AECF_TC_LAUNCH(128, 1); }
#undef AECF_TC_LAUNCH
    count_launch();
    AECF_CUDA_OK(cudaGetLastError());
    if (defer != nullptr) {
        if (partial) *defer = GemmPartials{static_cast<const float*>(workspace), pl.splits, static_cast<long long>(pl.tiles_m) * BM * d->n};
        else *defer = GemmPartials{static_cast<const float*>(C), 1, 0};
        return AECF_OK;
    }
    if (!partial) return AECF_OK;
    GemmEpilogue ep = make_epilogue(d, bias, C);
    return launch_splitk_reduce(static_cast<const float*>(workspace), d->m, d->n, pl.splits,
                                static_cast<long long>(pl.tiles_m) * BM * d->n, ep, s);
}

}  // namespace aecf
