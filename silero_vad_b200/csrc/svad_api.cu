// svad_api.cu -- CUDA kernel instantiations and the C ABI (include/silero_vad_b200.h) of the
// B200-native Silero-VAD engine.  Build: nvcc -gencode arch=compute_100a,code=sm_100a (see build.py).
//
// Kernel `svad_fused_fp32<SR16, RM>`: one persistent CTA (256 threads, ~214 KB dynamic shared memory,
// one CTA per SM) per tile of 4*RM streams; the whole per-chunk forward pass (STFT -> 4 conv -> LSTM ->
// head) for all T chunks runs inside the launch with (h, c) and the audio context resident on the SM.
// The weights are a linear "tape" in global memory (L2-resident, 0.89 MB) that thread 0 streams into a
// two-stage shared-memory ring with cp.async.bulk (TMA bulk copy, completion on an mbarrier) one slab
// ahead of the FFMA loops.  HBM traffic is the audio read once plus 4 B per chunk of probabilities.
#include <cuda_runtime.h>
#include <cooperative_groups.h>

#include <cstdarg>
#include <cstdio>
#include <cstdlib>
#include <atomic>
#include <chrono>
#include <exception>
#include <new>
#include <string>
#include <vector>

#include "../../include/silero_vad_b200.h"
#include "svad_tc.h"
#include "svad_small.h"
#include "svad_h16.cuh"
#include "svad_train.cuh"

using namespace svad;

// ------------------------------------------------------------------------------------------ device
namespace {

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

template <bool SR16, bool FEAT = false>
struct GpuEnv {
    static constexpr int kNslab = FEAT ? Geo<SR16>::nslab_enc : Geo<SR16>::nslab;   // slabs per step (run_cta's FEAT)
    float* sm;
    uint64_t* full;   // [kStages] "slab landed" mbarriers (TMA transaction count)
    uint64_t* empty;  // [kStages] "slab consumed" mbarriers (one arrival per warp)
    const float* tape;
    int tid_;
    __device__ __forceinline__ int tid() const { return tid_; }
    __device__ __forceinline__ float* smem() { return sm; }
    __device__ __forceinline__ void sync() { __syncthreads(); }
    __device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
    __device__ __forceinline__ void issue(long it) {  // one thread
        const int idx = (int)(it % kNslab), stage = (int)(it % kStages);
        const uint32_t bytes = (uint32_t)Tape<SR16>::slab_len(idx) * 4u;
        const uint32_t bar = smem_u32(full + stage);
        const uint32_t dst = smem_u32(sm + SmemMap::stage + stage * SmemMap::stage_floats);
        const float* src = tape + Tape<SR16>::slab_off(idx);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                     "l"(src), "r"(bytes), "r"(bar)
                     : "memory");
    }
    __device__ __forceinline__ static void mbar_wait(uint32_t bar, uint32_t parity) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "WAIT_%=:\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
            "@p bra DONE_%=;\n"
            "bra WAIT_%=;\n"
            "DONE_%=:\n"
            "}\n" ::"r"(bar),
            "r"(parity)
            : "memory");
    }
    __device__ __forceinline__ const float* slab_acquire(long it, long total) {
        if (tid_ == 0 && it >= 1 && it + 1 < total) {
            const long prev = it - 1;   // slab it+1 goes into the stage slab it-1 occupied
            mbar_wait(smem_u32(empty + (prev % kStages)), (uint32_t)((prev / kStages) & 1));
            issue(it + 1);
        }
        const int stage = (int)(it % kStages);
        mbar_wait(smem_u32(full + stage), (uint32_t)((it / kStages) & 1));
        return sm + SmemMap::stage + stage * SmemMap::stage_floats;
    }
    __device__ __forceinline__ void slab_done(long it) {   // one arrival per warp once all its lanes are done reading
        __syncwarp();
        if ((tid_ & 31) == 0)
            asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(empty + (it % kStages))) : "memory");
    }
};

constexpr size_t kSmemBytes = (size_t)SmemMap::total_floats * 4 + 64;

template <bool SR16, int RM, typename S, bool FEAT = false>
__global__ void __launch_bounds__(kThreads, 1) svad_fused_fp32(TileArgs a, int ntiles) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    float* sm = reinterpret_cast<float*>(smem_raw);
    uint64_t* full = reinterpret_cast<uint64_t*>(smem_raw + (size_t)SmemMap::total_floats * 4);
    uint64_t* empty = full + kStages;
    GpuEnv<SR16, FEAT> env{sm, full, empty, a.tape, (int)threadIdx.x};
    int my_tiles = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) my_tiles++;
    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; s++) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(full + s)) : "memory");
            asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" ::"r"(smem_u32(empty + s)), "r"(kThreads / 32) : "memory");
        }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
        const long total = (long)my_tiles * a.T * GpuEnv<SR16, FEAT>::kNslab;
        for (long i = 0; i < kStages && i < total; i++) env.issue(i);
    }
    __syncthreads();
    run_cta<SR16, RM, S, FEAT>(env, a, (int)blockIdx.x, (int)gridDim.x, ntiles);
}


// ------------------------------------------------------------------------------------------ tensor-core kernel
// Shared-memory matrix descriptor (tcgen05): start address, leading / stride byte offsets (>>4), version 1,
// layout type 2 = SWIZZLE_128B (K-major weight tiles), 1 = SWIZZLE_128B_BASE32B (MN-major tf32 activation rows).
__device__ __forceinline__ uint64_t umma_desc(uint32_t saddr, uint32_t lbo, uint32_t sbo, uint32_t layout) {
    return (uint64_t)((saddr >> 4) & 0x3FFF) | ((uint64_t)((lbo >> 4) & 0x3FFF) << 16) | ((uint64_t)((sbo >> 4) & 0x3FFF) << 32) |
           ((uint64_t)1 << 46) | ((uint64_t)layout << 61);
}
// instruction descriptor: D fp32, A/B tf32, A K-major, B MN-major, N = 32, M = 128
constexpr uint32_t kIdescTf32 = (1u << 4) | (2u << 7) | (2u << 10) | (0u << 15) | (1u << 16) | ((32u >> 3) << 17) | ((128u >> 4) << 24);
constexpr uint32_t kTmemCols = 512;   // enc0 D 0..127, LSTM gates 128..255, enc0 D2 (w_lo terms) 256..383

template <bool SR16>
struct GpuEnvTC {
    float* sm;
    uint64_t* full;    // [kTcStages] slab landed (TMA tx)
    uint64_t* mdone;   // [kTcStages] MMAs that read the stage have completed (tcgen05.commit)
    uint64_t* accb;    // layer accumulators complete
    const float* tape;
    const int4* tab;   // per slab of a step: {dep_delta | buffer << 8, bytes, shared-memory destination, tape offset} (built once per CTA)
    int tid_;
    uint32_t tmem;
    // warp-0 bookkeeping (identical in all its lanes): next slab to issue / last slab known consumed, their position in
    // the per-step schedule, parity bits of the mdone barriers, parity of the accumulator barrier
    int issued, issued_idx, freed;
    uint32_t mpar, fpar, acc_phase;   // parity bits: consumed barriers (ring warp), landed barriers (every consumer), accumulators
    __device__ __forceinline__ int tid() const { return tid_; }
    __device__ __forceinline__ float* smem() { return sm; }
    __device__ __forceinline__ void sync() { __syncthreads(); }
    __device__ __forceinline__ void prefetch_l2(const void* p) { asm volatile("prefetch.global.L2 [%0];" ::"l"(p)); }
    __device__ __forceinline__ void fence_async() { asm volatile("fence.proxy.async.shared::cta;" ::: "memory"); }
    __device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
    __device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
    __device__ __forceinline__ static bool elect() {   // one lane of a fully converged warp
        uint32_t pred;
        asm volatile("{\n.reg .pred P;\nelect.sync _|P, 0xffffffff;\nselp.u32 %0, 1, 0, P;\n}\n" : "=r"(pred));
        return pred != 0;
    }
    __device__ __forceinline__ static void mbar_wait(uint32_t bar, uint32_t parity) {
        asm volatile(
            "{\n"
            ".reg .pred p;\n"
            "WAIT_%=:\n"
            "mbarrier.try_wait.parity.shared::cta.b64 p, [%0], %1;\n"
            "@p bra DONE_%=;\n"
            "bra WAIT_%=;\n"
            "DONE_%=:\n"
            "}\n" ::"r"(bar),
            "r"(parity)
            : "memory");
    }
    __device__ __forceinline__ void issue(int idx) {   // one lane
        using TP = TapeTC<SR16>;
        const int b = TP::buf(idx);
        const uint32_t bytes = (uint32_t)TP::slab_len(idx) * 4u;
        const uint32_t bar = smem_u32(full + b);
        const uint32_t dst = smem_u32(sm + TP::template buf_off<SmemMapTC>(b));
        const float* src = tape + TP::slab_off(idx);
        asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(bytes) : "memory");
        asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(dst),
                     "l"(src), "r"(bytes), "r"(bar)
                     : "memory");
    }
    // consumers: wait for the slab with per-step index idx; one parity bit per buffer, flipped at every visit
    __device__ __forceinline__ const float* slab_wait(int idx) {
        using TP = TapeTC<SR16>;
        const int b = TP::buf(idx);
        mbar_wait(smem_u32(full + b), (fpar >> b) & 1u);
        fpar ^= 1u << b;
        return sm + TP::template buf_off<SmemMapTC>(b);
    }
    __device__ __forceinline__ void skip_phase(uint32_t mask, int) { fpar ^= mask; }
    __device__ __forceinline__ void slab_pass(int idx) { fpar ^= 1u << TapeTC<SR16>::buf(idx); }
    // ring warp
    __device__ __forceinline__ void wait_consumed_group(int idx, int n) {   // slabs are released in order
        for (int i = 0; i < n - 1; i++) mpar ^= 1u << TapeTC<SR16>::buf(idx + i);   // their phases complete before the last one's
        const int b = TapeTC<SR16>::buf(idx + n - 1);
        mbar_wait(smem_u32(mdone + b), (mpar >> b) & 1u);
        mpar ^= 1u << b;
    }
    __device__ __forceinline__ void ring_freed(int total) {
        using TP = TapeTC<SR16>;
        freed++;
        while (issued < total) {
            const int4 e = tab[issued_idx];   // table lookup: the branchy constexpr slab maps cost the ring warp ~150 cycles per slab
            if (issued - (e.x & 0xff) > freed) break;
            if (elect()) {
                const uint32_t bar = smem_u32(full + (e.x >> 8));
                asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" ::"r"(bar), "r"(e.y) : "memory");
                asm volatile("cp.async.bulk.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1], %2, [%3];" ::"r"(e.z),
                             "l"(tape + e.w), "r"(e.y), "r"(bar)
                             : "memory");
            }
            issued++;
            if (++issued_idx == TP::nslab) issued_idx = 0;
        }
    }
    // descriptors: low word carries the address; a k-step advances A by 32 B and B by 8 rows = 1024 B
    __device__ __forceinline__ uint64_t mma_a(const float* tile) const { return umma_desc(smem_u32(tile), 16, 1024, 2); }
    // B: N atoms of 32 slots (consecutive frames for enc0) at stride lbo_bytes, 4-row k groups 512 B apart
    __device__ __forceinline__ uint64_t mma_b(const float* rows, int lbo_bytes) const { return umma_desc(smem_u32(rows), (uint32_t)lbo_bytes, 512, 1); }
    template <int MM = 128>
    __device__ __forceinline__ void mma(int col, uint64_t ad, uint64_t bd, int ks, bool acc, int ncols) {
        const uint64_t a2 = ad + (uint64_t)(ks * 2), b2 = bd + (uint64_t)(ks * 64);
        const uint32_t accf = acc ? 1u : 0u;
        const uint32_t idesc = (kIdescTf32 & ~((0x3Fu << 17) | (0x1Fu << 24))) | ((uint32_t)(ncols >> 3) << 17) | ((uint32_t)(MM >> 4) << 24);
        if (elect())
            asm volatile(
                "{\n"
                ".reg .pred p;\n"
                "setp.ne.b32 p, %4, 0;\n"
                "tcgen05.mma.cta_group::1.kind::tf32 [%0], %1, %2, %3, p;\n"
                "}\n" ::"r"(tmem + (uint32_t)col),
                "l"(a2), "l"(b2), "r"(idesc), "r"(accf)
                : "memory");
    }
    // The 4 k-steps of one 32-wide k-chunk in ONE elected region: per k-step up to three (A, B) descriptor pairs (w_hi x_hi,
    // w_hi x_lo, w_lo x_hi), all into the same accumulator.  One elect / one descriptor transfer to the uniform registers
    // per chunk instead of per instruction: the per-instruction issue sequence (~30 SASS instructions, ~130 cycles) was
    // what bounded the MMA phases, not the tensor pipe.
#define SVAD_MMA(A, B, P) "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], " A ", " B ", %7, " P ";\n"
#define SVAD_MMB(A, B, P) "@q tcgen05.mma.cta_group::1.kind::tf32 [%0], " A ", " B ", %9, " P ";\n"
#define SVAD_KSTEP(N) "add.s64 a0, %1, " #N "*2; add.s64 b0, %2, " #N "*64; add.s64 a1, %3, " #N "*2; add.s64 b1, %4, " #N "*64; add.s64 a2, %5, " #N "*2; add.s64 b2, %6, " #N "*64;\n"
    template <int MM, int NP>
    __device__ __forceinline__ void mma_ks4(int col, uint64_t a0, uint64_t b0, uint64_t a1, uint64_t b1, uint64_t a2, uint64_t b2, bool acc_first, int ncols, int ncols12 = 0) {
        const uint32_t idesc = (kIdescTf32 & ~((0x3Fu << 17) | (0x1Fu << 24))) | ((uint32_t)(ncols >> 3) << 17) | ((uint32_t)(MM >> 4) << 24);
        const uint32_t idesc12 = ncols12 ? ((idesc & ~(0x3Fu << 17)) | ((uint32_t)(ncols12 >> 3) << 17)) : idesc;   // pairs 1, 2 may use another N
        const uint32_t d = tmem + (uint32_t)col, accf = acc_first ? 1u : 0u;
        if constexpr (NP == 3) {
            asm volatile("{\n.reg .pred q, p, t;\n.reg .b64 a0, b0, a1, b1, a2, b2;\nelect.sync _|q, 0xffffffff;\nsetp.ne.b32 p, %8, 0;\nsetp.eq.u32 t, %8, %8;\n"
                         SVAD_KSTEP(0) SVAD_MMA("a0", "b0", "p") SVAD_MMB("a1", "b1", "t") SVAD_MMB("a2", "b2", "t")
                         SVAD_KSTEP(1) SVAD_MMA("a0", "b0", "t") SVAD_MMB("a1", "b1", "t") SVAD_MMB("a2", "b2", "t")
                         SVAD_KSTEP(2) SVAD_MMA("a0", "b0", "t") SVAD_MMB("a1", "b1", "t") SVAD_MMB("a2", "b2", "t")
                         SVAD_KSTEP(3) SVAD_MMA("a0", "b0", "t") SVAD_MMB("a1", "b1", "t") SVAD_MMB("a2", "b2", "t") "}\n"
                         ::"r"(d), "l"(a0), "l"(b0), "l"(a1), "l"(b1), "l"(a2), "l"(b2), "r"(idesc), "r"(accf), "r"(idesc12) : "memory");
        } else if constexpr (NP == 2) {
            asm volatile("{\n.reg .pred q, p, t;\n.reg .b64 a0, b0, a1, b1, a2, b2;\nelect.sync _|q, 0xffffffff;\nsetp.ne.b32 p, %8, 0;\nsetp.eq.u32 t, %8, %8;\n"
                         SVAD_KSTEP(0) SVAD_MMA("a0", "b0", "p") SVAD_MMB("a1", "b1", "t")
                         SVAD_KSTEP(1) SVAD_MMA("a0", "b0", "t") SVAD_MMB("a1", "b1", "t")
                         SVAD_KSTEP(2) SVAD_MMA("a0", "b0", "t") SVAD_MMB("a1", "b1", "t")
                         SVAD_KSTEP(3) SVAD_MMA("a0", "b0", "t") SVAD_MMB("a1", "b1", "t") "}\n"
                         ::"r"(d), "l"(a0), "l"(b0), "l"(a1), "l"(b1), "l"(a2), "l"(b2), "r"(idesc), "r"(accf), "r"(idesc12) : "memory");
        } else {
            asm volatile("{\n.reg .pred q, p, t;\n.reg .b64 a0, b0, a1, b1, a2, b2;\nelect.sync _|q, 0xffffffff;\nsetp.ne.b32 p, %8, 0;\nsetp.eq.u32 t, %8, %8;\n"
                         SVAD_KSTEP(0) SVAD_MMA("a0", "b0", "p")
                         SVAD_KSTEP(1) SVAD_MMA("a0", "b0", "t")
                         SVAD_KSTEP(2) SVAD_MMA("a0", "b0", "t")
                         SVAD_KSTEP(3) SVAD_MMA("a0", "b0", "t") "}\n"
                         ::"r"(d), "l"(a0), "l"(b0), "l"(a1), "l"(b1), "l"(a2), "l"(b2), "r"(idesc), "r"(accf), "r"(idesc12) : "memory");
        }
    }
#undef SVAD_MMA
#undef SVAD_MMB
#undef SVAD_KSTEP
    __device__ __forceinline__ void mma_slab_done(int it) {
        if (elect())
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(mdone + TapeTC<SR16>::buf(it))) : "memory");
    }
    __device__ __forceinline__ void slab_skip(int it) {   // an MMA warp that does not read this slab still releases it
        if (elect()) asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" ::"r"(smem_u32(mdone + TapeTC<SR16>::buf(it))) : "memory");
    }
    __device__ __forceinline__ void acc_commit() {
        if (elect())
            asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];" ::"r"(smem_u32(accb)) : "memory");
    }
    __device__ __forceinline__ void acc_wait() {
        mbar_wait(smem_u32(accb), acc_phase);
        acc_phase ^= 1u;
        tc_fence_after();
    }
    __device__ __forceinline__ void tmem_ld16(int lq, int col, float (&v)[16]) {
        uint32_t r[16];
        const uint32_t taddr = tmem + ((uint32_t)(lq * 32) << 16) + (uint32_t)col;
        asm volatile(
            "tcgen05.ld.sync.aligned.32x32b.x16.b32 {%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15}, [%16];"
            : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]), "=r"(r[8]), "=r"(r[9]),
              "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15])
            : "r"(taddr));
        asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory");
#pragma unroll
        for (int i = 0; i < 16; i++) v[i] = __uint_as_float(r[i]);
    }
};

constexpr size_t kSmemBytesTC = (size_t)SmemMapTC::total_floats * 4 + 256 + 80 * 16;   // + mbarriers, TMEM slot, slab table

template <bool SR16, int RM, typename S>
__global__ void __launch_bounds__(kThreads, 1) svad_fused_tc(TileArgs a, int ntiles) {
    extern __shared__ __align__(1024) unsigned char smem_raw[];
    float* sm = reinterpret_cast<float*>(smem_raw);
    uint64_t* bars = reinterpret_cast<uint64_t*>(smem_raw + (size_t)SmemMapTC::total_floats * 4);
    constexpr int NB = TapeTC<SR16>::kBufs;
    uint32_t* tmem_slot = reinterpret_cast<uint32_t*>(bars + 2 * NB + 2);
    int4* tab = reinterpret_cast<int4*>(smem_raw + (size_t)SmemMapTC::total_floats * 4 + 256);
    static_assert(TapeTC<SR16>::nslab <= 80, "slab table size");
    if ((int)threadIdx.x < TapeTC<SR16>::nslab) {
        using TP = TapeTC<SR16>;
        const int i = (int)threadIdx.x, b = TP::buf(i);
        tab[i] = make_int4(TP::dep_delta(i) | (b << 8), TP::slab_len(i) * 4, (int)smem_u32(sm + TP::template buf_off<SmemMapTC>(b)), TP::slab_off(i));
    }
    GpuEnvTC<SR16> env{sm, bars, bars + NB, bars + 2 * NB, a.tape, tab, (int)threadIdx.x, 0u, 0, 0, -2, 0u, 0u, 0u};
    int my_tiles = 0;
    for (int tile = blockIdx.x; tile < ntiles; tile += gridDim.x) my_tiles++;
    if (threadIdx.x == 0) {
        for (int s = 0; s < NB; s++) {
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bars + s)) : "memory");          // landed: TMA
            asm volatile("mbarrier.init.shared::cta.b64 [%0], 1;" ::"r"(smem_u32(bars + NB + s)) : "memory");     // consumed: the one MMA warp that reads it
        }
        asm volatile("mbarrier.init.shared::cta.b64 [%0], 4;" ::"r"(smem_u32(bars + 2 * NB)) : "memory");         // accumulators: 4 MMA warps
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
        asm volatile("fence.proxy.async.shared::cta;" ::: "memory");
    }
    __syncthreads();
    if ((threadIdx.x >> 5) == kRingWarp) {   // the ring warp primes every buffer whose first slab has no predecessor
        const int total = (int)((long)my_tiles * a.T * TapeTC<SR16>::nslab);
        env.ring_freed(total);   // freed: -2 -> -1
    }
    if (threadIdx.x < 32) {   // warp 0 owns the TMEM allocation
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;" ::"r"(smem_u32(tmem_slot)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory");
    env.tmem = *tmem_slot;
    run_cta_tc<SR16, RM, S>(env, a, (int)blockIdx.x, (int)gridDim.x, ntiles);
    asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory");
    __syncthreads();
    if (threadIdx.x < 32) asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" ::"r"(env.tmem), "r"(kTmemCols) : "memory");
}


// ------------------------------------------------------------------------------------------ small-batch cluster kernel
namespace cg = cooperative_groups;

// Mailbox of the persistent single-cluster variant (svad_stream_*): mapped pinned host memory.  The host writes chunk `q` into
// in[q % kMailRing] and publishes seq_in = q + 1; every CTA of the cluster polls seq_in, builds the window from the mailbox and its
// own copy of the carried context, and rank 0 answers with out[q % kMailRing] and seq_out = q + 1.  seq_in < 0 ends the kernel.
constexpr int kMailRing = 4;
struct SmallMail {
    volatile long long* seq_in;    // host -> device
    volatile long long* seq_out;   // device -> host
    volatile int* flags;           // [kMailRing] bit 0: reset state and context before this chunk
    const float* in;               // [kMailRing][kSmallNS][n]
    volatile float* out;           // [kMailRing][kSmallNS]
};

template <bool SR16, typename S, bool MB = false>
__global__ void __launch_bounds__(kSmallThreads, 1) svad_small_cluster(TileArgs a, const float* __restrict__ blobs, SmallMail mb = SmallMail{}) {
    using G = Geo<SR16>;
    using M = SmallMap<SR16>;
    extern __shared__ __align__(16) float sm[];
    cg::cluster_group cluster = cg::this_cluster();
    const int r = (int)cluster.block_rank();
    const int cid = (int)blockIdx.x / kSmallCtas;
    const int tid = (int)threadIdx.x, warp = tid >> 5, lane = tid & 31;
    const int g0 = cid * kSmallNS;
    const S* audio = static_cast<const S*>(a.audio);

    {   // this CTA's slice of every layer -> shared memory, resident for the whole launch
        const float4* src = reinterpret_cast<const float4*>(blobs + (size_t)r * M::blob_floats);
        float4* dst = reinterpret_cast<float4*>(sm);
        for (int i = tid; i < M::blob_floats / 4; i += kSmallThreads) dst[i] = __ldg(src + i);
    }
    float* peer[kSmallCtas];
#pragma unroll
    for (int q = 0; q < kSmallCtas; q++) peer[q] = cluster.map_shared_rank(sm, q);
    // h lives twice (ping-pong by step parity) so the gather of h' never races the peers still reading h
    float* hbuf[2] = {sm + M::a_xh + 128 * 4, sm + M::a_h2};
    for (int i = tid; i < 128 * 4; i += kSmallThreads) {
        const int j = i >> 2, st = i & 3, g = g0 + st;
        hbuf[0][i] = (a.state_in && g < a.B) ? a.state_in[(long)g * kHid + j] : 0.0f;
    }
    if (tid < 64) {
        const int u = tid >> 2, st = tid & 3, g = g0 + st;
        sm[M::a_c + tid] = (a.state_in && g < a.B) ? a.state_in[((long)a.B + g) * kHid + 16 * r + u] : 0.0f;
    }
    __syncthreads();
    cluster.sync();

    const float4* xp4 = reinterpret_cast<const float4*>(sm + M::a_xp);
    const float4* mag4 = reinterpret_cast<const float4*>(sm + M::a_mag);
    const float4* e04 = reinterpret_cast<const float4*>(sm + M::a_e0);
    const float4* e14 = reinterpret_cast<const float4*>(sm + M::a_e1);
    const float4* e24 = reinterpret_cast<const float4*>(sm + M::a_e2);
    const float4* e34 = reinterpret_cast<const float4*>(sm + M::a_xh);
    float4* red = reinterpret_cast<float4*>(sm + M::a_red);
    // all-gather one float4 (4 streams of one channel) into the same offset of all 8 CTAs
    auto gather = [&](int off_floats, float4 v) {
#pragma unroll
        for (int q = 0; q < kSmallCtas; q++) *reinterpret_cast<float4*>(peer[q] + off_floats) = v;
    };
    auto relu4b = [](float4 v, float b) { return make_float4(fmaxf(v.x + b, 0.f), fmaxf(v.y + b, 0.f), fmaxf(v.z + b, 0.f), fmaxf(v.w + b, 0.f)); };
    const float4 zero4 = make_float4(0.f, 0.f, 0.f, 0.f);

#define SM_STAMP(k) do { if (a.dbg && blockIdx.x == 0 && t == 2 && tid == 0) a.dbg[k] = clock64(); } while (0)
    float* ctxbuf = sm + M::total_floats;   // mailbox mode: carried context [ctx][4]
    __shared__ int s_cmd;
    if (MB) {
        for (int i = tid; i < G::ctx * 4; i += kSmallThreads) ctxbuf[i] = 0.0f;
        for (int i = tid; i < (G::L1 + G::N / 4) * 4; i += kSmallThreads) sm[M::a_xp + i] = 0.0f;   // slots of absent streams stay zero
        __syncthreads();
        cluster.sync();
    }
    for (long t = 0; MB || t < a.T; t++) {
        const int cur = (int)(t & 1);
        SM_STAMP(0);
        if constexpr (MB) {
            // Rank 0 waits for chunk t -- ONE mailbox word carries the sequence number and the reset bit, a PCIe read per poll paces
            // the loop, ~30 s without a chunk ends the kernel -- fetches the samples with coalesced 16-byte reads (a few dozen PCIe
            // transactions instead of thousands of 4-byte ones) and writes them, with the command, into all 8 CTAs through
            // distributed shared memory: the cluster takes every decision together.
            if (r == 0) {
                if (tid == 0) {
                    int cmd = -1;
                    for (long spin = 0; spin < (1L << 24); spin++) {
                        const long long v = *mb.seq_in;
                        if (v < 0) break;
                        if ((v >> 1) > t) { cmd = (int)(v & 1); break; }
                    }
                    s_cmd = cmd;
                }
                __syncthreads();
                const int cmd0 = s_cmd;
                if (cmd0 >= 0) {
                    const float4* chunk4 = reinterpret_cast<const float4*>(mb.in + (size_t)(t % kMailRing) * kSmallNS * G::n);
                    for (int idx = tid; idx < a.B * (G::n / 4); idx += kSmallThreads) {
                        const int st = idx / (G::n / 4), kk = (idx % (G::n / 4)) * 4;
                        const float4 v = __ldcv(chunk4 + st * (G::n / 4) + kk / 4);
                        const int off = M::a_xp + (G::ctx + kk) * 4 + st;
#pragma unroll
                        for (int q = 0; q < kSmallCtas; q++) {
                            float* d = peer[q] + off;
                            d[0] = v.x; d[4] = v.y; d[8] = v.z; d[12] = v.w;
                        }
                    }
                }
                if (tid == 0) {
#pragma unroll
                    for (int q = 1; q < kSmallCtas; q++) *cluster.map_shared_rank(&s_cmd, q) = cmd0;
                }
            }
            cluster.sync();
            const int cmd = s_cmd;
            if (cmd < 0) break;
            if (cmd & 1) {        // new call on this line: zero (h, c) and the context
                for (int i = tid; i < G::ctx * 4; i += kSmallThreads) ctxbuf[i] = 0.0f;
                for (int i = tid; i < 128 * 4; i += kSmallThreads) hbuf[cur][i] = 0.0f;
                if (tid < 64) sm[M::a_c + tid] = 0.0f;
                __syncthreads();
            }
            // context rows from the carried copy, reflect rows xp[L1 + j] = xp[L1 - 2 - j] from the chunk rows just delivered
            for (int i = tid; i < G::ctx * 4; i += kSmallThreads) sm[M::a_xp + i] = ctxbuf[i];
            for (int i = tid; i < (G::N / 4) * 4; i += kSmallThreads) {
                const int j = i >> 2, st = i & 3;
                sm[M::a_xp + (G::L1 + j) * 4 + st] = sm[M::a_xp + (G::L1 - 2 - j) * 4 + st];
            }
            __syncthreads();
            for (int i = tid; i < G::ctx * 4; i += kSmallThreads) ctxbuf[i] = sm[M::a_xp + (G::L1 - G::ctx) * 4 + i];
        } else {
        // 1. padded window [context | chunk | reflect] of the 4 streams
        for (int i = tid; i < (G::L1 + G::N / 4) * 4; i += kSmallThreads) {
            const int k = i >> 2, st = i & 3, g = g0 + st;
            float v = 0.0f;
            if (g < a.B) v = window_sample<SR16, S>(audio + (long)g * a.ld, a.L, a.ctx_in ? a.ctx_in + (long)g * a.ctx_ld : nullptr, t, k, a.dec);
            sm[M::a_xp + i] = v;
        }
        }
        __syncthreads();
        SM_STAMP(1);
        // 2. STFT slice: thread = (basis row, frame), full K = N
        if (tid < M::RB * 4) {
            const int row = tid % M::RB, f = tid / M::RB;
            float4 acc = zero4;
            dotT(sm + M::w_basis, M::RB, row, xp4 + f * G::hop, 0, G::N, acc);
            red[tid] = acc;
        }
        __syncthreads();
        if (tid < M::BPC * 4) {
            const int lb = tid % M::BPC, f = tid / M::BPC, bin = r * M::BPC + lb;
            if (bin < G::F) {
                const float4 re = red[f * M::RB + 2 * lb], im = red[f * M::RB + 2 * lb + 1];
                gather(M::a_mag + (f * G::F + bin) * 4, make_float4(sqrtf(re.x * re.x + im.x * im.x), sqrtf(re.y * re.y + im.y * im.y),
                                                                    sqrtf(re.z * re.z + im.z * im.z), sqrtf(re.w * re.w + im.w * im.w)));
            }
        }
        SM_STAMP(2);
        cluster.sync();
        SM_STAMP(3);
        // 3. enc0 slice: thread = (channel o, out frame tt, k-part kp of 4); live taps only
        {
            const int o = tid & 15, tt = (tid >> 4) & 3, kp = tid >> 6;
            constexpr int Cc = (G::F + 3) / 4;
            const int c0 = kp * Cc, c1 = (c0 + Cc < G::F) ? c0 + Cc : G::F;
            float4 acc = zero4;
#pragma unroll
            for (int j = 0; j < 3; j++) {
                const int f = tt + j - 1;
                if (f < 0 || f > 3) continue;
                dotT(sm + M::w_e0 + j * G::F * 16, 16, o, mag4 + f * G::F, c0, c1, acc);
            }
            red[tid] = acc;
        }
        __syncthreads();
        if (tid < 64) {
            const int o = tid & 15, tt = tid >> 4;
            const float4 v = add4(add4(red[tid], red[tid + 64]), add4(red[tid + 128], red[tid + 192]));
            gather(M::a_e0 + (tt * 128 + 16 * r + o) * 4, relu4b(v, sm[M::w_b0 + o]));
        }
        SM_STAMP(4);
        cluster.sync();
        SM_STAMP(5);
        // 4. enc1 slice (stride 2): thread = (o 8, tt 2, kp 16): out frame tt reads frames 2 tt + j - 1, 8 channels per part
        {
            const int o = tid & 7, tt = (tid >> 3) & 1, kp = tid >> 4;
            float4 acc = zero4;
#pragma unroll
            for (int j = 0; j < 3; j++) {
                const int f = 2 * tt + j - 1;
                if (f < 0) continue;
                dotT(sm + M::w_e1 + j * 128 * 8, 8, o, e04 + f * 128, kp * 8, kp * 8 + 8, acc);
            }
            red[tid] = acc;
        }
        __syncthreads();
        if (tid < 16) {
            float4 v = zero4;
#pragma unroll
            for (int kp = 0; kp < 16; kp++) v = add4(v, red[tid + 16 * kp]);
            gather(M::a_e1 + ((tid >> 3) * 64 + 8 * r + (tid & 7)) * 4, relu4b(v, sm[M::w_b1 + (tid & 7)]));
        }
        cluster.sync();
        // 5. enc2 slice (taps 1, 2 live): thread = (o 8, kp 32): K = 2 x 64 in parts of 4
        {
            const int o = tid & 7, kp = tid >> 3;
            float4 acc = zero4;
            dotT(sm + M::w_e2, 8, o, e14, kp * 4, kp * 4 + 4, acc);   // rows k = jj*64 + c line up with e1[jj][c]
            red[tid] = acc;
        }
        __syncthreads();
        if (tid < 8) {
            float4 v = zero4;
#pragma unroll
            for (int kp = 0; kp < 32; kp++) v = add4(v, red[tid + 8 * kp]);
            gather(M::a_e2 + (8 * r + tid) * 4, relu4b(v, sm[M::w_b2 + tid]));
        }
        cluster.sync();
        // 6. enc3 slice (tap 1 live) -> first half of the LSTM input: thread = (o 16, kp 16)
        {
            const int o = tid & 15, kp = tid >> 4;
            float4 acc = zero4;
            dotT(sm + M::w_e3, 16, o, e24, kp * 4, kp * 4 + 4, acc);
            red[tid] = acc;
        }
        __syncthreads();
        if (tid < 16) {
            float4 v = zero4;
#pragma unroll
            for (int kp = 0; kp < 16; kp++) v = add4(v, red[tid + 16 * kp]);
            gather(M::a_xh + (16 * r + tid) * 4, relu4b(v, sm[M::w_b3 + tid]));
        }
        cluster.sync();
        SM_STAMP(6);
        // 7. LSTM: this CTA's 16 hidden units x 4 gates: thread = (row 64, kp 4), K = [e3 ; h]
        {
            const int row = tid & 63, kp = tid >> 6;
            float4 acc = zero4;
            if (kp < 2) dotT(sm + M::w_l, 64, row, e34, kp * 64, kp * 64 + 64, acc);
            else dotT(sm + M::w_l + 128 * 64, 64, row, reinterpret_cast<const float4*>(hbuf[cur]), (kp - 2) * 64, (kp - 2) * 64 + 64, acc);
            red[tid] = acc;
        }
        __syncthreads();
        if (tid < 64) {
            const float b = sm[M::w_bl + tid];
            const float4 v = add4(add4(red[tid], red[tid + 64]), add4(red[tid + 128], red[tid + 192]));
            *reinterpret_cast<float4*>(sm + M::a_gates + tid * 4) = make_float4(v.x + b, v.y + b, v.z + b, v.w + b);
        }
        __syncthreads();
        if (tid < 64) {
            const int u = tid >> 2, st = tid & 3;
            const float* gt = sm + M::a_gates + (u * 4) * 4 + st;
            const float ig = sigmoid_acc(gt[0]), fg = sigmoid_acc(gt[4]), gg = tanhf(gt[8]), og = sigmoid_acc(gt[12]);
            const float cn = fmaf(fg, sm[M::a_c + tid], ig * gg);
            sm[M::a_c + tid] = cn;
            const float hn = og * tanhf(cn);
            const int off = (int)(hbuf[cur ^ 1] - sm) + (16 * r + u) * 4 + st;
#pragma unroll
            for (int q = 0; q < kSmallCtas; q++) peer[q][off] = hn;
        }
        SM_STAMP(7);
        cluster.sync();
        SM_STAMP(8);
        // 8. head (rank 0): 128 threads = (hidden unit j), then a 4-stream reduction through shared memory
        if (r == 0) {
            if (tid < 128) {
                const float4 hv = reinterpret_cast<const float4*>(hbuf[cur ^ 1])[tid];
                const float wv = sm[M::w_out + tid];
                red[tid] = make_float4(wv * fmaxf(hv.x, 0.f), wv * fmaxf(hv.y, 0.f), wv * fmaxf(hv.z, 0.f), wv * fmaxf(hv.w, 0.f));
            }
            __syncthreads();
            if (tid < 32) {
                float4 v = add4(add4(red[tid], red[tid + 32]), add4(red[tid + 64], red[tid + 96]));
#pragma unroll
                for (int o2 = 16; o2 > 0; o2 >>= 1) {
                    v.x += __shfl_xor_sync(0xffffffffu, v.x, o2); v.y += __shfl_xor_sync(0xffffffffu, v.y, o2);
                    v.z += __shfl_xor_sync(0xffffffffu, v.z, o2); v.w += __shfl_xor_sync(0xffffffffu, v.w, o2);
                }
                const float b = sm[M::w_out + 128];
                if (tid < kSmallNS && g0 + tid < a.B) {
                    const float x = tid == 0 ? v.x : (tid == 1 ? v.y : (tid == 2 ? v.z : v.w));
                    if constexpr (MB) mb.out[(t % kMailRing) * kSmallNS + tid] = sigmoid_acc(x + b);
                    else a.probs[(long)(g0 + tid) * a.ldp + t] = sigmoid_acc(x + b);
                }
                if constexpr (MB) {   // publish: probabilities first, then the sequence number the host spins on
                    __threadfence_system();
                    __syncwarp();
                    if (tid == 0) *mb.seq_out = t + 1;
                }
            }
        }
        SM_STAMP(9);
    }
#undef SM_STAMP
    // carry state / context out
    const int fin = (int)(a.T & 1);
    if (a.state_out) {
        if (r == 0)
            for (int i = tid; i < 128 * 4; i += kSmallThreads) {
                const int j = i >> 2, st = i & 3, g = g0 + st;
                if (g < a.B) a.state_out[(long)g * kHid + j] = hbuf[fin][i];
            }
        if (tid < 64) {
            const int u = tid >> 2, st = tid & 3, g = g0 + st;
            if (g < a.B) a.state_out[((long)a.B + g) * kHid + 16 * r + u] = sm[M::a_c + tid];
        }
    }
    if (a.ctx_out && r == 0) {
        for (int i = tid; i < kSmallNS * G::ctx; i += kSmallThreads) {
            const int st = i / G::ctx, k = i % G::ctx, g = g0 + st;
            if (g < a.B) {
                const float* cx = a.ctx_in ? a.ctx_in + (long)g * a.ctx_ld : nullptr;
                a.ctx_out[(long)g * G::ctx + k] = (a.T > 0) ? window_sample<SR16, S>(audio + (long)g * a.ld, a.L, cx, a.T - 1, G::n + k, a.dec) : (cx ? cx[k] : 0.0f);
            }
        }
    }
    cluster.sync();   // nobody exits while a peer may still address its shared memory
}

}  // namespace

// ------------------------------------------------------------------------------------------ host
static thread_local std::string g_err;
static int fail(int code, const char* fmt, ...) {
    char buf[512];
    va_list ap;
    va_start(ap, fmt);
    vsnprintf(buf, sizeof buf, fmt, ap);
    va_end(ap);
    g_err = buf;
    return code;
}
#define CUDA_TRY(x)                                                                               \
    do {                                                                                          \
        cudaError_t err__ = (x);                                                                  \
        if (err__ != cudaSuccess) return fail(SVAD_ECUDA, "%s: %s", #x, cudaGetErrorString(err__)); \
    } while (0)

struct svad_engine {
    int device = 0, sms = 0, tile_rows = 0;
    float* d_tape[2] = {nullptr, nullptr};    // 0: 16 kHz, 1: 8 kHz   (fp32 CUDA-core kernel)
    float* d_consts[2] = {nullptr, nullptr};
    float* d_tape_tc[2] = {nullptr, nullptr};  // tensor-core kernel
    float* d_consts_tc[2] = {nullptr, nullptr};
    unsigned char* d_h16_f[2] = {nullptr, nullptr};   // fp16 split kernel: front / back weight tapes, constants
    unsigned char* d_h16_b[2] = {nullptr, nullptr};
    float* d_h16_c[2] = {nullptr, nullptr};
    float* d_small[2] = {nullptr, nullptr};    // small-batch cluster kernel: 8 per-CTA weight slices
    int small_max = 256;                       // streams up to which the cluster kernel is used (0 = never); crossover with the tile kernels measured at ~256
    int h16_pair = getenv("SVAD_H16_PAIR") ? atoi(getenv("SVAD_H16_PAIR")) : 1;   // svad_fused_h16 in CTA pairs sharing the weight streams
    int kernel = 2;                            // 0 = fp32 CUDA cores, 1 = tcgen05 split-TF32, 2 = tcgen05 split-fp16 two-loop kernel (default)
    long long* dbg = nullptr;
    int64_t launches = 0;
    // staging for the host-buffer entry points
    void *h_pin = nullptr, *d_buf = nullptr;
    size_t pin_bytes = 0, dbuf_bytes = 0;
    cudaStream_t stream = nullptr, stream_copy = nullptr;
    cudaEvent_t ev[8] = {};
};
constexpr int kMaxSlices = 8;

extern "C" int svad_abi_version(void) { return 1; }
extern "C" const char* svad_last_error(void) { return g_err.c_str(); }

static int engine_upload(svad_engine* e, int device, int sms, const TensorMap& tm, PackedBranch* pb, PackedBranch* pbt);
static int engine_create_impl(const char* weights_path, int device, svad_engine** out);

extern "C" int svad_engine_create(const char* weights_path, int device, svad_engine** out) {
    try {
        return engine_create_impl(weights_path, device, out);
    } catch (const std::bad_alloc&) {
        return fail(SVAD_ENOMEM, "out of memory while loading %s", weights_path ? weights_path : "(null)");
    } catch (const std::exception& ex) {
        return fail(SVAD_EWEIGHTS, "%s", ex.what());
    }
}

static int engine_create_impl(const char* weights_path, int device, svad_engine** out) {
    if (!weights_path || !out) return fail(SVAD_EINVAL, "null argument");
    *out = nullptr;
    TensorMap tm;
    std::string err;
    if (!read_container(weights_path, tm, err)) return fail(SVAD_EWEIGHTS, "%s", err.c_str());
    PackedBranch pb[2], pbt[2];
    if (!pack_branch<true>(tm, pb[0], err) || !pack_branch<false>(tm, pb[1], err)) return fail(SVAD_EWEIGHTS, "%s", err.c_str());
    if (!pack_branch_tc<true>(tm, pbt[0], err) || !pack_branch_tc<false>(tm, pbt[1], err)) return fail(SVAD_EWEIGHTS, "%s", err.c_str());
    int ndev = 0;
    if (cudaGetDeviceCount(&ndev) != cudaSuccess || ndev == 0)
        return fail(SVAD_ECUDA, "no CUDA device: silero_vad_b200 has no CPU fallback");
    if (device < 0 || device >= ndev) return fail(SVAD_EINVAL, "device %d out of range (%d devices)", device, ndev);
    CUDA_TRY(cudaSetDevice(device));
    cudaDeviceProp prop;
    CUDA_TRY(cudaGetDeviceProperties(&prop, device));
    if ((size_t)prop.sharedMemPerBlockOptin < kSmemBytes)
        return fail(SVAD_ECUDA, "device offers %zu B shared memory per block, kernel needs %zu", (size_t)prop.sharedMemPerBlockOptin, kSmemBytes);
    svad_engine* e = new (std::nothrow) svad_engine();
    if (!e) return fail(SVAD_ENOMEM, "out of memory");
    const int rc = engine_upload(e, device, prop.multiProcessorCount, tm, pb, pbt);
    if (rc != SVAD_OK) { svad_engine_destroy(e); return rc; }   // every partially created resource is released
    *out = e;
    return SVAD_OK;
}

static int engine_upload(svad_engine* e, int device, int sms, const TensorMap& tm, PackedBranch* pb, PackedBranch* pbt) {
    e->device = device;
    e->sms = sms;
    for (int b = 0; b < 2; b++) {
        CUDA_TRY(cudaMalloc(&e->d_tape[b], pb[b].tape.size() * 4));
        CUDA_TRY(cudaMalloc(&e->d_consts[b], pb[b].consts.size() * 4));
        CUDA_TRY(cudaMemcpy(e->d_tape[b], pb[b].tape.data(), pb[b].tape.size() * 4, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(e->d_consts[b], pb[b].consts.data(), pb[b].consts.size() * 4, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMalloc(&e->d_tape_tc[b], pbt[b].tape.size() * 4));
        CUDA_TRY(cudaMalloc(&e->d_consts_tc[b], pbt[b].consts.size() * 4));
        CUDA_TRY(cudaMemcpy(e->d_tape_tc[b], pbt[b].tape.data(), pbt[b].tape.size() * 4, cudaMemcpyHostToDevice));
        CUDA_TRY(cudaMemcpy(e->d_consts_tc[b], pbt[b].consts.data(), pbt[b].consts.size() * 4, cudaMemcpyHostToDevice));
        {
            PackedH16 ph;
            std::string err;
            if (!(b == 0 ? pack_branch_h16<true>(tm, ph, err) : pack_branch_h16<false>(tm, ph, err))) return fail(SVAD_EWEIGHTS, "%s", err.c_str());
            CUDA_TRY(cudaMalloc(&e->d_h16_f[b], ph.tapeF.size()));
            CUDA_TRY(cudaMalloc(&e->d_h16_b[b], ph.tapeB.size()));
            CUDA_TRY(cudaMalloc(&e->d_h16_c[b], ph.consts.size() * 4));
            CUDA_TRY(cudaMemcpy(e->d_h16_f[b], ph.tapeF.data(), ph.tapeF.size(), cudaMemcpyHostToDevice));
            CUDA_TRY(cudaMemcpy(e->d_h16_b[b], ph.tapeB.data(), ph.tapeB.size(), cudaMemcpyHostToDevice));
            CUDA_TRY(cudaMemcpy(e->d_h16_c[b], ph.consts.data(), ph.consts.size() * 4, cudaMemcpyHostToDevice));
        }
        std::vector<float> blobs;
        if (b == 0) pack_small<true>(tm, blobs); else pack_small<false>(tm, blobs);
        CUDA_TRY(cudaMalloc(&e->d_small[b], blobs.size() * 4));
        CUDA_TRY(cudaMemcpy(e->d_small[b], blobs.data(), blobs.size() * 4, cudaMemcpyHostToDevice));
    }
    CUDA_TRY(cudaStreamCreateWithFlags(&e->stream, cudaStreamNonBlocking));
    CUDA_TRY(cudaStreamCreateWithFlags(&e->stream_copy, cudaStreamNonBlocking));
    for (int i = 0; i < kMaxSlices; i++) CUDA_TRY(cudaEventCreateWithFlags(&e->ev[i], cudaEventDisableTiming));
    return SVAD_OK;
}

extern "C" void svad_engine_destroy(svad_engine* e) {
    if (!e) return;
    cudaSetDevice(e->device);
    for (int b = 0; b < 2; b++) { cudaFree(e->d_tape[b]); cudaFree(e->d_consts[b]); cudaFree(e->d_tape_tc[b]); cudaFree(e->d_consts_tc[b]); cudaFree(e->d_small[b]);
                                  cudaFree(e->d_h16_f[b]); cudaFree(e->d_h16_b[b]); cudaFree(e->d_h16_c[b]); }
    if (e->h_pin) cudaFreeHost(e->h_pin);
    if (e->d_buf) cudaFree(e->d_buf);
    if (e->stream) cudaStreamDestroy(e->stream);
    if (e->stream_copy) cudaStreamDestroy(e->stream_copy);
    for (int i = 0; i < kMaxSlices; i++) if (e->ev[i]) cudaEventDestroy(e->ev[i]);
    delete e;
}

extern "C" int svad_engine_set_tile_rows(svad_engine* e, int rows) {
    if (!e || !(rows == 0 || (rows >= 4 && rows <= 8))) return fail(SVAD_EINVAL, "tile rows must be 0 or 4..8");
    e->tile_rows = rows;
    return SVAD_OK;
}
extern "C" int svad_engine_set_kernel(svad_engine* e, int kernel) {
    if (!e || kernel < 0 || kernel > 2) return fail(SVAD_EINVAL, "kernel must be 0 (fp32 CUDA cores), 1 (tcgen05 split-TF32) or 2 (tcgen05 split-fp16, two-loop)");
    e->kernel = kernel;
    return SVAD_OK;
}
// profiling hook (not part of the public header): device buffer of 16 int64 clock stamps written by CTA 0
extern "C" int svad_engine_set_debug_buffer(svad_engine* e, long long* d_buf) {
    if (!e) return SVAD_EINVAL;
    e->dbg = d_buf;
    return SVAD_OK;
}
extern "C" int svad_engine_set_pair_mode(svad_engine* e, int on) {
    if (!e) return fail(SVAD_EINVAL, "null engine");
    e->h16_pair = on ? 1 : 0;
    return SVAD_OK;
}

extern "C" int svad_engine_set_small_batch_max(svad_engine* e, int streams) {
    if (!e || streams < 0) return fail(SVAD_EINVAL, "small-batch limit must be >= 0");
    e->small_max = streams;
    return SVAD_OK;
}
extern "C" int svad_engine_sm_count(const svad_engine* e) { return e ? e->sms : 0; }
extern "C" int64_t svad_engine_launch_count(const svad_engine* e) { return e ? e->launches : 0; }

template <bool SR16, int RM, typename S, bool FEAT = false>
static int launch(svad_engine* e, const TileArgs& a, cudaStream_t st) {
    auto kern = svad_fused_fp32<SR16, RM, S, FEAT>;
    static bool configured[16] = {};  // per device
    if (!configured[e->device & 15]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytes));
        configured[e->device & 15] = true;
    }
    const int ntiles = (a.B + 4 * RM - 1) / (4 * RM);
    const int grid = ntiles < e->sms ? ntiles : e->sms;
    kern<<<grid, kThreads, kSmemBytes, st>>>(a, ntiles);
    CUDA_TRY(cudaGetLastError());
    e->launches++;
    return SVAD_OK;
}

template <bool SR16, int RM, typename S>
static int launch_tc(svad_engine* e, const TileArgs& a, cudaStream_t st) {
    auto kern = svad_fused_tc<SR16, RM, S>;
    static bool configured[16] = {};
    if (!configured[e->device & 15]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)kSmemBytesTC));
        configured[e->device & 15] = true;
    }
    const int ntiles = (a.B + 4 * RM - 1) / (4 * RM);
    const int grid = ntiles < e->sms ? ntiles : e->sms;
    kern<<<grid, kThreads, kSmemBytesTC, st>>>(a, ntiles);
    CUDA_TRY(cudaGetLastError());
    e->launches++;
    return SVAD_OK;
}

template <bool SR16, typename S>
static int launch_small(svad_engine* e, const TileArgs& a, cudaStream_t st) {
    auto kern = svad_small_cluster<SR16, S>;
    const size_t smem = (size_t)SmallMap<SR16>::total_floats * 4;
    static bool configured[16] = {};
    if (!configured[e->device & 15]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured[e->device & 15] = true;
    }
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3((unsigned)((a.B + kSmallNS - 1) / kSmallNS * kSmallCtas));
    cfg.blockDim = dim3(kSmallThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = kSmallCtas; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, a, (const float*)e->d_small[SR16 ? 0 : 1], SmallMail{}));
    e->launches++;
    return SVAD_OK;
}

// fp16 split kernel: streams per tile chosen so that the tiles fill whole waves of SMs (B = 4096 on 148 SMs: 147 tiles of 28).
// Streams per tile of svad_fused_h16.  A CTA's step costs the same for 1 or 32 streams (the MMAs run at N = 32 per frame and the epilogue
// threads cover 32 slots either way), so tiles are always full: B = 4096 takes 128 CTAs, not 148 -- measured the same kernel time
// (1.183 vs 1.172 ms), 13 % fewer weight streams out of L2, and 20 SMs left for whatever else the device runs (the asynchronous
// all-gather of a multi-GPU job, copies).  `grid` = CTAs that walk `waves` tiles each (even for CTA pairs).
static int pick_bt(const svad_engine* e, int B) {
    if (e->tile_rows) return 4 * e->tile_rows;
    return B < 32 ? (B < 1 ? 1 : B) : 32;
}
static void pick_grid(int ntiles, int sms, bool pairs, int* grid, int* ntiles_eff) {
    const int waves = (ntiles + sms - 1) / sms;
    int g = (ntiles + waves - 1) / waves;
    if (pairs) g = ((g + 1) / 2) * 2;
    if (g > sms) g = sms;
    *grid = g;
    *ntiles_eff = pairs ? ((ntiles + g - 1) / g) * g : ntiles;   // a pair walks the same number of tiles (surplus ones lie past the batch)
}

template <bool SR16, typename S>
static int launch_h16(svad_engine* e, const TileArgs& a, cudaStream_t st) {
    auto kern = svad_fused_h16<SR16, S>;
    static bool configured[16] = {};
    if (!configured[e->device & 15]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)H16Map::total));
        configured[e->device & 15] = true;
    }
    const int br = SR16 ? 0 : 1;
    if (e->h16_pair && a.B >= 64) {
        // CTA pairs (clusters of 2) share the weight streams: each CTA fetches half of every slab and multicasts it to both, which halves
        // the bytes read out of L2.  Both CTAs of a pair must walk the same number of tiles, so every CTA gets ceil(ntiles / grid) of
        // them; the surplus ones lie past the batch (every load and store of such a tile is masked).
        auto kp = svad_fused_h16<SR16, S, true>;
        static bool configured_p[16] = {};
        static int pairs[16] = {};
        cudaLaunchConfig_t cfg{};
        cfg.blockDim = dim3(kH16Threads); cfg.dynamicSmemBytes = H16Map::total; cfg.stream = st;
        cudaLaunchAttribute attr[1];
        attr[0].id = cudaLaunchAttributeClusterDimension;
        attr[0].val.clusterDim.x = 2; attr[0].val.clusterDim.y = 1; attr[0].val.clusterDim.z = 1;
        cfg.attrs = attr; cfg.numAttrs = 1;
        if (!configured_p[e->device & 15]) {
            CUDA_TRY(cudaFuncSetAttribute(kp, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)H16Map::total));
            cfg.gridDim = dim3(2 * (e->sms / 2));
            int n = 0;
            if (cudaOccupancyMaxActiveClusters(&n, kp, &cfg) != cudaSuccess) { (void)cudaGetLastError(); n = 0; }   // no pairs: single CTAs below
            pairs[e->device & 15] = n;
            configured_p[e->device & 15] = true;
            if (getenv("SVAD_VERBOSE")) fprintf(stderr, "svad: h16 pair mode: %d co-resident CTA pairs on %d SMs\n", n, e->sms);
        }
        const int np = pairs[e->device & 15];
        if (np >= 1) {
            const int bt = pick_bt(e, a.B);
            const int ntiles = (a.B + bt - 1) / bt;
            int grid, ntiles_eff;
            pick_grid(ntiles, 2 * np, true, &grid, &ntiles_eff);
            cfg.gridDim = dim3(grid);
            if (cudaLaunchKernelEx(&cfg, kp, a, (const unsigned char*)e->d_h16_f[br], (const unsigned char*)e->d_h16_b[br], ntiles_eff, bt) == cudaSuccess) {
                e->launches++;
                return SVAD_OK;
            }
            (void)cudaGetLastError();   // the cluster launch was refused (e.g. a partitioned device): single CTAs from now on
            e->h16_pair = 0;
        }
    }
    const int bt = pick_bt(e, a.B);
    const int ntiles = (a.B + bt - 1) / bt;
    int grid, ntiles_eff;
    pick_grid(ntiles, e->sms, false, &grid, &ntiles_eff);
    kern<<<grid, kH16Threads, H16Map::total, st>>>(a, e->d_h16_f[br], e->d_h16_b[br], ntiles, bt);
    CUDA_TRY(cudaGetLastError());
    e->launches++;
    return SVAD_OK;
}

// rows per thread that minimises (waves x rows): the FFMA work of a CTA step is proportional to RM.
static int pick_rows(const svad_engine* e, int B) {
    if (e->tile_rows) return e->tile_rows;
    int best = 8;
    long best_cost = -1;
    for (int rm = 8; rm >= 4; rm--) {
        const long tiles = (B + 4 * rm - 1) / (4 * rm);
        const long waves = (tiles + e->sms - 1) / e->sms;
        const long cost = waves * rm;
        if (best_cost < 0 || cost < best_cost) { best_cost = cost; best = rm; }
    }
    return best;
}

template <bool SR16, typename S>
static int launch_rm(svad_engine* e, const TileArgs& a, cudaStream_t st) {
    if (a.B <= e->small_max) return launch_small<SR16, S>(e, a, st);
    if (e->kernel == 2) return launch_h16<SR16, S>(e, a, st);
    if (e->kernel == 1) {   // tensor-core kernel: MMA cost does not depend on the tile rows; only 7 and 8 are built
        if (a.T > 4000000) return fail(SVAD_EINVAL, "tensor-core kernel: at most 4e6 chunks per call (feed long streams in pieces)");
        const int rm = e->tile_rows ? e->tile_rows : pick_rows(e, a.B);
        return rm >= 8 ? launch_tc<SR16, 8, S>(e, a, st) : launch_tc<SR16, 7, S>(e, a, st);
    }
    switch (pick_rows(e, a.B)) {
        case 4: return launch<SR16, 4, S>(e, a, st);
        case 5: return launch<SR16, 5, S>(e, a, st);
        case 6: return launch<SR16, 6, S>(e, a, st);
        case 7: return launch<SR16, 7, S>(e, a, st);
        default: return launch<SR16, 8, S>(e, a, st);
    }
}

enum SampleFmt { kF32 = 0, kI16 = 1 };
static size_t fmt_size(int fmt) { return fmt == kI16 ? 2 : 4; }

// `Lraw` stored samples per row, of which every `dec`-th is read: the model sees L = ceil(Lraw / dec) samples (x[:, ::dec]).
static int forward_impl(svad_engine* e, int sr, int B, int64_t Lraw, int64_t ld, const void* d_audio, int fmt, const float* d_state_in,
                        const float* d_ctx_in, int64_t ctx_ld, float* d_state_out, float* d_ctx_out, float* d_probs,
                        int64_t ldp, cudaStream_t st, int dec = 1) {
    if (!e) return fail(SVAD_EINVAL, "null engine");
    if (sr != 16000 && sr != 8000) return fail(SVAD_EINVAL, "Supported sampling rates: [8000, 16000] (got %d)", sr);
    if (B < 0 || Lraw < 0 || dec < 1) return fail(SVAD_EINVAL, "negative size");
    const int64_t L = (Lraw + dec - 1) / dec;
    const int n = sr == 16000 ? 512 : 256;
    const int64_t T = (L + n - 1) / n;
    if (B == 0 || (T == 0 && !d_state_out && !d_ctx_out)) return SVAD_OK;
    if ((T > 0 && (!d_audio || !d_probs)) || ld < Lraw || ldp < T) return fail(SVAD_EINVAL, "bad audio/probs pointer or stride");
    CUDA_TRY(cudaSetDevice(e->device));
    const int br = sr == 16000 ? 0 : 1;
    TileArgs a{};
    a.audio = d_audio; a.ld = ld; a.L = L; a.dec = dec; a.B = B; a.T = T;
    a.state_in = d_state_in; a.ctx_in = d_ctx_in; a.ctx_ld = ctx_ld;
    a.state_out = d_state_out; a.ctx_out = d_ctx_out;
    a.probs = d_probs; a.ldp = ldp; a.dbg = e->dbg;
    a.tape = e->kernel == 1 ? e->d_tape_tc[br] : e->d_tape[br];
    a.consts = e->kernel == 2 && B > e->small_max ? e->d_h16_c[br] : (e->kernel == 1 ? e->d_consts_tc[br] : e->d_consts[br]);
    if (fmt == kI16) return sr == 16000 ? launch_rm<true, int16_t>(e, a, st) : launch_rm<false, int16_t>(e, a, st);
    return sr == 16000 ? launch_rm<true, float>(e, a, st) : launch_rm<false, float>(e, a, st);
}

extern "C" int svad_forward_device(svad_engine* e, int sr, int B, int64_t L, int64_t ld, const float* d_audio,
                                   const float* d_state_in, const float* d_ctx_in, float* d_state_out, float* d_ctx_out,
                                   float* d_probs, int64_t ldp, void* stream) {
    return forward_impl(e, sr, B, L, ld, d_audio, kF32, d_state_in, d_ctx_in, sr == 16000 ? 64 : 32, d_state_out, d_ctx_out,
                        d_probs, ldp, (cudaStream_t)stream);
}

extern "C" int svad_forward_device_pcm16(svad_engine* e, int sr, int B, int64_t L, int64_t ld, const int16_t* d_audio,
                                         const float* d_state_in, const float* d_ctx_in, float* d_state_out, float* d_ctx_out,
                                         float* d_probs, int64_t ldp, void* stream) {
    return forward_impl(e, sr, B, L, ld, d_audio, kI16, d_state_in, d_ctx_in, sr == 16000 ? 64 : 32, d_state_out, d_ctx_out,
                        d_probs, ldp, (cudaStream_t)stream);
}

// sample_format: 0 = f32, 1 = int16 PCM; sample_stride k >= 1 reads every k-th stored sample (sr = k * 16000 input).
extern "C" int svad_forward_device_ex(svad_engine* e, int sr, int B, int64_t L, int64_t ld, const void* d_audio, int sample_format,
                                      int sample_stride, const float* d_state_in, const float* d_ctx_in, float* d_state_out,
                                      float* d_ctx_out, float* d_probs, int64_t ldp, void* stream) {
    if (sample_format != kF32 && sample_format != kI16) return fail(SVAD_EINVAL, "sample_format must be 0 (f32) or 1 (int16 PCM)");
    if (sample_stride < 1) return fail(SVAD_EINVAL, "sample_stride must be >= 1");
    return forward_impl(e, sr, B, L, ld, d_audio, sample_format, d_state_in, d_ctx_in, sr == 16000 ? 64 : 32, d_state_out, d_ctx_out,
                        d_probs, ldp, (cudaStream_t)stream, sample_stride);
}

extern "C" int svad_step_device(svad_engine* e, int sr, int B, const float* d_input, const float* d_state_in, float* d_prob,
                                float* d_state_out, void* stream) {
    if (sr != 16000 && sr != 8000) return fail(SVAD_EINVAL, "Supported sampling rates: [8000, 16000] (got %d)", sr);
    const int n = sr == 16000 ? 512 : 256, ctx = n / 8;
    if (B > 0 && (!d_input || !d_prob)) return fail(SVAD_EINVAL, "null input/prob");
    // input rows are [context | chunk]: the chunk is the "audio", the context the carried-in samples
    return forward_impl(e, sr, B, n, ctx + n, d_input + ctx, kF32, d_state_in, d_input, ctx + n, d_state_out, nullptr, d_prob, 1,
                        (cudaStream_t)stream);
}

// ---- host-buffer twins -------------------------------------------------------------------------
// Page-locked caller buffers (cudaHostAlloc / cudaHostRegister / torch pin_memory) are DMA'd directly;
// pageable ones are staged through the engine's pinned buffer first.  The audio goes over in time slices
// (all streams x a few chunks) on a copy stream while the previous slice is being computed with the LSTM
// state and audio context carried on the device, so PCIe and the SMs overlap.
static bool is_pinned(const void* p) {
    cudaPointerAttributes at;
    if (cudaPointerGetAttributes(&at, p) != cudaSuccess) { cudaGetLastError(); return false; }
    return at.type == cudaMemoryTypeHost;
}

static int ensure_staging(svad_engine* e, size_t pin_bytes, size_t dev_bytes) {
    if (pin_bytes > e->pin_bytes) {
        if (e->h_pin) cudaFreeHost(e->h_pin);
        e->h_pin = nullptr; e->pin_bytes = 0;
        CUDA_TRY(cudaMallocHost(&e->h_pin, pin_bytes));
        e->pin_bytes = pin_bytes;
    }
    if (dev_bytes > e->dbuf_bytes) {
        if (e->d_buf) cudaFree(e->d_buf);
        e->d_buf = nullptr; e->dbuf_bytes = 0;
        CUDA_TRY(cudaMalloc(&e->d_buf, dev_bytes));
        e->dbuf_bytes = dev_bytes;
    }
    return SVAD_OK;
}

static int forward_host_impl(svad_engine* e, int sr, int B, int64_t L, int64_t ld, const void* audio, int fmt, const float* state_in,
                             const float* ctx_in, float* state_out, float* ctx_out, float* probs, int64_t ldp) {
    if (!e) return fail(SVAD_EINVAL, "null engine");
    if (sr != 16000 && sr != 8000) return fail(SVAD_EINVAL, "Supported sampling rates: [8000, 16000] (got %d)", sr);
    if (B < 0 || L < 0 || ld < L) return fail(SVAD_EINVAL, "bad size");
    if (B == 0) return SVAD_OK;
    const int n = sr == 16000 ? 512 : 256, ctx = n / 8;
    const int64_t T = (L + n - 1) / n;
    if (T > 0 && (!audio || !probs || ldp < T)) return fail(SVAD_EINVAL, "bad audio/probs");
    CUDA_TRY(cudaSetDevice(e->device));
    const size_t es = fmt_size(fmt);
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    // device: audio [B][L] | state [2][B][128] | ctx [B][ctx] | probs [B][T]      pinned host: same map
    const size_t o_audio = 0, o_state = al((size_t)B * L * es), o_ctx = o_state + al((size_t)2 * B * 128 * 4),
                 o_probs = o_ctx + al((size_t)B * ctx * 4), total = o_probs + al((size_t)B * T * 4);
    const bool audio_direct = T > 0 && is_pinned(audio);
    const bool probs_direct = T > 0 && ldp == T && is_pinned(probs);
    int rc = ensure_staging(e, total, total);
    if (rc) return rc;
    char *hp = (char*)e->h_pin, *dp = (char*)e->d_buf;
    float *d_state = (float*)(dp + o_state), *d_ctx = (float*)(dp + o_ctx), *d_probs = (float*)(dp + o_probs);
    cudaStream_t sc = e->stream_copy, sk = e->stream;
    // small inputs first (compute stream)
    if (state_in) {
        memcpy(hp + o_state, state_in, (size_t)2 * B * 128 * 4);
        CUDA_TRY(cudaMemcpyAsync(d_state, hp + o_state, (size_t)2 * B * 128 * 4, cudaMemcpyHostToDevice, sk));
    } else {
        CUDA_TRY(cudaMemsetAsync(d_state, 0, (size_t)2 * B * 128 * 4, sk));
    }
    if (ctx_in) {
        memcpy(hp + o_ctx, ctx_in, (size_t)B * ctx * 4);
        CUDA_TRY(cudaMemcpyAsync(d_ctx, hp + o_ctx, (size_t)B * ctx * 4, cudaMemcpyHostToDevice, sk));
    } else {
        CUDA_TRY(cudaMemsetAsync(d_ctx, 0, (size_t)B * ctx * 4, sk));
    }
    // time slices: at least 4 chunks each, at most kMaxSlices of them
    const int64_t per = T <= 8 ? T : (T + kMaxSlices - 1) / kMaxSlices < 4 ? 4 : (T + kMaxSlices - 1) / kMaxSlices;
    int slice = 0;
    for (int64_t t0 = 0; t0 < T; t0 += per, slice++) {
        const int64_t t1 = t0 + per < T ? t0 + per : T;
        const int64_t c0 = t0 * n, c1 = t1 * n < L ? t1 * n : L;     // sample columns of this slice
        const size_t width = (size_t)(c1 - c0) * es;
        const char* src = (const char*)audio + (size_t)c0 * es;
        size_t spitch = (size_t)ld * es;
        if (!audio_direct) {   // stage this slice's columns through pinned memory (rows packed at pitch L)
            for (int b = 0; b < B; b++) memcpy(hp + o_audio + ((size_t)b * L + c0) * es, src + (size_t)b * spitch, width);
            src = hp + o_audio + (size_t)c0 * es;
            spitch = (size_t)L * es;
        }
        CUDA_TRY(cudaMemcpy2DAsync(dp + o_audio + (size_t)c0 * es, (size_t)L * es, src, spitch, width, (size_t)B, cudaMemcpyHostToDevice, sc));
        cudaEvent_t ev = e->ev[slice % kMaxSlices];
        CUDA_TRY(cudaEventRecord(ev, sc));
        CUDA_TRY(cudaStreamWaitEvent(sk, ev, 0));
        rc = forward_impl(e, sr, B, c1 - c0, L, dp + o_audio + (size_t)c0 * es, fmt, d_state, d_ctx, ctx, d_state, d_ctx, d_probs + t0, T, sk);
        if (rc) return rc;
    }
    if (T > 0) CUDA_TRY(cudaMemcpyAsync(probs_direct ? (void*)probs : (void*)(hp + o_probs), d_probs, (size_t)B * T * 4, cudaMemcpyDeviceToHost, sk));
    if (state_out) CUDA_TRY(cudaMemcpyAsync(hp + o_state, d_state, (size_t)2 * B * 128 * 4, cudaMemcpyDeviceToHost, sk));
    if (ctx_out) CUDA_TRY(cudaMemcpyAsync(hp + o_ctx, d_ctx, (size_t)B * ctx * 4, cudaMemcpyDeviceToHost, sk));
    CUDA_TRY(cudaStreamSynchronize(sk));
    CUDA_TRY(cudaStreamSynchronize(sc));
    if (T > 0 && !probs_direct)
        for (int b = 0; b < B; b++) memcpy(probs + (size_t)b * ldp, hp + o_probs + (size_t)b * T * 4, (size_t)T * 4);
    if (state_out) memcpy(state_out, hp + o_state, (size_t)2 * B * 128 * 4);
    if (ctx_out) memcpy(ctx_out, hp + o_ctx, (size_t)B * ctx * 4);
    return SVAD_OK;
}

extern "C" int svad_forward_host(svad_engine* e, int sr, int B, int64_t L, int64_t ld, const float* audio, const float* state_in,
                                 const float* ctx_in, float* state_out, float* ctx_out, float* probs, int64_t ldp) {
    return forward_host_impl(e, sr, B, L, ld, audio, kF32, state_in, ctx_in, state_out, ctx_out, probs, ldp);
}
extern "C" int svad_forward_host_pcm16(svad_engine* e, int sr, int B, int64_t L, int64_t ld, const int16_t* audio, const float* state_in,
                                       const float* ctx_in, float* state_out, float* ctx_out, float* probs, int64_t ldp) {
    return forward_host_impl(e, sr, B, L, ld, audio, kI16, state_in, ctx_in, state_out, ctx_out, probs, ldp);
}

extern "C" int svad_step_host(svad_engine* e, int sr, int B, const float* input, const float* state_in, float* prob,
                              float* state_out) {
    if (!e) return fail(SVAD_EINVAL, "null engine");
    if (sr != 16000 && sr != 8000) return fail(SVAD_EINVAL, "Supported sampling rates: [8000, 16000] (got %d)", sr);
    if (B < 0) return fail(SVAD_EINVAL, "bad size");
    if (B == 0) return SVAD_OK;
    if (!input || !prob) return fail(SVAD_EINVAL, "null input/prob");
    const int n = sr == 16000 ? 512 : 256, ctx = n / 8, W = ctx + n;
    CUDA_TRY(cudaSetDevice(e->device));
    auto al = [](size_t x) { return (x + 255) & ~(size_t)255; };
    const size_t o_in = 0, o_state = al((size_t)B * W * 4), o_prob = o_state + al((size_t)2 * B * 128 * 4), total = o_prob + al((size_t)B * 4);
    int rc = ensure_staging(e, total, total);
    if (rc) return rc;
    char *hp = (char*)e->h_pin, *dp = (char*)e->d_buf;
    memcpy(hp + o_in, input, (size_t)B * W * 4);
    if (state_in) memcpy(hp + o_state, state_in, (size_t)2 * B * 128 * 4);
    cudaStream_t st = e->stream;
    CUDA_TRY(cudaMemcpyAsync(dp + o_in, hp + o_in, (size_t)B * W * 4, cudaMemcpyHostToDevice, st));
    if (state_in) CUDA_TRY(cudaMemcpyAsync(dp + o_state, hp + o_state, (size_t)2 * B * 128 * 4, cudaMemcpyHostToDevice, st));
    rc = svad_step_device(e, sr, B, (const float*)(dp + o_in), state_in ? (const float*)(dp + o_state) : nullptr, (float*)(dp + o_prob),
                          state_out ? (float*)(dp + o_state) : nullptr, st);
    if (rc) return rc;
    CUDA_TRY(cudaMemcpyAsync(hp + o_prob, dp + o_prob, (size_t)B * 4, cudaMemcpyDeviceToHost, st));
    if (state_out) CUDA_TRY(cudaMemcpyAsync(hp + o_state, dp + o_state, (size_t)2 * B * 128 * 4, cudaMemcpyDeviceToHost, st));
    CUDA_TRY(cudaStreamSynchronize(st));
    memcpy(prob, hp + o_prob, (size_t)B * 4);
    if (state_out) memcpy(state_out, hp + o_state, (size_t)2 * B * 128 * 4);
    return SVAD_OK;
}

// ------------------------------------------------------------------------------------------ collect_chunks / drop_chunks
// One gather launch over a segment table (reference: src/silero_vad/utils_vad.py:552-646, `torch.cat([wav[s:e] ...])`).
// plan[i] = {source element offset, destination element offset, length}; a CTA takes 8192 consecutive output elements,
// finds its first piece by bisection (once, thread 0) and walks forward: reads and writes are coalesced, HBM-bound.
namespace {
constexpr int kGatherUnit = 8192;
template <typename E>
__global__ void __launch_bounds__(256) svad_gather_segments(const E* __restrict__ src, E* __restrict__ dst, const long long* __restrict__ plan,
                                                            long long npieces, long long total) {
    __shared__ long long s_first;
    for (long long i0 = (long long)blockIdx.x * kGatherUnit; i0 < total; i0 += (long long)gridDim.x * kGatherUnit) {
        if (threadIdx.x == 0) {
            long long lo = 0, hi = npieces - 1;   // last piece whose destination offset is <= i0
            while (lo < hi) {
                const long long mid = (lo + hi + 1) >> 1;
                if (plan[3 * mid + 1] <= i0) lo = mid; else hi = mid - 1;
            }
            s_first = lo;
        }
        __syncthreads();
        long long pc = s_first;
        const long long iend = i0 + kGatherUnit < total ? i0 + kGatherUnit : total;
        for (long long i = i0 + threadIdx.x; i < iend; i += blockDim.x) {
            while (pc + 1 < npieces && plan[3 * (pc + 1) + 1] <= i) pc++;
            dst[i] = src[plan[3 * pc] + (i - plan[3 * pc + 1])];
        }
        __syncthreads();
    }
}
}  // namespace

extern "C" int svad_collect_chunks_device(svad_engine* e, const void* d_wav, int elem_bytes, int64_t B, int64_t ld, const int64_t* row_len,
                                          const int64_t* seg_rows, const int64_t* seg_bounds, int64_t n_seg, int drop, void* d_out,
                                          int64_t out_cap, int64_t* out_offsets, void* stream) {
    if (!e && d_out) return fail(SVAD_EINVAL, "null engine");   // the sizing pass (d_out == NULL) is host-only and needs none
    if ((elem_bytes != 2 && elem_bytes != 4) || B < 0 || n_seg < 0 || !out_offsets || (B > 0 && !row_len) || (n_seg > 0 && (!seg_rows || !seg_bounds)))
        return fail(SVAD_EINVAL, "bad argument");
    try {
        std::vector<long long> plan;
        int64_t k = 0, n_out = 0;
        auto piece = [&](int64_t row, int64_t a, int64_t b) {   // wav[row][a:b] with Python's clamping of non-negative bounds
            const int64_t len = row_len[row];
            if (a > len) a = len;
            if (b > len) b = len;
            if (b > a) { plan.push_back(row * ld + a); plan.push_back(n_out); plan.push_back(b - a); n_out += b - a; }
        };
        for (int64_t row = 0; row < B; row++) {
            out_offsets[row] = n_out;
            if (row_len[row] < 0 || row_len[row] > ld) return fail(SVAD_EINVAL, "row_len out of range");
            int64_t cur = 0;
            for (; k < n_seg && seg_rows[k] == row; k++) {
                const int64_t a = seg_bounds[2 * k], b = seg_bounds[2 * k + 1];
                if (a < 0 || b < 0) return fail(SVAD_EINVAL, "negative segment bound");
                if (drop) { piece(row, cur, a); cur = b; } else piece(row, a, b);
            }
            if (drop) piece(row, cur, row_len[row]);
        }
        if (k != n_seg) return fail(SVAD_EINVAL, "seg_rows must be sorted and < B");
        out_offsets[B] = n_out;
        if (!d_out || n_out == 0) return SVAD_OK;   // sizing pass
        if (n_out > out_cap) return fail(SVAD_EINVAL, "output buffer too small: need %lld elements", (long long)n_out);
        if (!d_wav) return fail(SVAD_EINVAL, "null audio");
        CUDA_TRY(cudaSetDevice(e->device));
        cudaStream_t st = (cudaStream_t)stream;
        long long* d_plan = nullptr;
        CUDA_TRY(cudaMallocAsync(&d_plan, plan.size() * sizeof(long long), st));
        cudaError_t err = cudaMemcpyAsync(d_plan, plan.data(), plan.size() * sizeof(long long), cudaMemcpyHostToDevice, st);
        if (err == cudaSuccess) {
            const long long npieces = (long long)(plan.size() / 3);
            long long units = (n_out + kGatherUnit - 1) / kGatherUnit;
            const int grid = (int)(units < (long long)e->sms * 8 ? units : (long long)e->sms * 8);
            if (elem_bytes == 4) svad_gather_segments<uint32_t><<<grid, 256, 0, st>>>((const uint32_t*)d_wav, (uint32_t*)d_out, d_plan, npieces, n_out);
            else svad_gather_segments<uint16_t><<<grid, 256, 0, st>>>((const uint16_t*)d_wav, (uint16_t*)d_out, d_plan, npieces, n_out);
            err = cudaGetLastError();
            e->launches++;
        }
        // the plan lives in pageable host memory: the copy above has been staged by the time cudaMemcpyAsync returns
        cudaFreeAsync(d_plan, st);
        if (err != cudaSuccess) return fail(SVAD_ECUDA, "collect_chunks: %s", cudaGetErrorString(err));
        return SVAD_OK;
    } catch (const std::bad_alloc&) {
        return fail(SVAD_ENOMEM, "out of memory");
    }
}

// ------------------------------------------------------------------------------------------ persistent streaming (BASELINE configs[1])
// One cluster of 8 CTAs stays resident and serves up to 4 live streams chunk by chunk through a mailbox in mapped pinned memory:
// no kernel launch, no cudaMemcpy and no stream synchronisation per 32 ms chunk -- the caller of the reference's streaming loop
// (VADIterator.__call__, src/silero_vad/utils_vad.py:507-549: one model call + .item() per chunk) pays one PCIe round trip.
struct svad_stream {
    svad_engine* e = nullptr;
    int sr = 0, ns = 0, n = 0;
    cudaStream_t st = nullptr;
    unsigned char* host = nullptr;
    SmallMail dev{};
    volatile long long* seq_in = nullptr;
    volatile long long* seq_out = nullptr;
    volatile int* flags = nullptr;
    float* in = nullptr;
    volatile float* out = nullptr;
    long long seq = 0;
    bool reset_next = true, dead = false;
};

template <bool SR16>
static int launch_stream_kernel(svad_stream* s) {
    auto kern = svad_small_cluster<SR16, float, true>;
    const size_t smem = (size_t)SmallMap<SR16>::total_floats * 4 + (size_t)Geo<SR16>::ctx * 4 * 4;
    CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
    TileArgs a{};
    a.B = s->ns; a.dec = 1;
    cudaLaunchConfig_t cfg{};
    cfg.gridDim = dim3(kSmallCtas);
    cfg.blockDim = dim3(kSmallThreads);
    cfg.dynamicSmemBytes = smem;
    cfg.stream = s->st;
    cudaLaunchAttribute at[1];
    at[0].id = cudaLaunchAttributeClusterDimension;
    at[0].val.clusterDim.x = kSmallCtas; at[0].val.clusterDim.y = 1; at[0].val.clusterDim.z = 1;
    cfg.attrs = at; cfg.numAttrs = 1;
    CUDA_TRY(cudaLaunchKernelEx(&cfg, kern, a, (const float*)s->e->d_small[SR16 ? 0 : 1], s->dev));
    s->e->launches++;
    return SVAD_OK;
}

extern "C" int svad_stream_close(svad_stream* s) {
    if (!s) return SVAD_OK;
    if (s->seq_in) {
        std::atomic_thread_fence(std::memory_order_release);
        *s->seq_in = -1;
    }
    if (s->st) { cudaStreamSynchronize(s->st); cudaStreamDestroy(s->st); }
    if (s->host) cudaFreeHost(s->host);
    delete s;
    return SVAD_OK;
}

extern "C" int svad_stream_open(svad_engine* e, int sr, int nstreams, svad_stream** out) {
    if (!e || !out) return fail(SVAD_EINVAL, "null argument");
    *out = nullptr;
    if (sr != 16000 && sr != 8000) return fail(SVAD_EINVAL, "Supported sampling rates: [8000, 16000] (got %d)", sr);
    if (nstreams < 1 || nstreams > kSmallNS) return fail(SVAD_EINVAL, "a streaming session serves 1..%d streams", kSmallNS);
    CUDA_TRY(cudaSetDevice(e->device));
    svad_stream* s = new (std::nothrow) svad_stream();
    if (!s) return fail(SVAD_ENOMEM, "out of memory");
    s->e = e; s->sr = sr; s->ns = nstreams; s->n = sr == 16000 ? 512 : 256;
    const size_t in_bytes = (size_t)kMailRing * kSmallNS * s->n * 4, bytes = 256 + in_bytes + (size_t)kMailRing * kSmallNS * 4;
    int rc = SVAD_OK;
    do {
        if (cudaHostAlloc((void**)&s->host, bytes, cudaHostAllocMapped) != cudaSuccess) { rc = fail(SVAD_ENOMEM, "cudaHostAlloc(mapped) failed"); break; }
        memset(s->host, 0, bytes);
        unsigned char* d = nullptr;
        if (cudaHostGetDevicePointer((void**)&d, s->host, 0) != cudaSuccess) { rc = fail(SVAD_ECUDA, "cudaHostGetDevicePointer failed"); break; }
        s->seq_in = reinterpret_cast<volatile long long*>(s->host);
        s->seq_out = reinterpret_cast<volatile long long*>(s->host + 64);
        s->flags = reinterpret_cast<volatile int*>(s->host + 128);
        s->in = reinterpret_cast<float*>(s->host + 256);
        s->out = reinterpret_cast<volatile float*>(s->host + 256 + in_bytes);
        s->dev.seq_in = reinterpret_cast<volatile long long*>(d);
        s->dev.seq_out = reinterpret_cast<volatile long long*>(d + 64);
        s->dev.flags = reinterpret_cast<volatile int*>(d + 128);
        s->dev.in = reinterpret_cast<const float*>(d + 256);
        s->dev.out = reinterpret_cast<volatile float*>(d + 256 + in_bytes);
        if (cudaStreamCreateWithFlags(&s->st, cudaStreamNonBlocking) != cudaSuccess) { rc = fail(SVAD_ECUDA, "cudaStreamCreate failed"); break; }
        rc = sr == 16000 ? launch_stream_kernel<true>(s) : launch_stream_kernel<false>(s);
    } while (0);
    if (rc != SVAD_OK) { s->seq_in = nullptr; svad_stream_close(s); return rc; }
    *out = s;
    return SVAD_OK;
}

extern "C" int svad_stream_reset(svad_stream* s) {
    if (!s) return fail(SVAD_EINVAL, "null stream");
    s->reset_next = true;   // applied by the kernel before the next chunk
    return SVAD_OK;
}

// chunk f32[nstreams][n] (host) -> prob f32[nstreams]; blocks until the persistent kernel has answered (one PCIe round trip + ~13 us of compute)
extern "C" int svad_stream_push(svad_stream* s, const float* chunk, float* prob) {
    if (!s || !chunk || !prob) return fail(SVAD_EINVAL, "null argument");
    if (s->dead) return fail(SVAD_ECUDA, "streaming session has ended (timed out); open a new one");
    const int slot = (int)(s->seq % kMailRing);
    float* dst = s->in + (size_t)slot * kSmallNS * s->n;
    memcpy(dst, chunk, (size_t)s->ns * s->n * 4);
    const long long word = ((s->seq + 1) << 1) | (s->reset_next ? 1 : 0);   // sequence number and reset bit travel in ONE word
    s->reset_next = false;
    std::atomic_thread_fence(std::memory_order_release);
    *s->seq_in = word;
    const auto t0 = std::chrono::steady_clock::now();
    for (unsigned spin = 1;; spin++) {
        if (*s->seq_out == s->seq + 1) break;
        if ((spin & 0xFFFF) == 0) {
            if (cudaStreamQuery(s->st) != cudaErrorNotReady) { s->dead = true; return fail(SVAD_ECUDA, "the persistent streaming kernel is not running any more"); }
            if (std::chrono::steady_clock::now() - t0 > std::chrono::seconds(10)) { s->dead = true; return fail(SVAD_ECUDA, "streaming kernel did not answer within 10 s"); }
        }
    }
    std::atomic_thread_fence(std::memory_order_acquire);
    for (int i = 0; i < s->ns; i++) prob[i] = s->out[slot * kSmallNS + i];
    s->seq++;
    return SVAD_OK;
}

// ------------------------------------------------------------------------------------------ decoder fine-tuning
// Encoder features: the fp32 tile kernel in features mode, whatever set_kernel / set_small_batch_max say (the inference kernels
// never hold the post-ReLU enc3 rows in fp32).
template <bool SR16>
static int launch_features(svad_engine* e, const TileArgs& a, cudaStream_t st) {
    switch (pick_rows(e, a.B)) {
        case 4: return launch<SR16, 4, float, true>(e, a, st);
        case 5: return launch<SR16, 5, float, true>(e, a, st);
        case 6: return launch<SR16, 6, float, true>(e, a, st);
        case 7: return launch<SR16, 7, float, true>(e, a, st);
        default: return launch<SR16, 8, float, true>(e, a, st);
    }
}

extern "C" int svad_features_device(svad_engine* e, int sr, int B, int64_t L, int64_t ld, const float* d_audio, const float* d_ctx_in,
                                    float* d_feat, void* stream) {
    if (!e) return fail(SVAD_EINVAL, "null engine");
    if (sr != 16000 && sr != 8000) return fail(SVAD_EINVAL, "Supported sampling rates: [8000, 16000] (got %d)", sr);
    const int n = sr == 16000 ? 512 : 256;
    if (B < 0 || L < 0 || L % n) return fail(SVAD_EINVAL, "features: B >= 0 and L a multiple of %d samples required (got B=%d, L=%lld)", n, B, (long long)L);
    if (B == 0 || L == 0) return SVAD_OK;
    if (!d_audio || !d_feat || ld < L) return fail(SVAD_EINVAL, "bad audio/feature pointer or stride");
    CUDA_TRY(cudaSetDevice(e->device));
    const int br = sr == 16000 ? 0 : 1;
    TileArgs a{};
    a.audio = d_audio; a.ld = ld; a.L = L; a.dec = 1; a.B = B; a.T = L / n;
    a.ctx_in = d_ctx_in; a.ctx_ld = sr == 16000 ? 64 : 32;
    a.probs = d_feat; a.ldp = a.T;   // features mode: [B][T][128]
    a.tape = e->d_tape[br]; a.consts = e->d_consts[br];
    return sr == 16000 ? launch_features<true>(e, a, (cudaStream_t)stream) : launch_features<false>(e, a, (cudaStream_t)stream);
}

// streams per CTA of the scans: one while the streams fit on the SMs, then 2 or 4 (a CTA's step costs little more for 4 streams)
static int dec_group(const svad_engine* e, int B) { return B <= e->sms ? 1 : (B <= 2 * e->sms ? 2 : 4); }
static long dec_chunks(long N) { return (N + kWgChunk - 1) / kWgChunk; }

extern "C" int64_t svad_decoder_tape_floats(int B, int64_t T) { return (B < 0 || T < 0) ? SVAD_EINVAL : (int64_t)B * T * (kGates + kHid); }

extern "C" int64_t svad_decoder_workspace_bytes(int B, int64_t T, int backward) {
    if (B < 0 || T < 0) return SVAD_EINVAL;
    const long N = (long)B * T;
    if (!backward) return (int64_t)N * kGates * 4;   // Gx
    return ((int64_t)N * kGates + (int64_t)B * (kHid + 1) + (int64_t)dec_chunks(N) * kGates * (2 * kHid + 1)) * 4;
}

template <class K>
static int dec_configure(svad_engine* e, K kern, size_t smem, bool* configured) {
    if (!configured[e->device & 15]) {
        CUDA_TRY(cudaFuncSetAttribute(kern, cudaFuncAttributeMaxDynamicSharedMemorySize, (int)smem));
        configured[e->device & 15] = true;
    }
    return SVAD_OK;
}

template <int G>
static int dec_forward(svad_engine* e, int B, long T, const float* w_hh, const float* w_head, const float* b_head, const float* drop, float* probs,
                       float* tape, const float* gx, cudaStream_t st) {
    static bool configured[16] = {};
    auto kern = dec_fwd<G>;
    if (int rc = dec_configure(e, kern, dec_fwd_smem_bytes<G>(), configured)) return rc;
    float* tg = tape;
    float* tc = tape ? tape + (long)B * T * kGates : nullptr;
    kern<<<(B + G - 1) / G, kDecThreads, dec_fwd_smem_bytes<G>(), st>>>(gx, w_hh, w_head, b_head, drop, probs, tg, tc, B, T);
    CUDA_TRY(cudaGetLastError());
    e->launches++;
    return SVAD_OK;
}

template <int G>
static int dec_backward(svad_engine* e, int B, long T, const float* w_hh, const float* w_head, const float* drop, const float* probs,
                        const float* dprobs, const float* tape, float* dgates, float* head_part, cudaStream_t st) {
    static bool configured[16] = {};
    auto kern = dec_bwd<G>;
    if (int rc = dec_configure(e, kern, dec_bwd_smem_bytes<G>(), configured)) return rc;
    kern<<<(B + G - 1) / G, kDecThreads, dec_bwd_smem_bytes<G>(), st>>>(w_hh, w_head, drop, probs, dprobs, tape, tape + (long)B * T * kGates,
                                                                    dgates, head_part, B, T);
    CUDA_TRY(cudaGetLastError());
    e->launches++;
    return SVAD_OK;
}

extern "C" int svad_decoder_forward_device(svad_engine* e, int B, int64_t T, const float* d_feat, const float* d_w_ih, const float* d_w_hh,
                                           const float* d_b_ih, const float* d_b_hh, const float* d_w_head, const float* d_b_head,
                                           const float* d_drop, float* d_probs, float* d_tape, void* d_work, void* stream) {
    if (!e) return fail(SVAD_EINVAL, "null engine");
    if (B < 0 || T < 0) return fail(SVAD_EINVAL, "negative size");
    if (B == 0 || T == 0) return SVAD_OK;
    if (!d_feat || !d_w_ih || !d_w_hh || !d_b_ih || !d_b_hh || !d_w_head || !d_b_head || !d_probs || !d_work)
        return fail(SVAD_EINVAL, "null feature, parameter, probability or workspace pointer");
    CUDA_TRY(cudaSetDevice(e->device));
    const cudaStream_t st = (cudaStream_t)stream;
    const long N = (long)B * T;
    float* gx = static_cast<float*>(d_work);
    dec_inproj<<<dim3((unsigned)((N + 63) / 64), kGates / 64), 256, 0, st>>>(d_feat, d_w_ih, d_b_ih, d_b_hh, gx, N);
    CUDA_TRY(cudaGetLastError());
    e->launches++;
    switch (dec_group(e, B)) {
        case 1: return dec_forward<1>(e, B, T, d_w_hh, d_w_head, d_b_head, d_drop, d_probs, d_tape, gx, st);
        case 2: return dec_forward<2>(e, B, T, d_w_hh, d_w_head, d_b_head, d_drop, d_probs, d_tape, gx, st);
        default: return dec_forward<4>(e, B, T, d_w_hh, d_w_head, d_b_head, d_drop, d_probs, d_tape, gx, st);
    }
}

extern "C" int svad_decoder_backward_device(svad_engine* e, int B, int64_t T, const float* d_feat, const float* d_w_hh, const float* d_w_head,
                                            const float* d_drop, const float* d_probs, const float* d_dprobs, const float* d_tape, void* d_work,
                                            float* d_dw_ih, float* d_dw_hh, float* d_db, float* d_dw_head, float* d_db_head, void* stream) {
    if (!e) return fail(SVAD_EINVAL, "null engine");
    if (B < 1 || T < 1) return fail(SVAD_EINVAL, "backward needs B >= 1 and T >= 1 (got B=%d, T=%lld)", B, (long long)T);
    if (!d_feat || !d_w_hh || !d_w_head || !d_probs || !d_dprobs || !d_tape || !d_work || !d_dw_ih || !d_dw_hh || !d_db || !d_dw_head || !d_db_head)
        return fail(SVAD_EINVAL, "null pointer argument");
    CUDA_TRY(cudaSetDevice(e->device));
    const cudaStream_t st = (cudaStream_t)stream;
    const long N = (long)B * T, nch = dec_chunks(N);
    if (nch > 65535) return fail(SVAD_EINVAL, "backward: at most %ld steps in total", 65535L * kWgChunk);
    float* dgates = static_cast<float*>(d_work);
    float* head_part = dgates + N * kGates;
    float* wg_part = head_part + (long)B * (kHid + 1);
    int rc;
    switch (dec_group(e, B)) {
        case 1: rc = dec_backward<1>(e, B, T, d_w_hh, d_w_head, d_drop, d_probs, d_dprobs, d_tape, dgates, head_part, st); break;
        case 2: rc = dec_backward<2>(e, B, T, d_w_hh, d_w_head, d_drop, d_probs, d_dprobs, d_tape, dgates, head_part, st); break;
        default: rc = dec_backward<4>(e, B, T, d_w_hh, d_w_head, d_drop, d_probs, d_dprobs, d_tape, dgates, head_part, st); break;
    }
    if (rc) return rc;
    dec_wgrad<<<dim3(kGates / 64, 2 * kHid / 64, (unsigned)nch), 256, 0, st>>>(dgates, d_feat, d_tape, d_tape + N * kGates, wg_part, T, N);
    CUDA_TRY(cudaGetLastError());
    const int tot = kGates * (2 * kHid + 1) + kHid + 1;
    dec_reduce<<<(tot + 255) / 256, 256, 0, st>>>(wg_part, (int)nch, head_part, B, d_dw_ih, d_dw_hh, d_db, d_dw_head, d_db_head);
    CUDA_TRY(cudaGetLastError());
    e->launches += 2;
    return SVAD_OK;
}

extern "C" int svad_threshold_grid_device(const float* d_probs, const float* d_targets, const int64_t* d_offsets, int64_t files,
                                          const double* d_grid, int64_t* d_counts, void* stream) {
    if (files < 0 || files > 0x7fffffff) return fail(SVAD_EINVAL, "files out of range (got %lld)", (long long)files);
    if (files == 0) return SVAD_OK;
    if (!d_probs || !d_targets || !d_offsets || !d_grid || !d_counts) return fail(SVAD_EINVAL, "null pointer argument");
    threshold_grid<<<(unsigned)files, 192, 0, (cudaStream_t)stream>>>(d_probs, d_targets, reinterpret_cast<const long long*>(d_offsets), d_grid,
                                                                    reinterpret_cast<long long*>(d_counts));
    CUDA_TRY(cudaGetLastError());
    return SVAD_OK;
}
