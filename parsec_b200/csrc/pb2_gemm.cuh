// pb2_gemm.cuh -- tensor-core (tcgen05 / TMEM / TMA) engine kernel for PB2_BODY_GEMM_BF16 windows.
//
// The task body restates what the reference reaches through `dyld=cublasDgemm` / cublasDgemm_v2
// (tests/dsl/dtd/dtd_test_simple_gemm.c:450,527; tests/runtime/cuda/nvlink.jdf:136-152): one tile
// GEMM per task, C(M x N) += A(M x K) * B(K x N).  Here in bf16 with fp32 accumulation in TMEM
// (BASELINE config 3); tiles are K-contiguous for both operands: A row-major [M][K], B stored
// [N][K] (== column-major K x N, what a "TN" cuBLAS call consumes), C row-major [M][N].
//
// One CTA per SM is one worker.  Warp roles (192 threads):
//   warp 0      : scheduler (ring pop / dependency release / retire) + TMA producer (one lane)
//   warp 1      : TMEM allocator + tcgen05.mma issuer (one lane)
//   warps 2..5  : epilogue: tcgen05.ld accumulators, C += acc in fp32, bf16 store
// A task is executed as ceil(M/128) x ceil(N/256) accumulator sub-tiles of 128 x 256 fp32 (256 TMEM
// columns); two accumulator buffers (512 columns) let the epilogue of sub-tile s overlap the MMAs
// of sub-tile s+1.  Operands stream through a 4-stage smem ring of {A 128x64, B 256x64} bf16
// 128B-swizzled boxes filled by TMA (`cp.async.bulk.tensor.2d`) from per-tile tensor maps.
#pragma once
#include <cuda.h>
#include "pb2_worker.cuh"

namespace pb2 {

namespace gemm {

constexpr int BM = 128, BN = 256, BK = 64, UK = 16;
constexpr int kStages = 4;
constexpr int kAStageBytes = BM * BK * 2;          // 16 KiB
constexpr int kBStageBytes = BN * BK * 2;          // 32 KiB
constexpr int kStageBytes = kAStageBytes + kBStageBytes;
constexpr int kThreads = 192;
constexpr int kEpiWarp0 = 2;
constexpr int kTmemCols = 512;
constexpr int kSmemBytes = kStages * kStageBytes + 1024 /*align*/ + 256 /*barriers*/;

__device__ __forceinline__ uint32_t smem_u32(const void* p) { return (uint32_t)__cvta_generic_to_shared(p); }

__device__ __forceinline__ void mbar_init(uint64_t* bar, uint32_t count) {
    asm volatile("mbarrier.init.shared::cta.b64 [%0], %1;" :: "r"(smem_u32(bar)), "r"(count) : "memory");
}
__device__ __forceinline__ void mbar_expect_tx(uint64_t* bar, uint32_t bytes) {
    asm volatile("mbarrier.arrive.expect_tx.shared::cta.b64 _, [%0], %1;" :: "r"(smem_u32(bar)), "r"(bytes) : "memory");
}
__device__ __forceinline__ void mbar_arrive(uint64_t* bar) {
    asm volatile("mbarrier.arrive.shared::cta.b64 _, [%0];" :: "r"(smem_u32(bar)) : "memory");
}
__device__ __forceinline__ bool mbar_try_wait(uint64_t* bar, uint32_t parity) {
    uint32_t ok;
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "mbarrier.try_wait.parity.shared::cta.b64 p, [%1], %2;\n"
        "selp.u32 %0, 1, 0, p;\n"
        "}\n" : "=r"(ok) : "r"(smem_u32(bar)), "r"(parity) : "memory");
    return ok != 0;
}
__device__ __forceinline__ void mbar_wait(uint64_t* bar, uint32_t parity) {
    while (!mbar_try_wait(bar, parity)) { }
}
__device__ __forceinline__ void tma_load_2d(void* smem_dst, const CUtensorMap* tmap, uint64_t* bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        :: "r"(smem_u32(smem_dst)), "l"(tmap), "r"(smem_u32(bar)), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void fence_proxy_async() { asm volatile("fence.proxy.async;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_before() { asm volatile("tcgen05.fence::before_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_fence_after() { asm volatile("tcgen05.fence::after_thread_sync;" ::: "memory"); }
__device__ __forceinline__ void tc_commit(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::1.mbarrier::arrive::one.shared::cluster.b64 [%0];"
                 :: "r"(smem_u32(bar)) : "memory");
}
// D[tmem] (+)= A[smem] * B[smem], M=128, N=256, K=16, bf16 x bf16 -> fp32
__device__ __forceinline__ void tc_mma(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::1.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" :: "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
__device__ __forceinline__ void tc_ld_32x32b_x32(uint32_t taddr, uint32_t (&r)[32]) {
    asm volatile(
        "tcgen05.ld.sync.aligned.32x32b.x32.b32 "
        "{%0,%1,%2,%3,%4,%5,%6,%7,%8,%9,%10,%11,%12,%13,%14,%15,"
        "%16,%17,%18,%19,%20,%21,%22,%23,%24,%25,%26,%27,%28,%29,%30,%31}, [%32];"
        : "=r"(r[0]), "=r"(r[1]), "=r"(r[2]), "=r"(r[3]), "=r"(r[4]), "=r"(r[5]), "=r"(r[6]), "=r"(r[7]),
          "=r"(r[8]), "=r"(r[9]), "=r"(r[10]), "=r"(r[11]), "=r"(r[12]), "=r"(r[13]), "=r"(r[14]), "=r"(r[15]),
          "=r"(r[16]), "=r"(r[17]), "=r"(r[18]), "=r"(r[19]), "=r"(r[20]), "=r"(r[21]), "=r"(r[22]), "=r"(r[23]),
          "=r"(r[24]), "=r"(r[25]), "=r"(r[26]), "=r"(r[27]), "=r"(r[28]), "=r"(r[29]), "=r"(r[30]), "=r"(r[31])
        : "r"(taddr) : "memory");
}
__device__ __forceinline__ void tc_wait_ld() { asm volatile("tcgen05.wait::ld.sync.aligned;" ::: "memory"); }

// K-major, 128B-swizzled operand descriptor (cute/arch/mma_sm100_desc.hpp SmemDescriptor):
// start>>4 [0,14) | LBO=1 [16,30) | SBO=1024>>4 [32,46) | version=1 [46,48) | SWIZZLE_128B=2 [61,64)
__device__ __forceinline__ uint64_t make_desc(uint32_t smem_addr) {
    return (uint64_t)((smem_addr & 0x3ffffu) >> 4) | (1ull << 16) | ((uint64_t)(1024 >> 4) << 32) | (1ull << 46) | (2ull << 61);
}
// kind::f16 instruction descriptor (InstrDescriptor): D=f32 [4,6)=1, A=bf16 [7,10)=1, B=bf16 [10,13)=1,
// A,B K-major (bits 15,16 = 0), N>>3 [17,23), M>>4 [24,29)
__device__ __forceinline__ constexpr uint32_t make_idesc(int M, int N) {
    return (1u << 4) | (1u << 7) | (1u << 10) | ((uint32_t)(N >> 3) << 17) | ((uint32_t)(M >> 4) << 24);
}

__device__ __forceinline__ float bf16_lo(uint32_t v) { return __uint_as_float(v << 16); }
__device__ __forceinline__ float bf16_hi(uint32_t v) { return __uint_as_float(v & 0xffff0000u); }
__device__ __forceinline__ uint32_t pack_bf16(float lo, float hi) {
    uint32_t r;
    asm("cvt.rn.bf16x2.f32 %0, %1, %2;" : "=r"(r) : "f"(hi), "f"(lo));
    return r;
}

struct Shared {
    alignas(16) pb2_task_t task;    // filled with four 16-byte loads
    uint64_t full[kStages];
    uint64_t empty[kStages];
    uint64_t tmem_full[2];
    uint64_t tmem_empty[2];
    uint32_t tmem_base;
    int32_t  id;
    int32_t  need;
    int32_t  decide;
    int32_t  last;
    uint32_t red[32];
};

}  // namespace gemm

__global__ void __launch_bounds__(gemm::kThreads, 1)
pb2_engine_gemm_kernel(WinDev w, const CUtensorMap* __restrict__ tmaps) {
    using namespace gemm;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    __shared__ Shared sh;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages; ++s) { mbar_init(&sh.full[s], 1); mbar_init(&sh.empty[s], 1); }
        for (int a = 0; a < 2; ++a) { mbar_init(&sh.tmem_full[a], 1); mbar_init(&sh.tmem_empty[a], 4); }
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 1) {
        asm volatile("tcgen05.alloc.cta_group::1.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"(smem_u32(&sh.tmem_base)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::1.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    __syncthreads();
    tc_fence_after();
    const uint32_t tmem_base = sh.tmem_base;

    // pipeline state persists across tasks
    uint32_t p_stage = 0, p_phase = 0;     // producer
    uint32_t c_stage = 0, c_phase = 0;     // MMA consumer
    uint32_t m_acc = 0, m_acc_phase = 0;   // MMA accumulator buffer
    uint32_t e_acc = 0, e_acc_phase = 0;   // epilogue accumulator buffer

    for (;;) {
        if (threadIdx.x == 0) {
            const int32_t id = pop_task(w);
            if (id != kEmpty) {
                __threadfence();
                w.start_seq[id] = (uint32_t)atomicAdd(&w.ctl->evt.v, 1ull);
                w.worker[id] = (int32_t)blockIdx.x;
            }
            sh.id = id;
        }
        __syncthreads();
        const int32_t id = sh.id;
        if (id == kEmpty) break;
        if (threadIdx.x < 4) reinterpret_cast<uint4*>(&sh.task)[threadIdx.x] =
            __ldg(reinterpret_cast<const uint4*>(&w.tasks[id]) + threadIdx.x);
        __syncthreads();
        const pb2_task_t& t = sh.task;

        // ---- stage in (same protocol as the HBM kernel) ----
        if (threadIdx.x == 0) {
            int need = 0;
            for (int f = 0; f < t.nb_flows; ++f)
                if (t.tile[f] >= 0 && needs_stage_in(&w.tiles[t.tile[f]], t.access[f])) need |= 1 << f;
            sh.need = need;
        }
        __syncthreads();
        {
            const int need = sh.need;
            for (int f = 0; f < t.nb_flows; ++f) {
                if (t.tile[f] < 0) continue;
                pb2_tile_t* tile = &w.tiles[t.tile[f]];
                if ((need >> f) & 1) stage_in_flow(stage_ctx(w), tile, t.access[f], &sh.decide);
                if (threadIdx.x == 0)
                    w.seen_version[id * PB2_MAX_FLOWS + f] = *reinterpret_cast<volatile uint32_t*>(&tile->version);
            }
            if (need) { fence_proxy_async(); __syncthreads(); }
        }

        const bool is_gemm = (t.body == PB2_BODY_GEMM_BF16);
        unsigned long long hbm_result = 0;
        if (!is_gemm && t.body != PB2_BODY_NOP) {
            // GEMM windows may carry a few HBM-bound tasks of the same DAG (e.g. a panel task): run them in place
            BodyArgs a;
            for (int f = 0; f < PB2_MAX_FLOWS; ++f) {
                const bool has = f < t.nb_flows && t.tile[f] >= 0;
                a.flow[f] = has ? w.tiles[t.tile[f]].dev_ptr : nullptr;
                a.bytes[f] = has ? w.tiles[t.tile[f]].bytes : 0;
            }
            a.elem0 = 0; a.part = 0;
            a.iparam[0] = t.iparam[0]; a.iparam[1] = t.iparam[1]; a.iparam[2] = t.iparam[2]; a.fparam = t.fparam;
            hbm_result = run_hbm_body(t.body, a, sh.red);
            fence_proxy_async();
            __syncthreads();
        }
        const int M = t.iparam[0], N = t.iparam[1], K = t.iparam[2];
        const int mblocks = is_gemm ? (M + BM - 1) / BM : 0;
        const int nblocks = is_gemm ? (N + BN - 1) / BN : 0;
        const int kblocks = (K + BK - 1) / BK;
        const int nsub = mblocks * nblocks;

        if (warp == 0) {
            // ===== TMA producer =====
            if (lane == 0 && nsub > 0) {
                fence_proxy_async();    // operand tiles may have been written by generic-proxy stores
                const CUtensorMap* mapA = &tmaps[t.tile[0]];
                const CUtensorMap* mapB = &tmaps[t.tile[1]];
                for (int sub = 0; sub < nsub; ++sub) {
                    const int mb = sub / nblocks, nb = sub % nblocks;
                    for (int kb = 0; kb < kblocks; ++kb) {
                        mbar_wait(&sh.empty[p_stage], p_phase ^ 1);
                        uint8_t* sa = smem + p_stage * kStageBytes;
                        uint8_t* sb = sa + kAStageBytes;
                        mbar_expect_tx(&sh.full[p_stage], kStageBytes);
                        tma_load_2d(sa, mapA, &sh.full[p_stage], kb * BK, mb * BM);
                        tma_load_2d(sb, mapB, &sh.full[p_stage], kb * BK, nb * BN);
                        tma_load_2d(sb + kAStageBytes, mapB, &sh.full[p_stage], kb * BK, nb * BN + 128);
                        if (++p_stage == kStages) { p_stage = 0; p_phase ^= 1; }
                    }
                }
            }
        } else if (warp == 1) {
            // ===== MMA issuer =====
            if (lane == 0 && nsub > 0) {
                constexpr uint32_t idesc = make_idesc(BM, BN);
                for (int sub = 0; sub < nsub; ++sub) {
                    mbar_wait(&sh.tmem_empty[m_acc], m_acc_phase ^ 1);
                    tc_fence_after();
                    const uint32_t d = tmem_base + m_acc * BN;
                    for (int kb = 0; kb < kblocks; ++kb) {
                        mbar_wait(&sh.full[c_stage], c_phase);
                        tc_fence_after();
                        const uint32_t sa = smem_u32(smem + c_stage * kStageBytes);
                        const uint64_t da = make_desc(sa), db = make_desc(sa + kAStageBytes);
#pragma unroll
                        for (int k = 0; k < BK / UK; ++k)
                            tc_mma(d, da + (uint64_t)(k * UK * 2 >> 4), db + (uint64_t)(k * UK * 2 >> 4), idesc,
                                   (kb | k) != 0 ? 1u : 0u);
                        tc_commit(&sh.empty[c_stage]);         // smem slot free once these MMAs retire
                        if (++c_stage == kStages) { c_stage = 0; c_phase ^= 1; }
                    }
                    tc_commit(&sh.tmem_full[m_acc]);           // accumulator ready for the epilogue
                    if (++m_acc == 2) { m_acc = 0; m_acc_phase ^= 1; }
                }
            }
        } else {
            // ===== epilogue warps: TMEM -> registers -> C += acc -> bf16 =====
            if (nsub > 0) {
                const int q = warp & 3;                         // TMEM lane quadrant this warp may access
                uint8_t* Cbase = reinterpret_cast<uint8_t*>(w.tiles[t.tile[2]].dev_ptr);
                for (int sub = 0; sub < nsub; ++sub) {
                    const int mb = sub / nblocks, nb = sub % nblocks;
                    mbar_wait(&sh.tmem_full[e_acc], e_acc_phase);
                    tc_fence_after();
                    const int row = mb * BM + q * 32 + lane;
                    const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16) + e_acc * BN;
#pragma unroll 1
                    for (int c = 0; c < BN / 32; ++c) {
                        uint32_t acc[32];
                        tc_ld_32x32b_x32(taddr + c * 32, acc);
                        tc_wait_ld();
                        const int col0 = nb * BN + c * 32;
                        if (row < M && col0 < N) {
                            uint4* cp = reinterpret_cast<uint4*>(Cbase + ((size_t)row * N + col0) * 2);
                            const int nv = (N - col0 >= 32) ? 4 : (N - col0) / 8;
#pragma unroll
                            for (int v = 0; v < 4; ++v) {
                                if (v < nv) {
                                    uint4 cv = ld_stream(cp + v);
                                    uint4 o;
                                    o.x = pack_bf16(bf16_lo(cv.x) + __uint_as_float(acc[v * 8 + 0]), bf16_hi(cv.x) + __uint_as_float(acc[v * 8 + 1]));
                                    o.y = pack_bf16(bf16_lo(cv.y) + __uint_as_float(acc[v * 8 + 2]), bf16_hi(cv.y) + __uint_as_float(acc[v * 8 + 3]));
                                    o.z = pack_bf16(bf16_lo(cv.z) + __uint_as_float(acc[v * 8 + 4]), bf16_hi(cv.z) + __uint_as_float(acc[v * 8 + 5]));
                                    o.w = pack_bf16(bf16_lo(cv.w) + __uint_as_float(acc[v * 8 + 6]), bf16_hi(cv.w) + __uint_as_float(acc[v * 8 + 7]));
                                    st_stream(cp + v, o);
                                }
                            }
                        }
                    }
                    tc_fence_before();
                    __syncwarp();
                    if (lane == 0) mbar_arrive(&sh.tmem_empty[e_acc]);
                    if (++e_acc == 2) { e_acc = 0; e_acc_phase ^= 1; }
                }
                fence_proxy_async();   // C may be consumed through TMA by a later task on another SM
            }
        }
        __syncthreads();

        // ---- pushout (PARSEC_PUSHOUT on the last k, dtd_test_simple_gemm.c:687) ----
        for (int f = 0; f < t.nb_flows; ++f) {
            if (pushes_out(t, f)) pushout(w.ctl, w.tiles[t.tile[f]].src_ptr, w.tiles[t.tile[f]].dev_ptr, w.tiles[t.tile[f]].bytes);
        }
        __syncthreads();

        if (threadIdx.x < 32) {
            __threadfence();
            if (threadIdx.x == 0) {
                // a body id validate_window accepts but run_hbm_body does not know (result ~0) does not abort here
                record_result(w, t.body, id, 0, 1, hbm_result);
                sh.last = retire_task(w, t, id) ? 1 : 0;
                __threadfence();
            }
            __syncwarp();
            release_successors_warp(w, t);
            release_remote_warp(w, id);
            if (threadIdx.x == 0 && sh.last) finish_window(w);
        }
        __syncthreads();
    }

    tc_fence_before();
    __syncthreads();
    if (warp == 1) {
        asm volatile("tcgen05.dealloc.cta_group::1.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}

static inline int pb2_gemm_nworkers(int sm_count) { return sm_count; }

static inline int pb2_gemm_launch(const WinDev& w, const CUtensorMap* tmaps, int nworkers, cudaStream_t stream) {
    static bool attr_set = false;
    if (!attr_set) {
        if (cudaFuncSetAttribute(pb2_engine_gemm_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize,
                                 gemm::kSmemBytes) != cudaSuccess) return PB2_ERR_DEVICE;
        attr_set = true;
    }
    pb2_engine_gemm_kernel<<<nworkers, gemm::kThreads, gemm::kSmemBytes, stream>>>(w, tmaps);
    return cudaGetLastError() == cudaSuccess ? PB2_SUCCESS : PB2_ERR_DEVICE;
}

}  // namespace pb2
