// pb2_gemm2.cuh -- tensor-core engine kernel v2 for PB2_BODY_GEMM_BF16 windows: CTA pairs + fused k-chains.
//
// What changes against v1 (pb2_gemm.cuh):
//   * a worker is a CLUSTER OF TWO CTAs on one TPC issuing `tcgen05.mma.cta_group::2` (M = 256, N = 256): each CTA
//     stages only its half of A and of B per k-block, halving L2->smem traffic per flop;
//   * the host groups GEMM tasks into UNITS: a maximal chain of tasks that accumulate into the same C tile and whose
//     only missing dependency is the previous link (the C(i,j) k-chain of dtd_test_simple_gemm.c:675-696, the k-chains
//     of a tile Cholesky).  A unit is executed by `nparts` independent row-parts of 256 rows; each part keeps its
//     256 x N fp32 accumulator in TMEM (128 lanes x 512 columns in each CTA) across ALL the members of the chain and
//     touches C once: C_out = bf16(C_in + sum_k A_k B_k^T).  This is the reference's "keep the released successor for
//     the same execution stream" (es->next_task, scheduling.c:517-530) taken to its conclusion: 32 dependent tasks
//     become one accumulation.  Members still retire one by one, in chain order, with their own sequence numbers,
//     versions and out-edges (the dependency trace is unchanged); only the intermediate bf16 roundings of C disappear.
//   * scheduling entities on the device are units (counter-mode dependency words), ring entries are (part, unit).
#pragma once
#include <cuda.h>
#include "pb2_worker.cuh"
#include "pb2_gemm.cuh"

namespace pb2 {

struct GUnit {                  // 48 bytes, read-only
    int32_t seg_begin, seg_count;   // members, in chain order
    int32_t succ_begin, succ_count; // out-edges of all members (chain links removed): target unit ids
    int32_t dep_goal;               // in-edges from other units
    int32_t nparts;
    int32_t tileC;                  // GEMM units: the C tile; -1 otherwise
    int32_t M, N, K;
    int32_t flags;                  // bit0 is_gemm, bit1 pushout C
    int32_t pad;
};
struct GSeg { int32_t task, tileA, tileB, pad; };

struct Win2Dev {
    WinDev w;                       // task-level arrays (descriptors, tiles, outputs, ctl, ring)
    const GUnit* units;
    const GSeg*  segs;
    const int32_t* usucc;
    int32_t* udep;
    int32_t* parts_left;
    const CUtensorMap* tmaps;
    int32_t nunits;
    int32_t debug;                  // development only (PB2_GEMM_DEBUG): 1 = no TMA loads, 2 = no MMAs, 4 = no epilogue
};

namespace gemm2 {
using namespace gemm;

constexpr int kThreads2 = 256;
constexpr int kStages2 = 4;
constexpr int kAStage = 128 * BK * 2;      // this CTA's 128 rows of A
constexpr int kBHalf = 128 * BK * 2;       // this CTA's 128 rows of one N=256 half of B
constexpr int kStage2 = kAStage + 2 * kBHalf;   // 48 KiB
constexpr int kSmem2 = kStages2 * kStage2 + 1024 + 256;

struct Job {
    int32_t unit, part, stop, is_gemm;
    int32_t seg_begin, seg_count, tileC, m0;
    int32_t M, N, K, pushout;
    int32_t n0, Nj, pad0, pad1;     // this part's columns [n0, n0 + Nj) of the N-wide tile (Nj <= 512: TMEM columns)
};

struct Shared2 {
    alignas(16) Job job;
    alignas(16) pb2_task_t task;    // non-GEMM units: the single member's descriptor
    uint64_t full[kStages2];
    uint64_t empty[kStages2];
    uint64_t tmem_full;
    uint32_t tmem_base;
    int32_t  need, decide;
    uint32_t red[32];
};

__device__ __forceinline__ uint32_t cluster_ctarank() { uint32_t r; asm volatile("mov.u32 %0, %%cluster_ctarank;" : "=r"(r)); return r; }
__device__ __forceinline__ void cluster_sync_all() {
    asm volatile("barrier.cluster.arrive.release.aligned;" ::: "memory");
    asm volatile("barrier.cluster.wait.acquire.aligned;" ::: "memory");
}
__device__ __forceinline__ uint32_t mapa(uint32_t saddr, uint32_t rank) {
    uint32_t r; asm volatile("mapa.shared::cluster.u32 %0, %1, %2;" : "=r"(r) : "r"(saddr), "r"(rank)); return r;
}
__device__ __forceinline__ void st_cluster_u32(uint32_t addr, uint32_t v) {
    asm volatile("st.shared::cluster.u32 [%0], %1;" :: "r"(addr), "r"(v) : "memory");
}
__device__ __forceinline__ void mbar_arrive_cluster(uint32_t addr) {
    // no cluster-scope release: the arrival publishes no data (the TMA bytes are tracked by complete_tx)
    asm volatile("mbarrier.arrive.shared::cluster.b64 _, [%0];" :: "r"(addr) : "memory");
}
// TMA load of this CTA's share into its own smem; completion bytes are credited to the LEADER's barrier
__device__ __forceinline__ void tma_load_2sm(void* smem_dst, const CUtensorMap* tmap, uint32_t leader_bar, int c0, int c1) {
    asm volatile(
        "cp.async.bulk.tensor.2d.cta_group::2.shared::cluster.global.mbarrier::complete_tx::bytes [%0], [%1, {%3, %4}], [%2];"
        :: "r"(smem_u32(smem_dst)), "l"(tmap), "r"(leader_bar), "r"(c0), "r"(c1) : "memory");
}
__device__ __forceinline__ void tc_mma2(uint32_t tmem_d, uint64_t desc_a, uint64_t desc_b, uint32_t idesc, uint32_t accumulate) {
    asm volatile(
        "{\n"
        ".reg .pred p;\n"
        "setp.ne.b32 p, %4, 0;\n"
        "tcgen05.mma.cta_group::2.kind::f16 [%0], %1, %2, %3, p;\n"
        "}\n" :: "r"(tmem_d), "l"(desc_a), "l"(desc_b), "r"(idesc), "r"(accumulate) : "memory");
}
// arrive (when all prior MMAs of the pair retire) on the barrier at the same smem offset in BOTH CTAs
__device__ __forceinline__ void tc_commit2(uint64_t* bar) {
    asm volatile("tcgen05.commit.cta_group::2.mbarrier::arrive::one.shared::cluster.multicast::cluster.b64 [%0], %1;"
                 :: "r"(smem_u32(bar)), "h"((uint16_t)0x3) : "memory");
}

// whole warp: the unit is complete (all parts): retire its members in chain order, release its out-edges
__device__ __forceinline__ void retire_unit_warp(const Win2Dev& g, const GUnit& u, int unit_id) {
    const WinDev& w = g.w;
    const int lane = threadIdx.x & 31;
    const int L = u.seg_count;
    unsigned long long ebase = 0, rbase = 0;
    if (lane == 0) {
        ebase = atomicAdd(&w.ctl->evt.v, (unsigned long long)(2 * L));
        rbase = atomicAdd(&w.ctl->retired.v, (unsigned long long)L);
        *reinterpret_cast<volatile unsigned long long*>(&w.ctl->progress_ns.v) = globaltimer_ns();
    }
    ebase = __shfl_sync(0xffffffffu, ebase, 0);
    rbase = __shfl_sync(0xffffffffu, rbase, 0);
    const uint32_t cver = (u.flags & 1) ? *reinterpret_cast<volatile uint32_t*>(&w.tiles[u.tileC].version) : 0u;
    for (int i = lane; i < L; i += 32) {
        const GSeg s = g.segs[u.seg_begin + i];
        const pb2_task_t& t = w.tasks[s.task];
        w.start_seq[s.task] = (uint32_t)(ebase + 2 * i);
        w.end_seq[s.task] = (uint32_t)(ebase + 2 * i + 1);
        w.retire_log[rbase + i] = s.task;
        w.worker[s.task] = (int32_t)blockIdx.x;
        if (u.flags & 1) {
            w.seen_version[s.task * PB2_MAX_FLOWS + 0] = *reinterpret_cast<volatile uint32_t*>(&w.tiles[s.tileA].version);
            w.seen_version[s.task * PB2_MAX_FLOWS + 1] = *reinterpret_cast<volatile uint32_t*>(&w.tiles[s.tileB].version);
            w.seen_version[s.task * PB2_MAX_FLOWS + 2] = cver + (uint32_t)i;
            w.result[s.task] = 0;
        } else {
            for (int f = 0; f < t.nb_flows; ++f)
                if (t.tile[f] >= 0) {
                    pb2_tile_t* tile = &w.tiles[t.tile[f]];
                    const uint32_t v = *reinterpret_cast<volatile uint32_t*>(&tile->version);
                    w.seen_version[s.task * PB2_MAX_FLOWS + f] = v;
                    if (t.access[f] & PB2_FLOW_ACCESS_WRITE) {
                        *reinterpret_cast<volatile uint32_t*>(&tile->version) = v + 1;
                        st_relaxed_gpu(&tile->state, PB2_TILE_VALID);
                    }
                }
        }
    }
    if (lane == 0 && (u.flags & 1)) {
        *reinterpret_cast<volatile uint32_t*>(&w.tiles[u.tileC].version) = cver + (uint32_t)L;
        st_relaxed_gpu(&w.tiles[u.tileC].state, PB2_TILE_VALID);
    }
    __threadfence();
    __syncwarp();
    // release: parsec_update_deps_with_counter on the successor units; a ready unit contributes nparts ring entries
    for (int e0 = 0; e0 < u.succ_count; e0 += 32) {
        const int e = e0 + lane;
        int nparts = 0, sid = -1;
        if (e < u.succ_count) {
            sid = g.usucc[u.succ_begin + e];
            if (atomicSub(&g.udep[sid], 1) == 1) nparts = g.units[sid].nparts;
        }
        push_ready_warp<true>(w, sid, nparts);
    }
    // out-edges into other GPUs' windows, member by member (a member with remote successors is always the last of
    // its unit: build_gemm2_units does not fuse across it)
    if (w.rs_begin) for (int i = 0; i < L; ++i) release_remote_warp(w, g.segs[u.seg_begin + i].task);
    if (lane == 0 && (int32_t)(rbase + L) == w.ntasks) finish_window(w);
    (void)unit_id;
}

}  // namespace gemm2

__global__ void __cluster_dims__(2, 1, 1) __launch_bounds__(gemm2::kThreads2, 1)
pb2_engine_gemm2_kernel(Win2Dev g) {
    using namespace gemm2;
    const WinDev& w = g.w;
    extern __shared__ uint8_t smem_raw[];
    uint8_t* smem = reinterpret_cast<uint8_t*>((reinterpret_cast<uintptr_t>(smem_raw) + 1023) & ~uintptr_t(1023));
    __shared__ Shared2 sh;

    const int warp = threadIdx.x >> 5, lane = threadIdx.x & 31;
    const uint32_t rank = cluster_ctarank();
    const bool leader = rank == 0;

    if (threadIdx.x == 0) {
        for (int s = 0; s < kStages2; ++s) { mbar_init(&sh.full[s], 2); mbar_init(&sh.empty[s], 1); }
        mbar_init(&sh.tmem_full, 1);
        asm volatile("fence.mbarrier_init.release.cluster;" ::: "memory");
    }
    if (warp == 2) {
        asm volatile("tcgen05.alloc.cta_group::2.sync.aligned.shared::cta.b32 [%0], %1;"
                     :: "r"(smem_u32(&sh.tmem_base)), "r"(kTmemCols) : "memory");
        asm volatile("tcgen05.relinquish_alloc_permit.cta_group::2.sync.aligned;" ::: "memory");
    }
    tc_fence_before();
    cluster_sync_all();
    tc_fence_after();
    const uint32_t tmem_base = sh.tmem_base;

    uint32_t p_stage = 0, p_phase = 0, c_stage = 0, c_phase = 0, tfull_phase = 0;

    for (;;) {
        // ---------------- leader: pop the next (part, unit), stage tiles in, publish the job to both CTAs
        if (leader) {
            if (threadIdx.x == 0) {
                Job j; memset(&j, 0, sizeof j);
                const int32_t e = pop_task(w);
                if (e == kEmpty) { j.stop = 1; }
                else {
                    __threadfence();
                    j.unit = PB2_SUCC_TASK((uint32_t)e); j.part = PB2_SUCC_FLOW((uint32_t)e);
                    const GUnit u = g.units[j.unit];
                    j.is_gemm = u.flags & 1; j.pushout = (u.flags >> 1) & 1;
                    j.seg_begin = u.seg_begin; j.seg_count = u.seg_count; j.tileC = u.tileC;
                    const int mparts = (u.M + 255) / 256;
                    j.m0 = (j.part % mparts) * 256; j.M = u.M; j.N = u.N; j.K = u.K;
                    j.n0 = (j.part / mparts) * 512; j.Nj = min(512, u.N - j.n0);
                }
                sh.job = j;
            }
            __syncthreads();
            if (!sh.job.stop) {
                // stage in every INVALID tile the job reads (same protocol as the other kernels); leader CTA only
                const int nseg = sh.job.is_gemm ? sh.job.seg_count : 0;
                for (int i = -1; i < 2 * nseg; ++i) {
                    int tile_id; uint8_t acc;
                    if (i < 0) { if (!sh.job.is_gemm) break; tile_id = sh.job.tileC; acc = PB2_FLOW_ACCESS_RW; }
                    else { const GSeg s = g.segs[sh.job.seg_begin + (i >> 1)]; tile_id = (i & 1) ? s.tileB : s.tileA; acc = PB2_FLOW_ACCESS_READ; }
                    pb2_tile_t* tile = &w.tiles[tile_id];
                    if (threadIdx.x == 0) sh.need = needs_stage_in(tile, acc);
                    __syncthreads();
                    if (sh.need) {
                        const int ns = tile_slices(w, tile->bytes);
                        if (ns == 1) stage_in_flow(stage_ctx(w), tile, acc, &sh.decide);
                        else stage_in_slices(stage_ctx(w), tile_id, ns, 0, ns, &sh.decide);     // take what nobody has claimed, wait for the rest
                        fence_proxy_async();
                    }
                    __syncthreads();
                }
                if (!sh.job.is_gemm) {
                    const GSeg s = g.segs[sh.job.seg_begin];
                    if (threadIdx.x < 4) reinterpret_cast<uint4*>(&sh.task)[threadIdx.x] =
                        __ldg(reinterpret_cast<const uint4*>(&w.tasks[s.task]) + threadIdx.x);
                    __syncthreads();
                    const pb2_task_t& t = sh.task;
                    for (int f = 0; f < t.nb_flows; ++f) {
                        if (t.tile[f] < 0 || !(t.access[f] & PB2_FLOW_ACCESS_READ)) continue;
                        pb2_tile_t* tile = &w.tiles[t.tile[f]];
                        if (threadIdx.x == 0) sh.need = needs_stage_in(tile, t.access[f]);
                        __syncthreads();
                        if (sh.need) { stage_in_flow(stage_ctx(w), tile, t.access[f], &sh.decide); fence_proxy_async(); }
                        __syncthreads();
                    }
                }
            }
            if (threadIdx.x < (int)(sizeof(Job) / 4)) {          // copy the job into the peer CTA's shared memory
                const uint32_t v = reinterpret_cast<const uint32_t*>(&sh.job)[threadIdx.x];
                st_cluster_u32(mapa(smem_u32(reinterpret_cast<uint32_t*>(&sh.job) + threadIdx.x), 1), v);
            }
        }
        cluster_sync_all();
        const Job job = sh.job;
        if (job.stop) break;

        if (job.is_gemm) {
            const int kblocks = (job.K + BK - 1) / BK;
            const int nhalves = (job.Nj + 255) / 256;
            if (warp == 1) {
                // ===== TMA producer (both CTAs): my 128 rows of A, my half of each N=256 block of B
                if (lane == 0) {
                    fence_proxy_async();
                    const uint32_t leader_full0 = smem_u32(&sh.full[0]) & 0xFEFFFFFFu;    // same offset in CTA 0
                    for (int s = 0; s < job.seg_count; ++s) {
                        const GSeg sg = g.segs[job.seg_begin + s];
                        const CUtensorMap* mapA = &g.tmaps[sg.tileA];
                        const CUtensorMap* mapB = &g.tmaps[sg.tileB];
                        if (s + 1 < job.seg_count) {        // the next member's descriptors: fetch them now, not on first use
                            const GSeg nx = g.segs[job.seg_begin + s + 1];
                            asm volatile("prefetch.tensormap [%0];" :: "l"(&g.tmaps[nx.tileA]) : "memory");
                            asm volatile("prefetch.tensormap [%0];" :: "l"(&g.tmaps[nx.tileB]) : "memory");
                        }
                        for (int kb = 0; kb < kblocks; ++kb) {
                            mbar_wait(&sh.empty[p_stage], p_phase ^ 1);
                            uint8_t* sa = smem + p_stage * kStage2;
                            const uint32_t bar = leader_full0 + p_stage * 8;
                            if (g.debug & 1) {
                                if (leader) mbar_arrive(&sh.full[p_stage]); else mbar_arrive_cluster(bar);
                            } else {
                            if (leader) mbar_expect_tx(&sh.full[p_stage], (uint32_t)(kAStage + nhalves * kBHalf) * 2);
                            else        mbar_arrive_cluster(bar);
                            tma_load_2sm(sa, mapA, bar, kb * BK, job.m0 + (int)rank * 128);
                            for (int h = 0; h < nhalves; ++h) {
                                const int nh = min(256, job.Nj - 256 * h);
                                tma_load_2sm(sa + kAStage + h * kBHalf, mapB, bar, kb * BK, job.n0 + 256 * h + (int)rank * (nh / 2));
                            }
                            }
                            if (++p_stage == kStages2) { p_stage = 0; p_phase ^= 1; }
                        }
                    }
                }
            } else if (warp == 2) {
                // ===== MMA issuer (leader CTA only, one thread, for the pair)
                if (leader && lane == 0) {
                    for (int s = 0; s < job.seg_count; ++s) {
                        for (int kb = 0; kb < kblocks; ++kb) {
                            mbar_wait(&sh.full[c_stage], c_phase);
                            tc_fence_after();
                            const uint32_t sa = smem_u32(smem + c_stage * kStage2);
                            const uint64_t da = make_desc(sa);
                            for (int h = 0; h < nhalves && !(g.debug & 2); ++h) {
                                const int nh = min(256, job.Nj - 256 * h);
                                const uint32_t idesc = make_idesc(256, nh);
                                const uint64_t db = make_desc(sa + kAStage + h * kBHalf);
#pragma unroll
                                for (int k = 0; k < BK / UK; ++k)
                                    tc_mma2(tmem_base + h * 256, da + (uint64_t)(k * UK * 2 >> 4), db + (uint64_t)(k * UK * 2 >> 4), idesc,
                                            (s | kb | k) != 0 ? 1u : 0u);
                            }
                            tc_commit2(&sh.empty[c_stage]);
                            if (++c_stage == kStages2) { c_stage = 0; c_phase ^= 1; }
                        }
                    }
                    tc_commit2(&sh.tmem_full);
                }
                if (!leader) {   // keep the consumer-side pipeline state in step with the leader
                    const int n = job.seg_count * kblocks;
                    for (int i = 0; i < n; ++i) if (++c_stage == kStages2) { c_stage = 0; c_phase ^= 1; }
                }
            } else if (warp >= 4) {
                // ===== epilogue (both CTAs): C rows m0 + rank*128 + quadrant*32 + lane
                const int q = warp & 3;
                uint8_t* Cbase = reinterpret_cast<uint8_t*>(w.tiles[job.tileC].dev_ptr);
                const int row = job.m0 + (int)rank * 128 + q * 32 + lane;
                // these warps idle during the main loop: pull this thread's C row into L2 now, so that the
                // read-modify-write below does not pay DRAM latency sixteen times in a row
                if (row < job.M)
                    for (int b = 0; b < job.Nj * 2; b += 128)
                        asm volatile("prefetch.global.L2 [%0];" :: "l"(Cbase + ((size_t)row * job.N + job.n0) * 2 + b));
                mbar_wait(&sh.tmem_full, tfull_phase);
                tc_fence_after();
                const uint32_t taddr = tmem_base + ((uint32_t)(q * 32) << 16);
                const int nchunks = (g.debug & 4) ? 0 : (job.Nj + 31) / 32;
                const bool row_ok = row < job.M;
                uint4 cv[4];
                auto load_c = [&](int c) {
                    const int col0 = c * 32;
                    const uint4* cp = reinterpret_cast<const uint4*>(Cbase + ((size_t)row * job.N + job.n0 + col0) * 2);
#pragma unroll
                    for (int v = 0; v < 4; ++v) cv[v] = (row_ok && col0 + v * 8 < job.Nj) ? ld_stream(cp + v) : make_uint4(0, 0, 0, 0);
                };
                load_c(0);
#pragma unroll 1
                for (int c = 0; c < nchunks; ++c) {
                    uint32_t acc[32];
                    tc_ld_32x32b_x32(taddr + c * 32, acc);
                    uint4 cur[4];
#pragma unroll
                    for (int v = 0; v < 4; ++v) cur[v] = cv[v];
                    if (c + 1 < nchunks) load_c(c + 1);           // next chunk's C values are in flight during this one
                    tc_wait_ld();
                    const int col0 = c * 32;
                    if (row_ok) {
                        uint4* cp = reinterpret_cast<uint4*>(Cbase + ((size_t)row * job.N + job.n0 + col0) * 2);
#pragma unroll
                        for (int v = 0; v < 4; ++v) {
                            if (col0 + v * 8 < job.Nj) {
                                uint4 o;
                                o.x = pack_bf16(bf16_lo(cur[v].x) + __uint_as_float(acc[v * 8 + 0]), bf16_hi(cur[v].x) + __uint_as_float(acc[v * 8 + 1]));
                                o.y = pack_bf16(bf16_lo(cur[v].y) + __uint_as_float(acc[v * 8 + 2]), bf16_hi(cur[v].y) + __uint_as_float(acc[v * 8 + 3]));
                                o.z = pack_bf16(bf16_lo(cur[v].z) + __uint_as_float(acc[v * 8 + 4]), bf16_hi(cur[v].z) + __uint_as_float(acc[v * 8 + 5]));
                                o.w = pack_bf16(bf16_lo(cur[v].w) + __uint_as_float(acc[v * 8 + 6]), bf16_hi(cur[v].w) + __uint_as_float(acc[v * 8 + 7]));
                                st_stream(cp + v, o);
                            }
                        }
                    }
                }
                tc_fence_before();
                fence_proxy_async();
            }
            tfull_phase ^= 1;      // one accumulator hand-over per GEMM job, tracked by every thread
        } else if (leader) {
            // ---------------- a non-GEMM member of the DAG (e.g. a panel stand-in): the leader CTA runs it in place
            const pb2_task_t& t = sh.task;
            BodyArgs a;
            for (int f = 0; f < PB2_MAX_FLOWS; ++f) {
                const bool has = f < t.nb_flows && t.tile[f] >= 0;
                a.flow[f] = has ? w.tiles[t.tile[f]].dev_ptr : nullptr;
                a.bytes[f] = has ? w.tiles[t.tile[f]].bytes : 0;
            }
            a.elem0 = 0; a.part = 0;
            a.iparam[0] = t.iparam[0]; a.iparam[1] = t.iparam[1]; a.iparam[2] = t.iparam[2]; a.fparam = t.fparam;
            const unsigned long long r = run_hbm_body(t.body, a, sh.red);
            // as in the v1 kernel, an unknown body id does not abort the window
            if (threadIdx.x == 0) record_result(w, t.body, g.segs[job.seg_begin].task, 0, 1, r);
            fence_proxy_async();
            for (int f = 0; f < t.nb_flows; ++f)
                if (pushes_out(t, f)) pushout(w.ctl, w.tiles[t.tile[f]].src_ptr, w.tiles[t.tile[f]].dev_ptr, w.tiles[t.tile[f]].bytes);
        }
        __threadfence();
        cluster_sync_all();          // every store of the part (both CTAs) is done and visible

        // ---------------- part complete: pushout of this part's C rows, then unit retirement by the last part
        if (leader) {
            if (job.is_gemm && job.pushout) {
                pb2_tile_t* tile = &w.tiles[job.tileC];
                const size_t row_bytes = (size_t)job.N * 2;
                const int rows = min(256, job.M - job.m0);
                if (rows > 0 && job.Nj == job.N) {
                    pushout(w.ctl, reinterpret_cast<uint8_t*>(tile->src_ptr) + (size_t)job.m0 * row_bytes,
                            reinterpret_cast<const uint8_t*>(tile->dev_ptr) + (size_t)job.m0 * row_bytes, (size_t)rows * row_bytes);
                } else if (rows > 0) {
                    // a column block of a tile wider than 512: row segments
                    for (int r = 0; r < rows; ++r) {
                        const size_t o = (size_t)(job.m0 + r) * row_bytes + (size_t)job.n0 * 2;
                        cta_copy<false>(reinterpret_cast<uint8_t*>(tile->src_ptr) + o, reinterpret_cast<const uint8_t*>(tile->dev_ptr) + o, (size_t)job.Nj * 2);
                    }
                    if (threadIdx.x == 0) atomicAdd(&w.ctl->bytes_d2h.v, (unsigned long long)rows * (unsigned long long)job.Nj * 2ull);
                }
                __syncthreads();
            }
            if (warp == 0) {
                int last = 0;
                if (lane == 0) { __threadfence(); last = atomicSub(&g.parts_left[job.unit], 1) == 1; }
                last = __shfl_sync(0xffffffffu, last, 0);
                if (last) { __threadfence(); retire_unit_warp(g, g.units[job.unit], job.unit); }
            }
        }
    }

    tc_fence_before();
    cluster_sync_all();
    if (warp == 2) {
        asm volatile("tcgen05.dealloc.cta_group::2.sync.aligned.b32 %0, %1;" :: "r"(tmem_base), "r"(kTmemCols) : "memory");
    }
}

static inline int pb2_gemm2_launch(const Win2Dev& g, int nworkers_ctas, cudaStream_t stream) {
    static bool attr_set = false;
    if (!attr_set) {
        if (cudaFuncSetAttribute(pb2_engine_gemm2_kernel, cudaFuncAttributeMaxDynamicSharedMemorySize, gemm2::kSmem2) != cudaSuccess) return PB2_ERR_DEVICE;
        attr_set = true;
    }
    const int grid = nworkers_ctas & ~1;       // whole clusters
    if (grid < 2) return PB2_ERR_BAD_PARAM;
    pb2_engine_gemm2_kernel<<<grid, gemm2::kThreads2, gemm2::kSmem2, stream>>>(g);
    return cudaGetLastError() == cudaSuccess ? PB2_SUCCESS : PB2_ERR_DEVICE;
}

}  // namespace pb2
