// pb2_engine.cu -- the persistent sm_100a DAG-execution kernel and its C ABI (include/pb2_engine.h).
//
// What it replaces in the reference (file:line in /root/reference):
//   * the manager thread's check_in_deps / exec / get_data_out / complete_task loop,
//     parsec/mca/device/device_gpu.c:3438-3562, and the 3-stage stream ring of
//     parsec_device_progress_stream (:2592-2731): here every CTA is a worker that pops a task id
//     from a device-resident ring, stages in, runs the body and retires the task itself;
//   * parsec_device_data_stage_in / parsec_default_gpu_stage_in (:1799, :1623): the worker that first
//     touches an INVALID tile moves it (host-pinned or peer memory -> its HBM slot) inside the kernel;
//   * parsec_release_dep_fct -> parsec_release_local_OUT_dependencies -> update_deps_with_counter /
//     _with_mask (parsec/parsec.c:1836, :1749, :1609, :1656): warp 0 of the worker walks the task's
//     out-edges, one lane per edge, atomically decrements / ORs the successor's dependency word and
//     pushes newly-ready successors into the ring with one warp-aggregated tail reservation;
//   * parsec_device_kernel_pop / _epilog (:2943, :3179): pushout flows are copied back to their
//     home location by the worker, versions are bumped for WRITE flows, the task id is appended to the
//     retire log that the host drains in batches to run __parsec_complete_execution bookkeeping.
#include <cuda_runtime.h>
#include <cuda.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <string>
#include <vector>
#include <mutex>
#include <map>
#include <algorithm>

#include "../../include/pb2_engine.h"
#include "pb2_sched.cuh"
#include "pb2_worker.cuh"
#include "pb2_gemm.cuh"
#include "pb2_gemm2.cuh"

namespace pb2 {

// ---------------------------------------------------------------------------------------------
// reset: (re)arm one window.  dep words, ring, counters, tile table.
// ---------------------------------------------------------------------------------------------
__global__ void pb2_window_reset_kernel(WinDev w, const pb2_tile_t* tiles_init,
                                        const int32_t* ready, int32_t nready) {
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t gsz = (size_t)gridDim.x * blockDim.x;
    for (size_t i = gid; i < (size_t)w.ntasks; i += gsz) {
        const pb2_task_t& t = w.tasks[i];
        // counter mode counts down from the goal (parsec.c:1625-1633); mask mode ORs up from 0 (:1693-1703)
        w.dep[i] = (t.flags & PB2_TASK_DEPS_MASK) ? 0 : t.dep_goal;
        if (w.parts_left) w.parts_left[i] = task_nparts(w, (int32_t)i);
        w.start_seq[i] = 0; w.end_seq[i] = 0; w.result[i] = 0; w.worker[i] = -1; w.retire_log[i] = -1;
        for (int f = 0; f < PB2_MAX_FLOWS; ++f) w.seen_version[i * PB2_MAX_FLOWS + f] = 0;
    }
    for (size_t i = gid; i <= (size_t)w.cap_mask; i += gsz)
        w.ring[i] = (i < (size_t)nready) ? ready[i] : kEmpty;
    for (size_t i = gid; i < (size_t)w.ntiles; i += gsz) {
        w.tiles[i] = tiles_init[i];
        if (w.slice_claim) reset_tile_slices(w, i);
    }
    if (gid == 0) {
        w.ctl->head.v = 0; w.ctl->tail.v = (unsigned long long)nready; w.ctl->evt.v = 0;
        w.ctl->retired.v = 0; w.ctl->done.v = (w.ntasks == 0) ? kDoneOK : 0;
        w.ctl->progress_ns.v = globaltimer_ns();
        w.ctl->bytes_h2d.v = 0; w.ctl->bytes_d2d.v = 0; w.ctl->bytes_d2h.v = 0;
        w.ctl->stage_ins.v = 0; w.ctl->body_errors.v = 0;
    }
}

// ---------------------------------------------------------------------------------------------
// the persistent engine kernel, HBM-bound bodies
// ---------------------------------------------------------------------------------------------
// 64-thread workers, 12 per SM (<= 80 registers, no spills): a worker keeps PB2_CHECK_UNROLL = 16 (read-only bodies) or
// PB2_UNROLL = 4 (read-modify-write bodies) 16-byte requests per thread in flight -- bytes in flight per SM are what
// the L2-bound Ex05 window responds to (r02 sweep in DESIGN.md: 20 x 4 requests 0.76 ms, 20 x 6 0.62 ms, 12 x 16 0.60 ms),
// while many small workers still overlap the serial pop / release sections of one task with the streaming of the others.
// What one worker does with a task is in pb2_worker.cuh (shared with the streaming kernel of pb2_stream.cu).
#ifndef PB2_HBM_MINB
#define PB2_HBM_MINB 12
#endif
#ifndef PB2_HBM_THREADS
#define PB2_HBM_THREADS 64
#endif
__global__ void __launch_bounds__(PB2_HBM_THREADS, PB2_HBM_MINB)
pb2_engine_hbm_kernel(WinDev w) {
    __shared__ TaskSmem s;
    __shared__ BulkSmem bulk;
    if (threadIdx.x == 0) bulk_init(bulk);
    __syncthreads();

    for (;;) {
        if (threadIdx.x == 0) {
            const int32_t e = pop_task(w);
            if (e != kEmpty) __threadfence();   // acquire side: order the tile reads below after the slot read
            s.entry = e;
        }
        __syncthreads();
        const int32_t entry = s.entry;
        if (entry == kEmpty) break;
        const int32_t id = w.nparts ? PB2_ENT_TASK(entry) : entry;
        const int part = w.nparts ? PB2_ENT_PART(entry) : 0;
        if (threadIdx.x < 4) reinterpret_cast<uint4*>(&s.task)[threadIdx.x] =
            __ldg(reinterpret_cast<const uint4*>(&w.tasks[id]) + threadIdx.x);
        if (threadIdx.x == 0 && part == 0) {
            w.start_seq[id] = (uint32_t)atomicAdd(&w.ctl->evt.v, 1ull);
            w.worker[id] = (int32_t)blockIdx.x;
        }
        __syncthreads();
        const int nparts = task_nparts(w, id);
        const unsigned long long r = run_task_part(w, s, &bulk, id, part, nparts);

        if (threadIdx.x < 32) {
            __threadfence();   // release side: the body's stores (all threads, ordered by the barrier) become
                               // visible before any successor can observe its dependency word / ring slot
            if (threadIdx.x == 0) {
                const pb2_task_t& t = s.task;
                store_result(w, t, id, part, nparts, r);
                // the last part to finish retires the task (fence / RMW chain orders every part's stores before it)
                int last = 1;
                if (nparts > 1) { last = atomicSub(&w.parts_left[id], 1) == 1; __threadfence(); }
                s.window_done = 0; s.last = last;
                if (last) {
                    s.window_done = retire_task(w, t, id) ? 1 : 0;
                    __threadfence();
                }
            }
            __syncwarp();
        }
        if (w.ps_begin != nullptr) {
            // tiles this task wrote for readers on other GPUs go out before those readers are released
            __syncthreads();
            if (s.last && w.ps_begin[id + 1] > w.ps_begin[id]) push_written_tiles(w.tiles, w.ctl, w.ps_begin, w.ps, id, &bulk);
        }
        if (threadIdx.x < 32) {
            if (s.last) { release_successors_warp(w, s.task); release_remote_warp(w, id); }
            if (threadIdx.x == 0 && s.window_done) finish_window(w);
        }
        __syncthreads();
    }
}

// re-arm the unit-level scheduling state of a v2 GEMM window (after pb2_window_reset_kernel re-armed the rest)
__global__ void pb2_window2_reset_kernel(Win2Dev g, const int32_t* ready_entries, int32_t nentries) {
    const size_t gid = (size_t)blockIdx.x * blockDim.x + threadIdx.x;
    const size_t gsz = (size_t)gridDim.x * blockDim.x;
    for (size_t i = gid; i < (size_t)g.nunits; i += gsz) { g.udep[i] = g.units[i].dep_goal; g.parts_left[i] = g.units[i].nparts; }
    for (size_t i = gid; i <= (size_t)g.w.cap_mask; i += gsz) g.w.ring[i] = (i < (size_t)nentries) ? ready_entries[i] : kEmpty;
    if (gid == 0) g.w.ctl->tail.v = (unsigned long long)nentries;
}

// The same bodies as a stand-alone kernel on a caller's stream: what a BODY [type=CUDA] enqueues when it runs under a
// device module that is not ours (the reference's stream engine), see pb2_body_launch.
struct LaunchArgs { void* ptr[PB2_MAX_FLOWS]; unsigned long long bytes[PB2_MAX_FLOWS]; int32_t iparam[3]; float fparam; int32_t body; int32_t nb; };
__device__ unsigned long long g_body_launch_errors;
__global__ void __launch_bounds__(256)
pb2_body_launch_kernel(LaunchArgs la) {
    __shared__ uint32_t red[32];
    __shared__ BodyArgs a;
    // every flow is cut at the same 16-byte aligned offsets, one slice per CTA
    unsigned long long widest = 0;
    for (int f = 0; f < la.nb; ++f) widest = la.bytes[f] > widest ? la.bytes[f] : widest;
    const unsigned long long per = ((widest / gridDim.x) + 15ull) & ~15ull;
    if (threadIdx.x == 0) {
        for (int f = 0; f < PB2_MAX_FLOWS; ++f) {
            const unsigned long long b = f < la.nb ? la.bytes[f] : 0;
            const unsigned long long off = per * blockIdx.x < b ? per * blockIdx.x : b;
            const unsigned long long len = (blockIdx.x == gridDim.x - 1) ? b - off : (off + per <= b ? per : b - off);
            a.flow[f] = f < la.nb ? reinterpret_cast<uint8_t*>(la.ptr[f]) + off : nullptr;
            a.bytes[f] = (uint32_t)len;
            if (f == 0) a.elem0 = (uint32_t)(off >> 2);
        }
        a.part = blockIdx.x; a.iparam[0] = la.iparam[0]; a.iparam[1] = la.iparam[1]; a.iparam[2] = la.iparam[2]; a.fparam = la.fparam;
    }
    __syncthreads();
    const unsigned long long r = run_hbm_body(la.body, a, red);
    if (threadIdx.x == 0 && (la.body == PB2_BODY_CHECK_I32 || la.body == PB2_BODY_CHECK_F32) && (r >> 32))
        atomicAdd(&g_body_launch_errors, r >> 32);
}

struct CopyDesc { void* dst; const void* src; unsigned long long bytes; };

__global__ void __launch_bounds__(256, 4)
pb2_copy_batch_kernel(const CopyDesc* __restrict__ d, int32_t n) {
    for (int32_t i = blockIdx.x; i < n; i += gridDim.x) {
        const CopyDesc c = d[i];
        cta_copy<true>(c.dst, c.src, (size_t)c.bytes);
    }
}

}  // namespace pb2

// =============================================================================================
// Host side
// =============================================================================================
using namespace pb2;

#include "pb2_engine_priv.hpp"

struct pb2_window_s {
    pb2_engine_t* e = nullptr;
    int kind = 0;
    int32_t ntasks = 0, nsucc = 0, ntiles = 0, nready = 0, nready_entries = 0;
    WinDev d{};
    pb2_task_t* d_tasks = nullptr;
    uint32_t* d_succ = nullptr;
    pb2_tile_t* d_tiles = nullptr;
    pb2_tile_t* d_tiles_init = nullptr;
    int32_t* d_ready = nullptr;
    cudaEvent_t ev0 = nullptr, ev1 = nullptr, ev2 = nullptr;
    CUtensorMap* d_tmaps = nullptr;     // kind 1: one 2-D bf16 tensor map per tile (box 64 x 128, 128B swizzle)
    bool v2 = false;                    // kind 1 executed by the CTA-pair kernel on units
    Win2Dev g{};
    int32_t* d_ready_entries = nullptr;
    int32_t nentries = 0;
    bool launched = false;
    bool shared = false;
    std::vector<int32_t> task_entry;          // per task: its ring entry with (parts - 1) in the part field
    std::vector<void*> allocs;
    std::vector<void*> peer_ptrs;
    std::vector<pb2_tile_t*> peer_tiles;     // per rank: its tile table as mapped here (nullptr: none / self)
    std::vector<int32_t> peer_ntiles;
};

template <class T>
static int dev_alloc_copy(pb2_window_t* w, T** dptr, const T* host, size_t n) {
    pb2_engine_t* e = w->e;
    void* p = nullptr;
    // stream-ordered pool allocation: after the first window of a size class this costs microseconds, whereas
    // cudaMalloc/cudaFree next to a 170 GB slab cost hundreds of microseconds each and synchronise the device
    if (w->shared) { PB2_CUDA(e, cudaMalloc(&p, (n ? n : 1) * sizeof(T))); }     // IPC needs cudaMalloc memory
    else PB2_CUDA(e, cudaMallocAsync(&p, (n ? n : 1) * sizeof(T), e->up_stream));
    w->allocs.push_back(p);
    if (host && n) PB2_CUDA(e, cudaMemcpyAsync(p, host, n * sizeof(T), cudaMemcpyHostToDevice, e->up_stream));
    *dptr = reinterpret_cast<T*>(p);
    return PB2_SUCCESS;
}

static int validate_window(pb2_engine_t* e, int kind, const pb2_task_t* tasks, int32_t ntasks,
                           const uint32_t* succ, int32_t nsucc, int32_t ntiles,
                           const int32_t* ready, int32_t nready) {
    if (ntasks < 0 || nsucc < 0 || ntiles < 0 || nready < 0) return PB2_ERR_BAD_PARAM;
    if (ntasks >= (1 << 27)) return PB2_ERR_VALUE_OUT_OF_BOUNDS;
    // ready-ring entries of the HBM kernel carry the task id in 22 bits (PB2_ENT_MAKE: part << 22 | task)
    if (kind == 0 && ntasks >= (1 << 22)) { e->last_error = "an HBM window holds at most 4194303 tasks (22-bit task id in the ready ring)"; return PB2_ERR_VALUE_OUT_OF_BOUNDS; }
    for (int32_t i = 0; i < ntasks; ++i) {
        const pb2_task_t& t = tasks[i];
        if (t.nb_flows > PB2_MAX_FLOWS) { e->last_error = "task with more than PB2_MAX_FLOWS flows"; return PB2_ERR_BAD_PARAM; }
        if (t.succ_count < 0 || t.succ_begin < 0 || (int64_t)t.succ_begin + t.succ_count > nsucc) {
            e->last_error = "successor range out of bounds"; return PB2_ERR_VALUE_OUT_OF_BOUNDS; }
        for (int f = 0; f < t.nb_flows; ++f)
            if (t.tile[f] >= ntiles) { e->last_error = "tile id out of bounds"; return PB2_ERR_VALUE_OUT_OF_BOUNDS; }
        if (t.body >= PB2_BODY_MAX || t.body == PB2_BODY_USER) { e->last_error = "unknown body id"; return PB2_ERR_BAD_PARAM; }
        if (kind == 0 && t.body == PB2_BODY_GEMM_BF16) {
            e->last_error = "GEMM body in an HBM-kind window (use kind 1)"; return PB2_ERR_BAD_PARAM; }
    }
    for (int32_t i = 0; i < nsucc; ++i)
        if (PB2_SUCC_TASK(succ[i]) >= ntasks) { e->last_error = "successor id out of bounds"; return PB2_ERR_VALUE_OUT_OF_BOUNDS; }
    for (int32_t i = 0; i < nready; ++i)
        if (ready[i] < 0 || ready[i] >= ntasks) { e->last_error = "ready id out of bounds"; return PB2_ERR_VALUE_OUT_OF_BOUNDS; }
    return PB2_SUCCESS;
}


// One tensor map per tile used as a GEMM operand: global tensor [rows][inner] bf16, row pitch inner*2 bytes,
// box {64 (inner, 128 bytes), 128 rows}, 128-byte swizzle: exactly the K-major SWIZZLE_128B smem layout the
// UMMA descriptors in pb2_gemm.cuh describe.  OOB rows/columns of ragged tiles are zero-filled by TMA.
typedef CUresult (*pb2_encode_tiled_fn)(CUtensorMap*, CUtensorMapDataType, cuuint32_t, void*, const cuuint64_t*,
                                        const cuuint64_t*, const cuuint32_t*, const cuuint32_t*, CUtensorMapInterleave,
                                        CUtensorMapSwizzle, CUtensorMapL2promotion, CUtensorMapFloatOOBfill);

static int build_tensor_maps(pb2_window_t* w, const pb2_task_t* tasks, int32_t ntasks,
                             const pb2_tile_t* tiles, int32_t ntiles) {
    pb2_engine_t* e = w->e;
    static pb2_encode_tiled_fn encode = nullptr;
    if (!encode) {
        void* fn = nullptr;
        cudaDriverEntryPointQueryResult q;
        PB2_CUDA(e, cudaGetDriverEntryPoint("cuTensorMapEncodeTiled", &fn, cudaEnableDefault, &q));
        if (!fn || q != cudaDriverEntryPointSuccess) { e->last_error = "cuTensorMapEncodeTiled not available"; return PB2_ERR_NOT_SUPPORTED; }
        encode = reinterpret_cast<pb2_encode_tiled_fn>(fn);
    }
    std::vector<int32_t> rows(ntiles, 0), inner(ntiles, 0);
    for (int32_t i = 0; i < ntasks; ++i) {
        const pb2_task_t& t = tasks[i];
        if (t.body != PB2_BODY_GEMM_BF16) continue;
        if (t.nb_flows < 3 || t.tile[0] < 0 || t.tile[1] < 0 || t.tile[2] < 0) { e->last_error = "GEMM task needs 3 data flows"; return PB2_ERR_BAD_PARAM; }
        const int M = t.iparam[0], N = t.iparam[1], K = t.iparam[2];
        if (M <= 0 || N <= 0 || K <= 0 || (K % 8) || (N % 8)) { e->last_error = "GEMM tile: need M,N,K > 0, K % 8 == 0, N % 8 == 0"; return PB2_ERR_NOT_SUPPORTED; }
        const int32_t need[2][2] = {{M, K}, {N, K}};
        for (int f = 0; f < 2; ++f) {
            const int32_t id = t.tile[f];
            if (rows[id] == 0) { rows[id] = need[f][0]; inner[id] = need[f][1]; }
            else if (rows[id] != need[f][0] || inner[id] != need[f][1]) { e->last_error = "tile used with two different operand shapes"; return PB2_ERR_NOT_SUPPORTED; }
            if ((uint64_t)need[f][0] * need[f][1] * 2 > tiles[id].bytes) { e->last_error = "GEMM operand larger than its tile"; return PB2_ERR_VALUE_OUT_OF_BOUNDS; }
        }
        if ((uint64_t)M * N * 2 > tiles[t.tile[2]].bytes) { e->last_error = "GEMM C larger than its tile"; return PB2_ERR_VALUE_OUT_OF_BOUNDS; }
    }
    std::vector<CUtensorMap> maps(ntiles ? ntiles : 1);
    memset(maps.data(), 0, maps.size() * sizeof(CUtensorMap));
    for (int32_t i = 0; i < ntiles; ++i) {
        if (rows[i] == 0) continue;
        if ((uintptr_t)tiles[i].dev_ptr & 15) { e->last_error = "GEMM tile not 16-byte aligned"; return PB2_ERR_BAD_PARAM; }
        cuuint64_t gdim[2] = {(cuuint64_t)inner[i], (cuuint64_t)rows[i]};
        cuuint64_t gstride[1] = {(cuuint64_t)inner[i] * 2};
        cuuint32_t box[2] = {64, 128};
        cuuint32_t estr[2] = {1, 1};
        CUresult r = encode(&maps[i], CU_TENSOR_MAP_DATA_TYPE_BFLOAT16, 2, tiles[i].dev_ptr, gdim, gstride, box, estr,
                            CU_TENSOR_MAP_INTERLEAVE_NONE, CU_TENSOR_MAP_SWIZZLE_128B,
                            CU_TENSOR_MAP_L2_PROMOTION_L2_256B, CU_TENSOR_MAP_FLOAT_OOB_FILL_NONE);
        if (r != CUDA_SUCCESS) { e->last_error = "cuTensorMapEncodeTiled failed"; return PB2_ERR_DEVICE; }
    }
    return dev_alloc_copy(w, &w->d_tmaps, maps.data(), maps.size());
}


// ---------------------------------------------------------------------------------------------
// v2 GEMM windows: group tasks into units (fused k-chains), see pb2_gemm2.cuh
// ---------------------------------------------------------------------------------------------
static int build_gemm2_units(pb2_window_t* w, const pb2_task_t* tasks, int32_t ntasks, const uint32_t* succ,
                             const int32_t* ready, int32_t nready, bool fuse, uint32_t* ring_cap_needed,
                             const int32_t* rs_begin) {
    std::vector<int32_t> indeg((size_t)ntasks, 0), cpred((size_t)ntasks, -1), ccons((size_t)ntasks, 0), next((size_t)ntasks, -1);
    auto is_gemm = [&](int32_t t) { return tasks[t].body == PB2_BODY_GEMM_BF16; };
    for (int32_t u = 0; u < ntasks; ++u)
        for (int32_t e = 0; e < tasks[u].succ_count; ++e) {
            const uint32_t s = succ[tasks[u].succ_begin + e];
            const int32_t t = PB2_SUCC_TASK(s);
            indeg[t]++;
            if (PB2_SUCC_FLOW(s) == 2 && is_gemm(u) && is_gemm(t) && tasks[u].tile[2] == tasks[t].tile[2]) { ccons[u]++; cpred[t] = u; }
        }
    // A window that peers release into: the tasks' dependency goals (counter mode, set by the partitioner) also
    // count the in-edges that come from other GPUs; the local CSR does not show them.
    if (w->shared)
        for (int32_t t = 0; t < ntasks; ++t) {
            const int32_t need = (tasks[t].flags & PB2_TASK_DEPS_MASK) ? __builtin_popcount((unsigned)tasks[t].dep_goal) : tasks[t].dep_goal;
            if (need < indeg[t]) { w->e->last_error = "dependency goal smaller than the in-window in-degree"; return PB2_ERR_BAD_PARAM; }
            indeg[t] = need;
        }
    if (fuse)
        for (int32_t t = 0; t < ntasks; ++t) {
            const int32_t u = cpred[t];
            if (u < 0 || indeg[t] != 1 || ccons[u] != 1) continue;                 // the chain link must be t's only missing input
            if (rs_begin && rs_begin[u + 1] > rs_begin[u]) continue;               // u's result is awaited on another GPU: retire it on its own
            if (tasks[u].access[2] & PB2_FLOW_PUSHOUT) continue;                   // u's C has to reach the host: flush there
            if (memcmp(tasks[u].iparam, tasks[t].iparam, sizeof tasks[u].iparam)) continue;
            next[u] = t;
        }
    std::vector<uint8_t> has_pred((size_t)ntasks, 0);
    for (int32_t u = 0; u < ntasks; ++u) if (next[u] >= 0) has_pred[next[u]] = 1;
    std::vector<GUnit> units; std::vector<GSeg> segs; std::vector<int32_t> unit_of((size_t)ntasks, -1);
    for (int32_t h = 0; h < ntasks; ++h) {
        if (has_pred[h]) continue;
        GUnit u{}; u.seg_begin = (int32_t)segs.size(); u.dep_goal = indeg[h];
        const bool g = is_gemm(h);
        u.flags = g ? 1 : 0; u.tileC = g ? tasks[h].tile[2] : -1;
        u.M = tasks[h].iparam[0]; u.N = tasks[h].iparam[1]; u.K = tasks[h].iparam[2];
        u.nparts = g ? ((u.M + 255) / 256) * ((u.N + 511) / 512) : 1;       // 256-row x 512-column blocks of C (TMEM: 512 columns)
        if (g && ((u.N % 16) || u.nparts > 16)) return PB2_ERR_NOT_SUPPORTED;       // caller falls back to the v1 kernel
        for (int32_t t = h; t >= 0; t = next[t]) {
            unit_of[t] = (int32_t)units.size();
            segs.push_back(GSeg{t, g ? tasks[t].tile[0] : -1, g ? tasks[t].tile[1] : -1, 0});
            if (g && (tasks[t].access[2] & PB2_FLOW_PUSHOUT)) u.flags |= 2;
        }
        u.seg_count = (int32_t)segs.size() - u.seg_begin;
        units.push_back(u);
    }
    std::vector<int32_t> usucc;
    for (GUnit& u : units) {
        u.succ_begin = (int32_t)usucc.size();
        for (int32_t i = 0; i < u.seg_count; ++i) {
            const int32_t t = segs[u.seg_begin + i].task;
            for (int32_t e = 0; e < tasks[t].succ_count; ++e) {
                const int32_t d = PB2_SUCC_TASK(succ[tasks[t].succ_begin + e]);
                if (d == next[t] && PB2_SUCC_FLOW(succ[tasks[t].succ_begin + e]) == 2) continue;   // the fused link
                usucc.push_back(unit_of[d]);
            }
        }
        u.succ_count = (int32_t)usucc.size() - u.succ_begin;
    }
    std::vector<int32_t> entries;
    uint32_t total_parts = 0;
    for (const GUnit& u : units) total_parts += (uint32_t)u.nparts;
    // Ready GEMM units enter the ring in Z-order of their (locals[0], locals[1]) = C(i,j) coordinates: the ~37 units
    // that run concurrently then form a compact block of C tiles that shares A rows and B columns in L2 (a FIFO
    // ring keeps whatever order the host gives it; the reference's priority hint mt*nt*kt - i*nt + j plays the
    // same role for its sorted pending list, device_gpu.c:2169-2174).
    std::vector<std::pair<uint64_t, int32_t>> order;
    auto morton = [](uint32_t x, uint32_t y) {
        uint64_t r = 0;
        for (int b = 0; b < 16; ++b) r |= ((uint64_t)((x >> b) & 1) << (2 * b + 1)) | ((uint64_t)((y >> b) & 1) << (2 * b));
        return r;
    };
    for (int32_t i = 0; i < nready; ++i) {
        const int32_t uid = unit_of[ready[i]];
        if (units[uid].dep_goal != 0) { w->e->last_error = "ready task has in-window predecessors"; return PB2_ERR_BAD_PARAM; }
        const pb2_task_t& t = tasks[ready[i]];
        const uint64_t key = (units[uid].flags & 1) ? morton((uint32_t)t.locals[0], (uint32_t)t.locals[1]) : 0;
        order.emplace_back(key, uid);
    }
    std::stable_sort(order.begin(), order.end(), [](const std::pair<uint64_t, int32_t>& a, const std::pair<uint64_t, int32_t>& b) { return a.first < b.first; });
    for (auto& o : order)
        for (int32_t p = 0; p < units[o.second].nparts; ++p) entries.push_back((int32_t)PB2_SUCC_MAKE(o.second, p));
    *ring_cap_needed = total_parts;
    int rc;
    GUnit* d_units = nullptr; GSeg* d_segs = nullptr; int32_t* d_usucc = nullptr;
    if ((rc = dev_alloc_copy(w, &d_units, units.data(), units.size())) != PB2_SUCCESS) return rc;
    if ((rc = dev_alloc_copy(w, &d_segs, segs.data(), segs.size())) != PB2_SUCCESS) return rc;
    if ((rc = dev_alloc_copy(w, &d_usucc, usucc.data(), usucc.size())) != PB2_SUCCESS) return rc;
    if ((rc = dev_alloc_copy(w, &w->d_ready_entries, entries.data(), entries.size())) != PB2_SUCCESS) return rc;
    if ((rc = dev_alloc_copy(w, &w->g.udep, (const int32_t*)nullptr, units.size())) != PB2_SUCCESS) return rc;
    if ((rc = dev_alloc_copy(w, &w->g.parts_left, (const int32_t*)nullptr, units.size())) != PB2_SUCCESS) return rc;
    w->task_entry.assign((size_t)ntasks, -1);
    for (int32_t t = 0; t < ntasks; ++t) w->task_entry[(size_t)t] = (int32_t)PB2_SUCC_MAKE(unit_of[t], units[(size_t)unit_of[t]].nparts - 1);
    w->g.units = d_units; w->g.segs = d_segs; w->g.usucc = d_usucc; w->g.nunits = (int32_t)units.size();
    w->nentries = (int32_t)entries.size();
    return PB2_SUCCESS;
}

extern "C" {

int pb2_engine_create(pb2_engine_t** engine, int cuda_device, const pb2_engine_params_t* params) {
    if (!engine) return PB2_ERR_BAD_PARAM;
    *engine = nullptr;
    int ndev = 0;
    cudaError_t err = cudaGetDeviceCount(&ndev);
    if (err != cudaSuccess || ndev == 0) {
        // The product path never falls back to a CPU implementation: no GPU => loud failure.
        fprintf(stderr, "pb2_engine_create: no CUDA device (%s)\n", cudaGetErrorString(err));
        return PB2_ERR_DEVICE;
    }
    if (cuda_device < 0 || cuda_device >= ndev) return PB2_ERR_BAD_PARAM;
    pb2_engine_t* e = new pb2_engine_s();
    e->cuda_device = cuda_device;
    PB2_CUDA(e, cudaSetDevice(cuda_device));
    PB2_CUDA(e, cudaGetDeviceProperties(&e->prop, cuda_device));
    if (e->prop.major != 10) {
        fprintf(stderr, "pb2_engine_create: device %d is sm_%d%d; this library only carries sm_100a code\n",
                cuda_device, e->prop.major, e->prop.minor);
        delete e;
        return PB2_ERR_NOT_SUPPORTED;
    }
    pb2_engine_params_t p{};
    if (params) p = *params;
    if (p.workers_per_sm <= 0) p.workers_per_sm = PB2_HBM_MINB;
    if (p.threads <= 0 || p.threads > PB2_HBM_THREADS) p.threads = PB2_HBM_THREADS;     // the kernel is compiled for this CTA size
    p.threads = (p.threads + 31) & ~31;
    if (p.timeout_ms <= 0) p.timeout_ms = 20000;
    if (p.part_bytes == 0) p.part_bytes = 256 * 1024;
    e->params = p;
    if (const char* sl = getenv("PB2_STAGE_SLICE_BYTES")) e->stage_slice_bytes = atoi(sl);
    if (const char* sm = getenv("PB2_STAGE_MODE")) e->params.stage_mode = atoi(sm);      // 1: SIMT mover (development aid)
    PB2_CUDA(e, cudaStreamCreateWithFlags(&e->own_stream, cudaStreamNonBlocking));
    PB2_CUDA(e, cudaStreamCreateWithFlags(&e->up_stream, cudaStreamNonBlocking));
    PB2_CUDA(e, cudaStreamCreateWithFlags(&e->dma_stream, cudaStreamNonBlocking));
    PB2_CUDA(e, cudaEventCreateWithFlags(&e->dma_ev, cudaEventDisableTiming));
    e->stream = e->own_stream;
    {   // keep freed window scratch cached in the default mempool instead of returning it to the driver
        cudaMemPool_t pool;
        if (cudaDeviceGetDefaultMemPool(&pool, cuda_device) == cudaSuccess) {
            unsigned long long thr = ~0ull;
            cudaMemPoolSetAttribute(pool, cudaMemPoolAttrReleaseThreshold, &thr);
        }
    }
    int occ = 0;
    PB2_CUDA(e, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pb2_engine_hbm_kernel, p.threads, 0));
    int per_sm = occ < p.workers_per_sm ? occ : p.workers_per_sm;
    if (per_sm < 1) per_sm = 1;
    e->nworkers = e->prop.multiProcessorCount * per_sm;
    if (p.max_workers > 0 && p.max_workers < e->nworkers) e->nworkers = p.max_workers;
    e->nworkers_gemm = pb2_gemm_nworkers(e->prop.multiProcessorCount);
    if (p.max_workers > 0 && p.max_workers < e->nworkers_gemm) e->nworkers_gemm = p.max_workers;
    if (p.gemm_mode != 1 && e->nworkers_gemm < 2) e->nworkers_gemm = 2;      // v2 workers are CTA pairs
    *engine = e;
    return PB2_SUCCESS;
}

int pb2_engine_destroy(pb2_engine_t* e) {
    if (!e) return PB2_ERR_BAD_PARAM;
    cudaSetDevice(e->cuda_device);
    for (auto& kv : e->registered) cudaHostUnregister(kv.first);
    if (e->own_stream) cudaStreamDestroy(e->own_stream);
    if (e->up_stream) cudaStreamDestroy(e->up_stream);
    if (e->dma_stream) cudaStreamDestroy(e->dma_stream);
    if (e->dma_ev) cudaEventDestroy(e->dma_ev);
    delete e;
    return PB2_SUCCESS;
}

int pb2_engine_info(pb2_engine_t* e, pb2_engine_info_t* info) {
    if (!e || !info) return PB2_ERR_BAD_PARAM;
    memset(info, 0, sizeof *info);
    info->cuda_device = e->cuda_device;
    info->sm_count = e->prop.multiProcessorCount;
    info->cc_major = e->prop.major; info->cc_minor = e->prop.minor;
    info->nworkers = e->nworkers; info->nworkers_gemm = e->nworkers_gemm;
    info->can_map_host = e->prop.canMapHostMemory;
    size_t f = 0, t = 0;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    PB2_CUDA(e, cudaMemGetInfo(&f, &t));
    info->total_mem = t; info->free_mem = f;
    return PB2_SUCCESS;
}

const char* pb2_engine_last_error(pb2_engine_t* e) { return e ? e->last_error.c_str() : "null engine"; }

int pb2_engine_malloc(pb2_engine_t* e, size_t bytes, void** dev_ptr) {
    if (!e || !dev_ptr) return PB2_ERR_BAD_PARAM;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    cudaError_t err = cudaMalloc(dev_ptr, bytes ? bytes : 16);
    if (err == cudaErrorMemoryAllocation) { cudaGetLastError(); *dev_ptr = nullptr; return PB2_ERR_OUT_OF_RESOURCE; }
    PB2_CUDA(e, err);
    return PB2_SUCCESS;
}

int pb2_engine_free(pb2_engine_t* e, void* dev_ptr) {
    if (!e) return PB2_ERR_BAD_PARAM;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    PB2_CUDA(e, cudaFree(dev_ptr));
    return PB2_SUCCESS;
}

int pb2_engine_host_register(pb2_engine_t* e, void* host_ptr, size_t bytes, void** dev_alias) {
    if (!e || !host_ptr || !bytes) return PB2_ERR_BAD_PARAM;
    std::lock_guard<std::mutex> lk(e->mu);
    auto it = e->registered.find(host_ptr);
    if (it != e->registered.end()) {   // idempotent, like dc->memory_registration_status
        if (dev_alias) *dev_alias = it->second.second;
        return PB2_SUCCESS;
    }
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    cudaError_t err = cudaHostRegister(host_ptr, bytes, cudaHostRegisterPortable | cudaHostRegisterMapped);
    if (err == cudaErrorHostMemoryAlreadyRegistered) { cudaGetLastError(); }   // e.g. torch pinned memory
    else PB2_CUDA(e, err);
    void* alias = nullptr;
    PB2_CUDA(e, cudaHostGetDevicePointer(&alias, host_ptr, 0));
    if (err != cudaErrorHostMemoryAlreadyRegistered) e->registered[host_ptr] = {bytes, alias};
    if (dev_alias) *dev_alias = alias;
    return PB2_SUCCESS;
}

int pb2_engine_host_unregister(pb2_engine_t* e, void* host_ptr) {
    if (!e) return PB2_ERR_BAD_PARAM;
    std::lock_guard<std::mutex> lk(e->mu);
    auto it = e->registered.find(host_ptr);
    if (it == e->registered.end()) return PB2_ERR_NOT_FOUND;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    PB2_CUDA(e, cudaHostUnregister(host_ptr));
    e->registered.erase(it);
    return PB2_SUCCESS;
}

int pb2_engine_memcpy_h2d(pb2_engine_t* e, void* dev, const void* host, size_t bytes) {
    if (!e) return PB2_ERR_BAD_PARAM;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    PB2_CUDA(e, cudaMemcpyAsync(dev, host, bytes, cudaMemcpyHostToDevice, e->stream));
    return PB2_SUCCESS;
}

int pb2_engine_prefetch_h2d(pb2_engine_t* e, void* dev, size_t dev_pitch, const void* host, size_t host_pitch,
                            size_t width_bytes, size_t rows) {
    if (!e || !dev || !host || !width_bytes || !rows) return PB2_ERR_BAD_PARAM;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    if (rows == 1 || (dev_pitch == width_bytes && host_pitch == width_bytes))
        PB2_CUDA(e, cudaMemcpyAsync(dev, host, width_bytes * rows, cudaMemcpyHostToDevice, e->dma_stream));
    else
        PB2_CUDA(e, cudaMemcpy2DAsync(dev, dev_pitch, host, host_pitch, width_bytes, rows, cudaMemcpyHostToDevice, e->dma_stream));
    e->dma_pending = true;
    return PB2_SUCCESS;
}

int pb2_engine_memcpy_d2h(pb2_engine_t* e, void* host, const void* dev, size_t bytes) {
    if (!e) return PB2_ERR_BAD_PARAM;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    PB2_CUDA(e, cudaMemcpyAsync(host, dev, bytes, cudaMemcpyDeviceToHost, e->stream));
    PB2_CUDA(e, cudaStreamSynchronize(e->stream));
    return PB2_SUCCESS;
}

int pb2_engine_copy_batch(pb2_engine_t* e, void* const* dst, const void* const* src, const uint64_t* bytes, int32_t n) {
    if (!e || n < 0 || (n && (!dst || !src || !bytes))) return PB2_ERR_BAD_PARAM;
    if (n == 0) return PB2_SUCCESS;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    std::vector<CopyDesc> h((size_t)n);
    for (int32_t i = 0; i < n; ++i) h[i] = CopyDesc{dst[i], src[i], bytes[i]};
    CopyDesc* d = nullptr;
    PB2_CUDA(e, cudaMallocAsync(reinterpret_cast<void**>(&d), sizeof(CopyDesc) * (size_t)n, e->stream));
    PB2_CUDA(e, cudaMemcpyAsync(d, h.data(), sizeof(CopyDesc) * (size_t)n, cudaMemcpyHostToDevice, e->stream));
    PB2_CUDA(e, cudaStreamSynchronize(e->stream));     // h is pageable: make sure the staging copy is done
    const int grid = n < e->nworkers ? n : e->nworkers;
    pb2_copy_batch_kernel<<<grid, 256, 0, e->stream>>>(d, n);
    PB2_CUDA(e, cudaGetLastError());
    PB2_CUDA(e, cudaFreeAsync(d, e->stream));
    return PB2_SUCCESS;
}

int pb2_engine_ipc_export(pb2_engine_t* e, void* dev_ptr, unsigned char handle[64]) {
    if (!e || !dev_ptr || !handle) return PB2_ERR_BAD_PARAM;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    cudaIpcMemHandle_t ih;
    PB2_CUDA(e, cudaIpcGetMemHandle(&ih, dev_ptr));
    memcpy(handle, &ih, 64);
    return PB2_SUCCESS;
}
int pb2_engine_ipc_open(pb2_engine_t* e, const unsigned char handle[64], void** dev_ptr) {
    if (!e || !dev_ptr || !handle) return PB2_ERR_BAD_PARAM;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    cudaIpcMemHandle_t ih;
    memcpy(&ih, handle, 64);
    PB2_CUDA(e, cudaIpcOpenMemHandle(dev_ptr, ih, cudaIpcMemLazyEnablePeerAccess));
    return PB2_SUCCESS;
}
int pb2_engine_ipc_close(pb2_engine_t* e, void* dev_ptr) {
    if (!e || !dev_ptr) return PB2_ERR_BAD_PARAM;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    PB2_CUDA(e, cudaIpcCloseMemHandle(dev_ptr));
    return PB2_SUCCESS;
}
int pb2_engine_enable_peer(pb2_engine_t* e, int peer_cuda_device) {
    if (!e) return PB2_ERR_BAD_PARAM;
    if (peer_cuda_device == e->cuda_device) return PB2_SUCCESS;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    int can = 0;
    PB2_CUDA(e, cudaDeviceCanAccessPeer(&can, e->cuda_device, peer_cuda_device));
    if (!can) return PB2_ERR_NOT_SUPPORTED;
    cudaError_t err = cudaDeviceEnablePeerAccess(peer_cuda_device, 0);
    if (err == cudaErrorPeerAccessAlreadyEnabled) { cudaGetLastError(); return PB2_SUCCESS; }
    PB2_CUDA(e, err);
    return PB2_SUCCESS;
}

int pb2_body_launch(void* cuda_stream, int body, int nb_args, void* const* ptrs, const uint64_t* bytes,
                    const int32_t* iparam3, float fparam) {
    if (body < 0 || body >= PB2_BODY_MAX || body == PB2_BODY_GEMM_BF16 || body == PB2_BODY_USER) return PB2_ERR_NOT_SUPPORTED;
    if (nb_args < 0 || nb_args > PB2_MAX_FLOWS || (nb_args && (!ptrs || !bytes))) return PB2_ERR_BAD_PARAM;
    LaunchArgs la;
    memset(&la, 0, sizeof la);
    unsigned long long widest = 0;
    for (int f = 0; f < nb_args; ++f) {
        if (bytes[f] >= (1ull << 32)) return PB2_ERR_VALUE_OUT_OF_BOUNDS;
        la.ptr[f] = ptrs[f]; la.bytes[f] = bytes[f];
        widest = bytes[f] > widest ? bytes[f] : widest;
    }
    if (iparam3) { la.iparam[0] = iparam3[0]; la.iparam[1] = iparam3[1]; la.iparam[2] = iparam3[2]; }
    la.fparam = fparam; la.body = body; la.nb = nb_args;
    if (body == PB2_BODY_NOP) return PB2_SUCCESS;
    int grid = (int)((widest + 32767) / 32768);             // 32 KiB per CTA
    if (grid < 1) grid = 1;
    if (grid > 1184) grid = 1184;
    if (body == PB2_BODY_ADD_AT_I32) grid = 1;
    pb2_body_launch_kernel<<<grid, 256, 0, reinterpret_cast<cudaStream_t>(cuda_stream)>>>(la);
    return cudaGetLastError() == cudaSuccess ? PB2_SUCCESS : PB2_ERR_DEVICE;
}

int pb2_body_launch_errors(uint64_t* errors, int reset) {
    unsigned long long v = 0;
    if (cudaMemcpyFromSymbol(&v, g_body_launch_errors, sizeof v) != cudaSuccess) return PB2_ERR_DEVICE;
    if (errors) *errors = v;
    if (reset) { v = 0; if (cudaMemcpyToSymbol(g_body_launch_errors, &v, sizeof v) != cudaSuccess) return PB2_ERR_DEVICE; }
    return PB2_SUCCESS;
}

int pb2_engine_set_stage_slice_bytes(pb2_engine_t* e, int32_t bytes) {
    if (!e) return PB2_ERR_BAD_PARAM;
    e->stage_slice_bytes = bytes;
    return PB2_SUCCESS;
}
int pb2_engine_set_part_bytes(pb2_engine_t* e, int32_t part_bytes) {
    if (!e) return PB2_ERR_BAD_PARAM;
    e->params.part_bytes = part_bytes == 0 ? 256 * 1024 : part_bytes;
    return PB2_SUCCESS;
}
int pb2_engine_set_shared_windows(pb2_engine_t* e, int on, const int32_t* next_rs_begin) {
    if (!e) return PB2_ERR_BAD_PARAM;
    e->shared_windows = on != 0; e->next_rs_begin = on ? next_rs_begin : nullptr;
    return PB2_SUCCESS;
}

int pb2_window_task_entries(pb2_window_t* w, int32_t* entry) {
    if (!w || !entry) return PB2_ERR_BAD_PARAM;
    if ((int32_t)w->task_entry.size() != w->ntasks) return PB2_ERR_NOT_SUPPORTED;
    memcpy(entry, w->task_entry.data(), w->task_entry.size() * sizeof(int32_t));
    return PB2_SUCCESS;
}

int pb2_engine_set_stream(pb2_engine_t* e, void* cuda_stream) {
    if (!e) return PB2_ERR_BAD_PARAM;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    PB2_CUDA(e, cudaStreamSynchronize(e->stream));
    e->stream = cuda_stream ? reinterpret_cast<cudaStream_t>(cuda_stream) : e->own_stream;
    return PB2_SUCCESS;
}

void* pb2_engine_get_stream(pb2_engine_t* e) { return e ? reinterpret_cast<void*>(e->stream) : nullptr; }

int pb2_engine_synchronize(pb2_engine_t* e) {
    if (!e) return PB2_ERR_BAD_PARAM;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    PB2_CUDA(e, cudaStreamSynchronize(e->stream));
    return PB2_SUCCESS;
}

// ---------------------------------------------------------------------------------------------
// windows
// ---------------------------------------------------------------------------------------------
int pb2_window_create(pb2_engine_t* e, pb2_window_t** window, int kind,
                      const pb2_task_t* tasks, int32_t ntasks,
                      const uint32_t* succ, int32_t nsucc,
                      const pb2_tile_t* tiles, int32_t ntiles,
                      const int32_t* ready, int32_t nready) {
    if (!e || !window) return PB2_ERR_BAD_PARAM;
    *window = nullptr;
    if ((ntasks && !tasks) || (nsucc && !succ) || (ntiles && !tiles) || (nready && !ready)) return PB2_ERR_BAD_PARAM;
    int rc = validate_window(e, kind, tasks, ntasks, succ, nsucc, ntiles, ready, nready);
    if (rc != PB2_SUCCESS) return rc;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    pb2_window_t* w = new pb2_window_s();
    w->shared = e->shared_windows;
    w->e = e; w->kind = kind; w->ntasks = ntasks; w->nsucc = nsucc; w->ntiles = ntiles; w->nready = nready;
#define TRY(x) do { rc = (x); if (rc != PB2_SUCCESS) { pb2_window_destroy(w); return rc; } } while (0)
    // wide tasks (HBM windows): the parts of a task are the tile_parts of its widest tile
    std::vector<pb2_task_t> dtasks(tasks, tasks + ntasks);
    std::vector<uint16_t> nparts((size_t)ntasks, 1);
    std::vector<int32_t> entries;
    uint32_t extra_parts = 0;
    for (int32_t i = 0; i < ntasks; ++i) {
        pb2_task_t& t = dtasks[i];
        t.flags &= 0x07;
        if (kind != 0 || t.body == PB2_BODY_NOP || e->params.part_bytes < 0 || ntasks >= (1 << 22)) continue;
        uint32_t big = 0;
        for (int f = 0; f < t.nb_flows; ++f) if (t.tile[f] >= 0 && tiles[t.tile[f]].bytes > big) big = tiles[t.tile[f]].bytes;
        const int np = tile_parts(big, e->params.part_bytes);
        if (np > 1) { nparts[(size_t)i] = (uint16_t)np; extra_parts += (uint32_t)np - 1; }
    }
    for (int32_t i = 0; i < nready; ++i)
        for (int p = 0; p < (int)nparts[(size_t)ready[i]]; ++p) entries.push_back(PB2_ENT_MAKE(ready[i], p));
    w->task_entry.resize((size_t)ntasks);
    for (int32_t i = 0; i < ntasks; ++i) w->task_entry[(size_t)i] = PB2_ENT_MAKE(i, (int)nparts[(size_t)i] - 1);
    TRY(dev_alloc_copy(w, &w->d_tasks, dtasks.data(), (size_t)ntasks));
    TRY(dev_alloc_copy(w, &w->d_succ, succ, (size_t)nsucc));
    TRY(dev_alloc_copy(w, &w->d_tiles_init, tiles, (size_t)ntiles));
    TRY(dev_alloc_copy(w, &w->d_tiles, (const pb2_tile_t*)nullptr, (size_t)ntiles));
    TRY(dev_alloc_copy(w, &w->d_ready, entries.data(), entries.size()));
    w->nready_entries = (int32_t)entries.size();
    uint32_t parts_needed = 0;
    if (kind == 1) {
        TRY(build_tensor_maps(w, tasks, ntasks, tiles, ntiles));
        if (e->params.gemm_mode != 1) {
            rc = build_gemm2_units(w, tasks, ntasks, succ, ready, nready, e->params.gemm_mode == 0, &parts_needed,
                                   w->shared ? e->next_rs_begin : nullptr);
            if (rc == PB2_SUCCESS) w->v2 = true;
            else if (rc != PB2_ERR_NOT_SUPPORTED) { pb2_window_destroy(w); return rc; }     // NOT_SUPPORTED: v1 kernel
        }
    }
    const int maxw = e->nworkers > e->nworkers_gemm ? e->nworkers : e->nworkers_gemm;
    uint32_t cap = 1024;
    while (cap < (uint32_t)ntasks + extra_parts + parts_needed + (uint32_t)maxw + 2u) cap <<= 1;   // every slot is used at most once per run
    WinDev& d = w->d;
    d.tasks = w->d_tasks; d.succ = w->d_succ; d.tiles = w->d_tiles;
    TRY(dev_alloc_copy(w, &d.dep, (const int32_t*)nullptr, (size_t)ntasks));
    TRY(dev_alloc_copy(w, &d.ring, (const int32_t*)nullptr, (size_t)cap));
    TRY(dev_alloc_copy(w, &d.ctl, (const Ctl*)nullptr, 1));
    TRY(dev_alloc_copy(w, &d.retire_log, (const int32_t*)nullptr, (size_t)ntasks));
    TRY(dev_alloc_copy(w, &d.start_seq, (const uint32_t*)nullptr, (size_t)ntasks));
    TRY(dev_alloc_copy(w, &d.end_seq, (const uint32_t*)nullptr, (size_t)ntasks));
    TRY(dev_alloc_copy(w, &d.seen_version, (const uint32_t*)nullptr, (size_t)ntasks * PB2_MAX_FLOWS));
    TRY(dev_alloc_copy(w, &d.result, (const unsigned long long*)nullptr, (size_t)ntasks));
    TRY(dev_alloc_copy(w, &d.worker, (const int32_t*)nullptr, (size_t)ntasks));
    d.parts_left = nullptr; d.rs_begin = nullptr; d.rs_rank = nullptr; d.rs_target = nullptr; d.peers = nullptr; d.shared = w->shared ? 1 : 0;
    d.ps_begin = nullptr; d.ps = nullptr;
    d.slice_claim = nullptr; d.slice_done = nullptr; d.part_bytes = e->params.part_bytes;
    d.nparts = nullptr; d.remote_units = 0;
    if (kind == 0 && extra_parts) {
        uint16_t* d_np = nullptr;
        TRY(dev_alloc_copy(w, &d_np, nparts.data(), (size_t)ntasks));
        d.nparts = d_np;
        TRY(dev_alloc_copy(w, &d.parts_left, (const int32_t*)nullptr, (size_t)ntasks));
    }
    if (kind == 0) {
        // Stage-in is cut finer than tasks are: a tile that has to come from the host or a peer GPU is pulled in slices
        // of stage_slice_bytes by EVERY worker that needs it (claim bit per slice), so the readers of a tile share the
        // transfer instead of one moving it while the others wait.
        int32_t slice = e->stage_slice_bytes > 0 ? e->stage_slice_bytes : 0;
        if (e->params.part_bytes > 0 && (slice == 0 || e->params.part_bytes < slice)) slice = e->params.part_bytes;
        bool sliced = false;
        for (int32_t i = 0; i < ntiles && !sliced; ++i)
            sliced = slice > 0 && tiles[i].state != PB2_TILE_VALID && tiles[i].bytes > (uint32_t)slice;
        if (sliced || extra_parts) {
            d.part_bytes = slice > 0 ? slice : e->params.part_bytes;
            TRY(dev_alloc_copy(w, &d.slice_claim, (const uint32_t*)nullptr, (size_t)ntiles * PB2_SLICE_WORDS));
            TRY(dev_alloc_copy(w, &d.slice_done, (const uint32_t*)nullptr, (size_t)ntiles * (PB2_SLICE_WORDS + 1)));
        }
    }
    if (kind == 1 && w->v2) {
        // operand tiles that have to be staged in (host or peer GPU) are pulled in 64 KiB slices by every CTA pair
        // that needs them (the parts of one unit, the units that share an operand) instead of by one CTA alone
        d.part_bytes = 64 * 1024;
        TRY(dev_alloc_copy(w, &d.slice_claim, (const uint32_t*)nullptr, (size_t)ntiles * PB2_SLICE_WORDS));
        TRY(dev_alloc_copy(w, &d.slice_done, (const uint32_t*)nullptr, (size_t)ntiles * (PB2_SLICE_WORDS + 1)));
    }
#undef TRY
    d.cap_mask = cap - 1; d.ntasks = ntasks; d.ntiles = ntiles; d.stage_mode = e->params.stage_mode;
    d.timeout_ns = (unsigned long long)e->params.timeout_ms * 1000000ull;
    if (w->v2) { w->g.w = d; w->g.tmaps = w->d_tmaps; w->g.debug = getenv("PB2_GEMM_DEBUG") ? atoi(getenv("PB2_GEMM_DEBUG")) : 0; }
    PB2_CUDA(e, cudaEventCreate(&w->ev0));
    PB2_CUDA(e, cudaEventCreate(&w->ev1));
    PB2_CUDA(e, cudaEventCreate(&w->ev2));
    // every descriptor array is on the device when this returns (the host vectors above are temporaries); the
    // upload stream is not ordered behind the engine stream, so creating the next window does not wait for the
    // window that is running
    PB2_CUDA(e, cudaStreamSynchronize(e->up_stream));
    *window = w;
    return PB2_SUCCESS;
}

int pb2_window_destroy(pb2_window_t* w) {
    if (!w) return PB2_ERR_BAD_PARAM;
    cudaSetDevice(w->e->cuda_device);
    if (w->launched) cudaEventSynchronize(w->ev2);        // this window only: a later one may be running
    for (void* p : w->peer_ptrs) cudaIpcCloseMemHandle(p);
    for (void* p : w->allocs) { if (w->shared) cudaFree(p); else cudaFreeAsync(p, w->e->stream); }
    if (w->ev0) cudaEventDestroy(w->ev0);
    if (w->ev1) cudaEventDestroy(w->ev1);
    if (w->ev2) cudaEventDestroy(w->ev2);
    delete w;
    return PB2_SUCCESS;
}

int pb2_window_arm(pb2_window_t* w) {
    if (!w) return PB2_ERR_BAD_PARAM;
    pb2_engine_t* e = w->e;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    if (e->dma_pending) {                       // prefetches queued for this window land before its first worker starts
        PB2_CUDA(e, cudaEventRecord(e->dma_ev, e->dma_stream));
        PB2_CUDA(e, cudaStreamWaitEvent(e->stream, e->dma_ev, 0));
        e->dma_pending = false;
    }
    PB2_CUDA(e, cudaEventRecord(w->ev0, e->stream));
    {
        const int threads = 256;
        size_t n = (size_t)w->ntasks > (size_t)w->d.cap_mask + 1 ? (size_t)w->ntasks : (size_t)w->d.cap_mask + 1;
        int blocks = (int)((n + threads - 1) / threads);
        if (blocks > e->prop.multiProcessorCount * 8) blocks = e->prop.multiProcessorCount * 8;
        if (blocks < 1) blocks = 1;
        pb2_window_reset_kernel<<<blocks, threads, 0, e->stream>>>(w->d, w->d_tiles_init, w->d_ready, w->nready_entries);
        PB2_CUDA(e, cudaGetLastError());
    }
    if (w->ntasks > 0 && w->kind == 1 && w->v2) {
        pb2_window2_reset_kernel<<<64, 256, 0, e->stream>>>(w->g, w->d_ready_entries, w->nentries);
        PB2_CUDA(e, cudaGetLastError());
    }
    PB2_CUDA(e, cudaEventRecord(w->ev1, e->stream));
    return PB2_SUCCESS;
}

int pb2_window_start(pb2_window_t* w) {
    if (!w) return PB2_ERR_BAD_PARAM;
    pb2_engine_t* e = w->e;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    if (w->ntasks > 0) {
        if (w->kind == 0) {
            pb2_engine_hbm_kernel<<<e->nworkers, e->params.threads, 0, e->stream>>>(w->d);
            PB2_CUDA(e, cudaGetLastError());
        } else if (w->v2) {
            int rc = pb2_gemm2_launch(w->g, e->nworkers_gemm, e->stream);
            if (rc != PB2_SUCCESS) { e->last_error = "gemm v2 window launch failed"; return rc; }
        } else {
            int rc = pb2_gemm_launch(w->d, w->d_tmaps, e->nworkers_gemm, e->stream);
            if (rc != PB2_SUCCESS) { e->last_error = "gemm window launch failed"; return rc; }
        }
    }
    PB2_CUDA(e, cudaEventRecord(w->ev2, e->stream));
    w->launched = true;
    return PB2_SUCCESS;
}

int pb2_window_launch(pb2_window_t* w) {
    int rc = pb2_window_arm(w);
    return rc == PB2_SUCCESS ? pb2_window_start(w) : rc;
}

int pb2_window_export(pb2_window_t* w, pb2_window_handle_t* h) {
    if (!w || !h) return PB2_ERR_BAD_PARAM;
    pb2_engine_t* e = w->e;
    if (!w->shared) { e->last_error = "window was not created with shared windows enabled"; return PB2_ERR_NOT_SUPPORTED; }
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    memset(h, 0, sizeof *h);
    cudaIpcMemHandle_t ih;
    PB2_CUDA(e, cudaIpcGetMemHandle(&ih, w->v2 ? w->g.udep : w->d.dep));  memcpy(h->dep, &ih, 64);   // fused-GEMM windows: unit words
    PB2_CUDA(e, cudaIpcGetMemHandle(&ih, w->d.ring)); memcpy(h->ring, &ih, 64);
    PB2_CUDA(e, cudaIpcGetMemHandle(&ih, w->d.ctl));  memcpy(h->ctl, &ih, 64);
    if (w->d.tiles && w->ntiles > 0) { PB2_CUDA(e, cudaIpcGetMemHandle(&ih, w->d.tiles)); memcpy(h->tiles, &ih, 64); h->ntiles = w->ntiles; }
    h->cap_mask = w->d.cap_mask; h->ntasks = w->ntasks; h->entry_kind = w->v2 ? 1 : 0;
    return PB2_SUCCESS;
}

int pb2_window_set_push(pb2_window_t* w, const int32_t* ps_begin, const pb2_push_t* push, int32_t npush) {
    if (!w || !ps_begin || npush < 0 || (npush && !push)) return PB2_ERR_BAD_PARAM;
    pb2_engine_t* e = w->e;
    if (w->v2 || !w->d.peers) { e->last_error = "pushes need an HBM window whose remote edges are set (pb2_window_set_remote)"; return PB2_ERR_NOT_SUPPORTED; }
    if (ps_begin[w->ntasks] != npush) return PB2_ERR_BAD_PARAM;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    std::vector<PushDev> pd((size_t)npush);
    for (int32_t i = 0; i < npush; ++i) {
        const pb2_push_t& p = push[i];
        if (p.rank < 0 || (size_t)p.rank >= w->peer_tiles.size() || !w->peer_tiles[(size_t)p.rank]) { e->last_error = "push to a rank whose tile table is not mapped"; return PB2_ERR_BAD_PARAM; }
        if (p.desc < 0 || p.desc >= w->peer_ntiles[(size_t)p.rank] || p.src_tile < 0 || p.src_tile >= w->ntiles) { e->last_error = "push descriptor out of bounds"; return PB2_ERR_VALUE_OUT_OF_BOUNDS; }
        memset(&pd[(size_t)i], 0, sizeof(PushDev));
        pd[(size_t)i].dst = reinterpret_cast<void*>(p.dst);
        pd[(size_t)i].dst_state = &w->peer_tiles[(size_t)p.rank][p.desc].state;
        pd[(size_t)i].bytes = p.bytes; pd[(size_t)i].src_tile = p.src_tile;
    }
    int rc;
    int32_t* d_b = nullptr; PushDev* d_p = nullptr;
    if ((rc = dev_alloc_copy(w, &d_b, ps_begin, (size_t)w->ntasks + 1)) != PB2_SUCCESS) return rc;
    if ((rc = dev_alloc_copy(w, &d_p, pd.data(), pd.size())) != PB2_SUCCESS) return rc;
    PB2_CUDA(e, cudaStreamSynchronize(e->up_stream));
    w->d.ps_begin = npush ? d_b : nullptr; w->d.ps = d_p;
    return PB2_SUCCESS;
}

int pb2_window_set_remote(pb2_window_t* w, int32_t my_rank, int32_t nranks, const pb2_window_handle_t* peers,
                          const int32_t* rs_begin, const int32_t* rs_rank, const uint32_t* rs_target, int32_t nrs) {
    if (!w || nranks <= 0 || my_rank < 0 || my_rank >= nranks || !peers || !rs_begin || nrs < 0) return PB2_ERR_BAD_PARAM;
    pb2_engine_t* e = w->e;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    const int32_t my_kind = w->v2 ? 1 : 0;
    for (int32_t r = 0; r < nranks; ++r)
        if (r != my_rank && peers[r].entry_kind != my_kind) { e->last_error = "peers run a different kind of window (fused GEMM units vs tasks)"; return PB2_ERR_NOT_SUPPORTED; }
    for (int32_t i = 0; i < nrs; ++i) {
        if (rs_rank[i] < 0 || rs_rank[i] >= nranks || rs_rank[i] == my_rank) { e->last_error = "remote edge to a bad rank"; return PB2_ERR_BAD_PARAM; }
        const int32_t idx = my_kind ? (int32_t)PB2_SUCC_TASK(rs_target[i]) : (int32_t)(rs_target[i] & 0x3FFFFFu);
        if (idx >= peers[rs_rank[i]].ntasks) { e->last_error = "remote edge target out of bounds"; return PB2_ERR_VALUE_OUT_OF_BOUNDS; }
    }
    if (rs_begin[w->ntasks] != nrs) return PB2_ERR_BAD_PARAM;
    std::vector<PeerWin> pw((size_t)nranks);
    for (int32_t r = 0; r < nranks; ++r) {
        memset(&pw[r], 0, sizeof(PeerWin));
        if (r == my_rank) continue;
        void *pd = nullptr, *pr = nullptr, *pc = nullptr, *pt = nullptr;
        cudaIpcMemHandle_t ih;
        memcpy(&ih, peers[r].dep, 64);  PB2_CUDA(e, cudaIpcOpenMemHandle(&pd, ih, cudaIpcMemLazyEnablePeerAccess));
        memcpy(&ih, peers[r].ring, 64); PB2_CUDA(e, cudaIpcOpenMemHandle(&pr, ih, cudaIpcMemLazyEnablePeerAccess));
        memcpy(&ih, peers[r].ctl, 64);  PB2_CUDA(e, cudaIpcOpenMemHandle(&pc, ih, cudaIpcMemLazyEnablePeerAccess));
        memcpy(&ih, peers[r].tiles, 64);
        {   // a window without tiles exports an all-zero handle
            bool any = false;
            for (int b = 0; b < 64; ++b) any |= peers[r].tiles[b] != 0;
            if (any) { PB2_CUDA(e, cudaIpcOpenMemHandle(&pt, ih, cudaIpcMemLazyEnablePeerAccess)); w->peer_ptrs.push_back(pt); }
        }
        w->peer_ptrs.push_back(pd); w->peer_ptrs.push_back(pr); w->peer_ptrs.push_back(pc);
        pw[r].tiles = reinterpret_cast<pb2_tile_t*>(pt);
        w->peer_tiles.resize((size_t)nranks, nullptr); w->peer_tiles[(size_t)r] = reinterpret_cast<pb2_tile_t*>(pt);
        w->peer_ntiles.resize((size_t)nranks, 0); w->peer_ntiles[(size_t)r] = peers[r].ntiles;
        pw[r].dep = reinterpret_cast<int32_t*>(pd); pw[r].ring = reinterpret_cast<int32_t*>(pr);
        pw[r].ctl = reinterpret_cast<Ctl*>(pc); pw[r].cap_mask = peers[r].cap_mask;
    }
    int rc;
    PeerWin* d_pw = nullptr; int32_t* d_b = nullptr; int32_t* d_r = nullptr; uint32_t* d_t = nullptr;
    if ((rc = dev_alloc_copy(w, &d_pw, pw.data(), pw.size())) != PB2_SUCCESS) return rc;
    if ((rc = dev_alloc_copy(w, &d_b, rs_begin, (size_t)w->ntasks + 1)) != PB2_SUCCESS) return rc;
    if ((rc = dev_alloc_copy(w, &d_r, rs_rank, (size_t)nrs)) != PB2_SUCCESS) return rc;
    if ((rc = dev_alloc_copy(w, &d_t, rs_target, (size_t)nrs)) != PB2_SUCCESS) return rc;
    PB2_CUDA(e, cudaStreamSynchronize(e->up_stream));
    w->d.peers = d_pw; w->d.rs_begin = d_b; w->d.rs_rank = d_r; w->d.rs_target = d_t; w->d.remote_units = my_kind;
    if (w->v2) w->g.w = w->d;
    return PB2_SUCCESS;
}

int pb2_window_wait(pb2_window_t* w, pb2_window_stats_t* stats) {
    if (!w) return PB2_ERR_BAD_PARAM;
    pb2_engine_t* e = w->e;
    if (!w->launched) return PB2_ERR_BAD_PARAM;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    PB2_CUDA(e, cudaEventSynchronize(w->ev2));
    Ctl c;
    PB2_CUDA(e, cudaMemcpy(&c, w->d.ctl, sizeof c, cudaMemcpyDeviceToHost));
    if (stats) {
        memset(stats, 0, sizeof *stats);
        stats->tasks_retired = c.retired.v;
        stats->bytes_h2d = c.bytes_h2d.v; stats->bytes_d2d = c.bytes_d2d.v; stats->bytes_d2h = c.bytes_d2h.v;
        stats->stage_ins = c.stage_ins.v; stats->body_errors = c.body_errors.v;
        cudaEventElapsedTime(&stats->reset_ms, w->ev0, w->ev1);
        cudaEventElapsedTime(&stats->kernel_ms, w->ev1, w->ev2);
    }
    const int32_t done = (int32_t)c.done.v;
    if (done == kDoneTimeout) { e->last_error = "window watchdog: no task retired within timeout (malformed DAG?)"; return PB2_ERR_DEVICE; }
    if (done == kDoneBadBody) { e->last_error = "window ran a task with an unknown body id"; return PB2_ERR_BAD_PARAM; }
    if ((int64_t)c.retired.v != (int64_t)w->ntasks) { e->last_error = "window ended before all tasks retired"; return PB2_ERROR; }
    return PB2_SUCCESS;
}

int pb2_window_results(pb2_window_t* w, int32_t* retire_order, uint32_t* start_seq, uint32_t* end_seq,
                       uint32_t* seen_version, uint64_t* result, int32_t* worker, pb2_tile_t* tiles_out) {
    if (!w) return PB2_ERR_BAD_PARAM;
    pb2_engine_t* e = w->e;
    PB2_CUDA(e, cudaSetDevice(e->cuda_device));
    const size_t n = (size_t)w->ntasks;
    if (retire_order && n) PB2_CUDA(e, cudaMemcpy(retire_order, w->d.retire_log, n * 4, cudaMemcpyDeviceToHost));
    if (start_seq && n) PB2_CUDA(e, cudaMemcpy(start_seq, w->d.start_seq, n * 4, cudaMemcpyDeviceToHost));
    if (end_seq && n) PB2_CUDA(e, cudaMemcpy(end_seq, w->d.end_seq, n * 4, cudaMemcpyDeviceToHost));
    if (seen_version && n) PB2_CUDA(e, cudaMemcpy(seen_version, w->d.seen_version, n * 4 * PB2_MAX_FLOWS, cudaMemcpyDeviceToHost));
    if (result && n) PB2_CUDA(e, cudaMemcpy(result, w->d.result, n * 8, cudaMemcpyDeviceToHost));
    if (worker && n) PB2_CUDA(e, cudaMemcpy(worker, w->d.worker, n * 4, cudaMemcpyDeviceToHost));
    if (tiles_out && w->ntiles) PB2_CUDA(e, cudaMemcpy(tiles_out, w->d_tiles, (size_t)w->ntiles * sizeof(pb2_tile_t), cudaMemcpyDeviceToHost));
    return PB2_SUCCESS;
}

}  // extern "C"
