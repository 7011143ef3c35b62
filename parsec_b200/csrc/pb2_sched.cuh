// pb2_sched.cuh -- device-resident scheduling state and primitives shared by the engine kernels
// (HBM-body kernel in pb2_engine.cu, tensor-core kernel in pb2_gemm.cuh).
#pragma once
#include "../../include/pb2_engine.h"
#include "pb2_dev_utils.cuh"
#include "pb2_bodies.cuh"

namespace pb2 {

constexpr int32_t kEmpty = -1;
constexpr int32_t kDoneOK = 1;
constexpr int32_t kDoneTimeout = 2;
constexpr int32_t kDoneBadBody = 3;

// Hot control words, one per 128-byte line so that atomics on them do not false-share.
struct alignas(128) Line { unsigned long long v; unsigned long long pad[15]; };
struct Ctl {
    Line head;       // pop tickets handed out
    Line tail;       // push tickets handed out
    Line evt;        // global event counter (start/end sequence numbers)
    Line retired;    // tasks retired
    Line done;       // 0 running, kDone*
    Line progress_ns;// globaltimer of the last retirement (watchdog)
    Line bytes_h2d, bytes_d2d, bytes_d2h, stage_ins, body_errors;
};

struct WinDev {
    const pb2_task_t* tasks;
    const uint32_t*   succ;
    pb2_tile_t*       tiles;
    int32_t*          dep;
    int32_t*          ring;
    Ctl*              ctl;
    int32_t*          retire_log;
    uint32_t*         start_seq;
    uint32_t*         end_seq;
    uint32_t*         seen_version;
    unsigned long long* result;
    int32_t*          worker;
    uint32_t          cap_mask;
    int32_t           ntasks;
    int32_t           ntiles;
    int32_t           stage_mode;
    unsigned long long timeout_ns;
    int32_t*          parts_left;     // HBM windows: parts of a task still running (wide tasks)
    // remote out-edges (other GPUs' windows), see pb2_window_set_remote
    const int32_t*    rs_begin;
    const int32_t*    rs_rank;
    const uint32_t*   rs_target;
    const struct PeerWin* peers;
    // producer-side pushes (pb2_window_set_push): task t writes ps[ps_begin[t] .. ps_begin[t+1]) into its readers' slots
    const int32_t*    ps_begin;
    const struct PushDev* ps;
    int32_t           shared;         // scheduling arrays are written by peers: poll / publish at system scope
    // sliced stage-in of tiles larger than part_bytes (HBM windows): which slices are claimed / staged
    uint32_t*         slice_claim;
    uint32_t*         slice_done;
    int32_t           part_bytes;
    const uint16_t*   nparts;         // HBM windows with wide tasks: parts per task (null: every task is one part)
    int32_t           remote_units;   // remote targets are (parts-1) << 27 | unit of a fused-GEMM window, not << 22 | task
};

struct PeerWin { int32_t* dep; int32_t* ring; Ctl* ctl; uint32_t cap_mask; int32_t pad; pb2_tile_t* tiles; };
struct alignas(32) PushDev { void* dst; int32_t* dst_state; uint32_t bytes; int32_t src_tile; int32_t pad[2]; };

// A task whose tiles are large is executed as several PARTS (byte slices of its tiles) by different workers: one
// tile at HBM / NVLink speed needs the whole GPU (a 64-thread CTA keeps 4 KiB in flight; a 4 MiB tile is 1.3 us of
// the machine, not 1 ms of one CTA).  Parts per task (1..512) live in WinDev::nparts; ring entries of HBM windows
// are (part << 22) | task, so such a window holds at most 2^22 tasks when it has wide tasks.
#define PB2_MAX_PARTS 512
#define PB2_SLICE_WORDS (PB2_MAX_PARTS / 32)
#define PB2_ENT_MAKE(task, part) ((int32_t)(((uint32_t)(part) << 22) | (uint32_t)(task)))
#define PB2_ENT_TASK(e)          ((int32_t)((uint32_t)(e) & 0x3FFFFFu))
#define PB2_ENT_PART(e)          ((int)((uint32_t)(e) >> 22))

// Parts of a tile cut at part_bytes (> 0): the parts of a wide task (its widest tile) and the stage-in slices of a tile.
__host__ __device__ __forceinline__ int tile_parts(uint32_t bytes, int32_t part_bytes) {
    const uint32_t n = (bytes + (uint32_t)part_bytes - 1) / (uint32_t)part_bytes;
    return n > PB2_MAX_PARTS ? PB2_MAX_PARTS : (n < 1 ? 1 : (int)n);
}

// Slice i of n slices of `per` = slice_size bytes: [off, off + len); the last one takes the remainder.
__host__ __device__ __forceinline__ uint32_t slice_size(uint32_t bytes, int n) { return ((bytes / (uint32_t)n) + 15u) & ~15u; }
__host__ __device__ __forceinline__ void slice_bounds(uint32_t per, uint32_t bytes, int i, int n, uint32_t& off, uint32_t& len) {
    off = per * (uint32_t)i < bytes ? per * (uint32_t)i : bytes;
    len = (i == n - 1) ? bytes - off : (off + per <= bytes ? per : bytes - off);
}

// Stamp of index idx of a ring of `slots` entries (never 0).
__host__ __device__ __forceinline__ uint32_t ring_gen(unsigned long long idx, unsigned long long slots) {
    return (uint32_t)(idx / slots) + 1u;
}

__device__ __forceinline__ int task_nparts(const WinDev& w, int32_t id) { return w.nparts ? (int)w.nparts[id] : 1; }

// Whole warp: a lane with np > 0 pushes the entries of parts 0 .. np-1 of ready `sid`, one tail reservation per warp.
// UNITS: v2 GEMM units (PB2_SUCC_MAKE, <= 16 parts), written lane by lane: fewer registers in pb2_engine_gemm2_kernel.
template <bool UNITS>
__device__ __forceinline__ void push_ready_warp(const WinDev& w, int32_t sid, int np) {
    const int lane = threadIdx.x & 31;
    int incl = np;
    for (int o = 1; o < 32; o <<= 1) { const int v = __shfl_up_sync(0xffffffffu, incl, o); if (lane >= o) incl += v; }
    const int total = __shfl_sync(0xffffffffu, incl, 31);
    if (!total) return;
    unsigned long long base = 0;
    if (lane == 0) base = atomicAdd(&w.ctl->tail.v, (unsigned long long)total);
    base = __shfl_sync(0xffffffffu, base, 0);
    const uint32_t first = (uint32_t)base + (uint32_t)(incl - np);
    const unsigned many = UNITS ? 0u : __ballot_sync(0xffffffffu, np > 4);
    if (np > 0 && (UNITS || np <= 4))
        for (int p = 0; p < np; ++p)
            st_release_gpu(&w.ring[(first + (uint32_t)p) & w.cap_mask], UNITS ? (int32_t)PB2_SUCC_MAKE(sid, p) : PB2_ENT_MAKE(sid, p));
    for (unsigned m = many; m; m &= m - 1) {
        const int src = __ffs(m) - 1;
        const int32_t s2 = __shfl_sync(0xffffffffu, sid, src);
        const int n2 = __shfl_sync(0xffffffffu, np, src);
        const uint32_t f2 = __shfl_sync(0xffffffffu, first, src);
        for (int p = lane; p < n2; p += 32)
            st_release_gpu(&w.ring[(f2 + (uint32_t)p) & w.cap_mask], UNITS ? (int32_t)PB2_SUCC_MAKE(s2, p) : PB2_ENT_MAKE(s2, p));
    }
}

// ---------------------------------------------------------------------------------------------
// scheduling primitives shared by the HBM and the GEMM engine kernels
// ---------------------------------------------------------------------------------------------

// One thread: take the next pop ticket and wait for its slot.  Returns a task id, or kEmpty when the
// window is finished (or aborted).  Ticket order == push order, i.e. a strict FIFO ready queue.
__device__ __forceinline__ int32_t pop_task(const WinDev& w) {
    const uint32_t ticket = (uint32_t)atomicAdd(&w.ctl->head.v, 1ull);
    int32_t* slot = &w.ring[ticket & w.cap_mask];
    uint32_t spins = 0;
    int32_t id;
    while ((id = (w.shared ? ld_acquire_sys(slot) : ld_acquire_gpu(slot))) == kEmpty) {
        if (ld_relaxed_gpu(reinterpret_cast<const int32_t*>(&w.ctl->done.v)) != 0) return kEmpty;
        if ((++spins & 1023u) == 0) {
            // watchdog: a DAG whose dependency counts are wrong would spin forever
            const unsigned long long last = *reinterpret_cast<volatile unsigned long long*>(&w.ctl->progress_ns.v);
            // signed: %globaltimer read on another SM can be slightly behind the value a retiring SM just stored
            if ((long long)(globaltimer_ns() - last) > (long long)w.timeout_ns) {
                st_relaxed_gpu(reinterpret_cast<int32_t*>(&w.ctl->done.v), kDoneTimeout);
                return kEmpty;
            }
        }
        __nanosleep(spins < 64 ? 32 : 256);
    }
    return id;
}

// Whole warp: release the out-edges of task t (parsec_release_dep_fct semantics), push the newly
// ready successors.  Must be called after a __threadfence() that follows the body's stores.
__device__ __forceinline__ void release_successors_warp(const WinDev& w, const pb2_task_t& t) {
    const int lane = threadIdx.x & 31;
    for (int e0 = 0; e0 < t.succ_count; e0 += 32) {
        const int e = e0 + lane;
        bool ready = false;
        int32_t sid = -1;
        if (e < t.succ_count) {
            const uint32_t s = w.succ[t.succ_begin + e];
            sid = PB2_SUCC_TASK(s);
            const pb2_task_t& st = w.tasks[sid];
            if (st.flags & PB2_TASK_DEPS_MASK) {
                // parsec_update_deps_with_mask, parsec.c:1656-1720: OR the destination flow bit, the
                // task is ready when (word & goal) == goal; each bit is set exactly once (:1688 assert)
                const int32_t bit = 1 << PB2_SUCC_FLOW(s);
                const int32_t old = atomicOr(&w.dep[sid], bit);
                ready = (((old | bit) & st.dep_goal) == st.dep_goal) && ((old & st.dep_goal) != st.dep_goal);
            } else {
                // parsec_update_deps_with_counter, parsec.c:1609-1654: fetch_dec, ready at 0
                ready = (atomicSub(&w.dep[sid], 1) == 1);
            }
        }
        push_ready_warp<false>(w, sid, ready ? task_nparts(w, sid) : 0);
    }
}

// Whole warp: release the out-edges that lead into other GPUs' windows.  The activation message of the reference
// (remote_dep_mpi.c:1860 remote_dep_mpi_recv_activate -> release of the local successors) becomes a system-scope
// atomic on the peer's dependency word and, when it reaches zero, ring entries written into the peer's HBM over
// NVLink.  The tile itself is pulled by the peer's worker from this GPU's slot when the task runs (stage_in_flow).
__device__ __forceinline__ void release_remote_warp(const WinDev& w, int32_t id) {
    if (!w.rs_begin) return;
    const int lane = threadIdx.x & 31;
    const int32_t b = w.rs_begin[id], e1 = w.rs_begin[id + 1];
    if (b == e1) return;
    __threadfence_system();            // our tile bytes are visible to the peers before they can see the release
    for (int32_t e0 = b; e0 < e1; e0 += 32) {
        const int32_t e = e0 + lane;
        int np = 0;
        int32_t sid = 0;
        uint32_t first = 0;
        PeerWin pw = w.peers[w.rs_rank[e < e1 ? e : b]];
        if (e < e1) {
            const uint32_t tgt = w.rs_target[e];
            sid = w.remote_units ? (int32_t)PB2_SUCC_TASK(tgt) : PB2_ENT_TASK(tgt);
            if (atomicSub_system(&pw.dep[sid], 1) == 1) {
                np = (w.remote_units ? (int)PB2_SUCC_FLOW(tgt) : PB2_ENT_PART(tgt)) + 1;
                first = (uint32_t)atomicAdd_system(&pw.ctl->tail.v, (unsigned long long)np);
            }
        }
        // entries of one ready task go to ONE peer: lanes cooperate per ready lane, the ring pointer travels with it
        const unsigned many = __ballot_sync(0xffffffffu, np > 0);
        for (unsigned m = many; m; m &= m - 1) {
            const int src = __ffs(m) - 1;
            const int32_t s2 = __shfl_sync(0xffffffffu, sid, src);
            const int n2 = __shfl_sync(0xffffffffu, np, src);
            const uint32_t f2 = __shfl_sync(0xffffffffu, first, src);
            const unsigned long long rp = __shfl_sync(0xffffffffu, (unsigned long long)(uintptr_t)pw.ring, src);
            const uint32_t cm = __shfl_sync(0xffffffffu, pw.cap_mask, src);
            int32_t* ring = reinterpret_cast<int32_t*>((uintptr_t)rp);
            for (int p = lane; p < n2; p += 32)
                st_release_sys(&ring[(f2 + (uint32_t)p) & cm], w.remote_units ? (int32_t)PB2_SUCC_MAKE(s2, p) : PB2_ENT_MAKE(s2, p));
        }
    }
}

// Whole CTA, after the body of a task whose written tile other GPUs read: write the tile into every reader rank's slot
// (posted stores over NVLink through the bulk mover: local reads, remote writes, no round trip per chunk), then publish
// the slot's state at system scope.  The release of the remote successors follows (release_remote_warp): they find
// the tile VALID.  This is the PUT of remote_dep_mpi.c:2120 issued by the producer instead of a GET by each consumer.
static __device__ __noinline__ void push_written_tiles(const pb2_tile_t* tiles, Ctl* ctl, const int32_t* ps_begin, const PushDev* ps,
                                                       int32_t id, BulkSmem* bulk) {
    const int32_t b = ps_begin[id], e = ps_begin[id + 1];
    for (int32_t i = b; i < e; ++i) {
        const PushDev p = ps[i];
        cta_copy<false>(p.dst, tiles[p.src_tile].dev_ptr, p.bytes, bulk);
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence_system();
            st_release_sys(p.dst_state, PB2_TILE_VALID);
            atomicAdd(&ctl->bytes_d2d.v, (unsigned long long)p.bytes);
        }
    }
    __syncthreads();
}

// One thread, after the window's last task released its out-edges.
__device__ __forceinline__ void finish_window(const WinDev& w) {
    __threadfence();
    st_release_gpu(reinterpret_cast<int32_t*>(&w.ctl->done.v), kDoneOK);
}

__device__ __forceinline__ void reset_tile_slices(const WinDev& w, size_t tile) {
    for (int k = 0; k < PB2_SLICE_WORDS; ++k) w.slice_claim[tile * PB2_SLICE_WORDS + k] = 0;
    for (int k = 0; k <= PB2_SLICE_WORDS; ++k) w.slice_done[tile * (PB2_SLICE_WORDS + 1) + k] = 0;
}

// ---------------------------------------------------------------------------------------------
// stage-in / stage-out of one flow by the whole CTA
// ---------------------------------------------------------------------------------------------
// What the out-of-line stage-in helpers need from the window, passed BY VALUE in registers: a reference to the
// kernel-parameter struct would force a 300-byte local-memory copy of it in every caller.
struct StageCtx {
    pb2_tile_t* tiles; Ctl* ctl; uint32_t* slice_claim; uint32_t* slice_done; int32_t use_bulk; int32_t part_bytes;
};
__device__ __forceinline__ StageCtx stage_ctx(const WinDev& w) {
    return StageCtx{w.tiles, w.ctl, w.slice_claim, w.slice_done, w.stage_mode == 0 ? 1 : 0, w.part_bytes};
}

// parsec_device_data_stage_in, device_gpu.c:1799-2165: only a READ access needs the bytes;
// "finally we'll just overwrite w/o read" (data.c:427) for WRITE-only flows.
__device__ __forceinline__ bool needs_stage_in(const pb2_tile_t* tile, uint8_t access) {
    return (access & PB2_FLOW_ACCESS_READ) && ld_acquire_gpu(&tile->state) != PB2_TILE_VALID;
}

// One thread: wait for a tile or slice that another worker (SYS: a producer on another GPU) moves.
template <bool SYS>
__device__ __forceinline__ void wait_word(const int32_t* word, int32_t mask, int32_t want) {
    while (((SYS ? ld_acquire_sys(word) : ld_acquire_gpu(word)) & mask) != want) __nanosleep(64);
}

__device__ __forceinline__ void count_stage_in(Ctl* ctl, const pb2_tile_t* tile, uint32_t bytes) {
    atomicAdd(tile->src_kind == PB2_SRC_PEER ? &ctl->bytes_d2d.v : &ctl->bytes_h2d.v, (unsigned long long)bytes);
}

// Thread 0 decides (s_decide[0]): 1 = this CTA moves the tile, 0 = already valid (possibly after waiting)
static __device__ __noinline__ void stage_in_flow(const StageCtx w, pb2_tile_t* tile, uint8_t access, int* s_decide, BulkSmem* bulk = nullptr) {
    if (threadIdx.x == 0) {
        int decide = 0;
        if ((access & PB2_FLOW_ACCESS_READ) && tile->src_kind == PB2_SRC_PUSH) {
            // the producer writes this slot and publishes its state before it releases us: nothing to move
            wait_word<true>(&tile->state, -1, PB2_TILE_VALID);
        } else if (access & PB2_FLOW_ACCESS_READ) {
            int32_t st = atomicCAS(&tile->state, PB2_TILE_INVALID, PB2_TILE_STAGING);
            if (st == PB2_TILE_INVALID) {
                decide = 1;
            } else if (st != PB2_TILE_VALID) {
                // another worker is moving it: "data copy is already under transfer" (device_gpu.c:1873-1884)
                __nanosleep(64);
                wait_word<false>(&tile->state, -1, PB2_TILE_VALID);
            }
        }
        *s_decide = decide;
    }
    __syncthreads();
    if (*s_decide) {
        cta_copy<true>(tile->dev_ptr, tile->src_ptr, tile->bytes, w.use_bulk ? bulk : nullptr);
        __syncthreads();
        if (threadIdx.x == 0) {
            __threadfence();
            st_release_gpu(&tile->state, PB2_TILE_VALID);   // COMPLETE_TRANSFER (device_gpu.c:2358-2573)
            count_stage_in(w.ctl, tile, tile->bytes);
            atomicAdd(&w.ctl->stage_ins.v, 1ull);
        }
    }
    __syncthreads();
}


// Number of stage-in slices of a tile.
__device__ __forceinline__ int tile_slices_of(int32_t part_bytes, const uint32_t* slice_claim, uint32_t bytes) {
    if (part_bytes <= 0 || !slice_claim) return 1;
    return tile_parts(bytes, part_bytes);
}
__device__ __forceinline__ int tile_slices(const WinDev& w, uint32_t bytes) { return tile_slices_of(w.part_bytes, w.slice_claim, bytes); }

// Stage in the slices [s0, s1) of a tile larger than part_bytes.  Every slice is moved by exactly one CTA (claim
// bit), so the parts of a wide task -- and the parts of other readers of the same version -- pull the tile in
// parallel instead of one CTA moving 4 MiB alone; a CTA that finds a slice claimed by someone else only waits
// for it.  The worker whose slice completes the tile publishes PB2_TILE_VALID.
static __device__ __noinline__ void stage_in_slices(const StageCtx w, int32_t tile_id, int nslices, int s0, int s1, int* s_decide, BulkSmem* bulk = nullptr) {
    pb2_tile_t* tile = &w.tiles[tile_id];
    if (tile->src_kind == PB2_SRC_PUSH) {       // written by its producer (see stage_in_flow)
        if (threadIdx.x == 0) wait_word<true>(&tile->state, -1, PB2_TILE_VALID);
        __syncthreads();
        return;
    }
    const uint32_t bytes = tile->bytes;
    const uint32_t sper = slice_size(bytes, nslices);
    uint32_t* claim = w.slice_claim + (size_t)tile_id * PB2_SLICE_WORDS;
    uint32_t* done = w.slice_done + (size_t)tile_id * (PB2_SLICE_WORDS + 1);     // last word: number of staged slices
    for (int sl = s0; sl < s1; ++sl) {
        const uint32_t bit = 1u << (sl & 31);
        if (threadIdx.x == 0) *s_decide = (atomicOr(&claim[sl >> 5], bit) & bit) ? 0 : 1;
        __syncthreads();
        if (*s_decide) {
            uint32_t off, len;
            slice_bounds(sper, bytes, sl, nslices, off, len);
            cta_copy<true>(reinterpret_cast<uint8_t*>(tile->dev_ptr) + off, reinterpret_cast<const uint8_t*>(tile->src_ptr) + off, len, w.use_bulk ? bulk : nullptr);
            __syncthreads();
            if (threadIdx.x == 0) {
                __threadfence();
                atomicOr(&done[sl >> 5], bit);
                count_stage_in(w.ctl, tile, len);
                if ((int)atomicAdd(&done[PB2_SLICE_WORDS], 1u) + 1 == nslices) {
                    __threadfence();
                    st_release_gpu(&tile->state, PB2_TILE_VALID);
                    atomicAdd(&w.ctl->stage_ins.v, 1ull);
                }
            }
        }
        __syncthreads();
    }
    if (threadIdx.x == 0) {
        for (int sl = s0; sl < s1; ++sl) {
            const int32_t bit = (int32_t)(1u << (sl & 31));
            wait_word<false>(reinterpret_cast<const int32_t*>(&done[sl >> 5]), bit, bit);
        }
        __threadfence();
    }
    __syncthreads();
}

}  // namespace pb2
