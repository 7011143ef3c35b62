// pb2_worker.cuh -- what one worker CTA does with one (part of a) task: push (stage-in), exec (body), pop (pushout).
// Shared by the window kernel (pb2_engine.cu) and the streaming kernel (pb2_stream.cu); the two differ only in where
// ready tasks come from and in how a finished task is retired and its successors are released.
//
// Reference: parsec_device_kernel_push / _exec / _pop, parsec/mca/device/device_gpu.c:2745, :2873, :2943.
//
// Register discipline: the kernels run 24 CTAs of 64 threads per SM (<= 40 registers per thread).  Everything that is
// indexed by a run-time flow number lives in shared memory (TaskSmem), filled by one thread per flow, so that no
// array is demoted to local memory; tile payloads move through TMA (no payload registers) or 4 x 16-byte loads.
#pragma once
#include "pb2_sched.cuh"

namespace pb2 {

struct alignas(16) TaskSmem {
    pb2_task_t task;                 // four 16-byte loads
    BodyArgs   args;                 // this part's slice of every flow
    uint32_t   off[PB2_MAX_FLOWS];   // byte offset of the slice inside its tile
    uint32_t   tbytes[PB2_MAX_FLOWS];// whole-tile byte counts
    int32_t    entry;                // ring entry popped (kEmpty: leave)
    int32_t    need;                 // bit f: flow f has to be staged in
    int32_t    decide;               // scratch of the stage-in helpers
    int32_t    last;                 // this part retired the task
    int32_t    window_done;          // this task was the last of the window
    uint32_t   red[32];
};

__device__ __forceinline__ bool pushes_out(const pb2_task_t& t, int f) {
    return t.tile[f] >= 0 && (t.access[f] & PB2_FLOW_PUSHOUT) && (t.access[f] & PB2_FLOW_ACCESS_WRITE);
}

// All threads: parsec_device_kernel_pop stage_out (device_gpu.c:2943) of a written flow to its home copy.
__device__ __forceinline__ void pushout(Ctl* ctl, void* home, const void* dev, size_t bytes, BulkSmem* bulk = nullptr) {
    cta_copy<false>(home, dev, bytes, bulk);
    if (threadIdx.x == 0) atomicAdd(&ctl->bytes_d2h.v, (unsigned long long)bytes);
}

// All threads (uniform): stage in every flow whose bit is set in s.need.  One CTA-wide call per task at most.
static __device__ __noinline__ void stage_in_needed_flows(const StageCtx c, TaskSmem* sp, BulkSmem* bulk) {
    TaskSmem& s = *sp;
    const int need = s.need;
#pragma unroll 1
    for (int f = 0; f < PB2_MAX_FLOWS; ++f) {
        if (!((need >> f) & 1)) continue;
        const int32_t tid = s.task.tile[f];
        const uint32_t bytes = s.tbytes[f];
        const int ns = tile_slices_of(c.part_bytes, c.slice_claim, bytes);
        if (ns == 1) stage_in_flow(c, &c.tiles[tid], s.task.access[f], &s.decide, bulk);
        else {
            // slices [s0, s1) of the tile cover this part's bytes (the task may be cut differently from the tile
            // when its widest flow is another tile)
            const uint32_t sper = slice_size(bytes, ns);
            const uint32_t off = s.off[f], len = s.args.bytes[f];
            int s0 = (int)(off / sper), s1 = (int)((off + len + sper - 1) / sper);
            if (s0 > ns - 1) s0 = ns - 1;
            if (s1 > ns) s1 = ns;
            if (len == 0) s1 = s0;
            stage_in_slices(c, tid, ns, s0, s1, &s.decide, bulk);
        }
    }
}

// All threads.  On entry s.task holds the descriptor (published by a barrier).  Returns the body result (thread 0).
__device__ __forceinline__ unsigned long long
run_task_part(const WinDev& w, TaskSmem& s, BulkSmem* bulk, int32_t id, int part, int nparts) {
    const pb2_task_t& t = s.task;
    // ---- push: one thread per flow works out its slice and whether the tile has to be staged in -----------------
    if (threadIdx.x < 32) {
        const int f = (int)threadIdx.x;
        const bool mine = f < PB2_MAX_FLOWS && f < (int)t.nb_flows && t.tile[f < PB2_MAX_FLOWS ? f : 0] >= 0;
        pb2_tile_t* tile = mine ? &w.tiles[t.tile[f]] : nullptr;
        const uint32_t bytes = mine ? tile->bytes : 0u;
        // every flow is cut at the same byte offsets (those of the task's widest tile, 16-byte aligned, the last
        // part takes the remainder), so two-flow bodies pair equal offsets
        uint32_t widest = bytes;
        for (int o = 1; o < PB2_MAX_FLOWS; o <<= 1) {
            const uint32_t v = __shfl_xor_sync(0xffffffffu, widest, o);
            widest = v > widest ? v : widest;
        }
        uint32_t off, len;
        slice_bounds(slice_size(widest, nparts), bytes, part, nparts, off, len);
        const bool need = mine && needs_stage_in(tile, t.access[f]);
        const unsigned needmask = __ballot_sync(0xffffffffu, need);
        if (f < PB2_MAX_FLOWS) {
            s.args.flow[f] = mine ? reinterpret_cast<uint8_t*>(tile->dev_ptr) + off : nullptr;
            s.args.bytes[f] = len; s.off[f] = off; s.tbytes[f] = bytes;
            if (mine && part == 0)
                w.seen_version[(size_t)id * PB2_MAX_FLOWS + f] = *reinterpret_cast<volatile uint32_t*>(&tile->version);
        }
        if (f == 0) {
            s.need = (int32_t)needmask;
            s.args.part = (uint32_t)part; s.args.elem0 = off >> 2;
            s.args.iparam[0] = t.iparam[0]; s.args.iparam[1] = t.iparam[1]; s.args.iparam[2] = t.iparam[2];
            s.args.fparam = t.fparam;
        }
    }
    __syncthreads();
    // the cold path, out of line and called once: everything it needs is in shared memory, nothing of the caller's
    // has to survive the call in registers
    if (s.need) stage_in_needed_flows(stage_ctx(w), &s, bulk);

    // ---- exec: the body (parsec_device_kernel_exec -> submit) ----
    const unsigned long long r = run_hbm_body(t.body, s.args, s.red);
    __syncthreads();

    // ---- pop: pushout of written flows to their home copy (parsec_device_kernel_pop stage_out) ----
#pragma unroll
    for (int f = 0; f < PB2_MAX_FLOWS; ++f) {
        if (f < (int)t.nb_flows && pushes_out(t, f))
            pushout(w.ctl, reinterpret_cast<uint8_t*>(w.tiles[t.tile[f]].src_ptr) + s.off[f], s.args.flow[f], s.args.bytes[f], bulk);
    }
    __syncthreads();
    return r;
}

// Thread 0 of the part that finished last: version / coherency epilog of the written flows
// (version = candidate->version + 1 for WRITE flows, device_gpu.c:2148-2152).
__device__ __forceinline__ void epilog_written_flows(const WinDev& w, const pb2_task_t& t) {
    for (int f = 0; f < (int)t.nb_flows; ++f) {
        if (t.tile[f] < 0 || !(t.access[f] & PB2_FLOW_ACCESS_WRITE)) continue;
        pb2_tile_t* tile = &w.tiles[t.tile[f]];
        *reinterpret_cast<volatile uint32_t*>(&tile->version) = *reinterpret_cast<volatile uint32_t*>(&tile->version) + 1;
        if (!(t.access[f] & PB2_FLOW_ACCESS_READ)) st_relaxed_gpu(&tile->state, PB2_TILE_VALID);
    }
}

// Thread 0 of the part that finished last, before the out-edges are released, so that the retire log is a linear
// extension of the DAG's partial order (a successor can only retire after us).  True: the window's last task.
__device__ __forceinline__ bool retire_task(const WinDev& w, const pb2_task_t& t, int32_t id) {
    epilog_written_flows(w, t);
    w.end_seq[id] = (uint32_t)atomicAdd(&w.ctl->evt.v, 1ull);
    const uint32_t seq = (uint32_t)atomicAdd(&w.ctl->retired.v, 1ull);
    w.retire_log[seq] = id;
    *reinterpret_cast<volatile unsigned long long*>(&w.ctl->progress_ns.v) = globaltimer_ns();
    return (int32_t)(seq + 1) == w.ntasks;
}

// Thread 0: store the body result of this part (CHECK bodies add their mismatch counts over the parts).
__device__ __forceinline__ void record_result(const WinDev& w, int body, int32_t id, int part, int nparts, unsigned long long r) {
    if (body == PB2_BODY_CHECK_I32 || body == PB2_BODY_CHECK_F32) {
        if (nparts == 1) w.result[id] = r; else if (r) atomicAdd(&w.result[id], r);
        if (r >> 32) atomicAdd(&w.ctl->body_errors.v, r >> 32);
    } else if (part == 0) w.result[id] = r;
}

// Thread 0 of a task-part worker: record_result; an unknown body id (result ~0) aborts the window.
__device__ __forceinline__ void store_result(const WinDev& w, const pb2_task_t& t, int32_t id, int part, int nparts,
                                             unsigned long long r) {
    if (r == ~0ull) st_relaxed_gpu(reinterpret_cast<int32_t*>(&w.ctl->done.v), kDoneBadBody);
    record_result(w, t.body, id, part, nparts, r);
}

}  // namespace pb2
