// pb2_stream.cu -- the streaming engine: host-written command ring, ONE persistent sm_100a kernel per GPU, retire ring
// back to the host (include/pb2_stream.h).  Original design; what it stands in for in the reference:
//   parsec_device_progress_stream + the exec-stream rings            parsec/mca/device/device_gpu.c:2592-2731
//   parsec_device_kernel_push / _exec / _pop (per task, per stream)  device_gpu.c:2745, :2873, :2943
//   parsec_release_dep_fct for edges between in-flight GPU tasks     parsec/parsec.c:1836
//
// Device side: CTA 0 is the DISPATCHER (its warp 0 reads commands from pinned host memory, 32 at a time, fills the
// device-resident task / tile / edge tables and pushes ready tasks on the ready ring); every other CTA is a WORKER
// running pb2_worker.cuh::run_task_part on what it pops.  A worker that finishes a task closes the task's edge
// list, decrements its successors' dependency words, pushes the ones that reach zero, and only then publishes the
// retire record, so the host can recycle the ticket and the edge nodes as soon as it sees the record.
#include <cuda_runtime.h>
#include <stdio.h>
#include <stdlib.h>
#include <string.h>
#include <atomic>
#include <deque>
#include <mutex>
#include <vector>

#include "../../include/pb2_stream.h"
#include "pb2_engine_priv.hpp"
#include "pb2_worker.cuh"

namespace pb2 {

enum : uint8_t { CMD_NONE = 0, CMD_TASK = 1, CMD_TILE = 2, CMD_EDGE = 3 };
enum : uint32_t { HS_STOPPED = 0, HS_RUNNING = 1, HS_ERROR = 2 };
constexpr int32_t kEdgeEmpty = -1;
constexpr int32_t kEdgeDone = -2;

// 64 bytes, written by the host with plain stores; `stamp` (the generation of the ring index, never 0) is stored last.
struct alignas(64) Cmd {
    uint8_t  op, body, nb_flows, flags;
    uint16_t nparts, dep_goal;
    union {
        struct { int32_t ticket; int32_t tile[PB2_MAX_FLOWS]; uint8_t access[PB2_MAX_FLOWS];
                 int32_t iparam[3]; float fparam; int32_t locals[2]; } task;                    // 48 B
        struct { int32_t tile; int32_t state; uint32_t version; int32_t src_kind;
                 uint64_t dev_ptr; uint64_t src_ptr; uint32_t bytes; } tset;                     // 36 B (+4 pad)
        struct { int32_t pred, succ, node; } edge;
        uint32_t raw[12];
    } u;                    // 48 bytes at offset 8
    uint32_t pad;
    uint32_t stamp;         // offset 60
};
static_assert(sizeof(Cmd) == 64, "Cmd must be one 64-byte line");

// 32 bytes, written by a worker into pinned host memory; the 16 bytes holding `stamp` are stored last.
struct alignas(32) Retire {
    uint32_t seen[PB2_MAX_FLOWS];
    uint64_t result;
    int32_t  ticket;
    uint32_t stamp;        // generation of the retire index (never 0); low bit 31 set => bad body
};
static_assert(sizeof(Retire) == 32, "Retire must be 32 bytes");

// params.trace: one per retire index, written before the retire record of the same index
struct alignas(32) TraceRec { unsigned long long t_start, t_end; uint32_t smid; int32_t ticket; uint32_t pad[2]; };

struct HostCtl {            // pinned host memory, written by both sides
    volatile uint32_t state;        // HS_*
    volatile uint32_t stop_req;     // host -> device: park as soon as nothing is in flight
    volatile uint32_t error;        // kDone* code when state == HS_ERROR
    volatile uint32_t pad;
    char pad0[48];                  // `state` changes a few times per run and is read at every kick: its own line
    volatile unsigned long long cmd_consumed;   // device -> host: commands the dispatcher has taken (rewritten all the time)
    char pad1[56];
};

struct SCtl {               // device memory
    unsigned long long cmd_head;        // next command index (dispatcher only; survives a park)
    unsigned long long dispatched;      // tasks handed to the tables
    Line published;                     // tasks whose retire record is visible to the host
    Line released;                      // tasks made ready by a device-side decrement
    Line edges_late;                    // edges the dispatcher found already satisfied
};

struct StreamDev {
    WinDev w;
    const Cmd* cmd; uint32_t cmd_mask;
    Retire* ret;   uint32_t ret_mask;
    HostCtl* hctl;
    SCtl* sctl;
    int32_t* succ_head;     // per ticket: kEdgeEmpty, kEdgeDone or the first edge node
    int32_t* edge_next;     // per node
    int32_t* edge_succ;     // per node
    uint16_t* nparts_rw;    // == w.nparts, writable alias for the dispatcher
    pb2_task_t* tasks_rw;   // == w.tasks
    unsigned long long idle_ns;
    TraceRec* trace;        // pinned host memory, nullptr unless params.trace
};

__device__ __forceinline__ uint32_t ld_volatile_u32(const volatile uint32_t* p) { return *p; }
__device__ __forceinline__ void st_volatile_v8(void* p, const uint4& a, const uint4& b) {      // 32-byte aligned
    asm volatile("st.volatile.global.v8.b32 [%0], {%1,%2,%3,%4,%5,%6,%7,%8};"
                 :: "l"(p), "r"(a.x), "r"(a.y), "r"(a.z), "r"(a.w), "r"(b.x), "r"(b.y), "r"(b.z), "r"(b.w) : "memory");
}
__device__ __forceinline__ void st_volatile_v4(void* p, const uint4& v) {
    asm volatile("st.volatile.global.v4.u32 [%0], {%1,%2,%3,%4};" :: "l"(p), "r"(v.x), "r"(v.y), "r"(v.z), "r"(v.w) : "memory");
}

// One thread: push the ring entries of ready task `slot`.
__device__ __forceinline__ void push_ready(const WinDev& w, int32_t slot, int np) {
    const uint32_t first = (uint32_t)atomicAdd(&w.ctl->tail.v, (unsigned long long)np);
    for (int p = 0; p < np; ++p) st_release_gpu(&w.ring[(first + (uint32_t)p) & w.cap_mask], PB2_ENT_MAKE(slot, p));
}

// One thread: take the next pop ticket and wait for its slot; the slot is handed back empty (the ring wraps).
__device__ __forceinline__ int32_t stream_pop(const WinDev& w) {
    const uint32_t ticket = (uint32_t)atomicAdd(&w.ctl->head.v, 1ull);
    int32_t* slot = &w.ring[ticket & w.cap_mask];
    uint32_t spins = 0;
    int32_t id;
    while ((id = ld_acquire_gpu(slot)) == kEmpty) {
        if (ld_relaxed_gpu(reinterpret_cast<const int32_t*>(&w.ctl->done.v)) != 0) return kEmpty;
        ++spins;
        __nanosleep(spins < 64 ? 32 : 256);
    }
    st_relaxed_gpu(slot, kEmpty);
    return id;
}

// ---------------------------------------------------------------------------------------------
// dispatcher (warp 0 of CTA 0)
// ---------------------------------------------------------------------------------------------
__device__ __forceinline__ void dispatcher_warp(const StreamDev& sd) {
    const WinDev& w = sd.w;
    const int lane = threadIdx.x & 31;
    unsigned long long head = sd.sctl->cmd_head;
    unsigned long long dispatched = sd.sctl->dispatched;
    unsigned long long last_work = globaltimer_ns();
    if (lane == 0) { sd.hctl->state = HS_RUNNING; __threadfence_system(); }
    for (;;) {
        // phase 1: which of the next 32 commands are there?  (stamp == generation of the index, stored last)
        const unsigned long long idx = head + (unsigned long long)lane;
        const Cmd* c = &sd.cmd[idx & sd.cmd_mask];
        const uint32_t want = ring_gen(idx, sd.cmd_mask + 1ull);
        const uint32_t got = ld_volatile_u32(&c->stamp);
        const unsigned validm = __ballot_sync(0xffffffffu, got == want);
        const int n = (validm == 0xffffffffu) ? 32 : (__ffs(~validm) - 1);
        if (n == 0) {
            int leave = 0;
            if (lane == 0) {
                const unsigned long long now = globaltimer_ns();
                const unsigned long long pub = *reinterpret_cast<volatile unsigned long long*>(&sd.sctl->published.v);
                const bool quiet = (pub == dispatched);
                if (quiet && (ld_volatile_u32(&sd.hctl->stop_req) != 0 || (long long)(now - last_work) > (long long)sd.idle_ns)) {
                    // park: tell the host first, then look once more -- a command stored before the host saw STOPPED
                    // is either seen here (we stay) or the host relaunches (it re-reads the state after storing)
                    sd.hctl->state = HS_STOPPED;
                    __threadfence_system();
                    if (ld_volatile_u32(&sd.cmd[head & sd.cmd_mask].stamp) == ring_gen(head, sd.cmd_mask + 1ull)) {
                        sd.hctl->state = HS_RUNNING;
                        __threadfence_system();
                    } else leave = 1;
                } else if (!quiet) {
                    const unsigned long long last = *reinterpret_cast<volatile unsigned long long*>(&w.ctl->progress_ns.v);
                    const unsigned long long ref = last > last_work ? last : last_work;
                    if ((long long)(now - ref) > (long long)w.timeout_ns) {
                        sd.hctl->error = (uint32_t)kDoneTimeout; sd.hctl->state = HS_ERROR;
                        __threadfence_system();
                        st_relaxed_gpu(reinterpret_cast<int32_t*>(&w.ctl->done.v), kDoneTimeout);
                        leave = 2;
                    }
                } else if (ld_relaxed_gpu(reinterpret_cast<const int32_t*>(&w.ctl->done.v)) == kDoneBadBody) {
                    sd.hctl->error = (uint32_t)kDoneBadBody; sd.hctl->state = HS_ERROR;
                    __threadfence_system();
                    leave = 2;
                }
            }
            leave = __shfl_sync(0xffffffffu, leave, 0);
            if (leave) {
                if (lane == 0) {
                    sd.sctl->cmd_head = head; sd.sctl->dispatched = dispatched;
                    __threadfence();
                    if (leave == 1) st_release_gpu(reinterpret_cast<int32_t*>(&w.ctl->done.v), kDoneOK);
                }
                return;
            }
            __nanosleep(200);
            continue;
        }
        __threadfence_system();     // acquire: the payload reads below come after the stamp reads
        // phase 2: every lane < n loads its command (four 16-byte loads from pinned host memory)
        uint4 q0 = make_uint4(0, 0, 0, 0), q1 = q0, q2 = q0, q3 = q0;
        if (lane < n) {
            const uint4* p = reinterpret_cast<const uint4*>(c);
            q0 = ld_remote(p); q1 = ld_remote(p + 1); q2 = ld_remote(p + 2); q3 = ld_remote(p + 3);
        }
        const uint8_t op = (lane < n) ? (uint8_t)(q0.x & 0xffu) : (uint8_t)CMD_NONE;
        const int np = (int)(q0.y & 0xffffu), goal = (int)(q0.y >> 16);
        // phase A: tables (tiles, task descriptors, dependency words) -- no command of this batch is visible to a
        // worker yet, so the lanes may fill them in any order
        int32_t ticket = -1;
        if (op == CMD_TILE) {
            const int32_t tile = (int32_t)q0.z;
            if (tile >= 0 && tile < w.ntiles) {
                pb2_tile_t t;
                t.state = (int32_t)q0.w; t.version = q1.x; t.src_kind = (int32_t)q1.y;
                t.dev_ptr = reinterpret_cast<void*>(((unsigned long long)q1.w << 32) | q1.z);
                t.src_ptr = reinterpret_cast<void*>(((unsigned long long)q2.y << 32) | q2.x);
                t.bytes = q2.z;
                w.tiles[tile] = t;
                if (w.slice_claim && t.state != PB2_TILE_VALID) reset_tile_slices(w, (size_t)tile);
            }
        } else if (op == CMD_TASK) {
            ticket = (int32_t)q0.z;
            pb2_task_t t;
            t.dep_goal = goal; t.succ_begin = 0; t.succ_count = 0; t.priority = 0;
            t.body = (uint8_t)((q0.x >> 8) & 0xffu); t.nb_flows = (uint8_t)((q0.x >> 16) & 0xffu);
            t.flags = (uint8_t)(q0.x >> 24); t.class_id = 0;
            t.tile[0] = (int32_t)q0.w; t.tile[1] = (int32_t)q1.x; t.tile[2] = (int32_t)q1.y; t.tile[3] = (int32_t)q1.z;
            t.access[0] = (uint8_t)(q1.w & 0xffu); t.access[1] = (uint8_t)((q1.w >> 8) & 0xffu);
            t.access[2] = (uint8_t)((q1.w >> 16) & 0xffu); t.access[3] = (uint8_t)(q1.w >> 24);
            t.iparam[0] = (int32_t)q2.x; t.iparam[1] = (int32_t)q2.y; t.iparam[2] = (int32_t)q2.z;
            t.fparam = __uint_as_float(q2.w);
            t.locals[0] = (int32_t)q3.x; t.locals[1] = (int32_t)q3.y;
            sd.tasks_rw[ticket] = t;
            w.dep[ticket] = goal;
            sd.succ_head[ticket] = kEdgeEmpty;
            sd.nparts_rw[ticket] = (uint16_t)np;
            w.parts_left[ticket] = np;
            w.result[ticket] = 0;
        }
        __threadfence();
        __syncwarp();
        // phase B: ready tasks enter the ring in command order
        push_ready_warp<false>(w, ticket, (op == CMD_TASK && goal == 0) ? np : 0);
        // phase C: look-ahead edges.  A predecessor that has already closed its list counts as satisfied.
        if (op == CMD_EDGE) {
            const int32_t pred = (int32_t)q0.z, succ = (int32_t)q0.w, node = (int32_t)q1.x;
            sd.edge_succ[node] = succ;
            int32_t old = ld_acquire_gpu(&sd.succ_head[pred]);
            for (;;) {
                if (old == kEdgeDone) {
                    atomicAdd(&sd.sctl->edges_late.v, 1ull);
                    if (atomicSub(&w.dep[succ], 1) == 1) push_ready(w, succ, (int)sd.nparts_rw[succ]);
                    break;
                }
                sd.edge_next[node] = old;
                __threadfence();
                const int32_t seen = atomicCAS(&sd.succ_head[pred], old, node);
                if (seen == old) break;
                old = seen;
            }
        }
        const unsigned ntask = __popc(__ballot_sync(0xffffffffu, op == CMD_TASK));
        dispatched += ntask;
        head += (unsigned long long)n;
        last_work = globaltimer_ns();
        if (lane == 0) sd.hctl->cmd_consumed = head;       // posted write; the host only uses it for flow control
    }
}

// ---------------------------------------------------------------------------------------------
// the persistent streaming kernel
// ---------------------------------------------------------------------------------------------
#ifndef PB2_STREAM_MINB
#define PB2_STREAM_MINB 12
#endif
__global__ void __launch_bounds__(64, PB2_STREAM_MINB)
pb2_stream_kernel(StreamDev sd) {
    const WinDev& w = sd.w;
    if (blockIdx.x == 0) {                 // the dispatcher CTA
        if (threadIdx.x < 32) dispatcher_warp(sd);
        return;
    }
    __shared__ TaskSmem s;
    __shared__ BulkSmem bulk;
    if (threadIdx.x == 0) bulk_init(bulk);
    __syncthreads();
    for (;;) {
        if (threadIdx.x == 0) {
            const int32_t e = stream_pop(w);
            if (e != kEmpty) __threadfence();
            s.entry = e;
        }
        __syncthreads();
        const int32_t entry = s.entry;
        if (entry == kEmpty) break;
        const unsigned long long t_pop = (sd.trace != nullptr && threadIdx.x == 0) ? globaltimer_ns() : 0ull;
        const int32_t id = PB2_ENT_TASK(entry);
        const int part = PB2_ENT_PART(entry);
        // the task table is rewritten when tickets are recycled: read it at L2, never through a read-only path
        if (threadIdx.x < 4) reinterpret_cast<uint4*>(&s.task)[threadIdx.x] =
            __ldcg(reinterpret_cast<const uint4*>(&w.tasks[id]) + threadIdx.x);
        __syncthreads();
        const int nparts = (int)__ldcg(&w.nparts[id]);
        const unsigned long long r = run_task_part(w, s, &bulk, id, part, nparts);

        if (threadIdx.x == 0) {
            __threadfence();
            const pb2_task_t& t = s.task;
            store_result(w, t, id, part, nparts, r);
            int last = 1;
            if (nparts > 1) { last = atomicSub(&w.parts_left[id], 1) == 1; __threadfence(); }
            if (last) {
                epilog_written_flows(w, t);
                // the retire INDEX is taken before the out-edges are released (the host drains records in index
                // order, so its view is a linear extension of the DAG); the RECORD is published after the release
                // walk, so the host never recycles a ticket or an edge node this thread still reads
                const unsigned long long ridx = atomicAdd(&w.ctl->retired.v, 1ull);
                *reinterpret_cast<volatile unsigned long long*>(&w.ctl->progress_ns.v) = globaltimer_ns();
                __threadfence();
                int32_t node = atomicExch(&sd.succ_head[id], kEdgeDone);
                while (node >= 0) {
                    const int32_t succ = __ldcg(&sd.edge_succ[node]);
                    const int32_t next = __ldcg(&sd.edge_next[node]);
                    if (atomicSub(&w.dep[succ], 1) == 1) {
                        push_ready(w, succ, (int)__ldcg(&w.nparts[succ]));
                        atomicAdd(&sd.sctl->released.v, 1ull);
                    }
                    node = next;
                }
                if (sd.trace != nullptr) {
                    TraceRec* tr = &sd.trace[ridx & sd.ret_mask];
                    tr->t_start = t_pop; tr->t_end = globaltimer_ns(); tr->smid = smid(); tr->ticket = id;
                }
                Retire* rec = &sd.ret[ridx & sd.ret_mask];
                const uint32_t gen = ring_gen(ridx, sd.ret_mask + 1ull);
                const uint4 lo = __ldcg(reinterpret_cast<const uint4*>(&w.seen_version[(size_t)id * PB2_MAX_FLOWS]));
                const unsigned long long res = *reinterpret_cast<volatile unsigned long long*>(&w.result[id]);
                uint4 hi;
                hi.x = (uint32_t)res; hi.y = (uint32_t)(res >> 32); hi.z = (uint32_t)id;
                hi.w = (gen & 0x7fffffffu) | (r == ~0ull ? 0x80000000u : 0u);
                // What the host must see BEFORE the record -- bytes this task pushed out to host memory, its trace entry --
                // is ordered by one system-scope fence; a task that wrote nothing the host reads skips it.  The record
                // itself is ONE 32-byte store (a single sector write over PCIe): the host, which reads the stamp first,
                // never sees half of it, and the record is visible one posted write after the task ended.
                bool host_reads = sd.trace != nullptr;
                for (int f = 0; f < (int)t.nb_flows; ++f) host_reads |= (t.access[f] & PB2_FLOW_PUSHOUT) != 0;
                if (host_reads) __threadfence_system();
                st_volatile_v8(rec, lo, hi);
                __threadfence_system();
                atomicAdd(&sd.sctl->published.v, 1ull);
            }
        }
        __syncthreads();
    }
}

__global__ void pb2_stream_rearm_kernel(StreamDev sd) {
    // runs between two instances of the persistent kernel: every pop ticket of the parked instance is void
    sd.w.ctl->head.v = 0; sd.w.ctl->tail.v = 0; sd.w.ctl->done.v = 0;
    sd.w.ctl->progress_ns.v = globaltimer_ns();
}

}  // namespace pb2

// =============================================================================================
// host side
// =============================================================================================
using namespace pb2;

struct DryTask { pb2_task_t t; int32_t dep; std::vector<int32_t> succ; bool done; };

struct pb2_stream_s {
    pb2_engine_t* e = nullptr;
    pb2_stream_params_t p{};
    bool dry = false;
    std::string last_error;
    uint32_t slots = 0, ring_cap = 0;
    // pinned host memory
    Cmd* h_cmd = nullptr; Retire* h_ret = nullptr; HostCtl* h_ctl = nullptr; TraceRec* h_trace = nullptr;
    StreamDev d{};
    std::vector<void*> dev_allocs;
    cudaStream_t kstream = nullptr;
    int nworkers = 0;
    // Host bookkeeping, in two halves that two different threads may drive at the same time (include/pb2_stream.h):
    //   SUBMIT side (set_tile / submit / add_edge / kick): cmd_written, consumed_seen, free_tickets, the per-ticket arrays
    //   POLL side   (poll):                                ret_read
    // Tickets travel back from the poll side through a single-producer single-consumer ring; the in-flight counters are
    // atomics; per-ticket arrays are written before the command is published and read after its retire record arrived.
    unsigned long long cmd_written = 0;
    unsigned long long consumed_seen = 0;    // last value read from h_ctl->cmd_consumed (the device rewrites that line all the time)
    std::vector<int32_t> free_tickets, free_nodes;
    std::vector<uint64_t> cookie;            // per ticket
    std::vector<uint16_t> tk_parts;          // per ticket
    std::vector<std::vector<int32_t>> tk_nodes;   // per ticket: edge nodes that die with it
    std::vector<uint8_t> tk_live;
    alignas(64) unsigned long long ret_read = 0;
    std::vector<int32_t> freed;              // SPSC ring of tickets given back by poll, capacity `slots`
    alignas(64) std::atomic<uint64_t> freed_tail{0};   // written by poll
    alignas(64) std::atomic<uint64_t> freed_head{0};   // written by submit
    // counters: each side writes its own line; the other side reads it only when its last view is not good enough
    alignas(64) std::atomic<uint64_t> sub_tasks{0};     // submit side: tasks / ring entries handed to the device
    std::atomic<uint64_t> sub_entries{0};
    uint64_t ret_entries_seen = 0;                      // submit side's last view of ret_entries
    alignas(64) std::atomic<uint64_t> ret_tasks{0};     // poll side: tasks / ring entries whose record was read
    std::atomic<uint64_t> ret_entries{0};
    std::mutex launch_mu;                    // (re)launch of the persistent kernel: either side may find it parked
    std::mutex nodes_mu;                     // free_nodes: add_edge takes, poll gives back (look-ahead edges only)
    std::mutex dry_mu;                       // dry run: the emulated device is shared by both sides
    pb2_stream_stats_t st{};
    // dry run
    std::vector<DryTask> dry_tasks;
    std::deque<int32_t> dry_ready;
    std::vector<pb2_tile_t> dry_tiles;
    std::vector<uint32_t> tile_bytes;        // host mirror of the tile sizes (parts of wide tasks)
};

#define STREAM_CUDA(s, call)                                                                     \
    do {                                                                                         \
        cudaError_t err__ = (call);                                                              \
        if (err__ != cudaSuccess) {                                                              \
            char buf__[512];                                                                     \
            snprintf(buf__, sizeof buf__, "%s:%d %s -> %s", __FILE__, __LINE__, #call,           \
                     cudaGetErrorString(err__));                                                 \
            (s)->last_error = buf__;                                                             \
            fprintf(stderr, "pb2: CUDA error %s\n", buf__);                                      \
            return PB2_ERR_DEVICE;                                                               \
        }                                                                                        \
    } while (0)

template <class T>
static int sdev_alloc(pb2_stream_t* s, T** out, size_t n, int fill) {
    void* ptr = nullptr;
    STREAM_CUDA(s, cudaMalloc(&ptr, (n ? n : 1) * sizeof(T)));
    STREAM_CUDA(s, cudaMemset(ptr, fill, (n ? n : 1) * sizeof(T)));
    s->dev_allocs.push_back(ptr);
    *out = reinterpret_cast<T*>(ptr);
    return PB2_SUCCESS;
}

static uint32_t round_pow2(uint32_t v, uint32_t lo, uint32_t hi) {
    uint32_t r = lo;
    while (r < v && r < hi) r <<= 1;
    return r;
}

extern "C" {

const char* pb2_stream_last_error(pb2_stream_t* s) { return s ? s->last_error.c_str() : "null stream"; }

int pb2_stream_create(pb2_engine_t* e, const pb2_stream_params_t* params, pb2_stream_t** stream) {
    if (!stream) return PB2_ERR_BAD_PARAM;
    *stream = nullptr;
    pb2_stream_params_t p{};
    if (params) p = *params;
    if (!e && !p.dry_run) return PB2_ERR_BAD_PARAM;
    if (p.cmd_slots <= 0) p.cmd_slots = 65536;
    if (p.max_tiles <= 0) p.max_tiles = 65536;
    if (p.idle_us <= 0) p.idle_us = 2000;
    if (p.timeout_ms <= 0) p.timeout_ms = 20000;
    if (p.part_bytes == 0) p.part_bytes = 256 * 1024;
    pb2_stream_t* s = new pb2_stream_s();
    s->e = e; s->p = p; s->dry = p.dry_run != 0;
    s->slots = round_pow2((uint32_t)p.cmd_slots, 1024u, 1u << 21);
    s->ring_cap = s->slots * 4u;
    s->free_tickets.reserve(s->slots); s->free_nodes.reserve(s->slots);
    for (int32_t i = (int32_t)s->slots - 1; i >= 0; --i) { s->free_tickets.push_back(i); s->free_nodes.push_back(i); }
    s->tile_bytes.assign((size_t)p.max_tiles, 0);
    s->cookie.assign(s->slots, 0); s->tk_parts.assign(s->slots, 1); s->tk_nodes.resize(s->slots); s->tk_live.assign(s->slots, 0);
    s->freed.assign(s->slots, -1);
    if (s->dry) {
        s->dry_tasks.resize(s->slots);
        s->dry_tiles.resize((size_t)p.max_tiles);
        *stream = s;
        return PB2_SUCCESS;
    }
    STREAM_CUDA(s, cudaSetDevice(e->cuda_device));
    STREAM_CUDA(s, cudaHostAlloc(reinterpret_cast<void**>(&s->h_cmd), sizeof(Cmd) * s->slots, cudaHostAllocMapped | cudaHostAllocPortable));
    STREAM_CUDA(s, cudaHostAlloc(reinterpret_cast<void**>(&s->h_ret), sizeof(Retire) * s->slots, cudaHostAllocMapped | cudaHostAllocPortable));
    STREAM_CUDA(s, cudaHostAlloc(reinterpret_cast<void**>(&s->h_ctl), sizeof(HostCtl), cudaHostAllocMapped | cudaHostAllocPortable));
    memset(s->h_cmd, 0, sizeof(Cmd) * s->slots);
    memset(s->h_ret, 0, sizeof(Retire) * s->slots);
    memset((void*)s->h_ctl, 0, sizeof(HostCtl));
    StreamDev& d = s->d;
    void* alias = nullptr;
    STREAM_CUDA(s, cudaHostGetDevicePointer(&alias, s->h_cmd, 0)); d.cmd = reinterpret_cast<const Cmd*>(alias);
    STREAM_CUDA(s, cudaHostGetDevicePointer(&alias, s->h_ret, 0)); d.ret = reinterpret_cast<Retire*>(alias);
    STREAM_CUDA(s, cudaHostGetDevicePointer(&alias, (void*)s->h_ctl, 0)); d.hctl = reinterpret_cast<HostCtl*>(alias);
    d.cmd_mask = s->slots - 1; d.ret_mask = s->slots - 1;
    if (p.trace) {
        STREAM_CUDA(s, cudaHostAlloc(reinterpret_cast<void**>(&s->h_trace), sizeof(TraceRec) * s->slots, cudaHostAllocMapped | cudaHostAllocPortable));
        memset(s->h_trace, 0, sizeof(TraceRec) * s->slots);
        STREAM_CUDA(s, cudaHostGetDevicePointer(&alias, s->h_trace, 0)); d.trace = reinterpret_cast<TraceRec*>(alias);
    }
    int rc;
#define TRY(x) do { rc = (x); if (rc != PB2_SUCCESS) { pb2_stream_destroy(s); return rc; } } while (0)
    WinDev& w = d.w;
    memset(&w, 0, sizeof w);
    TRY(sdev_alloc(s, &d.tasks_rw, s->slots, 0)); w.tasks = d.tasks_rw;
    TRY(sdev_alloc(s, &w.tiles, (size_t)p.max_tiles, 0));
    TRY(sdev_alloc(s, &w.dep, s->slots, 0));
    TRY(sdev_alloc(s, &w.ring, s->ring_cap, 0xff));
    TRY(sdev_alloc(s, &w.ctl, 1, 0));
    TRY(sdev_alloc(s, &w.seen_version, (size_t)s->slots * PB2_MAX_FLOWS, 0));
    TRY(sdev_alloc(s, &w.result, s->slots, 0));
    TRY(sdev_alloc(s, &w.parts_left, s->slots, 0));
    TRY(sdev_alloc(s, &d.nparts_rw, s->slots, 0)); w.nparts = d.nparts_rw;
    TRY(sdev_alloc(s, &w.slice_claim, (size_t)p.max_tiles * PB2_SLICE_WORDS, 0));
    TRY(sdev_alloc(s, &w.slice_done, (size_t)p.max_tiles * (PB2_SLICE_WORDS + 1), 0));
    TRY(sdev_alloc(s, &d.sctl, 1, 0));
    TRY(sdev_alloc(s, &d.succ_head, s->slots, 0xff));
    TRY(sdev_alloc(s, &d.edge_next, s->slots, 0xff));
    TRY(sdev_alloc(s, &d.edge_succ, s->slots, 0xff));
#undef TRY
    w.cap_mask = s->ring_cap - 1; w.ntasks = (int32_t)s->slots; w.ntiles = p.max_tiles;
    w.stage_mode = e->params.stage_mode;
    // device-side slicing of stage-in (see pb2_window_create): finer than the parts of wide tasks
    w.part_bytes = (e->stage_slice_bytes > 0 && (p.part_bytes <= 0 || e->stage_slice_bytes < p.part_bytes)) ? e->stage_slice_bytes : p.part_bytes;
    w.timeout_ns = (unsigned long long)p.timeout_ms * 1000000ull;
    d.idle_ns = (unsigned long long)p.idle_us * 1000ull;
    STREAM_CUDA(s, cudaStreamCreateWithFlags(&s->kstream, cudaStreamNonBlocking));
    int occ = 0;
    STREAM_CUDA(s, cudaOccupancyMaxActiveBlocksPerMultiprocessor(&occ, pb2_stream_kernel, 64, 0));
    if (occ > PB2_STREAM_MINB) occ = PB2_STREAM_MINB;
    if (occ < 1) occ = 1;
    s->nworkers = e->prop.multiProcessorCount * occ;
    if (p.max_workers > 0 && p.max_workers + 1 < s->nworkers) s->nworkers = p.max_workers + 1;
    if (s->nworkers < 2) s->nworkers = 2;
    *stream = s;
    return PB2_SUCCESS;
}

int pb2_stream_destroy(pb2_stream_t* s) {
    if (!s) return PB2_ERR_BAD_PARAM;
    if (!s->dry) {
        cudaSetDevice(s->e->cuda_device);
        if (s->kstream) {
            if (s->h_ctl) s->h_ctl->stop_req = 1;
            cudaStreamSynchronize(s->kstream);
            cudaStreamDestroy(s->kstream);
        }
        for (void* p : s->dev_allocs) cudaFree(p);
        if (s->h_cmd) cudaFreeHost(s->h_cmd);
        if (s->h_ret) cudaFreeHost(s->h_ret);
        if (s->h_ctl) cudaFreeHost((void*)s->h_ctl);
        if (s->h_trace) cudaFreeHost(s->h_trace);
    }
    delete s;
    return PB2_SUCCESS;
}

static int stream_launch_if_parked(pb2_stream_t* s) {
    if (s->dry) return PB2_SUCCESS;
    std::atomic_thread_fence(std::memory_order_seq_cst);
    uint32_t st = s->h_ctl->state;
    if (st == HS_RUNNING) return PB2_SUCCESS;
    if (st == HS_ERROR) { s->last_error = "streaming kernel aborted (watchdog or unknown body)"; return PB2_ERR_DEVICE; }
    std::lock_guard<std::mutex> guard(s->launch_mu);
    st = s->h_ctl->state;                       // the other side may have relaunched it meanwhile
    if (st == HS_RUNNING) return PB2_SUCCESS;
    if (st == HS_ERROR) { s->last_error = "streaming kernel aborted (watchdog or unknown body)"; return PB2_ERR_DEVICE; }
    STREAM_CUDA(s, cudaSetDevice(s->e->cuda_device));
    s->h_ctl->state = HS_RUNNING;
    std::atomic_thread_fence(std::memory_order_seq_cst);
    pb2_stream_rearm_kernel<<<1, 1, 0, s->kstream>>>(s->d);
    pb2_stream_kernel<<<s->nworkers, 64, 0, s->kstream>>>(s->d);
    STREAM_CUDA(s, cudaGetLastError());
    s->st.kernel_launches++;
    return PB2_SUCCESS;
}

// reserve the next command slot (waits for the dispatcher when the ring is full)
static int stream_cmd_slot(pb2_stream_t* s, Cmd** out) {
    // flow control reads the device-written counter only when the last value seen says the ring could be full
    if (s->cmd_written - s->consumed_seen >= (unsigned long long)s->slots) s->consumed_seen = s->h_ctl->cmd_consumed;
    if (s->cmd_written - s->consumed_seen >= (unsigned long long)s->slots) {
        int rc = stream_launch_if_parked(s);
        if (rc != PB2_SUCCESS) return rc;
        unsigned long long spins = 0;
        while (s->cmd_written - s->h_ctl->cmd_consumed >= (unsigned long long)s->slots) {
            if (s->h_ctl->state == HS_ERROR) { s->last_error = "streaming kernel aborted"; return PB2_ERR_DEVICE; }
            if ((++spins & 0xfffff) == 0 && s->h_ctl->state == HS_STOPPED) { rc = stream_launch_if_parked(s); if (rc != PB2_SUCCESS) return rc; }
        }
        s->consumed_seen = s->h_ctl->cmd_consumed;
    }
    *out = &s->h_cmd[s->cmd_written & (s->slots - 1)];
    // the slots a few commands ahead: last read by the device a lap ago, nowhere near this core's cache
    __builtin_prefetch(&s->h_cmd[(s->cmd_written + 6) & (s->slots - 1)], 1, 3);
    return PB2_SUCCESS;
}
static void stream_cmd_publish(pb2_stream_t* s, Cmd* c) {
    const uint32_t gen = ring_gen(s->cmd_written, s->slots);
    std::atomic_thread_fence(std::memory_order_release);
    *reinterpret_cast<volatile uint32_t*>(&c->stamp) = gen;
    s->cmd_written++;
}

int pb2_stream_set_tile(pb2_stream_t* s, int32_t tile, const pb2_tile_t* desc) {
    if (!s || !desc || tile < 0 || tile >= s->p.max_tiles) return PB2_ERR_BAD_PARAM;
    s->tile_bytes[(size_t)tile] = desc->bytes;
    if (s->dry) { s->dry_tiles[(size_t)tile] = *desc; return PB2_SUCCESS; }
    Cmd* c;
    int rc = stream_cmd_slot(s, &c);
    if (rc != PB2_SUCCESS) return rc;
    memset(c, 0, 60);
    c->op = CMD_TILE;
    c->u.tset.tile = tile; c->u.tset.state = desc->state; c->u.tset.version = desc->version; c->u.tset.src_kind = desc->src_kind;
    c->u.tset.dev_ptr = (uint64_t)(uintptr_t)desc->dev_ptr; c->u.tset.src_ptr = (uint64_t)(uintptr_t)desc->src_ptr;
    c->u.tset.bytes = desc->bytes;
    stream_cmd_publish(s, c);
    return PB2_SUCCESS;
}

int pb2_stream_submit(pb2_stream_t* s, const pb2_task_t* task, uint64_t cookie, int32_t* ticket) {
    if (!s || !task) return PB2_ERR_BAD_PARAM;
    if (task->nb_flows > PB2_MAX_FLOWS) { s->last_error = "task with more than PB2_MAX_FLOWS flows"; return PB2_ERR_BAD_PARAM; }
    if (task->body >= PB2_BODY_MAX || task->body == PB2_BODY_USER || task->body == PB2_BODY_GEMM_BF16) {
        s->last_error = "body cannot run in the streaming kernel"; return PB2_ERR_NOT_SUPPORTED; }
    if (task->dep_goal < 0 || task->dep_goal > 0xffff) return PB2_ERR_VALUE_OUT_OF_BOUNDS;
    for (int f = 0; f < task->nb_flows; ++f)
        if (task->tile[f] >= s->p.max_tiles) { s->last_error = "tile id out of bounds"; return PB2_ERR_VALUE_OUT_OF_BOUNDS; }
    if (s->free_tickets.empty()) {              // take back what the poll side has retired
        uint64_t h = s->freed_head.load(std::memory_order_relaxed);
        const uint64_t t = s->freed_tail.load(std::memory_order_acquire);
        for (; h != t; ++h) s->free_tickets.push_back(s->freed[h & (s->slots - 1)]);
        s->freed_head.store(h, std::memory_order_release);
        if (s->free_tickets.empty()) return PB2_ERR_OUT_OF_RESOURCE;
    }
    // parts: the tile_parts of the widest tile, the rule the device applies to the slices of a tile
    uint32_t np = 1;
    if (s->p.part_bytes > 0 && task->body != PB2_BODY_NOP) {
        uint32_t big = 0;
        for (int f = 0; f < task->nb_flows; ++f)
            if (task->tile[f] >= 0 && s->tile_bytes[(size_t)task->tile[f]] > big) big = s->tile_bytes[(size_t)task->tile[f]];
        np = (uint32_t)tile_parts(big, s->p.part_bytes);
    }
    {   // ready-ring capacity: entries in flight, with a view of the poll side's counter that is refreshed only when needed
        const uint64_t sub = s->sub_entries.load(std::memory_order_relaxed);
        if (sub - s->ret_entries_seen + np + 64 > (uint64_t)s->ring_cap / 2) {
            s->ret_entries_seen = s->ret_entries.load(std::memory_order_acquire);
            if (sub - s->ret_entries_seen + np + 64 > (uint64_t)s->ring_cap / 2) return PB2_ERR_OUT_OF_RESOURCE;
        }
    }
    const int32_t tk = s->free_tickets.back();
    if (s->dry) {
        std::lock_guard<std::mutex> guard(s->dry_mu);
        s->free_tickets.pop_back();
        s->cookie[(size_t)tk] = cookie; s->tk_parts[(size_t)tk] = (uint16_t)np; s->tk_live[(size_t)tk] = 1;
        s->sub_entries.store(s->sub_entries.load(std::memory_order_relaxed) + np, std::memory_order_relaxed);
        s->sub_tasks.store(s->sub_tasks.load(std::memory_order_relaxed) + 1, std::memory_order_release);
        if (ticket) *ticket = tk;
        DryTask& dt = s->dry_tasks[(size_t)tk];
        dt.t = *task; dt.dep = task->dep_goal; dt.succ.clear(); dt.done = false;
        if (dt.dep == 0) s->dry_ready.push_back(tk);
    } else {
        Cmd* c;
        int rc = stream_cmd_slot(s, &c);
        if (rc != PB2_SUCCESS) return rc;
        s->free_tickets.pop_back();
        s->cookie[(size_t)tk] = cookie; s->tk_parts[(size_t)tk] = (uint16_t)np; s->tk_live[(size_t)tk] = 1;
        memset(c, 0, 60);
        c->op = CMD_TASK; c->body = task->body; c->nb_flows = task->nb_flows; c->flags = task->flags;
        c->nparts = (uint16_t)np; c->dep_goal = (uint16_t)task->dep_goal;
        c->u.task.ticket = tk;
        for (int f = 0; f < PB2_MAX_FLOWS; ++f) { c->u.task.tile[f] = f < task->nb_flows ? task->tile[f] : -1; c->u.task.access[f] = task->access[f]; }
        c->u.task.iparam[0] = task->iparam[0]; c->u.task.iparam[1] = task->iparam[1]; c->u.task.iparam[2] = task->iparam[2];
        c->u.task.fparam = task->fparam; c->u.task.locals[0] = task->locals[0]; c->u.task.locals[1] = task->locals[1];
        s->sub_entries.store(s->sub_entries.load(std::memory_order_relaxed) + np, std::memory_order_relaxed);
        s->sub_tasks.store(s->sub_tasks.load(std::memory_order_relaxed) + 1, std::memory_order_release);
        if (ticket) *ticket = tk;               // before the command is visible: the caller's record may be recycled right after
        stream_cmd_publish(s, c);
    }
    return PB2_SUCCESS;
}

int pb2_stream_add_edge(pb2_stream_t* s, int32_t pred, int32_t succ) {
    if (!s || pred < 0 || succ < 0 || pred >= (int32_t)s->slots || succ >= (int32_t)s->slots) return PB2_ERR_BAD_PARAM;
    if (!s->tk_live[(size_t)pred] || !s->tk_live[(size_t)succ]) { s->last_error = "edge names a ticket that is not in flight"; return PB2_ERR_BAD_PARAM; }
    s->st.edges++;
    if (s->dry) {
        std::lock_guard<std::mutex> guard(s->dry_mu);
        DryTask& p = s->dry_tasks[(size_t)pred];
        if (p.done) { if (--s->dry_tasks[(size_t)succ].dep == 0) s->dry_ready.push_back(succ); }
        else p.succ.push_back(succ);
        return PB2_SUCCESS;
    }
    Cmd* c;
    int rc = stream_cmd_slot(s, &c);
    if (rc != PB2_SUCCESS) return rc;
    int32_t node;
    {
        std::lock_guard<std::mutex> guard(s->nodes_mu);
        if (s->free_nodes.empty()) return PB2_ERR_OUT_OF_RESOURCE;
        node = s->free_nodes.back(); s->free_nodes.pop_back();
        s->tk_nodes[(size_t)pred].push_back(node);
    }
    memset(c, 0, 60);
    c->op = CMD_EDGE; c->u.edge.pred = pred; c->u.edge.succ = succ; c->u.edge.node = node;
    stream_cmd_publish(s, c);
    return PB2_SUCCESS;
}

int pb2_stream_kick(pb2_stream_t* s) {
    if (!s) return PB2_ERR_BAD_PARAM;
    if (s->dry || s->cmd_written == 0) return PB2_SUCCESS;
    return stream_launch_if_parked(s);          // a fence and one read of a line that changes a few times per run
}

int pb2_stream_poll(pb2_stream_t* s, pb2_retire_t* out, int32_t max) {
    if (!s || (max > 0 && !out)) return PB2_ERR_BAD_PARAM;
    int n = 0;
    if (s->dry) {
        std::lock_guard<std::mutex> guard(s->dry_mu);
        while (n < max && !s->dry_ready.empty()) {
            const int32_t tk = s->dry_ready.front(); s->dry_ready.pop_front();
            DryTask& dt = s->dry_tasks[(size_t)tk];
            dt.done = true;
            pb2_retire_t& r = out[n++];
            memset(&r, 0, sizeof r);
            r.cookie = s->cookie[(size_t)tk]; r.ticket = tk; r.status = PB2_SUCCESS;
            for (int f = 0; f < dt.t.nb_flows && f < PB2_MAX_FLOWS; ++f) {
                if (dt.t.tile[f] < 0) continue;
                pb2_tile_t& tl = s->dry_tiles[(size_t)dt.t.tile[f]];
                r.seen_version[f] = tl.version;
                if (dt.t.access[f] & PB2_FLOW_ACCESS_WRITE) tl.version++;
                tl.state = PB2_TILE_VALID;
            }
            for (int32_t sc : dt.succ) if (--s->dry_tasks[(size_t)sc].dep == 0) s->dry_ready.push_back(sc);
            dt.succ.clear();
            s->tk_live[(size_t)tk] = 0;
            const uint64_t ft = s->freed_tail.load(std::memory_order_relaxed);
            s->freed[ft & (s->slots - 1)] = tk;
            s->freed_tail.store(ft + 1, std::memory_order_release);
            s->ret_entries.store(s->ret_entries.load(std::memory_order_relaxed) + s->tk_parts[(size_t)tk], std::memory_order_release);
            s->ret_tasks.store(s->ret_tasks.load(std::memory_order_relaxed) + 1, std::memory_order_release);
        }
        return n;
    }
    if (s->h_ctl->state == HS_ERROR) {
        s->last_error = s->h_ctl->error == (uint32_t)kDoneTimeout ? "streaming kernel watchdog: no task retired within timeout"
                                                                  : "streaming kernel ran a task with an unknown body id";
        return s->h_ctl->error == (uint32_t)kDoneTimeout ? PB2_ERR_DEVICE : PB2_ERR_BAD_PARAM;
    }
    if (s->h_ctl->state == HS_STOPPED && s->sub_tasks.load(std::memory_order_acquire) != s->ret_tasks.load(std::memory_order_relaxed)) {
        // nobody kicked: every retire record already written is in the ring; anything else needs the kernel
        const Retire* nxt = &s->h_ret[s->ret_read & (s->slots - 1)];
        const uint32_t g = ring_gen(s->ret_read, s->slots) & 0x7fffffffu;
        if ((*reinterpret_cast<const volatile uint32_t*>(&nxt->stamp) & 0x7fffffffu) != g) {
            int rc = stream_launch_if_parked(s);
            if (rc != PB2_SUCCESS) return rc;
        }
    }
    while (n < max) {
        const Retire* rec = &s->h_ret[s->ret_read & (s->slots - 1)];
        __builtin_prefetch(&s->h_ret[(s->ret_read + 8) & (s->slots - 1)], 0, 3);
        const uint32_t gen = ring_gen(s->ret_read, s->slots) & 0x7fffffffu;
        const uint32_t stamp = *reinterpret_cast<const volatile uint32_t*>(&rec->stamp);
        if ((stamp & 0x7fffffffu) != gen) break;
        std::atomic_thread_fence(std::memory_order_acquire);
        const int32_t tk = *reinterpret_cast<const volatile int32_t*>(&rec->ticket);
        pb2_retire_t& r = out[n++];
        r.cookie = s->cookie[(size_t)tk]; r.result = *reinterpret_cast<const volatile uint64_t*>(&rec->result);
        for (int f = 0; f < PB2_MAX_FLOWS; ++f) r.seen_version[f] = *reinterpret_cast<const volatile uint32_t*>(&rec->seen[f]);
        r.ticket = tk; r.status = (stamp & 0x80000000u) ? PB2_ERR_BAD_PARAM : PB2_SUCCESS;
        if (s->h_trace) {
            const volatile TraceRec* tr = &s->h_trace[s->ret_read & (s->slots - 1)];
            r.t_start_ns = tr->t_start; r.t_end_ns = tr->t_end; r.smid = tr->smid; r.pad = 0;
        } else { r.t_start_ns = 0; r.t_end_ns = 0; r.smid = 0; r.pad = 0; }
        if (!s->tk_nodes[(size_t)tk].empty()) {
            std::lock_guard<std::mutex> guard(s->nodes_mu);
            for (int32_t nd : s->tk_nodes[(size_t)tk]) s->free_nodes.push_back(nd);
            s->tk_nodes[(size_t)tk].clear();
        }
        s->tk_live[(size_t)tk] = 0;
        const uint64_t ft = s->freed_tail.load(std::memory_order_relaxed);
        s->freed[ft & (s->slots - 1)] = tk;
        s->freed_tail.store(ft + 1, std::memory_order_release);
        s->ret_entries.store(s->ret_entries.load(std::memory_order_relaxed) + s->tk_parts[(size_t)tk], std::memory_order_release);
        s->ret_tasks.store(s->ret_tasks.load(std::memory_order_relaxed) + 1, std::memory_order_release);
        s->ret_read++;
    }
    return n;
}

int pb2_stream_quiesce(pb2_stream_t* s) {
    if (!s) return PB2_ERR_BAD_PARAM;
    if (s->dry) return PB2_SUCCESS;
    STREAM_CUDA(s, cudaSetDevice(s->e->cuda_device));
    if (s->cmd_written != s->h_ctl->cmd_consumed) { int rc = stream_launch_if_parked(s); if (rc != PB2_SUCCESS) return rc; }
    s->h_ctl->stop_req = 1;
    std::atomic_thread_fence(std::memory_order_seq_cst);
    STREAM_CUDA(s, cudaStreamSynchronize(s->kstream));
    s->h_ctl->stop_req = 0;
    if (s->h_ctl->state == HS_ERROR) { s->last_error = "streaming kernel aborted"; return PB2_ERR_DEVICE; }
    // a relaunch may have been queued behind the instance that just parked with commands still unread
    if (s->cmd_written != s->h_ctl->cmd_consumed) return pb2_stream_quiesce(s);
    return PB2_SUCCESS;
}

int pb2_stream_inflight(pb2_stream_t* s) { return s ? (int)(s->sub_tasks.load() - s->ret_tasks.load()) : 0; }

int pb2_stream_stats(pb2_stream_t* s, pb2_stream_stats_t* out) {
    if (!s || !out) return PB2_ERR_BAD_PARAM;
    if (!s->dry) {
        STREAM_CUDA(s, cudaSetDevice(s->e->cuda_device));
        Ctl c; SCtl sc;
        cudaStream_t aux = s->e->up_stream;
        STREAM_CUDA(s, cudaMemcpyAsync(&c, s->d.w.ctl, sizeof c, cudaMemcpyDeviceToHost, aux));
        STREAM_CUDA(s, cudaMemcpyAsync(&sc, s->d.sctl, sizeof sc, cudaMemcpyDeviceToHost, aux));
        STREAM_CUDA(s, cudaStreamSynchronize(aux));
        s->st.bytes_h2d = c.bytes_h2d.v; s->st.bytes_d2d = c.bytes_d2d.v; s->st.bytes_d2h = c.bytes_d2h.v;
        s->st.stage_ins = c.stage_ins.v; s->st.body_errors = c.body_errors.v;
        s->st.edges_late = sc.edges_late.v; s->st.released_on_device = sc.released.v;
    }
    s->st.submitted = s->sub_tasks.load(); s->st.retired = s->ret_tasks.load();
    *out = s->st;
    return PB2_SUCCESS;
}

}  // extern "C"
