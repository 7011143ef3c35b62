/*
 * device_b200_module.c -- one parsec_device_module_t per B200 (parsec/mca/device/device.h:145-189), driven by the
 * streaming engine of libparsec_b200.so (include/pb2_stream.h): a host-written command ring, ONE persistent sm_100a
 * kernel per GPU, a retire ring back.
 *
 * What is ours and what is PaRSEC's:
 *   - kernel_scheduler and everything under it (manager election, residency of the flows on the device, the choice of
 *     a transfer source, eviction and write-back, the run of the body, the epilog and the hand-back to
 *     __parsec_complete_execution) is this file; it replaces parsec_device_kernel_scheduler and its helpers
 *     (parsec/mca/device/device_gpu.c:3375-3613, :2592-3292, transfer_gpu.c) for modules of this component;
 *   - the coherency protocol of parsec_data_t stays PaRSEC's own (parsec_data_start/end_transfer_ownership_to_copy,
 *     parsec/data.c:313-458): the CPU side of the runtime reads the same states;
 *   - the device heap is PaRSEC's zone allocator (parsec/utils/zone_malloc.c) through the base-class helpers
 *     parsec_device_memory_reserve / _release / parsec_device_flush_lru (device_gpu.c:866-1100), exactly like the
 *     cuda, hip and level_zero components use them.
 *
 * Threading (SURVEY.md 8b "Threading"): any worker thread may call kernel_scheduler concurrently.  A caller does for its
 * own task whatever needs no device-wide decision (task record, recording of the body, residency of the flows -- under
 * `alloc_lock` when replicas have to be made or filled), puts the record into the slot-ring inbox and adds one to `owed`.
 * Two roles then drive the device.  The STARTER (whoever holds `starter_active`) drains the inbox in order and owns the
 * submit side of the stream: tile descriptions, command ring, events of the copy-engine and lane paths.  The MANAGER (the
 * caller that takes `owed` from 0 to 1, until it is back to 0: every completed task subtracts one) owns the poll side:
 * retire ring, copy-engine pushouts, and the hand-over of finished tasks to the worker pool, where their epilog and
 * __parsec_complete_execution run (b200_epilog_hook).  The LRUs are shared by the starter and the epilogs (`lru_lock`).
 */
#include "parsec/parsec_config.h"
#include "parsec/parsec_internal.h"
#include "parsec/sys/atomic.h"
#include "parsec/utils/mca_param.h"
#include "parsec/utils/debug.h"
#include "parsec/utils/zone_malloc.h"
#include "parsec/constants.h"
#include "parsec/data_internal.h"
#include "parsec/scheduling.h"
#include "parsec/execution_stream.h"
#include "parsec/mca/device/device.h"
#include "parsec/mca/device/device_gpu.h"
#include "parsec/mca/device/b200/device_b200.h"
#include "parsec/mca/device/b200/device_b200_internal.h"

#include "pb2_engine.h"
#include "pb2_stream.h"

#include <cuda_runtime_api.h>
#include <stddef.h>
#include <stdlib.h>
#include <string.h>
#include <stdio.h>
#include <limits.h>
#include <time.h>
static inline uint64_t b200_now_ns(void) { struct timespec ts; clock_gettime(CLOCK_MONOTONIC, &ts); return (uint64_t)ts.tv_sec * 1000000000ull + (uint64_t)ts.tv_nsec; }
#include <x86intrin.h>
#define B200_TSC() __rdtsc()

/* device_b200_nvtx: the host side of a device as NVTX ranges of the domain "parsec_b200" (header-only NVTX3: the calls are
 * no-ops unless a tool injected itself; what parsec/profiling_nvtx.c does for the profiling keys of device_gpu.c:348-381) */
#include <nvtx3/nvToolsExt.h>
static nvtxDomainHandle_t b200_nvtx_domain = NULL;
static inline void b200_nvtx_attr(nvtxEventAttributes_t *a, const char *name)
{
    memset(a, 0, sizeof *a);
    a->version = NVTX_VERSION; a->size = NVTX_EVENT_ATTRIB_STRUCT_SIZE;
    a->messageType = NVTX_MESSAGE_TYPE_ASCII; a->message.ascii = name;
}
static inline void b200_nvtx_push(const char *name)
{
    if( parsec_b200_nvtx ) { nvtxEventAttributes_t a; b200_nvtx_attr(&a, name); (void)nvtxDomainRangePushEx(b200_nvtx_domain, &a); }
}
static inline void b200_nvtx_pop(void)
{
    if( parsec_b200_nvtx ) (void)nvtxDomainRangePop(b200_nvtx_domain);
}
static inline void b200_nvtx_mark(const char *name)
{
    if( parsec_b200_nvtx ) { nvtxEventAttributes_t a; b200_nvtx_attr(&a, name); nvtxDomainMarkEx(b200_nvtx_domain, &a); }
}

/* ------------------------------------------------------------------------------------------------------------------ */
/* types                                                                                                                */
/* ------------------------------------------------------------------------------------------------------------------ */
/* The two locks of a module are taken once or twice per task by every worker thread.  parsec_atomic_lock backs off with
 * nanosleep(): right for the rarely contended locks of the runtime, a 50 us stall here.  A ticket lock instead: FIFO
 * hand-over, waiters spin on a line only the holder writes. */
typedef struct b200_lock_s {
    volatile uint32_t next;    char pad0[60];
    volatile uint32_t serving; char pad1[60];
} b200_lock_t;
static inline void b200_lock(b200_lock_t *l)
{
    const uint32_t t = __atomic_fetch_add(&l->next, 1, __ATOMIC_RELAXED);
    while( __atomic_load_n(&l->serving, __ATOMIC_ACQUIRE) != t ) _mm_pause();
}
static inline void b200_unlock(b200_lock_t *l)
{
    __atomic_store_n(&l->serving, l->serving + 1, __ATOMIC_RELEASE);
}

enum {
    BT_NEW = 0,        /* popped from the inbox, nothing reserved yet                                   */
    BT_STAGED,         /* resident and described to the device, waiting for room in the command ring      */
    BT_DMA_IN,         /* copy-engine stage-in of unregistered host memory in progress (event)          */
    BT_INFLIGHT,       /* descriptor in the command ring / running in the persistent kernel             */
    BT_LANE,           /* opaque submit body enqueued on the lane stream (event)                        */
    BT_DMA_OUT         /* copy-engine pushout in progress (event)                                       */
};

/* One record per task handed to the device.  Laid out by who touches what: the manager's hot path (inbox, submit,
 * retire) reads the first two lines and `cmd`, the worker that runs the epilog reads `proxy` and the task itself. */
typedef struct b200_task_s {
    parsec_list_item_t   item;
    parsec_gpu_task_t   *gpu_task;
    int32_t              state;
    int32_t              ticket;          /* pb2_stream ticket, -1 when none */
    int32_t              body;            /* enum pb2_body_e recorded by parsec_b200_task_body, -1: opaque body */
    int32_t              prepared;        /* the caller found every flow resident: residency, readers and versions are settled */
    int32_t              cmd_built;       /* `cmd` is ready for pb2_stream_submit */
    int32_t              recorded;        /* the caller of kernel_scheduler already ran the submit function in record mode */
    int32_t              has_complete_stage;
    uint32_t             dma_out_mask;    /* pushout flows that need the copy engine (home not device-visible) */
    uint64_t             result;
    uint64_t             cold_bytes;      /* bytes this task stages in over PCIe / NVLink (throttle, see b200_start_task) */
    struct parsec_device_b200_module_s *dev;
    int32_t              is_kernel;       /* PARSEC_GPU_TASK_TYPE_KERNEL (not a prefetch / warm-up pseudo task) */
    int32_t              defer_tiles;     /* tile descriptions go to tdesc[]: the starter hands them to the device */
    int32_t              ntdesc;
    pb2_task_t           cmd __attribute__((aligned(64)));   /* the engine command of this task (built by whoever settles its flows) */
    parsec_task_t        proxy __attribute__((aligned(64))); /* the completion task the worker pool runs for this one (b200_epilog_hook) */
    /* start path of tasks the manager has to look at, lane / copy-engine paths */
    int32_t              nb_args;
    int32_t              arg_flow[PB2_MAX_FLOWS];
    int32_t              iparam[3];
    float                fparam;
    uint32_t             peer_src_mask;   /* flows whose source copy on a peer GPU holds a reader for us */
    parsec_data_copy_t  *peer_src[MAX_PARAM_COUNT];
    int32_t              custom_stage;    /* b200_user_stage_in || b200_user_stage_out */
    cudaEvent_t          ev;              /* created the first time a copy-engine / lane path needs it */
    int32_t              ev_dev;          /* CUDA device the event belongs to, -1: none */
    struct b200_task_s  *next_free;       /* per-thread free list */
    struct b200_task_s  *next_done;       /* chain of finished tasks one proxy completes / lane_done stack */
    struct { int32_t tile; pb2_tile_t desc; } tdesc[MAX_PARAM_COUNT];   /* see defer_tiles */
} b200_task_t;

typedef struct b200_host_range_s { char *base; size_t len; char *alias; int lazy; } b200_host_range_t;   /* lazy: unregistered by its owner, still pinned (registration cache) */

typedef struct b200_trace_ev_s {
    char     name[24];
    int32_t  locals[2];
    int32_t  body, smid;
    uint64_t t_start_ns, t_end_ns, cold_bytes;
} b200_trace_ev_t;
#define B200_LINE __attribute__((aligned(64)))
/* Laid out by who writes what: every group below starts on its own cache line. */
typedef struct parsec_device_b200_module_s {
    parsec_device_cuda_module_t super;    /* generated CUDA bodies read cuda_index / the exec stream through this layout */
    /* read-mostly */
    pb2_engine_t        *engine;
    pb2_stream_t        *stream;
    int                  dry_run;
    char                *slab_base;
    uint8_t             *tile_described;  /* per heap block: the device tile table entry of the replica that starts here is current */
    b200_task_t * volatile *inbox_ring;   /* callers take a slot index with one fetch-and-add and store their task record there;
                                           * the starter reads the slots in order (pointers side by side: it can prefetch the records) */
    cudaStream_t         dma_stream;
    parsec_cuda_exec_stream_t *lane;      /* exec_stream[0]: what submit functions receive */
    uint64_t             first_entry_ns, first_task_ns, last_done_ns;
    /* callers of kernel_scheduler */
    volatile int64_t     inbox_tail B200_LINE;       /* next slot a caller takes */
    volatile int32_t     owed B200_LINE;             /* tasks handed over and not completed: 0 -> 1 elects the manager */
    volatile int32_t     callers_inside B200_LINE;
    volatile int32_t     max_callers_inside;
    /* worker threads */
    volatile int64_t     epilogs_done B200_LINE;     /* epilogs the worker threads have ended */
    b200_lock_t          lru_lock B200_LINE;         /* gpu_mem_lru / gpu_mem_owned_lru: the starter and the workers' epilogs */
    /* RESIDENCY of the flows of a task (device heap, choice of a source, tile descriptions) is decided under this lock,
     * by the calling worker for engine tasks, by the starter for the others.  A caller pushes its task into the inbox
     * BEFORE it lets the lock go: the inbox holds the decisions in the order they were taken. */
    b200_lock_t          alloc_lock B200_LINE;
    /* Two roles drive a device.  The STARTER (inbox, residency, stage-in decisions, command ring, events of the stage-in
     * and lane paths) is whichever thread holds `starter_active`: a caller of kernel_scheduler takes it when it is free
     * and keeps it while tasks keep arriving; the manager takes it when tasks that had to wait may go on.  The MANAGER
     * (elected through `owed`) owns the retire side: retire ring, pushouts through the copy engine, completion. */
    volatile int32_t     handed_back B200_LINE;      /* tasks the starter gave back to the runtime (b200_forward_peer): the manager
                                                      * subtracts them from `owed` like completions */
    volatile int32_t     starter_active B200_LINE;
    volatile int32_t     fatal;           /* the starter hit a fatal device problem: the manager gives the device up */
    volatile int32_t     memory_pressure; /* the heap has been full since the last memory_release: LRU order is kept from here on */
    struct b200_task_s * volatile lane_done;   /* finished lane tasks, starter -> manager (lock-free stack) */
    volatile int32_t     retry_stalled B200_LINE;    /* something happened that may let a waiting task start (a retirement, a newcomer,
                                                      * the end of an epilog): set by anybody, cleared by the starter */
    volatile int64_t     cold_inflight B200_LINE;    /* bytes of stage-in handed to the device and not retired yet (starter adds, manager subtracts) */
    /* starter-private */
    volatile int64_t     inbox_head B200_LINE;       /* slots the starter has emptied (callers read it when the ring is full) */
    parsec_list_t        stalled B200_LINE;          /* b200_task_t not started yet: new ones, and ones waiting for memory or ring space */
    parsec_list_t        settled;         /* ... whose flows the caller settled (b200_prepare_resident): they only need ring space */
    parsec_list_t        cold_q;          /* ... whose caller decided a stage-in: FIFO behind the stage-in window */
    int32_t              nb_cold;
    parsec_list_t        waiting_event;   /* b200_task_t in BT_DMA_IN / BT_LANE, in event order */
    int32_t              nb_settled;
    int32_t              nb_stalled;
    int32_t              again_window;    /* the last AGAIN of b200_start_task came from the stage-in window, not from memory */
    int32_t              lane_pending;    /* staged batchable lane tasks waiting in lane->fifo_pending for b200_fire_lane */
    uint64_t             n_engine, n_lane, n_settled_by_caller;   /* statistics (folded into parsec_b200_stats_t on demand) */
    uint64_t             tsc_start[4];    /* start phase by step: reserve, stage-in decisions, record, command */
    uint64_t             tsc_s[3];        /* starter time by phase: inbox, start, events */
    /* manager-private */
    parsec_list_t        waiting_out B200_LINE;      /* b200_task_t in BT_DMA_OUT */
    parsec_task_t       *completion_ring; /* proxies of finished tasks, handed to the worker pool once per iteration */
    b200_task_t         *batch_head;      /* the finished tasks the next proxy will complete (a chain through next_done) */
    int32_t              batch_len;
    int32_t              completed_now;   /* completions of the current manager iteration, subtracted from owed at its end */
    int32_t              blocked_spins;   /* manager iterations since the last forced attempt to start a waiting task */
    int32_t              complete_inline; /* this retire pass found ONE finished task and an empty device: a serial stretch of the
                                           * DAG, where handing the completion to another thread only adds a hop to every edge */
    int64_t              epilogs_started; /* finished tasks handed to the worker pool */
    uint64_t             tsc[8];          /* manager time by phase: -, -, -, poll, finish, idle poll, schedule */
    /* observability (device_b200_trace): what the reference reports through PINS / profiling keys around stage-in, exec
     * and stage-out of a task (device_gpu.c:348-381) is kept here per task, stamped by the device clock */
    struct b200_trace_ev_s *trace_ev;
    size_t               trace_n, trace_cap;
    pb2_retire_t         retbuf[256];
    parsec_b200_stats_t  st B200_LINE;    /* rarely written counters */
} parsec_device_b200_module_t;

/* host ranges registered with memory_register: shared by the modules of the component (cudaHostRegisterPortable) */
static b200_host_range_t *b200_ranges = NULL;
static int b200_nb_ranges = 0, b200_cap_ranges = 0;
static parsec_atomic_lock_t b200_ranges_lock = PARSEC_ATOMIC_UNLOCKED;

static int  parsec_b200_submit_is_engine(parsec_advance_task_function_t fn);
static void parsec_b200_submit_set_engine(parsec_advance_task_function_t fn);

#define B200_DEV(gpu)   ((parsec_device_b200_module_t*)(gpu))
#define B200_BT(gt)     ((b200_task_t*)(uintptr_t)(gt)->last_data_check_epoch)

#define B200_CUDA(call, what, onerr)                                                              \
    do { cudaError_t e__ = (call); if( cudaSuccess != e__ ) {                                     \
        parsec_warning("device_b200: %s: %s", (what), cudaGetErrorString(e__)); onerr; } } while(0)

/* ------------------------------------------------------------------------------------------------------------------ */
/* small helpers                                                                                                        */
/* ------------------------------------------------------------------------------------------------------------------ */
int parsec_b200_is_b200_device(const parsec_device_module_t *device)
{
    return (NULL != device) && (device->component == &parsec_device_b200_component);
}

int parsec_b200_device_count(void)
{
    int n = 0;
    if( cudaSuccess != cudaGetDeviceCount(&n) ) { (void)cudaGetLastError(); return 0; }
    return n;
}

static char *b200_device_visible(const void *host_ptr, size_t len)
{
    char *res = NULL;
    parsec_atomic_lock(&b200_ranges_lock);
    for( int i = 0; i < b200_nb_ranges; i++ ) {
        const b200_host_range_t *r = &b200_ranges[i];
        if( (const char*)host_ptr >= r->base && (const char*)host_ptr + len <= r->base + r->len ) {
            res = r->alias + ((const char*)host_ptr - r->base);
            break;
        }
    }
    parsec_atomic_unlock(&b200_ranges_lock);
    return res;
}

/* where the kernel can reach the datum's host copy (its home, where a pushout goes): NULL when it has none */
static char *b200_home_alias(const parsec_data_t *original, size_t span)
{
    const parsec_data_copy_t *cpu = original->device_copies[0];
    return (NULL != cpu && NULL != cpu->device_private) ? b200_device_visible(cpu->device_private, span) : NULL;
}

/* the task brought its own stage_in / stage_out (device_gpu.h:75-91) */
static inline int b200_user_stage_in(const parsec_gpu_task_t *gt) { return NULL != gt->stage_in && gt->stage_in != parsec_default_gpu_stage_in; }
static inline int b200_user_stage_out(const parsec_gpu_task_t *gt) { return NULL != gt->stage_out && gt->stage_out != parsec_default_gpu_stage_out; }

#define B200_INBOX_SLOTS (1 << 16)
/* Task records live on PER-THREAD free lists: the worker that calls kernel_scheduler takes one, the worker that runs the
 * task's epilog gives it back -- both are threads of the same pool, so the lists stay balanced without any atomic. */
#define B200_TL_CACHE    8192
#define B200_FLAG_WRITER ((parsec_data_flag_t)1 << 4)   /* a task that writes this replica is in flight: the replica is on no LRU */
static __thread b200_task_t *b200_tl_free = NULL;
static __thread int          b200_tl_nfree = 0;
static __thread b200_task_t *b200_tl_recording = NULL;   /* the task whose submit function this thread is calling in record mode */

static parsec_hook_return_t b200_epilog_hook(parsec_execution_stream_t *es, parsec_task_t *task);
static const __parsec_chore_t b200_completion_chores[] = {
    { .type = PARSEC_DEV_CPU, .evaluate = NULL, .hook = b200_epilog_hook, .dyld = NULL, .dyld_fn = NULL },
    { .type = PARSEC_DEV_NONE, .evaluate = NULL, .hook = NULL, .dyld = NULL, .dyld_fn = NULL },
};
static const parsec_task_class_t b200_completion_tc = {
    .name = "b200 completion", .flags = 0, .task_class_id = 0, .nb_flows = 0, .nb_parameters = 0, .nb_locals = 0,
    .incarnations = b200_completion_chores,
};

static b200_task_t *b200_bt_new(parsec_device_b200_module_t *dev, parsec_gpu_task_t *gpu_task)
{
    b200_task_t *bt = b200_tl_free;
    if( NULL != bt ) { b200_tl_free = bt->next_free; b200_tl_nfree--; }
    else {
        if( 0 != posix_memalign((void**)&bt, 64, sizeof(b200_task_t)) ) abort();
        memset(bt, 0, sizeof(b200_task_t));
        PARSEC_OBJ_CONSTRUCT(&bt->item, parsec_list_item_t);
        PARSEC_OBJ_CONSTRUCT(&bt->proxy, parsec_task_t);
        bt->proxy.task_class = &b200_completion_tc;
        bt->proxy.priority = INT32_MAX;                 /* completions first: they release work */
        bt->proxy.status = PARSEC_TASK_STATUS_HOOK;     /* no prepare_input */
        bt->proxy.chore_mask = 1;
        bt->proxy.selected_chore = 0;
        bt->proxy.selected_device = parsec_mca_device_get(0);
        bt->proxy.load = 0;
        bt->proxy.repo_entry = NULL;
        bt->ev_dev = -1;
    }
    PARSEC_LIST_ITEM_SINGLETON(&bt->item);
    bt->dev = dev;
    bt->gpu_task = gpu_task; bt->state = BT_NEW; bt->ticket = -1; bt->body = -1; bt->nb_args = 0;
    bt->peer_src_mask = 0; bt->dma_out_mask = 0; bt->result = 0; bt->custom_stage = 0; bt->cold_bytes = 0;
    bt->recorded = 0; bt->prepared = 0; bt->cmd_built = 0; bt->defer_tiles = 0; bt->ntdesc = 0;
    bt->is_kernel = (NULL == gpu_task) || (PARSEC_GPU_TASK_TYPE_KERNEL == gpu_task->task_type);
    bt->has_complete_stage = (NULL != gpu_task) && (NULL != gpu_task->complete_stage);   /* recording the body may change it */
    if( NULL != gpu_task ) gpu_task->last_data_check_epoch = (uint64_t)(uintptr_t)bt;
    return bt;
}

static void b200_bt_free(b200_task_t *bt)
{
    bt->gpu_task = NULL;
    if( b200_tl_nfree < B200_TL_CACHE ) { bt->next_free = b200_tl_free; b200_tl_free = bt; b200_tl_nfree++; return; }
    if( bt->ev_dev >= 0 ) (void)cudaEventDestroy(bt->ev);
    free(bt);
}

/* CUDA calls are issued by whichever thread starts or finishes the task: make the module's GPU current first (only the
 * copy-engine / lane paths come here, never the engine fast path) */
static inline void b200_cuda_here(parsec_device_b200_module_t *dev)
{
    if( !dev->dry_run ) B200_CUDA(cudaSetDevice(dev->super.cuda_index), "cudaSetDevice", {});
}

/* the event of a task that takes a copy-engine / lane path (made on first use, remade when the record moves to another GPU) */
static cudaEvent_t b200_bt_event(parsec_device_b200_module_t *dev, b200_task_t *bt)
{
    if( bt->ev_dev != (int32_t)dev->super.cuda_index ) {
        if( bt->ev_dev >= 0 ) (void)cudaEventDestroy(bt->ev);
        bt->ev_dev = -1;
        b200_cuda_here(dev);
        B200_CUDA(cudaEventCreateWithFlags(&bt->ev, cudaEventDisableTiming), "cudaEventCreate", { return bt->ev; });
        bt->ev_dev = (int32_t)dev->super.cuda_index;
    }
    return bt->ev;
}

/* Every insertion into an LRU list first takes the replica off whatever list it is on (a no-op for a singleton): a
 * replica can never be linked twice, whatever order epilogs and starts interleave in. */
static inline void b200_lru_put(parsec_device_b200_module_t *dev, parsec_list_t *list, parsec_data_copy_t *copy)
{
    b200_lock(&dev->lru_lock);
    copy->flags &= (parsec_data_flag_t)~B200_FLAG_WRITER;
    parsec_list_item_ring_chop((parsec_list_item_t*)copy); PARSEC_LIST_ITEM_SINGLETON(copy);
    parsec_list_nolock_push_back(list, (parsec_list_item_t*)copy);
    b200_unlock(&dev->lru_lock);
}
/* off the lists; `for_writer`: until the writing task's epilog puts it back */
static inline void b200_lru_take(parsec_device_b200_module_t *dev, parsec_data_copy_t *copy, int for_writer)
{
    b200_lock(&dev->lru_lock);
    if( for_writer ) copy->flags |= B200_FLAG_WRITER;
    parsec_list_item_ring_chop((parsec_list_item_t*)copy); PARSEC_LIST_ITEM_SINGLETON(copy);
    b200_unlock(&dev->lru_lock);
}
/* a replica that was just read moves to the back of its list -- unless a writer has taken it off the lists meanwhile */
static inline void b200_lru_touch(parsec_device_b200_module_t *dev, parsec_data_copy_t *copy)
{
    b200_lock(&dev->lru_lock);
    if( !(copy->flags & B200_FLAG_WRITER) ) {
        parsec_list_t *l = (PARSEC_DATA_COHERENCY_OWNED == copy->coherency_state) ? &dev->super.super.gpu_mem_owned_lru
                                                                                  : &dev->super.super.gpu_mem_lru;
        parsec_list_item_ring_chop((parsec_list_item_t*)copy); PARSEC_LIST_ITEM_SINGLETON(copy);
        parsec_list_nolock_push_back(l, (parsec_list_item_t*)copy);
    }
    b200_unlock(&dev->lru_lock);
}

/* The manager walks objects other cores wrote a moment ago (gpu_task, parsec_task_t, data copies, parsec_data_t): every
 * first touch is a cache-to-cache transfer of 100+ ns, and one task touches half a dozen of them one after the other.
 * Both manager loops therefore run a four-deep software prefetch ahead of the task they work on, one pointer level
 * per step (each level needs the line the previous step asked for). */
#define B200_PF(p) __builtin_prefetch((const void*)(p), 0, 3)
#define B200_PFW(p) __builtin_prefetch((const void*)(p), 1, 3)
static inline void b200_pf1(const b200_task_t *bt)
{
    const char *g = (const char*)bt->gpu_task;
    if( NULL != g ) { B200_PF(g); B200_PF(g + 64); B200_PF(g + 128); }
}
static inline void b200_pf2(const b200_task_t *bt)
{
    const parsec_gpu_task_t *g = bt->gpu_task;
    if( NULL == g || NULL == g->ec ) return;
    const parsec_task_t *t = g->ec;
    B200_PF(t); B200_PF((const char*)t + 64);
    B200_PF(&t->data[0]); B200_PF((const char*)&t->data[0] + 64);
    B200_PF(g->flow_info);
}
static inline void b200_pf3(const b200_task_t *bt)
{
    const parsec_gpu_task_t *g = bt->gpu_task;
    if( NULL == g || NULL == g->ec ) return;
    const uint32_t n = g->nb_flows < 4 ? g->nb_flows : 4;
    for( uint32_t i = 0; i < n; i++ ) {
        if( NULL != g->ec->data[i].data_in ) B200_PF(g->ec->data[i].data_in);
        if( NULL != g->ec->data[i].data_out ) B200_PF(g->ec->data[i].data_out);
    }
}
static inline void b200_pf4(const b200_task_t *bt)
{
    const parsec_gpu_task_t *g = bt->gpu_task;
    if( NULL == g || NULL == g->ec ) return;
    const uint32_t n = g->nb_flows < 4 ? g->nb_flows : 4;
    for( uint32_t i = 0; i < n; i++ ) {
        const parsec_data_copy_t *c = (NULL != g->ec->data[i].data_in) ? g->ec->data[i].data_in : g->ec->data[i].data_out;
        if( NULL != c && NULL != c->original ) { B200_PF(c->original); B200_PF((const char*)c->original + 64); }
    }
}

static inline int32_t b200_tile_of(const parsec_device_b200_module_t *dev, const parsec_data_copy_t *gpu_copy)
{
    return (int32_t)(((char*)gpu_copy->device_private - dev->slab_base) / (ptrdiff_t)dev->super.super.mem_block_size);
}

/* a reader on a copy that may live on another device: refuse when its owner is reclaiming it (readers < 0) */
static int b200_copy_acquire_reader(parsec_data_copy_t *copy)
{
    int32_t r = copy->readers;
    while( r >= 0 ) {
        if( parsec_atomic_cas_int32(&copy->readers, r, r + 1) ) return 1;
        r = copy->readers;
    }
    return 0;
}

/* ------------------------------------------------------------------------------------------------------------------ */
/* eviction and write-back (replaces the tail of parsec_device_data_reserve_space, device_gpu.c:1330-1612, and the     */
/* W2R pseudo-tasks of transfer_gpu.c:224-362)                                                                         */
/* ------------------------------------------------------------------------------------------------------------------ */
static void b200_release_copy_memory(parsec_device_b200_module_t *dev, parsec_data_copy_t *copy)
{
    parsec_data_t *original = copy->original;
    if( NULL != original ) {
        parsec_atomic_lock(&original->lock);
        /* the replica holds one reference on its datum: detaching may destroy it, lock included */
        const int survives = original->super.obj_reference_count != 1;
        parsec_data_copy_detach(original, copy, dev->super.super.super.device_index);
        parsec_atomic_wmb();
        if( survives ) parsec_atomic_unlock(&original->lock);
    }
    if( NULL != dev->tile_described ) dev->tile_described[b200_tile_of(dev, copy)] = 0;
    zone_free(dev->super.super.memory, copy->device_private);
    copy->device_private = NULL;
    PARSEC_OBJ_RELEASE(copy);
    dev->super.super.super.nb_evictions++;
    dev->st.evictions++;
}

/* Write the oldest dirty replicas home with the copy engine and move them to the clean LRU.  Blocks the manager for
 * the duration of the copies (the persistent kernel keeps running beside them).  The replicas are off every list while
 * their bytes travel; the LRU lock is held for the list work only, never across the copies. */
static int b200_write_back_some(parsec_device_b200_module_t *dev, int how_many)
{
    parsec_list_item_t *it, *next;
    parsec_data_copy_t *moved[64];
    int done = 0;
    if( how_many > 64 ) how_many = 64;
    b200_lock(&dev->lru_lock);
    for( it = PARSEC_LIST_ITERATOR_FIRST(&dev->super.super.gpu_mem_owned_lru);
         it != PARSEC_LIST_ITERATOR_END(&dev->super.super.gpu_mem_owned_lru) && done < how_many; it = next ) {
        parsec_data_copy_t *copy = (parsec_data_copy_t*)it;
        next = PARSEC_LIST_ITERATOR_NEXT(it);
        if( 0 != copy->readers || (copy->flags & B200_FLAG_WRITER) ) continue;
        parsec_data_copy_t *cpu = copy->original->device_copies[0];
        if( NULL == cpu || (!dev->dry_run && NULL == cpu->device_private) ) continue;       /* nowhere to write it: keep it */
        parsec_list_nolock_remove(&dev->super.super.gpu_mem_owned_lru, it);
        PARSEC_LIST_ITEM_SINGLETON(it);
        moved[done++] = copy;
    }
    b200_unlock(&dev->lru_lock);
    if( 0 == done ) return 0;
    if( !dev->dry_run ) {
        b200_cuda_here(dev);
        for( int i = 0; i < done; i++ ) {
            parsec_data_copy_t *copy = moved[i], *cpu = copy->original->device_copies[0];
            B200_CUDA(cudaMemcpyAsync(cpu->device_private, copy->device_private, copy->original->span, cudaMemcpyDeviceToHost, dev->dma_stream),
                      "write-back cudaMemcpyAsync", { moved[i] = NULL; b200_lru_put(dev, &dev->super.super.gpu_mem_owned_lru, copy); continue; });
            (void)parsec_atomic_fetch_add_int64((volatile int64_t*)&dev->super.super.super.data_out_to_host, (int64_t)copy->original->span);
            dev->st.bytes_d2h_dma += copy->original->span;
        }
        B200_CUDA(cudaStreamSynchronize(dev->dma_stream), "write-back synchronize", {});
    }
    int n = 0;
    for( int i = 0; i < done; i++ ) {
        parsec_data_copy_t *copy = moved[i];
        if( NULL == copy ) continue;
        parsec_data_copy_t *cpu = copy->original->device_copies[0];
        parsec_atomic_lock(&copy->original->lock);
        if( cpu->version < copy->version ) cpu->version = copy->version;
        cpu->coherency_state = PARSEC_DATA_COHERENCY_SHARED;
        copy->coherency_state = PARSEC_DATA_COHERENCY_SHARED;
        if( copy->original->owner_device == (int8_t)dev->super.super.super.device_index ) copy->original->owner_device = 0;
        parsec_atomic_unlock(&copy->original->lock);
        b200_lru_put(dev, &dev->super.super.gpu_mem_lru, copy);
        dev->st.w2r_copies++;
        n++;
    }
    return n;
}

/* Free one replica nobody uses: oldest clean one first; if every clean replica is busy, write dirty ones home. */
static int b200_evict_one(parsec_device_b200_module_t *dev, const parsec_gpu_task_t *for_task)
{
    for( int pass = 0; pass < 2; pass++ ) {
        parsec_list_item_t *it, *next;
        parsec_data_copy_t *victim = NULL;
        b200_lock(&dev->lru_lock);
        for( it = PARSEC_LIST_ITERATOR_FIRST(&dev->super.super.gpu_mem_lru);
             it != PARSEC_LIST_ITERATOR_END(&dev->super.super.gpu_mem_lru); it = next ) {
            parsec_data_copy_t *copy = (parsec_data_copy_t*)it;
            next = PARSEC_LIST_ITERATOR_NEXT(it);
            if( PARSEC_DATA_STATUS_UNDER_TRANSFER == copy->data_transfer_status || (copy->flags & B200_FLAG_WRITER) ) continue;
            /* a task that has not run yet was handed this replica as its input (the repo retains it): keep it */
            if( copy->super.super.obj_reference_count > 1 ) continue;
            if( NULL != for_task ) {
                int mine = 0;
                for( uint32_t f = 0; f < for_task->nb_flows; f++ )
                    mine |= (for_task->ec->data[f].data_out == copy) || (for_task->ec->data[f].data_in == copy);
                if( mine ) continue;
            }
            /* tombstone: a peer GPU that wants this replica as a source sees readers < 0 and looks elsewhere */
            if( !parsec_atomic_cas_int32(&copy->readers, 0, INT_MIN / 2) ) continue;
            /* never drop the only up-to-date replica */
            parsec_data_copy_t *cpu = (NULL != copy->original) ? copy->original->device_copies[0] : NULL;
            if( NULL != copy->original && (NULL == cpu || cpu->version < copy->version) &&
                copy->original->owner_device == (int8_t)dev->super.super.super.device_index ) {
                copy->readers = 0;
                continue;
            }
            parsec_list_nolock_remove(&dev->super.super.gpu_mem_lru, it);
            PARSEC_LIST_ITEM_SINGLETON(it);
            victim = copy;
            break;
        }
        b200_unlock(&dev->lru_lock);
        if( NULL != victim ) {
            victim->readers = 0;
            b200_release_copy_memory(dev, victim);
            return 1;
        }
        if( 0 == b200_write_back_some(dev, 16) ) break;
    }
    return 0;
}

/* ------------------------------------------------------------------------------------------------------------------ */
/* residency: every flow gets a replica on this device (parsec_device_data_reserve_space, device_gpu.c:1209)           */
/* ------------------------------------------------------------------------------------------------------------------ */
static int b200_reserve(parsec_device_b200_module_t *dev, b200_task_t *bt)
{
    parsec_gpu_task_t *gpu_task = bt->gpu_task;
    parsec_task_t *this_task = gpu_task->ec;
    const uint8_t my = dev->super.super.super.device_index;
    parsec_data_copy_t *fresh[MAX_PARAM_COUNT];
    int nfresh = 0;

    for( uint32_t i = 0; i < gpu_task->nb_flows; i++ ) {
        const parsec_flow_t *flow = gpu_task->flow_info[i].flow;
        if( PARSEC_FLOW_ACCESS_NONE == (PARSEC_FLOW_ACCESS_MASK & flow->flow_flags) ) { gpu_task->flow_info[i].flow_span = 0; continue; }
        parsec_data_copy_t *in = this_task->data[i].data_in;
        if( NULL == in ) continue;
        if( in->device_index == my ) { this_task->data[i].data_out = in; continue; }
        parsec_data_t *master = in->original;
        parsec_atomic_lock(&master->lock);
        parsec_data_copy_t *gpu_elem = PARSEC_DATA_GET_COPY(master, my);
        parsec_atomic_unlock(&master->lock);
        if( NULL == gpu_elem ) {
            void *ptr;
            while( NULL == (ptr = zone_malloc(dev->super.super.memory, gpu_task->flow_info[i].flow_span)) ) {
                dev->memory_pressure = 1;
                if( !b200_evict_one(dev, gpu_task) ) {
                    /* nothing can be freed now: undo what this pass allocated and let the task wait for retirements */
                    for( int k = 0; k < nfresh; k++ ) {
                        b200_lru_take(dev, fresh[k], 0);
                        b200_release_copy_memory(dev, fresh[k]);
                        dev->super.super.super.nb_evictions--; dev->st.evictions--;
                    }
                    for( uint32_t k = 0; k < gpu_task->nb_flows; k++ )
                        if( NULL != this_task->data[k].data_in && this_task->data[k].data_in->device_index != my ) this_task->data[k].data_out = NULL;
                    return PARSEC_HOOK_RETURN_AGAIN;
                }
            }
            gpu_elem = PARSEC_OBJ_NEW(parsec_data_copy_t);
            gpu_elem->flags = PARSEC_DATA_FLAG_PARSEC_OWNED | PARSEC_DATA_FLAG_PARSEC_MANAGED;
            gpu_elem->device_private = ptr;
            gpu_elem->arena_chunk = (parsec_arena_chunk_t*)dev->super.super.memory;
            gpu_elem->coherency_state = PARSEC_DATA_COHERENCY_INVALID;
            gpu_elem->version = 0;
            gpu_elem->dtt = in->dtt;
            parsec_atomic_lock(&master->lock);
            parsec_data_copy_attach(master, gpu_elem, my);
            parsec_atomic_unlock(&master->lock);
            /* fresh replicas sit on the clean LRU; a reader or the write detach below protects them */
            b200_lru_put(dev, &dev->super.super.gpu_mem_lru, gpu_elem);
            fresh[nfresh++] = gpu_elem;
        }
        this_task->data[i].data_out = gpu_elem;
    }
    return PARSEC_HOOK_RETURN_DONE;
}

/* does starting this task require a fresh allocation on the device? */
static int b200_needs_memory(const parsec_device_b200_module_t *dev, const parsec_gpu_task_t *gpu_task)
{
    const uint8_t my = dev->super.super.super.device_index;
    for( uint32_t i = 0; i < gpu_task->nb_flows; i++ ) {
        const parsec_flow_t *flow = gpu_task->flow_info[i].flow;
        if( PARSEC_FLOW_ACCESS_NONE == (PARSEC_FLOW_ACCESS_MASK & flow->flow_flags) ) continue;
        const parsec_data_copy_t *in = gpu_task->ec->data[i].data_in;
        if( NULL == in || in->device_index == my ) continue;
        if( NULL == PARSEC_DATA_GET_COPY(in->original, my) ) return 1;
    }
    return 0;
}

/* ------------------------------------------------------------------------------------------------------------------ */
/* stage-in decisions (parsec_device_data_stage_in, device_gpu.c:1799-2165): who is the source, who moves the bytes     */
/* ------------------------------------------------------------------------------------------------------------------ */
/* a tile description decided by `bt`: straight to the device when the starter decides, kept in the record when the
 * calling worker does (the starter sends the descriptions of a record before anything that was decided after them) */
static int b200_emit_tile(parsec_device_b200_module_t *dev, b200_task_t *bt, int32_t tid, const pb2_tile_t *tile)
{
    if( !bt->defer_tiles ) return (PB2_SUCCESS == pb2_stream_set_tile(dev->stream, tid, tile)) ? 0 : -1;
    if( bt->ntdesc >= MAX_PARAM_COUNT ) return -1;
    bt->tdesc[bt->ntdesc].tile = tid; bt->tdesc[bt->ntdesc].desc = *tile; bt->ntdesc++;
    return 0;
}

/* what the device tile table says about the replica `out` of a flow of access `type`: the version before the task runs,
 * where its bytes come from / go to.  returns 0, -1 when the description cannot be sent */
static int b200_describe_tile(parsec_device_b200_module_t *dev, b200_task_t *bt, const parsec_data_copy_t *out, size_t span,
                              uint8_t type, char *src_ptr, int32_t src_kind, int32_t state)
{
    const pb2_tile_t tile = { .dev_ptr = out->device_private, .src_ptr = src_ptr, .bytes = (uint32_t)span, .state = state,
                              .version = (PARSEC_FLOW_ACCESS_WRITE & type) ? out->version - 1 : out->version, .src_kind = src_kind };
    const int32_t tid = b200_tile_of(dev, out);
    if( 0 != b200_emit_tile(dev, bt, tid, &tile) ) return -1;
    dev->tile_described[tid] = 1;
    return 0;
}

/* a flow whose input already is this device's replica: a writer bumps its version and takes it off the LRUs until it
 * retires, a reader holds it */
static void b200_use_resident_flow(parsec_device_b200_module_t *dev, parsec_data_copy_t *copy, uint8_t type)
{
    if( PARSEC_FLOW_ACCESS_WRITE & type ) {
        copy->version++;
        b200_lru_take(dev, copy, 1);
        parsec_atomic_lock(&copy->original->lock);
        copy->original->owner_device = dev->super.super.super.device_index; copy->coherency_state = PARSEC_DATA_COHERENCY_OWNED;
        parsec_atomic_unlock(&copy->original->lock);
    }
    if( PARSEC_FLOW_ACCESS_READ & type ) (void)parsec_atomic_fetch_inc_int32(&copy->readers);
}

/* the bytes of `copy` are here (callback_complete_push, device_gpu.c:2358-2573).  The caller holds the datum's lock. */
static void b200_transfer_done(parsec_device_b200_module_t *dev, parsec_data_copy_t *copy, uint8_t type)
{
    copy->data_transfer_status = PARSEC_DATA_STATUS_COMPLETE_TRANSFER;
    parsec_data_end_transfer_ownership_to_copy(copy->original, dev->super.super.super.device_index, type);
}

/* mode 0: engine task (the kernel pulls device-visible sources, the copy engine the others);
 * mode 1: lane task, default staging (copy engine on the lane stream); mode 2: lane task with a user stage_in: nothing is
 * copied here, the flows that need their bytes are left UNDER_TRANSFER for the callback.
 * returns 0 ok, 1 when a copy was enqueued or is owed (the task has to wait for bt->ev), <0 error / retry */
static int b200_stage_in(parsec_device_b200_module_t *dev, b200_task_t *bt, int mode)
{
    const int for_lane = (0 != mode);
    parsec_gpu_task_t *gpu_task = bt->gpu_task;
    parsec_task_t *this_task = gpu_task->ec;
    parsec_device_module_t *mod = &dev->super.super.super;
    const uint8_t my = mod->device_index;
    int used_dma = 0;
    uint32_t pre_acquired = 0;

    /* A task that was handed another GPU's replica needs that replica to stay: take the readers first, all or none,
     * before anything of the task's own state changes (a replica its owner is reclaiming makes the task wait) */
    for( uint32_t i = 0; i < gpu_task->nb_flows; i++ ) {
        const parsec_flow_t *flow = gpu_task->flow_info[i].flow;
        parsec_data_copy_t *in = this_task->data[i].data_in;
        if( NULL == in || NULL == this_task->data[i].data_out || in == this_task->data[i].data_out ) continue;
        if( !(PARSEC_FLOW_ACCESS_READ & flow->flow_flags) || !parsec_mca_device_is_gpu(in->device_index) ) continue;
        if( b200_copy_acquire_reader(in) ) { pre_acquired |= (1u << i); continue; }
        for( uint32_t k = 0; k < i; k++ )
            if( pre_acquired & (1u << k) ) (void)parsec_atomic_fetch_dec_int32(&this_task->data[k].data_in->readers);
        return PARSEC_HOOK_RETURN_AGAIN;
    }

    for( uint32_t i = 0; i < gpu_task->nb_flows; i++ ) {
        const parsec_flow_t *flow = gpu_task->flow_info[i].flow;
        const uint8_t type = (uint8_t)(flow->flow_flags & PARSEC_FLOW_ACCESS_MASK);
        if( PARSEC_FLOW_ACCESS_NONE == type ) continue;
        parsec_data_copy_t *in = this_task->data[i].data_in, *out = this_task->data[i].data_out;
        if( NULL == in || NULL == out ) continue;
        parsec_data_t *original = in->original;
        const size_t span = gpu_task->flow_info[i].flow_span;
        gpu_task->flow_info[i].source = NULL;

        if( in == out ) {      /* the input already is this device's replica */
            b200_use_resident_flow(dev, out, type);
            /* a replica filled on the stream lane (copy engine, opaque body): the kernel has not met it yet */
            if( !for_lane && !dev->tile_described[b200_tile_of(dev, out)] &&
                0 != b200_describe_tile(dev, bt, out, span, type, b200_home_alias(original, span), PB2_SRC_HOST, PB2_TILE_VALID) )
                return PARSEC_HOOK_RETURN_ERROR;
            continue;
        }

        parsec_atomic_lock(&original->lock);
        if( PARSEC_FLOW_ACCESS_WRITE & type ) {        /* a written replica leaves the LRUs until the task retires */
            b200_lru_take(dev, out, 1);
        }
        /* source: the copy the task was given, unless it is a host copy and a peer GPU we can read holds the same
         * version (device_gpu.c:1892-1975) */
        parsec_data_copy_t *src = in;
        int src_acquired = 0, src_detour = 0;
        if( (PARSEC_FLOW_ACCESS_READ & type) ) {
            if( parsec_mca_device_is_gpu(in->device_index) ) {
                /* the task was handed another GPU's replica: it IS the newest version (no pushout was asked for), so
                 * the bytes have to come from there -- in place over NVLink when this GPU can address it, through
                 * the copy engine otherwise; a replica its owner is reclaiming right now is retried later */
                src_acquired = (pre_acquired >> i) & 1;            /* taken above */
                src_detour = !(dev->super.super.peer_access_mask & (1 << in->device_index));
            } else if( !(PARSEC_FLOW_ACCESS_WRITE & type) ) {
                for( uint32_t t = 1; t < parsec_nb_devices; t++ ) {
                    parsec_data_copy_t *cand = original->device_copies[t];
                    if( t == my || NULL == cand || !(dev->super.super.peer_access_mask & (1 << t)) ) continue;
                    if( cand->version != in->version || PARSEC_DATA_COHERENCY_INVALID == cand->coherency_state ||
                        PARSEC_DATA_STATUS_UNDER_TRANSFER == cand->data_transfer_status ) continue;
                    if( b200_copy_acquire_reader(cand) ) { src = cand; src_acquired = 1; break; }
                }
            }
        }
        if( NULL == src ) { parsec_atomic_unlock(&original->lock); return PARSEC_HOOK_RETURN_ERROR; }

        int transfer_from = parsec_data_start_transfer_ownership_to_copy(original, my, type);
        /* what decides is the VERSION: the replica here is current iff it carries the version the task was given */
        if( -1 != transfer_from && out->version == src->version && PARSEC_DATA_STATUS_COMPLETE_TRANSFER == out->data_transfer_status ) transfer_from = -1;
        if( NULL == src->device_private ) transfer_from = -1;                /* NEW data nobody wrote yet */
        if( (NULL == this_task->data[i].source_repo_entry) && (NULL == original->dc) && (0 == in->version) ) transfer_from = -1;
        if( PARSEC_DATA_STATUS_UNDER_TRANSFER == out->data_transfer_status ) transfer_from = -1;   /* an earlier task brings it */
        mod->required_data_in += original->span;

        const int32_t src_kind = parsec_mca_device_is_gpu(src->device_index) ? PB2_SRC_PEER : PB2_SRC_HOST;
        char *pull_from = NULL;         /* set when the kernel pulls the bytes itself */
        if( -1 == transfer_from ) {
            if( src_acquired ) { (void)parsec_atomic_fetch_dec_int32(&src->readers); src_acquired = 0; }
            if( PARSEC_DATA_STATUS_UNDER_TRANSFER != out->data_transfer_status ) b200_transfer_done(dev, out, type);
            if( PARSEC_FLOW_ACCESS_WRITE & type ) out->version = src->version + 1;
        } else {
            char *visible = (PB2_SRC_PEER == src_kind) ? (char*)src->device_private
                                                       : b200_device_visible(src->device_private, span);
            mod->data_in_from_device[src->device_index] += span;
            mod->nb_data_faults += span;
            bt->cold_bytes += span;
            if( PB2_SRC_PEER == src_kind ) { if( src_detour ) dev->st.peer_detours++; else dev->st.peer_pulls++; }
            if( NULL != visible && !src_detour && !for_lane && !dev->dry_run ) {
                /* the persistent kernel pulls it (TMA bulk copy) when the task runs */
                pull_from = visible;
                out->data_transfer_status = PARSEC_DATA_STATUS_UNDER_TRANSFER;
                if( PB2_SRC_PEER == src_kind ) dev->st.bytes_d2d_kernel += span; else dev->st.bytes_h2d_kernel += span;
            } else if( 2 == mode ) {
                out->data_transfer_status = PARSEC_DATA_STATUS_UNDER_TRANSFER;       /* the user's stage_in moves it */
                used_dma = 1;
            } else if( !dev->dry_run ) {
                /* unregistered host memory, or an opaque body that needs the bytes before it is enqueued: copy engine */
                b200_cuda_here(dev);
                B200_CUDA(cudaMemcpyAsync(out->device_private, src->device_private, span,
                                          PB2_SRC_PEER == src_kind ? cudaMemcpyDeviceToDevice : cudaMemcpyHostToDevice,
                                          for_lane ? dev->lane->cuda_stream : dev->dma_stream),
                          "stage-in cudaMemcpyAsync", { parsec_atomic_unlock(&original->lock); return PARSEC_HOOK_RETURN_ERROR; });
                out->data_transfer_status = PARSEC_DATA_STATUS_UNDER_TRANSFER;
                dev->st.bytes_h2d_dma += span;
                used_dma = 1;
            } else {
                out->data_transfer_status = PARSEC_DATA_STATUS_UNDER_TRANSFER;
            }
            out->version = (PARSEC_FLOW_ACCESS_WRITE & type) ? src->version + 1 : src->version;
            gpu_task->flow_info[i].source = src;          /* what a user stage_in reads (stage_custom.jdf:28-60) */
            if( src_acquired ) { bt->peer_src_mask |= (1u << i); bt->peer_src[i] = src; }
        }
        /* The entry is written when the replica is new to the device or when a new pull has just been decided -- and
         * ONLY then: a second reader that arrives while the first one's pull is still running must find the entry as
         * the kernel left it (STAGING), not a fresh "VALID" from the host. */
        const int failed = !for_lane && (-1 != transfer_from || !dev->tile_described[b200_tile_of(dev, out)]) &&
            0 != b200_describe_tile(dev, bt, out, span, type, NULL != pull_from ? pull_from : b200_home_alias(original, span),
                                    src_kind, NULL != pull_from ? PB2_TILE_INVALID : PB2_TILE_VALID);
        parsec_atomic_unlock(&original->lock);
        if( failed ) return PARSEC_HOOK_RETURN_ERROR;
    }
    return used_dma;
}

/* ------------------------------------------------------------------------------------------------------------------ */
/* the body                                                                                                             */
/* ------------------------------------------------------------------------------------------------------------------ */
int parsec_b200_task_body(parsec_device_gpu_module_t *gpu_device, parsec_gpu_task_t *gpu_task,
                          parsec_gpu_exec_stream_t *gpu_stream,
                          int body, int nb_args, const int *flow_index, const int32_t *iparam, float fparam)
{
    if( NULL == gpu_device || NULL == gpu_task || nb_args < 0 || nb_args > PB2_MAX_FLOWS || body < 0 || body >= PB2_BODY_MAX )
        return PARSEC_HOOK_RETURN_ERROR;
    for( int a = 0; a < nb_args; a++ )
        if( flow_index[a] < 0 || (uint32_t)flow_index[a] >= gpu_task->nb_flows ) return PARSEC_HOOK_RETURN_ERROR;
    if( parsec_b200_is_b200_device(&gpu_device->super) ) {
        b200_task_t *bt = b200_tl_recording;
        if( NULL == bt || bt->gpu_task != gpu_task ) return PARSEC_HOOK_RETURN_ERROR;
        bt->body = body; bt->nb_args = nb_args;
        for( int a = 0; a < nb_args; a++ ) bt->arg_flow[a] = flow_index[a];
        bt->iparam[0] = iparam ? iparam[0] : 0; bt->iparam[1] = iparam ? iparam[1] : 0; bt->iparam[2] = iparam ? iparam[2] : 0;
        bt->fparam = fparam;
        return PARSEC_HOOK_RETURN_DONE;
    }
    /* any other GPU module (the reference's stream engine): the same body as a stand-alone kernel on its stream */
    {
        void *ptrs[PB2_MAX_FLOWS] = {NULL, NULL, NULL, NULL};
        uint64_t bytes[PB2_MAX_FLOWS] = {0, 0, 0, 0};
        int32_t ip[3] = { iparam ? iparam[0] : 0, iparam ? iparam[1] : 0, iparam ? iparam[2] : 0 };
        for( int a = 0; a < nb_args; a++ ) {
            ptrs[a] = gpu_task->ec->data[flow_index[a]].data_out->device_private;
            bytes[a] = gpu_task->flow_info[flow_index[a]].flow_span;
        }
        parsec_cuda_exec_stream_t *cs = (parsec_cuda_exec_stream_t*)gpu_stream;
        return (PB2_SUCCESS == pb2_body_launch((void*)cs->cuda_stream, body, nb_args, ptrs, bytes, ip, fparam))
               ? PARSEC_HOOK_RETURN_DONE : PARSEC_HOOK_RETURN_ERROR;
    }
}

uint64_t parsec_b200_task_result(const parsec_gpu_task_t *gpu_task)
{
    const b200_task_t *bt = (const b200_task_t*)(uintptr_t)gpu_task->last_data_check_epoch;
    return (NULL != bt) ? bt->result : 0;
}

/* ------------------------------------------------------------------------------------------------------------------ */
/* completion: epilog of the flows + hand-back to the runtime (parsec_device_kernel_pop / _epilog, device_gpu.c:2943,  */
/* :3179, and the complete_task tail of the scheduler, :3562-3590)                                                     */
/*                                                                                                                      */
/* The manager is one thread and every task passes through it twice; what it does per task decides the task rate of     */
/* the device.  The whole epilog -- coherency of every flow, LRU position, prepare_output / release_deps /               */
/* release_task -- therefore runs on the WORKER POOL: the manager only links the task record's embedded proxy task      */
/* (an ordinary parsec_task_t of a private class with one CPU incarnation) into a ring it schedules once per iteration. */
/* The proxy's hook does the epilog, calls __parsec_complete_execution on the real task (exactly once, with that         */
/* worker's execution stream) and returns ASYNC, so the runtime never tries to complete the proxy itself.  Every replica */
/* of the task keeps one reader until release_deps has given the successors their references: eviction cannot take it   */
/* away in between.                                                                                                      */
/* ------------------------------------------------------------------------------------------------------------------ */
static inline void b200_stat_add(uint64_t *counter, uint64_t v)
{
    (void)parsec_atomic_fetch_add_int64((volatile int64_t*)counter, (int64_t)v);
}

/* the flows of a finished task; fills held[] with the replicas that keep a reader until the caller lets them go */
static int b200_epilog_flows(parsec_device_b200_module_t *dev, b200_task_t *bt, parsec_data_copy_t **held)
{
    parsec_gpu_task_t *gpu_task = bt->gpu_task;
    parsec_task_t *this_task = gpu_task->ec;
    parsec_device_module_t *mod = &dev->super.super.super;
    int nheld = 0;

    for( uint32_t i = 0; i < gpu_task->nb_flows; i++ ) {
        const parsec_flow_t *flow = gpu_task->flow_info[i].flow;
        const uint8_t type = (uint8_t)(flow->flow_flags & PARSEC_FLOW_ACCESS_MASK);
        if( PARSEC_FLOW_ACCESS_NONE == type || NULL == this_task->data[i].data_in ) continue;
        parsec_data_copy_t *gpu_copy = this_task->data[i].data_out;
        if( NULL == gpu_copy ) continue;
        parsec_data_t *original = gpu_copy->original;
        /* The datum's lock (parsec_atomic_lock: nanosleep under contention) is taken when something of the protocol
         * changes -- the end of a transfer, a write.  The other readers of a replica that is simply there only move its
         * LRU position and let go of their reader: eight of them finishing together must not queue up on it. */
        const int locked = (PARSEC_FLOW_ACCESS_WRITE & type) || PARSEC_DATA_STATUS_UNDER_TRANSFER == gpu_copy->data_transfer_status;
        if( locked ) parsec_atomic_lock(&original->lock);
        if( PARSEC_DATA_STATUS_UNDER_TRANSFER == gpu_copy->data_transfer_status ) b200_transfer_done(dev, gpu_copy, type);
        if( bt->peer_src_mask & (1u << i) ) (void)parsec_atomic_fetch_dec_int32(&bt->peer_src[i]->readers);
        /* READ flows took their reader when the task started; a write-only flow takes one now */
        if( !(PARSEC_FLOW_ACCESS_READ & type) ) (void)parsec_atomic_fetch_inc_int32(&gpu_copy->readers);
        held[nheld++] = gpu_copy;
        if( PARSEC_FLOW_ACCESS_WRITE & type ) {
            b200_stat_add(&mod->required_data_out, gpu_task->flow_info[i].flow_span);
            if( gpu_task->pushout & (1 << i) ) {
                parsec_data_copy_t *cpu_copy = original->device_copies[0];
                if( NULL != cpu_copy ) {
                    cpu_copy->version = gpu_copy->version;
                    cpu_copy->coherency_state = PARSEC_DATA_COHERENCY_SHARED;
                    gpu_copy->coherency_state = PARSEC_DATA_COHERENCY_SHARED;
                    cpu_copy->data_transfer_status = PARSEC_DATA_STATUS_COMPLETE_TRANSFER;
                    b200_stat_add(&mod->data_out_to_host, gpu_task->flow_info[i].flow_span);
                    if( 0 == (parsec_mpi_allow_gpu_memory_communications & PARSEC_RUNTIME_SEND_GPU_MEMORY) )
                        this_task->data[i].data_out = cpu_copy;           /* successors consume the host copy */
                }
                b200_lru_put(dev, &dev->super.super.gpu_mem_lru, gpu_copy);
            } else {
                gpu_copy->coherency_state = PARSEC_DATA_COHERENCY_OWNED;
                b200_lru_put(dev, &dev->super.super.gpu_mem_owned_lru, gpu_copy);
            }
        } else if( dev->memory_pressure && 1 == gpu_copy->readers && 0 != (gpu_copy->flags & PARSEC_DATA_FLAG_PARSEC_OWNED) ) {
            /* least recently used goes to the front: the last reader of a replica moves it to the back of its list.  The
             * order only matters once something has to be evicted: until the heap has been full once the lists keep
             * their insertion order and the readers of a replica do not queue up on the LRU lock. */
            b200_lru_touch(dev, gpu_copy);
        }
        if( locked ) parsec_atomic_unlock(&original->lock);
    }
    return nheld;
}

/* epilog, runtime completion and release of one finished task; frees its record */
static void b200_finish_one(parsec_device_b200_module_t *dev, parsec_execution_stream_t *es, b200_task_t *bt, int run_complete_stage)
{
    parsec_gpu_task_t *gpu_task = bt->gpu_task;
    parsec_data_copy_t *held[MAX_PARAM_COUNT];
    const int nheld = b200_epilog_flows(dev, bt, held);
    if( run_complete_stage && NULL != gpu_task->complete_stage ) {
        parsec_gpu_task_t *gt = gpu_task;
        (void)gpu_task->complete_stage(&dev->super.super, &gt, &dev->lane->super);
    }
    (void)__parsec_complete_execution(es, gpu_task->ec);
    for( int i = 0; i < nheld; i++ ) (void)parsec_atomic_fetch_dec_int32(&held[i]->readers);
    gpu_task->last_data_check_epoch = 0;
    gpu_task->release_device_task(gpu_task);
    b200_bt_free(bt);
}

static parsec_hook_return_t b200_epilog_hook(parsec_execution_stream_t *es, parsec_task_t *task)
{
    b200_task_t *bt = (b200_task_t*)((char*)task - offsetof(b200_task_t, proxy));
    parsec_device_b200_module_t *dev = bt->dev;
    int64_t n = 0;
    b200_nvtx_push("b200 epilog batch");
    /* one proxy completes a short chain of finished tasks (B200_EPILOG_BATCH): scheduling a task costs the manager about
     * as much as everything else it does for one */
    while( NULL != bt ) {
        b200_task_t *next = bt->next_done;
        if( NULL != next ) { B200_PF(next); B200_PF(next->gpu_task); }
        b200_finish_one(dev, es, bt, 0);   /* the proxy lives in the record: nothing of it is touched after this hook returns ASYNC */
        bt = next;
        n++;
    }
    if( dev->nb_stalled > 0 && !dev->retry_stalled ) dev->retry_stalled = 1;   /* the readers just dropped may be what a waiting task needs evicted */
    parsec_atomic_wmb();
    (void)parsec_atomic_fetch_add_int64(&dev->epilogs_done, n);
    b200_nvtx_pop();
    return PARSEC_HOOK_RETURN_ASYNC;
}

#define B200_EPILOG_BATCH 4
/* the chain collected so far becomes one proxy task of the completion ring */
static inline void b200_close_batch(parsec_device_b200_module_t *dev)
{
    b200_task_t *bt = dev->batch_head;
    if( NULL == bt ) return;
    dev->batch_head = NULL; dev->batch_len = 0;
    PARSEC_LIST_ITEM_SINGLETON(&bt->proxy);
    if( NULL == dev->completion_ring ) dev->completion_ring = &bt->proxy;
    else parsec_list_item_ring_push((parsec_list_item_t*)dev->completion_ring, (parsec_list_item_t*)&bt->proxy);
}

/* manager side of a finished kernel task */
static void b200_complete(parsec_device_b200_module_t *dev, parsec_execution_stream_t *es, b200_task_t *bt)
{
    dev->super.super.super.executed_tasks++;
    dev->completed_now++;
    if( parsec_b200_parallel_completion && !bt->has_complete_stage && !dev->complete_inline ) {
        /* nothing of the task but its record is touched here */
        dev->epilogs_started++;
        bt->next_done = dev->batch_head; dev->batch_head = bt;
        if( ++dev->batch_len >= B200_EPILOG_BATCH ) b200_close_batch(dev);
        return;
    }
    /* in line: a user completion hook (device_gpu.h:41-43; dtd_test_simple_gemm.c:538) is called by the thread that
     * drives the device, like the reference does, and device_b200_parallel_completion = 0 asks for it */
    b200_finish_one(dev, es, bt, 1);
}

/* Copy-engine pushout of the flows in `mask` to their host copies, on `stream`; a user stage_out is called once per flow
 * (device_gpu.c:2980, :3138) and enqueues on the lane stream (stage_custom.jdf:62-95).  returns the number of flows that
 * had something enqueued, < 0 when a stage_out or a copy failed (the flows before it stay enqueued) */
static int b200_copy_home(parsec_device_b200_module_t *dev, b200_task_t *bt, uint32_t mask, cudaStream_t stream)
{
    parsec_gpu_task_t *gpu_task = bt->gpu_task;
    int n = 0;
    for( uint32_t i = 0; i < gpu_task->nb_flows; i++ ) {
        if( !(mask & (1u << i)) ) continue;
        if( b200_user_stage_out(gpu_task) ) {
            if( PARSEC_SUCCESS != gpu_task->stage_out(gpu_task, 1u << i, &dev->lane->super) ) return -1;
            n++;
            continue;
        }
        parsec_data_copy_t *gpu_copy = gpu_task->ec->data[i].data_out;
        parsec_data_copy_t *cpu_copy = gpu_copy->original->device_copies[0];
        if( NULL == cpu_copy || NULL == cpu_copy->device_private ) continue;
        B200_CUDA(cudaMemcpyAsync(cpu_copy->device_private, gpu_copy->device_private, gpu_task->flow_info[i].flow_span,
                                  cudaMemcpyDeviceToHost, stream), "pushout cudaMemcpyAsync", { return -1; });
        dev->st.bytes_d2h_dma += gpu_task->flow_info[i].flow_span;
        n++;
    }
    return n;
}

/* pushout flows whose host home the kernel cannot write (memory that was never registered): copy engine.  returns 1 when
 * the task has to wait for its event */
static int b200_dma_pushout(parsec_device_b200_module_t *dev, b200_task_t *bt)
{
    if( dev->dry_run ) return 0;
    b200_cuda_here(dev);
    cudaStream_t stream = b200_user_stage_out(bt->gpu_task) ? dev->lane->cuda_stream : dev->dma_stream;
    if( 0 == b200_copy_home(dev, bt, bt->dma_out_mask, stream) ) return 0;     /* after a failure: wait for what is enqueued */
    B200_CUDA(cudaEventRecord(b200_bt_event(dev, bt), stream), "cudaEventRecord", {});
    return 1;
}

/* ------------------------------------------------------------------------------------------------------------------ */
/* one task: from the inbox to the command ring / the lane                                                              */
/* ------------------------------------------------------------------------------------------------------------------ */
/* The engine command of a task whose flows all have their replica (data_out): tile ids, access modes, where a pushout
 * goes.  Touches nothing of the device: built by whoever settled the flows -- the calling worker for resident tasks. */
static void b200_build_cmd(parsec_device_b200_module_t *dev, b200_task_t *bt)
{
    parsec_gpu_task_t *gpu_task = bt->gpu_task;
    pb2_task_t *t = &bt->cmd;
    memset(t, 0, sizeof *t);
    t->body = (uint8_t)bt->body; t->nb_flows = (uint8_t)bt->nb_args;
    for( int a = 0; a < PB2_MAX_FLOWS; a++ ) t->tile[a] = -1;
    for( int a = 0; a < bt->nb_args; a++ ) {
        const int f = bt->arg_flow[a];
        const parsec_flow_t *flow = gpu_task->flow_info[f].flow;
        parsec_data_copy_t *out = gpu_task->ec->data[f].data_out;
        t->tile[a] = b200_tile_of(dev, out);
        t->access[a] = (uint8_t)(flow->flow_flags & PARSEC_FLOW_ACCESS_MASK);
        if( (gpu_task->pushout & (1 << f)) && (PARSEC_FLOW_ACCESS_WRITE & flow->flow_flags) ) {
            /* the tile has one src_ptr, the kernel stages in from it and pushes out to it: a flow pulled from a peer
             * goes home through the copy engine */
            if( !bt->custom_stage && NULL != b200_home_alias(out->original, gpu_task->flow_info[f].flow_span) &&
                !(bt->peer_src_mask & (1u << f)) )
                t->access[a] |= PB2_FLOW_PUSHOUT;            /* the worker CTA copies it home */
            else bt->dma_out_mask |= (1u << f);
        }
    }
    /* pushout flows the body does not name still have to reach the host */
    for( uint32_t f = 0; f < gpu_task->nb_flows; f++ ) {
        int named = 0;
        for( int a = 0; a < bt->nb_args; a++ ) named |= (bt->arg_flow[a] == (int)f);
        if( !named && (gpu_task->pushout & (1 << f)) && (PARSEC_FLOW_ACCESS_WRITE & gpu_task->flow_info[f].flow->flow_flags) &&
            NULL != gpu_task->ec->data[f].data_out ) bt->dma_out_mask |= (1u << f);
    }
    t->iparam[0] = bt->iparam[0]; t->iparam[1] = bt->iparam[1]; t->iparam[2] = bt->iparam[2]; t->fparam = bt->fparam;
    t->locals[0] = gpu_task->ec->locals[0].value; t->locals[1] = gpu_task->ec->locals[1].value;
    bt->cmd_built = 1;
}

/* manager only */
static int b200_push_engine(parsec_device_b200_module_t *dev, b200_task_t *bt)
{
    if( !bt->cmd_built ) b200_build_cmd(dev, bt);
    /* The instant the command is published the task may run and retire: the record is final BEFORE the submit. */
    const int32_t state_before = bt->state;
    bt->state = BT_INFLIGHT;
    int rc = pb2_stream_submit(dev->stream, &bt->cmd, (uint64_t)(uintptr_t)bt, &bt->ticket);
    if( PB2_SUCCESS != rc ) {
        bt->state = state_before;
        if( PB2_ERR_OUT_OF_RESOURCE == rc ) return PARSEC_HOOK_RETURN_AGAIN;
        parsec_warning("device_b200: submit failed: %s", pb2_stream_last_error(dev->stream));
        return PARSEC_HOOK_RETURN_ERROR;
    }
    dev->n_engine++;
    return PARSEC_HOOK_RETURN_DONE;
}

/* Called by the worker thread that hands the task over, BEFORE the hand-over.  A task whose every input already is this
 * device's replica (the data came from a task that ran here) needs no decision of the manager: nothing is allocated,
 * nothing moves.  The caller -- the thread that has the task, its flows and the replicas in its cache -- takes the
 * readers, bumps the versions of the written flows and builds the engine command; the manager only submits it.
 * returns 1 when the task is settled, 0 when the manager has to look at it (nothing was changed then). */
static int b200_prepare_resident(parsec_device_b200_module_t *dev, b200_task_t *bt)
{
    parsec_gpu_task_t *gpu_task = bt->gpu_task;
    parsec_task_t *this_task = gpu_task->ec;
    const uint8_t my = dev->super.super.super.device_index;
    if( NULL == dev->tile_described ) return 0;
    for( uint32_t i = 0; i < gpu_task->nb_flows; i++ ) {
        const parsec_flow_t *flow = gpu_task->flow_info[i].flow;
        if( PARSEC_FLOW_ACCESS_NONE == (PARSEC_FLOW_ACCESS_MASK & flow->flow_flags) ) continue;
        const parsec_data_copy_t *in = this_task->data[i].data_in;
        if( NULL == in ) continue;
        if( in->device_index != my || NULL == in->device_private || NULL == in->original ) return 0;
        if( !dev->tile_described[b200_tile_of(dev, in)] ) return 0;      /* filled on the stream lane: the kernel has not met it */
    }
    for( uint32_t i = 0; i < gpu_task->nb_flows; i++ ) {
        const parsec_flow_t *flow = gpu_task->flow_info[i].flow;
        const uint8_t type = (uint8_t)(flow->flow_flags & PARSEC_FLOW_ACCESS_MASK);
        if( PARSEC_FLOW_ACCESS_NONE == type ) { gpu_task->flow_info[i].flow_span = 0; continue; }
        parsec_data_copy_t *in = this_task->data[i].data_in;
        if( NULL == in ) continue;
        this_task->data[i].data_out = in;
        gpu_task->flow_info[i].source = NULL;
        b200_use_resident_flow(dev, in, type);
    }
    b200_build_cmd(dev, bt);
    bt->prepared = 1;
    return 1;
}

static int b200_chore_allows_batch(const parsec_task_t *task, const parsec_device_module_t *device)
{
    if( NULL == task || NULL == task->task_class || task->selected_chore < 0 ) return 0;
    const __parsec_chore_t *chore = &task->task_class->incarnations[task->selected_chore];
    return parsec_mca_device_type_supports_batch(device->type) && (0 != (chore->type & device->type)) &&
           (0 != (chore->type & PARSEC_DEV_CHORE_ALLOW_BATCH));
}

/* Call the submit function in RECORD mode: a body that names an engine body through parsec_b200_task_body enqueues
 * nothing and leaves it in the record; an opaque body enqueues its work on the lane stream.  returns the submit code */
static int b200_record_body(parsec_device_b200_module_t *dev, b200_task_t *bt)
{
    parsec_gpu_task_t *gpu_task = bt->gpu_task;
    b200_tl_recording = bt;
    const int rc = gpu_task->submit(&dev->super.super, gpu_task, &dev->lane->super);
    b200_tl_recording = NULL;
    bt->has_complete_stage = (NULL != gpu_task->complete_stage);     /* a body may install one (dtd_test_simple_gemm.c:538) */
    return rc;
}

/* after an opaque body has been enqueued on the lane stream: pushouts on the same stream, then the event */
static int b200_lane_after_submit(parsec_device_b200_module_t *dev, b200_task_t *bt)
{
    parsec_gpu_task_t *gpu_task = bt->gpu_task;
    uint32_t mask = 0;
    for( uint32_t i = 0; i < gpu_task->nb_flows; i++ )
        if( (gpu_task->pushout & (1 << i)) && (PARSEC_FLOW_ACCESS_WRITE & gpu_task->flow_info[i].flow->flow_flags) && NULL != gpu_task->ec->data[i].data_out )
            mask |= (1u << i);
    if( b200_copy_home(dev, bt, mask, dev->lane->cuda_stream) < 0 ) return PARSEC_HOOK_RETURN_ERROR;
    B200_CUDA(cudaEventRecord(b200_bt_event(dev, bt), dev->lane->cuda_stream), "cudaEventRecord", {});
    bt->state = BT_LANE;
    dev->n_lane++;
    parsec_list_nolock_push_back(&dev->waiting_event, &bt->item);
    return PARSEC_HOOK_RETURN_DONE;
}

/* the submit function of a staged lane task, and what follows it */
static int b200_lane_submit(parsec_device_b200_module_t *dev, b200_task_t *bt)
{
    parsec_gpu_task_t *gpu_task = bt->gpu_task;
    /* the submit hook may turn gpu_task into a batch ring: start from a clean singleton (device_gpu.c:2918-2922) */
    PARSEC_LIST_ITEM_SINGLETON(&gpu_task->list_item);
    const int src = b200_record_body(dev, bt);
    if( src < 0 && PARSEC_HOOK_RETURN_ASYNC != src ) return PARSEC_HOOK_RETURN_ERROR;
    if( bt->body >= 0 ) {
        /* first task of a class whose body names an engine body: remember it, and run THIS one in the kernel too
         * once its copy-engine stage-in has landed */
        parsec_b200_submit_set_engine(gpu_task->submit);
        for( uint32_t i = 0; i < gpu_task->nb_flows; i++ ) {
            parsec_data_copy_t *out = gpu_task->ec->data[i].data_out;
            if( NULL == out || NULL == gpu_task->ec->data[i].data_in ) continue;
            const size_t span = gpu_task->flow_info[i].flow_span;
            const uint8_t type = (uint8_t)(gpu_task->flow_info[i].flow->flow_flags & PARSEC_FLOW_ACCESS_MASK);
            if( 0 != b200_describe_tile(dev, bt, out, span, type, b200_home_alias(out->original, span), PB2_SRC_HOST, PB2_TILE_VALID) )
                return PARSEC_HOOK_RETURN_ERROR;
        }
        B200_CUDA(cudaEventRecord(b200_bt_event(dev, bt), dev->lane->cuda_stream), "cudaEventRecord", {});
        bt->state = BT_DMA_IN;
        parsec_list_nolock_push_back(&dev->waiting_event, &bt->item);
        return PARSEC_HOOK_RETURN_DONE;
    }
    /* opaque: its kernels are on the lane stream behind the copies.  A batching body has chained the tasks it took from
     * fifo_pending on the ring of its gpu_task: they ran with it, each of them completes like it. */
    parsec_list_item_t *ring = (parsec_list_item_t*)gpu_task->list_item.list_next;
    while( ring != &gpu_task->list_item ) {
        parsec_list_item_t *next = (parsec_list_item_t*)ring->list_next;
        parsec_gpu_task_t *member = (parsec_gpu_task_t*)ring;
        PARSEC_LIST_ITEM_SINGLETON(ring);
        dev->lane_pending--; dev->st.lane_batched++;
        if( PARSEC_HOOK_RETURN_DONE != b200_lane_after_submit(dev, B200_BT(member)) ) return PARSEC_HOOK_RETURN_ERROR;
        ring = next;
    }
    PARSEC_LIST_ITEM_SINGLETON(&gpu_task->list_item);
    return b200_lane_after_submit(dev, bt);
}

/* the staged batchable tasks of this pass: oldest first, each call may take more of them along */
static int b200_fire_lane(parsec_device_b200_module_t *dev)
{
    int n = 0;
    while( dev->lane_pending > 0 ) {
        parsec_gpu_task_t *head = (parsec_gpu_task_t*)parsec_list_nolock_pop_front(dev->lane->super.fifo_pending);
        if( NULL == head ) { dev->lane_pending = 0; break; }
        dev->lane_pending--;
        if( PARSEC_HOOK_RETURN_DONE != b200_lane_submit(dev, B200_BT(head)) ) return -1;
        n++;
    }
    return n;
}

static int b200_start_task(parsec_device_b200_module_t *dev, parsec_execution_stream_t *es, b200_task_t *bt)
{
    parsec_gpu_task_t *gpu_task = bt->gpu_task;
    int rc;
    (void)es;
    dev->again_window = 0;
    if( bt->prepared ) { bt->state = BT_STAGED; return b200_push_engine(dev, bt); }
    if( dev->cold_inflight >= (int64_t)parsec_b200_stage_window && b200_needs_memory(dev, gpu_task) ) { dev->again_window = 1; return PARSEC_HOOK_RETURN_AGAIN; }
    uint64_t c0 = B200_TSC(), c1;
    if( PARSEC_HOOK_RETURN_DONE != (rc = b200_reserve(dev, bt)) ) return rc;
    c1 = B200_TSC(); dev->tsc_start[0] += c1 - c0; c0 = c1;

    /* Which kind of body?  A body that names an engine body goes to the persistent kernel.  An opaque stream body has
     * enqueued its work on the lane stream the moment it was recorded, so its inputs must be there first -- such bodies
     * are therefore only probed after a copy-engine stage-in on the same stream. */
    const parsec_task_class_t *tc = gpu_task->ec->task_class;
    /* engine bodies are recognised by their submit function having been seen naming one (set below, the first time,
     * after a conservative copy-engine stage-in); dry-run modules never enqueue anything, so they always record */
    int known_engine = bt->recorded || dev->dry_run || (!bt->custom_stage && parsec_b200_submit_is_engine(gpu_task->submit));

    if( known_engine ) {
        rc = b200_stage_in(dev, bt, 0);
        if( rc < 0 ) return rc;
        c1 = B200_TSC(); dev->tsc_start[1] += c1 - c0; c0 = c1;
        if( bt->cold_bytes ) (void)parsec_atomic_fetch_add_int64(&dev->cold_inflight, (int64_t)bt->cold_bytes);
        int src = 0;
        if( !bt->recorded ) {             /* normally done by the thread that called kernel_scheduler */
            src = b200_record_body(dev, bt);
            bt->recorded = 1;
        }
        if( dev->dry_run && bt->body < 0 ) { bt->body = PB2_BODY_NOP; bt->nb_args = 0; }
        if( src < 0 || bt->body < 0 ) {
            parsec_warning("device_b200: body of task class %s stopped naming an engine body", tc ? tc->name : "?");
            return PARSEC_HOOK_RETURN_ERROR;
        }
        if( rc > 0 ) {                      /* unregistered host memory: wait for the copy engine, then push */
            B200_CUDA(cudaEventRecord(b200_bt_event(dev, bt), dev->dma_stream), "cudaEventRecord", {});
            bt->state = BT_DMA_IN;
            parsec_list_nolock_push_back(&dev->waiting_event, &bt->item);
            return PARSEC_HOOK_RETURN_DONE;
        }
        bt->state = BT_STAGED;
        c1 = B200_TSC(); dev->tsc_start[2] += c1 - c0; c0 = c1;
        rc = b200_push_engine(dev, bt);
        dev->tsc_start[3] += B200_TSC() - c0;
        return rc;
    }

    /* stream lane: stage in with the copy engine on the lane stream (or the user's stage_in), run submit, event */
    b200_cuda_here(dev);
    const int user_in = b200_user_stage_in(gpu_task);
    rc = b200_stage_in(dev, bt, user_in ? 2 : 1);
    if( rc < 0 ) return rc;
    if( bt->cold_bytes ) (void)parsec_atomic_fetch_add_int64(&dev->cold_inflight, (int64_t)bt->cold_bytes);
    if( user_in ) {
        uint32_t mask = 0;
        for( uint32_t i = 0; i < gpu_task->nb_flows; i++ )
            if( NULL != gpu_task->ec->data[i].data_out && PARSEC_DATA_STATUS_UNDER_TRANSFER == gpu_task->ec->data[i].data_out->data_transfer_status ) mask |= (1u << i);
        if( mask && PARSEC_SUCCESS != gpu_task->stage_in(gpu_task, mask, &dev->lane->super) ) return PARSEC_HOOK_RETURN_ERROR;
    }
    /* A body that may BATCH (chore flag PARSEC_DEV_CHORE_ALLOW_BATCH, `batch = true` in a JDF body) collects further
     * staged tasks of its kind with parsec_gpu_task_collect_batch (device_gpu.c:2228-2285), which looks for them in
     * the stream's fifo_pending.  Such a task is only STAGED here; its submit function is called when the pass has
     * staged everything it could (b200_fire_lane), so that the tasks behind it are there to be collected. */
    if( b200_chore_allows_batch(gpu_task->ec, &dev->super.super.super) && !parsec_b200_submit_is_engine(gpu_task->submit) ) {
        bt->state = BT_LANE;
        PARSEC_LIST_ITEM_SINGLETON(&gpu_task->list_item);
        parsec_list_nolock_push_back(dev->lane->super.fifo_pending, &gpu_task->list_item);
        dev->lane_pending++;
        return PARSEC_HOOK_RETURN_DONE;
    }
    return b200_lane_submit(dev, bt);
}

/* ------------------------------------------------------------------------------------------------------------------ */
/* submit functions known to name engine bodies (small open-addressed set, shared by the modules)                      */
/* ------------------------------------------------------------------------------------------------------------------ */
#define B200_SUBMIT_SET 256
static void * volatile b200_engine_submits[B200_SUBMIT_SET];
static int parsec_b200_submit_is_engine(parsec_advance_task_function_t fn)
{
    uintptr_t h = ((uintptr_t)fn >> 4) % B200_SUBMIT_SET;
    for( int p = 0; p < B200_SUBMIT_SET; p++ ) {
        void *v = b200_engine_submits[(h + p) % B200_SUBMIT_SET];
        if( v == (void*)fn ) return 1;
        if( NULL == v ) return 0;
    }
    return 0;
}
static void parsec_b200_submit_set_engine(parsec_advance_task_function_t fn)
{
    uintptr_t h = ((uintptr_t)fn >> 4) % B200_SUBMIT_SET;
    for( int p = 0; p < B200_SUBMIT_SET; p++ ) {
        void * volatile *slot = &b200_engine_submits[(h + p) % B200_SUBMIT_SET];
        if( *slot == (void*)fn ) return;
        if( NULL == *slot && parsec_atomic_cas_ptr(slot, NULL, (void*)fn) ) return;
    }
}

/* ------------------------------------------------------------------------------------------------------------------ */
/* pseudo tasks: data_advise PREFETCH / WARMUP (device.h:79-81; parsec_device_data_advise, device_gpu.c:713-777)        */
/* A prefetch is a task with one READ flow and an empty body: the persistent kernel pulls the tile in (TMA) like any    */
/* other stage-in, asynchronously, and later readers of the tile wait on its state on the device.                        */
/* ------------------------------------------------------------------------------------------------------------------ */
static const parsec_flow_t b200_prefetch_flow = {
    .name = "FLOW", .flow_flags = PARSEC_FLOW_ACCESS_READ, .flow_index = 0,
};
static parsec_task_class_t b200_prefetch_tc = {
    .name = "b200 data prefetch", .flags = 0, .task_class_id = 0, .nb_flows = 1, .nb_parameters = 0, .nb_locals = 0,
    .in = { &b200_prefetch_flow, NULL }, .out = { NULL },
};
static int b200_prefetch_submit(parsec_device_gpu_module_t *gpu_device, parsec_gpu_task_t *gpu_task, parsec_gpu_exec_stream_t *gpu_stream)
{
    static const int flow0 = 0;
    return parsec_b200_task_body(gpu_device, gpu_task, gpu_stream, PB2_BODY_NOP, 1, &flow0, NULL, 0.f);
}
static void b200_release_pseudo_task(parsec_gpu_task_t *gpu_task)
{
    if( NULL != gpu_task->ec ) {
        if( NULL != gpu_task->ec->data[0].data_in ) PARSEC_DATA_COPY_RELEASE(gpu_task->ec->data[0].data_in);
        free(gpu_task->ec);
        gpu_task->ec = NULL;
    }
    PARSEC_OBJ_RELEASE(gpu_task);
}

static parsec_hook_return_t b200_kernel_scheduler(parsec_device_module_t *module, parsec_execution_stream_t *es, void *_gpu_task);

static int b200_data_advise(parsec_device_module_t *module, parsec_data_t *data, int advice)
{
    switch( advice ) {
    case PARSEC_DEV_DATA_ADVICE_PREFERRED_DEVICE:
        data->preferred_device = module->device_index;
        return PARSEC_SUCCESS;
    case PARSEC_DEV_DATA_ADVICE_PREFETCH:
    case PARSEC_DEV_DATA_ADVICE_WARMUP: {
        parsec_data_copy_t *src = (data->owner_device >= 0) ? data->device_copies[data->owner_device] : data->device_copies[0];
        if( NULL == src ) return PARSEC_ERR_NOT_FOUND;
        parsec_gpu_task_t *gpu_task = (parsec_gpu_task_t*)PARSEC_OBJ_NEW(parsec_gpu_dsl_task_t);
        gpu_task->task_type = (PARSEC_DEV_DATA_ADVICE_PREFETCH == advice) ? PARSEC_GPU_TASK_TYPE_PREFETCH : PARSEC_GPU_TASK_TYPE_WARMUP;
        gpu_task->ec = (parsec_task_t*)calloc(1, sizeof(parsec_task_t));
        PARSEC_OBJ_CONSTRUCT(gpu_task->ec, parsec_task_t);
        gpu_task->ec->task_class = &b200_prefetch_tc;
        gpu_task->ec->selected_device = module;
        gpu_task->nb_flows = 1;
        gpu_task->flow_info[0].flow = &b200_prefetch_flow;
        gpu_task->flow_info[0].flow_span = data->span;
        gpu_task->stage_in = parsec_default_gpu_stage_in;
        gpu_task->stage_out = parsec_default_gpu_stage_out;
        gpu_task->submit = b200_prefetch_submit;
        gpu_task->release_device_task = b200_release_pseudo_task;
        PARSEC_DATA_COPY_RETAIN(src);
        gpu_task->ec->data[0].data_in = src;
        /* same path as any task: whoever is (or becomes) the manager stages it in; the calling thread may become it */
        (void)b200_kernel_scheduler(module, NULL, gpu_task);
        return PARSEC_SUCCESS;
    }
    default:
        return PARSEC_ERR_NOT_FOUND;
    }
}

/* ------------------------------------------------------------------------------------------------------------------ */
/* the manager loop                                                                                                     */
/* ------------------------------------------------------------------------------------------------------------------ */
static void b200_finish(parsec_device_b200_module_t *dev, parsec_execution_stream_t *es, b200_task_t *bt)
{
    if( bt->cold_bytes ) { (void)parsec_atomic_fetch_add_int64(&dev->cold_inflight, -(int64_t)bt->cold_bytes); bt->cold_bytes = 0; }
    if( !dev->retry_stalled ) dev->retry_stalled = 1;     /* a retirement frees ring space, reopens the stage-in window, unpins replicas */
    if( bt->is_kernel ) { b200_complete(dev, es, bt); return; }
    parsec_gpu_task_t *gpu_task = bt->gpu_task;
    /* pseudo task: the replica is resident and valid now; no runtime completion */
    parsec_data_copy_t *out = gpu_task->ec->data[0].data_out;
    if( NULL != out ) {
        parsec_atomic_lock(&out->original->lock);
        if( PARSEC_DATA_STATUS_UNDER_TRANSFER == out->data_transfer_status ) b200_transfer_done(dev, out, PARSEC_FLOW_ACCESS_READ);
        if( bt->peer_src_mask & 1u ) (void)parsec_atomic_fetch_dec_int32(&bt->peer_src[0]->readers);
        if( 1 == out->readers ) b200_lru_touch(dev, out);
        (void)parsec_atomic_fetch_dec_int32(&out->readers);
        parsec_atomic_unlock(&out->original->lock);
    }
    b200_bt_free(bt);
    gpu_task->last_data_check_epoch = 0;
    gpu_task->release_device_task(gpu_task);
    dev->completed_now++;
}

/* A task that cannot get memory here, all of whose non-resident inputs are replicas of ONE peer b200 device where it
 * needs no memory at all, runs THERE: two devices whose heaps are full of replicas that only tasks queued on the other
 * device still reference would otherwise wait for each other for ever (each replica is retained until its readers
 * have run).  Returns that device, or NULL. */
static parsec_device_b200_module_t *b200_forward_peer(parsec_device_b200_module_t *dev, const parsec_gpu_task_t *gpu_task)
{
    const uint8_t my = dev->super.super.super.device_index;
    parsec_device_b200_module_t *peer = NULL;
    if( PARSEC_GPU_TASK_TYPE_KERNEL != gpu_task->task_type ) return NULL;
    for( uint32_t i = 0; i < gpu_task->nb_flows; i++ ) {
        const parsec_flow_t *flow = gpu_task->flow_info[i].flow;
        if( PARSEC_FLOW_ACCESS_NONE == (PARSEC_FLOW_ACCESS_MASK & flow->flow_flags) ) continue;
        const parsec_data_copy_t *in = gpu_task->ec->data[i].data_in;
        if( NULL == in || in->device_index == my ) continue;
        if( !parsec_mca_device_is_gpu(in->device_index) ) {
            if( NULL != PARSEC_DATA_GET_COPY(in->original, my) ) continue;        /* resident here, would have to be there too */
            return NULL;
        }
        parsec_device_module_t *m = parsec_mca_device_get(in->device_index);
        if( !parsec_b200_is_b200_device(m) ) return NULL;
        if( NULL != peer && (parsec_device_module_t*)peer != m ) return NULL;
        peer = (parsec_device_b200_module_t*)m;
    }
    if( NULL == peer || peer->dry_run != dev->dry_run || b200_needs_memory(peer, gpu_task) ) return NULL;
    return peer;
}

/* starter: `bt` (in `stalled`, BT_NEW) is short of memory here.  If its inputs sit on a peer device where it needs none, the task
 * goes BACK TO THE RUNTIME with that peer as its selected device: the runtime runs its hook again (what a hook that returns
 * AGAIN gets, scheduling.c:445-467) and keeps an a-priori selected device (device.c:113-118).  returns 1 when the task left. */
static int b200_hand_back(parsec_device_b200_module_t *dev, parsec_execution_stream_t *es, b200_task_t *bt)
{
    parsec_device_b200_module_t *peer;
    if( NULL == es || BT_NEW != bt->state || NULL == (peer = b200_forward_peer(dev, bt->gpu_task)) ) return 0;
    parsec_gpu_task_t *gt = bt->gpu_task;
    parsec_task_t *task = gt->ec;
    parsec_list_nolock_remove(&dev->stalled, &bt->item);
    PARSEC_LIST_ITEM_SINGLETON(&bt->item);
    dev->nb_stalled--;
    b200_bt_free(bt);
    gt->last_data_check_epoch = UINT64_MAX;
    gt->release_device_task(gt);                       /* the hook builds a new one */
    (void)parsec_atomic_fetch_add_int64(&task->selected_device->device_load, -task->load);   /* __parsec_execute adds it again ... */
    task->selected_device = &peer->super.super.super;                 /* ... to the device it keeps (device.c: "a-priori selected_device") */
    (void)parsec_atomic_fetch_add_int32(&dev->handed_back, 1);      /* the manager takes it off `owed` */
    dev->st.forwarded++;
    b200_nvtx_mark("b200 task handed back to the runtime for a peer device");
    PARSEC_LIST_ITEM_SINGLETON(&task->super);
    (void)__parsec_reschedule(es, task);
    return 1;
}

/* inbox -> lists of tasks to start, in slot order (starter only).  A slot whose index has been taken but whose pointer
 * is not there yet ends the pass: its caller is a few instructions away from storing it.  The tile descriptions a caller
 * decided go to the device here, in the order of the decisions.  returns the number of records taken, < 0 on error */
static int b200_drain_inbox(parsec_device_b200_module_t *dev)
{
    int64_t head = dev->inbox_head;
    const int64_t head0 = head;
    for(;;) {
        b200_task_t * volatile *slot = &dev->inbox_ring[head & (B200_INBOX_SLOTS - 1)];
        b200_task_t *bt = *slot;
        if( NULL == bt ) break;
        parsec_atomic_rmb();
        *slot = NULL;
        head++;
        {   /* the records a few slots further on: written by other cores a moment ago */
            const char *la = (const char*)dev->inbox_ring[(head + 6) & (B200_INBOX_SLOTS - 1)];
            if( NULL != la ) { B200_PFW(la); B200_PFW(la + 64); B200_PF(la + offsetof(b200_task_t, cmd)); }
        }
        for( int k = 0; k < bt->ntdesc; k++ )
            if( PB2_SUCCESS != pb2_stream_set_tile(dev->stream, bt->tdesc[k].tile, &bt->tdesc[k].desc) ) return -1;
        bt->ntdesc = 0; bt->defer_tiles = 0;
        switch( bt->prepared ) {
        case 1:  parsec_list_nolock_push_back(&dev->settled, &bt->item); dev->nb_settled++; dev->n_settled_by_caller++; break;
        case 2:  parsec_list_nolock_push_back(&dev->cold_q, &bt->item); dev->nb_cold++; dev->n_settled_by_caller++; break;
        case 3:  bt->state = BT_DMA_IN; parsec_list_nolock_push_back(&dev->waiting_event, &bt->item);
                 if( bt->cold_bytes ) (void)parsec_atomic_fetch_add_int64(&dev->cold_inflight, (int64_t)bt->cold_bytes);
                 break;
        default: parsec_list_nolock_push_back(&dev->stalled, &bt->item); dev->nb_stalled++; break;
        }
    }
    if( head != head0 ) { dev->inbox_head = head; dev->retry_stalled = 1; }
    return (int)(head - head0);
}

#define B200_STARTS_PER_PASS 512       /* then look at the retire ring again */
/* Tasks whose caller settled their flows (`settled`, no stage-in) or decided their stage-in (`cold_q`) only need a slot
 * in the command ring: in order, behind the stage-in window.  The worker CTAs of the persistent kernel would happily
 * start thousands of PCIe pulls at once; they would then all finish together, tens of milliseconds later, and their
 * successors with them.  Keeping only a few link round-trips worth of cold bytes in flight makes tasks retire as a steady
 * stream.  returns 0 when the list is done or the window is closed, 1 when the command ring is full, 2 when the pass has
 * started enough, < 0 on error */
static int b200_push_queue(parsec_device_b200_module_t *dev, parsec_list_t *q, int32_t *nb, int *started)
{
    while( *nb > 0 ) {
        if( *started >= B200_STARTS_PER_PASS ) return 2;
        b200_task_t *bt = (b200_task_t*)PARSEC_LIST_ITERATOR_FIRST(q);
        parsec_list_item_t *la = PARSEC_LIST_ITERATOR_NEXT(&bt->item);
        if( la != PARSEC_LIST_ITERATOR_END(q) ) { la = PARSEC_LIST_ITERATOR_NEXT(la);
            if( la != PARSEC_LIST_ITERATOR_END(q) ) { B200_PF(la); B200_PF((const char*)la + offsetof(b200_task_t, cmd)); } }
        if( bt->cold_bytes && dev->cold_inflight >= (int64_t)parsec_b200_stage_window ) return 0;
        parsec_list_nolock_remove(q, &bt->item);
        PARSEC_LIST_ITEM_SINGLETON(&bt->item);
        if( BT_NEW == bt->state ) bt->state = BT_STAGED;
        const uint64_t cold = bt->cold_bytes;          /* the record may be recycled the moment the command is out */
        const int rc = b200_push_engine(dev, bt);
        if( PARSEC_HOOK_RETURN_AGAIN == rc ) { parsec_list_nolock_push_front(q, &bt->item); return 1; }
        if( PARSEC_HOOK_RETURN_DONE != rc ) return -1;
        if( cold ) (void)parsec_atomic_fetch_add_int64(&dev->cold_inflight, (int64_t)cold);
        (*nb)--;
        (*started)++;
    }
    return 0;
}

/* the copy-engine / lane event of a task: 1 it has happened, 0 not yet, -1 it failed */
static int b200_event_state(const b200_task_t *bt)
{
    const cudaError_t q = cudaEventQuery(bt->ev);
    if( cudaSuccess == q ) return 1;
    if( cudaErrorNotReady == q ) { (void)cudaGetLastError(); return 0; }
    parsec_warning("device_b200: event failed: %s", cudaGetErrorString(q));
    return -1;
}

/* The STARTER's pass: inbox, starts, events of the stage-in / lane paths.  Called with `starter_active` held.
 * returns the number of tasks it moved forward (0: nothing to do right now), < 0 on a fatal device problem */
static int b200_start_pass(parsec_device_b200_module_t *dev, parsec_execution_stream_t *es)
{
    uint64_t t0 = B200_TSC(), t1;
    int moved = 0;
    /* 1. inbox */
    {
        const int n = b200_drain_inbox(dev);
        if( n < 0 ) return -1;
        moved += n;
    }
    t1 = B200_TSC(); dev->tsc_s[0] += t1 - t0; t0 = t1;
    /* 2. start tasks.  Settled tasks first (they only need a slot in the command ring; the stage-ins in flight are for
     *    them), then the others, oldest first.  A task that cannot get device memory stays where it is and the
     *    ones behind it are tried: their inputs may be resident already (they hold references that keep
     *    replicas from being evicted), and their retirement is what frees memory.  A full command ring stops the pass,
     *    and so does the stage-in window (a throttle, not a shortage: retirements reopen it). */
    int started = 0;
    if( dev->retry_stalled && (dev->nb_settled > 0 || dev->nb_stalled > 0 || dev->nb_cold > 0) ) {
        dev->retry_stalled = 0;
        int stop = b200_push_queue(dev, &dev->settled, &dev->nb_settled, &started);
        if( 0 == stop ) stop = b200_push_queue(dev, &dev->cold_q, &dev->nb_cold, &started);
        if( stop < 0 ) return -1;
        const int ring_full = (1 == stop);
        int cut = (2 == stop);
        parsec_list_item_t *it = PARSEC_LIST_ITERATOR_FIRST(&dev->stalled), *next;
        int mem_blocked = 0;
        for( ; !ring_full && !cut && it != PARSEC_LIST_ITERATOR_END(&dev->stalled); it = next ) {
            b200_task_t *bt = (b200_task_t*)it;
            next = PARSEC_LIST_ITERATOR_NEXT(it);
            int rc;
            if( started >= B200_STARTS_PER_PASS ) { cut = 1; break; }
            if( next != PARSEC_LIST_ITERATOR_END(&dev->stalled) ) {
                /* look-ahead prefetch of what the full start path reads, one pointer level per position */
                parsec_list_item_t *la = next;
                b200_pf4((b200_task_t*)la); la = PARSEC_LIST_ITERATOR_NEXT(la);
                if( la != PARSEC_LIST_ITERATOR_END(&dev->stalled) ) { b200_pf3((b200_task_t*)la); la = PARSEC_LIST_ITERATOR_NEXT(la);
                if( la != PARSEC_LIST_ITERATOR_END(&dev->stalled) ) { b200_pf2((b200_task_t*)la); la = PARSEC_LIST_ITERATOR_NEXT(la);
                if( la != PARSEC_LIST_ITERATOR_END(&dev->stalled) ) { b200_pf1((b200_task_t*)la); } } }
            }
            /* once a task has failed to get memory in this pass, only tasks that need none are tried -- all of them:
             * the task whose retirement frees memory may be anywhere behind */
            if( mem_blocked && BT_NEW == bt->state && b200_needs_memory(dev, bt->gpu_task) ) {
                if( b200_hand_back(dev, es, bt) ) moved++;
                continue;
            }
            parsec_list_nolock_remove(&dev->stalled, it);
            PARSEC_LIST_ITEM_SINGLETON(it);
            if( BT_NEW == bt->state ) {
                /* residency is decided under the lock, after everything the callers have decided so far has reached the
                 * device (their records are in the inbox: they push before they let the lock go) */
                b200_lock(&dev->alloc_lock);
                const int n = b200_drain_inbox(dev);
                rc = (n < 0) ? PARSEC_HOOK_RETURN_ERROR : b200_start_task(dev, es, bt);
                b200_unlock(&dev->alloc_lock);
                if( n > 0 ) moved += n;
            } else rc = b200_push_engine(dev, bt);            /* staged, waiting for ring space */
            if( PARSEC_HOOK_RETURN_AGAIN == rc ) {
                /* back where it was */
                if( next == PARSEC_LIST_ITERATOR_END(&dev->stalled) ) parsec_list_nolock_push_back(&dev->stalled, it);
                else parsec_list_nolock_add_before(&dev->stalled, next, it);
                if( BT_NEW != bt->state ) break;            /* ring full */
                if( dev->again_window ) break;              /* throttled: every cold task behind this one is, too */
                if( b200_hand_back(dev, es, bt) ) { moved++; continue; }
                mem_blocked = 1;
                continue;
            }
            if( PARSEC_HOOK_RETURN_DONE != rc ) return -1;
            dev->nb_stalled--;
            started++;
        }
        if( cut ) dev->retry_stalled = 1;
    }
    if( dev->lane_pending > 0 ) { const int n = b200_fire_lane(dev); if( n < 0 ) return -1; moved += n; }
    if( started && PB2_SUCCESS != pb2_stream_kick(dev->stream) ) return -1;
    t1 = B200_TSC(); dev->tsc_s[1] += t1 - t0; t0 = t1;
    /* 3. copy-engine / lane events */
    if( !parsec_list_nolock_is_empty(&dev->waiting_event) ) {
        parsec_list_item_t *it = PARSEC_LIST_ITERATOR_FIRST(&dev->waiting_event), *next;
        for( ; it != PARSEC_LIST_ITERATOR_END(&dev->waiting_event); it = next ) {
            b200_task_t *bt = (b200_task_t*)it;
            next = PARSEC_LIST_ITERATOR_NEXT(it);
            const int ev = b200_event_state(bt);
            if( 0 == ev ) continue;
            if( ev < 0 ) return -1;
            parsec_list_nolock_remove(&dev->waiting_event, it);
            PARSEC_LIST_ITEM_SINGLETON(it);
            if( BT_DMA_IN == bt->state ) {
                /* the copy engine delivered the inputs: the replicas are valid, the task goes to the kernel */
                parsec_gpu_task_t *gt = bt->gpu_task;
                for( uint32_t i = 0; i < gt->nb_flows; i++ ) {
                    parsec_data_copy_t *out = gt->ec->data[i].data_out;
                    if( NULL == out || NULL == gt->ec->data[i].data_in || PARSEC_DATA_STATUS_UNDER_TRANSFER != out->data_transfer_status ) continue;
                    parsec_atomic_lock(&out->original->lock);
                    b200_transfer_done(dev, out, (uint8_t)(gt->flow_info[i].flow->flow_flags & PARSEC_FLOW_ACCESS_MASK));
                    parsec_atomic_unlock(&out->original->lock);
                }
                bt->state = BT_STAGED;
                int rc = b200_push_engine(dev, bt);
                if( PARSEC_HOOK_RETURN_AGAIN == rc ) { parsec_list_nolock_push_front(&dev->stalled, &bt->item); dev->nb_stalled++; dev->retry_stalled = 1; }
                else if( PARSEC_HOOK_RETURN_DONE != rc ) return -1;
                else if( PB2_SUCCESS != pb2_stream_kick(dev->stream) ) return -1;
            } else {
                /* BT_LANE: finished; completion belongs to the manager */
                b200_task_t *old;
                do { old = dev->lane_done; bt->next_done = old; } while( !parsec_atomic_cas_ptr(&dev->lane_done, old, bt) );
            }
            moved++;
        }
    }
    t1 = B200_TSC(); dev->tsc_s[2] += t1 - t0; t0 = t1;
    return moved + started;
}

static void b200_trace_task(parsec_device_b200_module_t *dev, const b200_task_t *bt, const pb2_retire_t *r)
{
    if( dev->trace_n == dev->trace_cap ) {
        dev->trace_cap = dev->trace_cap ? 2 * dev->trace_cap : 65536;
        dev->trace_ev = (b200_trace_ev_t*)realloc(dev->trace_ev, dev->trace_cap * sizeof(b200_trace_ev_t));
    }
    b200_trace_ev_t *e = &dev->trace_ev[dev->trace_n++];
    const parsec_task_t *t = bt->gpu_task->ec;
    memset(e, 0, sizeof *e);
    snprintf(e->name, sizeof e->name, "%s", (NULL != t && NULL != t->task_class && NULL != t->task_class->name) ? t->task_class->name : "?");
    if( NULL != t ) { e->locals[0] = t->locals[0].value; e->locals[1] = t->locals[1].value; }
    e->body = bt->body; e->smid = (int32_t)r->smid; e->t_start_ns = r->t_start_ns; e->t_end_ns = r->t_end_ns; e->cold_bytes = bt->cold_bytes;
}

/* <device_b200_trace>.<device index>.json, Chrome trace format (chrome://tracing, Perfetto): one complete event per
 * task, pid = device, tid = SM, ts / dur in microseconds of the device clock relative to the first event */
static void b200_trace_write(parsec_device_b200_module_t *dev)
{
    if( NULL == dev->trace_ev || 0 == dev->trace_n || NULL == parsec_b200_trace || '\0' == parsec_b200_trace[0] ) return;
    char path[1024];
    snprintf(path, sizeof path, "%s.%d.json", parsec_b200_trace, (int)dev->super.super.super.device_index);
    FILE *f = fopen(path, "w");
    if( NULL == f ) { parsec_warning("device_b200: cannot write the trace %s", path); return; }
    uint64_t t0 = UINT64_MAX;
    for( size_t i = 0; i < dev->trace_n; i++ ) if( dev->trace_ev[i].t_start_ns && dev->trace_ev[i].t_start_ns < t0 ) t0 = dev->trace_ev[i].t_start_ns;
    fprintf(f, "{\"displayTimeUnit\": \"ns\", \"traceEvents\": [\n");
    for( size_t i = 0; i < dev->trace_n; i++ ) {
        const b200_trace_ev_t *e = &dev->trace_ev[i];
        fprintf(f, "%s{\"name\": \"%s\", \"ph\": \"X\", \"pid\": %d, \"tid\": %d, \"ts\": %.3f, \"dur\": %.3f, "
                   "\"args\": {\"l0\": %d, \"l1\": %d, \"body\": %d, \"stage_in_bytes\": %lu}}",
                i ? ",\n" : "", e->name, (int)dev->super.super.super.device_index, e->smid,
                (double)(e->t_start_ns - t0) * 1e-3, (double)(e->t_end_ns - e->t_start_ns) * 1e-3,
                e->locals[0], e->locals[1], e->body, (unsigned long)e->cold_bytes);
    }
    fprintf(f, "\n]}\n");
    fclose(f);
}

/* The MANAGER's pass: retire ring, copy-engine pushouts, lane tasks the starter saw finish.
 * returns < 0 on a fatal device problem */
static int b200_retire_pass(parsec_device_b200_module_t *dev, parsec_execution_stream_t *es)
{
    uint64_t t0 = B200_TSC(), t1;
    if( dev->fatal ) return -1;
    if( NULL != dev->lane_done ) {
        b200_task_t *bt = dev->lane_done;
        while( !parsec_atomic_cas_ptr(&dev->lane_done, bt, NULL) ) bt = dev->lane_done;
        while( NULL != bt ) { b200_task_t *next = bt->next_done; b200_finish(dev, es, bt); bt = next; }
    }
    if( !parsec_list_nolock_is_empty(&dev->waiting_out) ) {
        parsec_list_item_t *it = PARSEC_LIST_ITERATOR_FIRST(&dev->waiting_out), *next;
        for( ; it != PARSEC_LIST_ITERATOR_END(&dev->waiting_out); it = next ) {
            b200_task_t *bt = (b200_task_t*)it;
            next = PARSEC_LIST_ITERATOR_NEXT(it);
            const int ev = b200_event_state(bt);
            if( 0 == ev ) continue;
            if( ev < 0 ) return -1;
            parsec_list_nolock_remove(&dev->waiting_out, it);
            PARSEC_LIST_ITEM_SINGLETON(it);
            b200_finish(dev, es, bt);
        }
    }
    for(;;) {
        int n = pb2_stream_poll(dev->stream, dev->retbuf, (int32_t)(sizeof(dev->retbuf) / sizeof(dev->retbuf[0])));
        if( n < 0 ) { parsec_warning("device_b200: %s", pb2_stream_last_error(dev->stream)); return -1; }
        t1 = B200_TSC(); dev->tsc[n ? 3 : 5] += t1 - t0; t0 = t1;
        dev->complete_inline = (1 == n) && (0 == pb2_stream_inflight(dev->stream)) && (dev->inbox_tail == dev->inbox_head);
        if( n > 0 ) b200_nvtx_push("b200 retire pass");
        for( int i = 0; i < n; i++ ) {
            b200_task_t *bt = (b200_task_t*)(uintptr_t)dev->retbuf[i].cookie;
            if( i + 5 < n ) { const char *la = (const char*)(uintptr_t)dev->retbuf[i + 5].cookie; B200_PFW(la); B200_PFW(la + 64); B200_PFW(la + offsetof(b200_task_t, proxy)); }
            if( NULL == bt->gpu_task || BT_INFLIGHT != bt->state ) {
                parsec_warning("device_b200: retire record %d/%d for a task that is not in flight (bt %p state %d ticket %d/%d gpu_task %p)",
                               i, n, (void*)bt, bt->state, bt->ticket, dev->retbuf[i].ticket, (void*)bt->gpu_task);
                return -1;
            }
            bt->result = dev->retbuf[i].result;
            if( NULL != dev->trace_ev || (NULL != parsec_b200_trace && '\0' != parsec_b200_trace[0]) ) b200_trace_task(dev, bt, &dev->retbuf[i]);
            if( (PB2_BODY_CHECK_I32 == bt->body || PB2_BODY_CHECK_F32 == bt->body) && (bt->result >> 32) ) dev->st.check_mismatches += bt->result >> 32;
            bt->ticket = -1;
            if( PB2_SUCCESS != dev->retbuf[i].status ) { parsec_warning("device_b200: task ran an unknown engine body"); return -1; }
            if( bt->dma_out_mask && b200_dma_pushout(dev, bt) > 0 ) {
                bt->state = BT_DMA_OUT;
                parsec_list_nolock_push_back(&dev->waiting_out, &bt->item);
            } else b200_finish(dev, es, bt);
        }
        if( n > 0 ) b200_nvtx_pop();
        t1 = B200_TSC(); dev->tsc[4] += t1 - t0; t0 = t1;
        if( n < (int)(sizeof(dev->retbuf) / sizeof(dev->retbuf[0])) ) break;
    }
    dev->complete_inline = 0;
    b200_close_batch(dev);
    return 0;
}

/* is there anything a starter could do right now? (racy reads: a wrong answer costs one empty pass or one iteration) */
static inline int b200_start_work(const parsec_device_b200_module_t *dev)
{
    return dev->inbox_tail != dev->inbox_head ||
           ((dev->nb_stalled > 0 || dev->nb_settled > 0 || dev->nb_cold > 0) && dev->retry_stalled) ||
           !parsec_list_nolock_is_empty((parsec_list_t*)&dev->waiting_event);
}

/* Take the starter role if it is free and run passes while they move something.  returns < 0 on a fatal problem. */
static int b200_try_start(parsec_device_b200_module_t *dev, parsec_execution_stream_t *es, int sticky)
{
    for(;;) {
        if( dev->starter_active || !parsec_atomic_cas_int32(&dev->starter_active, 0, 1) ) return 0;
        int rc;
        do { b200_nvtx_push("b200 start pass"); rc = b200_start_pass(dev, es); b200_nvtx_pop(); } while( rc > 0 && sticky );
        if( rc < 0 ) dev->fatal = 1;
        parsec_atomic_wmb();
        dev->starter_active = 0;
        parsec_mfence();
        if( rc < 0 ) return -1;
        /* a task that arrived between the last look at the inbox and the release of the role must not be left behind */
        if( dev->inbox_tail == dev->inbox_head ) return 0;
    }
}


static parsec_hook_return_t
b200_kernel_scheduler(parsec_device_module_t *module, parsec_execution_stream_t *es, void *_gpu_task)
{
    parsec_device_b200_module_t *dev = (parsec_device_b200_module_t*)module;
    parsec_gpu_task_t *gpu_task = (parsec_gpu_task_t*)_gpu_task;

    if( 0 == dev->first_entry_ns ) dev->first_entry_ns = b200_now_ns();
    int32_t inside = parsec_atomic_fetch_inc_int32(&dev->callers_inside) + 1;
    if( inside > dev->max_callers_inside ) dev->max_callers_inside = inside;
    /* 0. What does not need a decision of the manager is done here, by the calling thread, in parallel with every other
     *    caller -- it built the gpu_task a moment ago and ran prepare_input on the task: every line is in its cache,
     *    while the manager would have to pull each of them from here, and one thread paying a dozen cache-to-cache
     *    transfers per task is what bounds the task rate of a device.
     *      - the task record;
     *      - the RECORDING of the body: a submit function known to name an engine body is a pure function of the task
     *        (it enqueues nothing), so it can run before the flows are resident;
     *      - for a task whose inputs all are this device's replicas already: readers, versions, the engine command. */
    if( UINT64_MAX != gpu_task->last_data_check_epoch ) {
        parsec_warning("device_b200: gpu_task %p handed to kernel_scheduler twice (epoch %lx)", (void*)gpu_task, (unsigned long)gpu_task->last_data_check_epoch);
        abort();
    }
    b200_task_t *bt = b200_bt_new(dev, gpu_task);
    bt->proxy.taskpool = (NULL != gpu_task->ec) ? gpu_task->ec->taskpool : NULL;
    bt->custom_stage = b200_user_stage_in(gpu_task) || b200_user_stage_out(gpu_task);
    if( !bt->custom_stage && NULL != gpu_task->submit && (dev->dry_run || parsec_b200_submit_is_engine(gpu_task->submit)) ) {
        const int src = b200_record_body(dev, bt);
        if( src >= 0 && bt->body >= 0 ) bt->recorded = 1;
        else if( !dev->dry_run ) bt->body = -1;        /* the manager will say what is wrong with it */
        else { bt->recorded = 1; bt->body = PB2_BODY_NOP; bt->nb_args = 0; }   /* dry run: an opaque body is a no-op */
    }
    int decided = 0;
    if( bt->recorded && bt->is_kernel && !b200_prepare_resident(dev, bt) && dev->nb_stalled < 64 && !dev->memory_pressure &&
        dev->inbox_tail - dev->inbox_head < B200_INBOX_SLOTS - 4096 /* never wait for an inbox slot with the lock held */ ) {
        /*  - for an engine task that needs replicas made or filled: the same decisions the starter would take (heap,
         *    source, versions), under the residency lock.  The tile descriptions ride in the record. */
        b200_lock(&dev->alloc_lock);
        decided = 1;
        bt->defer_tiles = 1;
        if( PARSEC_HOOK_RETURN_DONE == b200_reserve(dev, bt) ) {
            const int rc = b200_stage_in(dev, bt, 0);
            if( 0 == rc ) { b200_build_cmd(dev, bt); bt->prepared = 2; }
            else if( rc > 0 ) {                      /* unregistered host memory: the copy engine brings it, the starter waits for the event */
                B200_CUDA(cudaEventRecord(b200_bt_event(dev, bt), dev->dma_stream), "cudaEventRecord", {});
                bt->prepared = 3;
            } else if( PARSEC_HOOK_RETURN_AGAIN != rc ) dev->fatal = 1;
            /* AGAIN: a peer replica is being reclaimed; nothing was changed, the starter retries */
        }
        if( 0 == bt->prepared ) bt->defer_tiles = (bt->ntdesc > 0);     /* descriptions decided before a failure still go first */
    }
    /* 1. one more task is owed, THEN it is handed over.  In this order the manager can never complete a task whose debt
     *    has not been booked yet: booking first keeps `owed` from dropping to zero -- and a second manager from being
     *    elected -- while a task is on its way into the inbox. */
    int32_t before = parsec_atomic_fetch_add_int32(&dev->owed, 1);
    {
        const int64_t idx = parsec_atomic_fetch_add_int64(&dev->inbox_tail, 1);
        while( idx - dev->inbox_head >= B200_INBOX_SLOTS ) { _mm_pause(); }   /* ring full: the starter is draining it */
        parsec_atomic_wmb();
        dev->inbox_ring[idx & (B200_INBOX_SLOTS - 1)] = bt;
    }
    if( decided ) b200_unlock(&dev->alloc_lock);
    (void)parsec_atomic_fetch_dec_int32(&dev->callers_inside);
    if( before > 0 ) {
        /* somebody manages the device and owes this task too.  If nobody is STARTING tasks right now, this thread does,
         * for as long as tasks keep arriving: starts and retirements then proceed on two cores. */
        (void)b200_try_start(dev, es, 1);
        return PARSEC_HOOK_RETURN_ASYNC;
    }

    /* 2. this thread is the manager until nothing is owed any more */
    dev->st.manager_entries++;
    b200_nvtx_mark("b200 manager elected");
    if( 0 == dev->first_task_ns ) dev->first_task_ns = b200_now_ns();
    if( NULL == es ) {
        /* data_advise comes without an execution stream and owes no runtime completion: it cannot complete other
         * threads' tasks, so it only drives the device until its own pseudo task is done */
        es = parsec_my_execution_stream();
        if( NULL == es && NULL != module->context ) es = module->context->virtual_processes[0]->execution_streams[0];
    }
    b200_cuda_here(dev);
    uint64_t idle_spins = 0;
    for(;;) {
        dev->completed_now = 0;
        if( 0 == (++idle_spins & 0x3ffffff) && NULL != getenv("PARSEC_B200_DEBUG") ) {
            fprintf(stderr, "b200 manager stuck? owed %d inbox %ld stalled %d settled %d starter %d retry %d stream inflight %d executed %lu\n",
                    dev->owed, (long)(dev->inbox_tail - dev->inbox_head), dev->nb_stalled, dev->nb_settled, dev->starter_active, dev->retry_stalled,
                    pb2_stream_inflight(dev->stream), (unsigned long)module->executed_tasks);
        }
        /* the starter role, when nobody has it: one pass, then back to the retire ring */
        if( (dev->nb_stalled > 0 || dev->nb_settled > 0 || dev->nb_cold > 0) && ++dev->blocked_spins >= 1024 ) {
            /* references that keep a replica from being evicted are also dropped where nobody tells the device (the data
             * repositories of the runtime): a waiting task is retried every so often whatever happened */
            dev->blocked_spins = 0; dev->retry_stalled = 1;
        }
        if( b200_start_work(dev) && b200_try_start(dev, es, 0) < 0 ) dev->fatal = 1;
        if( b200_retire_pass(dev, es) < 0 ) {
            parsec_warning("GPU[%d:%s]: the device engine reported a fatal error; giving up", module->device_index, module->name);
            return PARSEC_HOOK_RETURN_DISABLE;
        }
        if( NULL != dev->completion_ring ) {
            parsec_task_t *ring = dev->completion_ring;
            dev->completion_ring = NULL;
            const uint64_t ts0 = B200_TSC();
            __parsec_schedule(es, ring, 0);
            dev->tsc[6] += B200_TSC() - ts0;
        }
        /* `completed_now` belongs to the manager: take a private copy BEFORE the subtraction -- the instant `owed`
         * reaches zero another thread may become the manager and reset the field */
        int32_t done_now = dev->completed_now;
        if( dev->handed_back ) done_now += parsec_atomic_fetch_and_int32(&dev->handed_back, 0);
        if( done_now ) {
            idle_spins = 0;
            /* the subtraction that reaches zero is the LAST thing a manager does with the device */
            const int32_t left = parsec_atomic_fetch_sub_int32(&dev->owed, done_now) - done_now;
            if( 0 == left ) { dev->last_done_ns = b200_now_ns(); return PARSEC_HOOK_RETURN_ASYNC; }
            if( left < 0 ) {
                parsec_warning("GPU[%d:%s]: more tasks completed than were handed over (%d)", module->device_index, module->name, left);
                return PARSEC_HOOK_RETURN_DISABLE;
            }
        }
    }
}

/* ------------------------------------------------------------------------------------------------------------------ */
/* module entry points                                                                                                  */
/* ------------------------------------------------------------------------------------------------------------------ */
static int b200_set_device(parsec_device_gpu_module_t *gpu)
{
    parsec_device_b200_module_t *dev = B200_DEV(gpu);
    if( dev->dry_run ) return PARSEC_SUCCESS;
    B200_CUDA(cudaSetDevice(dev->super.cuda_index), "cudaSetDevice", { return PARSEC_ERROR; });
    return PARSEC_SUCCESS;
}
static int b200_memory_info(parsec_device_gpu_module_t *gpu, size_t *free_mem, size_t *total_mem)
{
    parsec_device_b200_module_t *dev = B200_DEV(gpu);
    if( dev->dry_run ) { *free_mem = *total_mem = (size_t)8 << 30; return PARSEC_SUCCESS; }
    pb2_engine_info_t info;
    if( PB2_SUCCESS != pb2_engine_info(dev->engine, &info) ) return PARSEC_ERROR;
    *free_mem = info.free_mem; *total_mem = info.total_mem;
    return PARSEC_SUCCESS;
}
static int b200_memory_allocate(parsec_device_gpu_module_t *gpu, size_t bytes, void **addr)
{
    parsec_device_b200_module_t *dev = B200_DEV(gpu);
    if( dev->dry_run ) { *addr = (void*)((uintptr_t)1 << 40); dev->slab_base = (char*)*addr; return PARSEC_SUCCESS; }   /* never dereferenced */
    if( PB2_SUCCESS != pb2_engine_malloc(dev->engine, bytes, addr) ) return PARSEC_ERR_OUT_OF_RESOURCE;
    dev->slab_base = (char*)*addr;
    return PARSEC_SUCCESS;
}
static int b200_memory_free(parsec_device_gpu_module_t *gpu, void *addr)
{
    parsec_device_b200_module_t *dev = B200_DEV(gpu);
    if( dev->dry_run ) return PARSEC_SUCCESS;
    return (PB2_SUCCESS == pb2_engine_free(dev->engine, addr)) ? PARSEC_SUCCESS : PARSEC_ERROR;
}
static void *b200_find_incarnation(parsec_device_gpu_module_t *gpu, const char *fname)
{
    (void)gpu;
    return parsec_device_find_function(fname, NULL, NULL);
}

static int b200_memory_register(parsec_device_module_t *device, parsec_data_collection_t *desc, void *ptr, size_t length)
{
    parsec_device_b200_module_t *dev = (parsec_device_b200_module_t*)device;
    if( desc->memory_registration_status == PARSEC_MEMORY_STATUS_REGISTERED ) return PARSEC_SUCCESS;
    /* Registration cache.  ptgpp-generated pools register their collections in the startup hook and unregister them in
     * the destructor (jdf2c.c: "Register all the data"), so an application that runs one pool after another over the
     * same matrix pays cudaHostRegister -- 40 to 400 ms per GiB on this host -- inside every parsec_context_add_taskpool.
     * Ranges given back with memory_unregister stay pinned (lazy) and are revived by the next registration of the same
     * range; a registration that merely overlaps a lazy range retires it first.  device_b200_registration_cache = 0
     * restores eager unpinning. */
    void *alias = ptr;
    int revived = 0;
    parsec_atomic_lock(&b200_ranges_lock);
    for( int i = 0; i < b200_nb_ranges; i++ ) {
        b200_host_range_t *r = &b200_ranges[i];
        if( !r->lazy ) continue;
        if( r->base == (char*)ptr && r->len >= length ) { r->lazy = 0; revived = 1; break; }
        if( (char*)ptr < r->base + r->len && r->base < (char*)ptr + length ) {      /* overlap: the old pinning goes */
            char *old = r->base;
            *r = b200_ranges[--b200_nb_ranges]; i--;
            if( !dev->dry_run ) { (void)pb2_stream_quiesce(dev->stream); (void)pb2_engine_host_unregister(dev->engine, old); }
        }
    }
    parsec_atomic_unlock(&b200_ranges_lock);
    if( revived ) { dev->st.registration_hits++; desc->memory_registration_status = PARSEC_MEMORY_STATUS_REGISTERED; return PARSEC_SUCCESS; }
    if( !dev->dry_run ) {
        if( PB2_SUCCESS != pb2_engine_host_register(dev->engine, ptr, length, &alias) ) return PARSEC_ERROR;
    }
    parsec_atomic_lock(&b200_ranges_lock);
    if( b200_nb_ranges == b200_cap_ranges ) {
        b200_cap_ranges = b200_cap_ranges ? 2 * b200_cap_ranges : 16;
        b200_ranges = (b200_host_range_t*)realloc(b200_ranges, sizeof(b200_host_range_t) * (size_t)b200_cap_ranges);
    }
    b200_ranges[b200_nb_ranges].base = (char*)ptr; b200_ranges[b200_nb_ranges].len = length; b200_ranges[b200_nb_ranges].alias = (char*)alias;
    b200_ranges[b200_nb_ranges].lazy = 0;
    b200_nb_ranges++;
    parsec_atomic_unlock(&b200_ranges_lock);
    desc->memory_registration_status = PARSEC_MEMORY_STATUS_REGISTERED;
    return PARSEC_SUCCESS;
}

static int b200_memory_unregister(parsec_device_module_t *device, parsec_data_collection_t *desc, void *ptr)
{
    parsec_device_b200_module_t *dev = (parsec_device_b200_module_t*)device;
    if( desc->memory_registration_status == PARSEC_MEMORY_STATUS_UNREGISTERED ) return PARSEC_SUCCESS;
    int found = 0;
    parsec_atomic_lock(&b200_ranges_lock);
    for( int i = 0; i < b200_nb_ranges; i++ ) {
        if( b200_ranges[i].base != (char*)ptr || b200_ranges[i].lazy ) continue;
        if( parsec_b200_registration_cache ) b200_ranges[i].lazy = 1;
        else { b200_ranges[i] = b200_ranges[--b200_nb_ranges]; found = 1; }
        break;
    }
    parsec_atomic_unlock(&b200_ranges_lock);
    if( found && !dev->dry_run ) {
        /* nothing of ours may be resident while CUDA unpins the range */
        (void)pb2_stream_quiesce(dev->stream);
        (void)pb2_engine_host_unregister(dev->engine, ptr);
    }
    desc->memory_registration_status = PARSEC_MEMORY_STATUS_UNREGISTERED;
    return PARSEC_SUCCESS;
}

/* module_fini: whatever the cache still pins is given back */
static void b200_registration_cache_drop(parsec_device_b200_module_t *dev)
{
    parsec_atomic_lock(&b200_ranges_lock);
    for( int i = 0; i < b200_nb_ranges; i++ ) {
        if( !b200_ranges[i].lazy ) continue;
        if( !dev->dry_run ) (void)pb2_engine_host_unregister(dev->engine, b200_ranges[i].base);
        b200_ranges[i] = b200_ranges[--b200_nb_ranges]; i--;
    }
    parsec_atomic_unlock(&b200_ranges_lock);
}

static void b200_profile_print(parsec_device_b200_module_t *dev)
{
    if( NULL == getenv("PARSEC_B200_PROFILE") ) return;
    uint64_t tot = 0; for( int i = 3; i < 7; i++ ) tot += dev->tsc[i];
    fprintf(stderr, "b200 starter Mcycles: inbox %.1f start %.1f events %.1f (total %.1f, %lu settled by their caller) | manager Mcycles: poll %.1f finish %.1f idle-poll %.1f schedule %.1f (total %.1f, %lu tasks so far, %lu manager entries)\n",
            dev->tsc_s[0] * 1e-6, dev->tsc_s[1] * 1e-6, dev->tsc_s[2] * 1e-6, (dev->tsc_s[0] + dev->tsc_s[1] + dev->tsc_s[2]) * 1e-6, (unsigned long)dev->n_settled_by_caller,
            dev->tsc[3] * 1e-6, dev->tsc[4] * 1e-6, dev->tsc[5] * 1e-6, dev->tsc[6] * 1e-6,
            tot * 1e-6, (unsigned long)dev->super.super.super.executed_tasks, (unsigned long)dev->st.manager_entries);
    memset(dev->tsc_s, 0, sizeof dev->tsc_s);
    fprintf(stderr, "b200 manager start Mcycles: reserve %.1f stage-in %.1f record %.1f command %.1f\n",
            dev->tsc_start[0] * 1e-6, dev->tsc_start[1] * 1e-6, dev->tsc_start[2] * 1e-6, dev->tsc_start[3] * 1e-6);
    memset(dev->tsc, 0, sizeof dev->tsc); memset(dev->tsc_start, 0, sizeof dev->tsc_start);
}

static int b200_memory_release(parsec_device_module_t *device)
{
    parsec_device_b200_module_t *dev = (parsec_device_b200_module_t*)device;
    b200_profile_print(dev);
    dev->first_task_ns = dev->first_entry_ns = 0;
    /* the tail of an epilog (letting go of the readers it held) may still be running on a worker thread */
    while( dev->epilogs_done < dev->epilogs_started ) { parsec_atomic_rmb(); }
    /* dirty replicas go home first: flush_lru would drop them with a warning (device_gpu.c:1033-1037) */
    if( !dev->dry_run ) (void)pb2_stream_quiesce(dev->stream);
    while( b200_write_back_some(dev, 64) > 0 ) { }
    const int rc = parsec_device_flush_lru(device);
    dev->memory_pressure = 0;
    if( NULL != dev->tile_described ) memset(dev->tile_described, 0, (size_t)dev->super.super.mem_nb_blocks);
    return rc;
}

static int b200_all_devices_attached(parsec_device_module_t *device)
{
    parsec_device_b200_module_t *dev = (parsec_device_b200_module_t*)device, *peer;
    dev->super.super.peer_access_mask = (int16_t)(1 << device->device_index);
    if( dev->dry_run ) {
        for( int j = 0; NULL != (peer = (parsec_device_b200_module_t*)parsec_device_b200_component.modules[j]); j++ )
            dev->super.super.peer_access_mask = (int16_t)(dev->super.super.peer_access_mask | (1 << peer->super.super.super.device_index));
        return PARSEC_SUCCESS;
    }
    for( int j = 0; NULL != (peer = (parsec_device_b200_module_t*)parsec_device_b200_component.modules[j]); j++ ) {
        if( peer == dev ) continue;
        if( PB2_SUCCESS == pb2_engine_enable_peer(dev->engine, peer->super.cuda_index) )
            dev->super.super.peer_access_mask = (int16_t)(dev->super.super.peer_access_mask | (1 << peer->super.super.super.device_index));
        else parsec_warning("GPU[%d:%s]: no peer access to %s: its replicas will be fetched through the copy engine",
                            device->device_index, device->name, peer->super.super.super.name);
    }
    return PARSEC_SUCCESS;
}

int parsec_b200_get_stats(const parsec_device_module_t *device, parsec_b200_stats_t *stats)
{
    if( !parsec_b200_is_b200_device(device) || NULL == stats ) return PARSEC_ERR_BAD_PARAM;
    parsec_device_b200_module_t *dev = (parsec_device_b200_module_t*)device;
    pb2_stream_stats_t ss;
    *stats = dev->st;
    stats->tasks_engine = dev->n_engine; stats->tasks_lane = dev->n_lane;
    stats->first_entry_ns = dev->first_entry_ns; stats->first_task_ns = dev->first_task_ns; stats->last_done_ns = dev->last_done_ns;
    stats->max_concurrent_callers = (uint64_t)dev->max_callers_inside;
    if( PB2_SUCCESS == pb2_stream_stats(dev->stream, &ss) ) {
        stats->kernel_launches = ss.kernel_launches; stats->released_on_device = ss.released_on_device;
        stats->bytes_h2d_kernel = ss.bytes_h2d; stats->bytes_d2d_kernel = ss.bytes_d2d; stats->bytes_d2h_kernel = ss.bytes_d2h;
    }
    return PARSEC_SUCCESS;
}

int parsec_b200_module_init(int dev_id, parsec_device_module_t **module)
{
    parsec_device_b200_module_t *dev = NULL;
    if( 0 != posix_memalign((void**)&dev, 64, sizeof(parsec_device_b200_module_t)) ) return PARSEC_ERR_OUT_OF_RESOURCE;
    memset(dev, 0, sizeof(parsec_device_b200_module_t));
    parsec_device_gpu_module_t *gpu = &dev->super.super;
    parsec_device_module_t *device = &gpu->super;
    *module = NULL;
    PARSEC_OBJ_CONSTRUCT(device, parsec_device_module_t);
    dev->dry_run = parsec_b200_dry_run > 0;
    dev->super.cuda_index = (uint8_t)dev_id;
    dev->super.major = 10; dev->super.minor = 0;
    if( -1 == asprintf(&device->name, "b200(%d)", dev_id) ) { free(dev); return PARSEC_ERROR; }

    if( !dev->dry_run ) {
        pb2_engine_params_t ep;
        memset(&ep, 0, sizeof ep);
        if( PB2_SUCCESS != pb2_engine_create(&dev->engine, dev_id, &ep) ) {
            parsec_warning("device_b200: CUDA device %d is not usable by the engine (needs sm_100)", dev_id);
            free(device->name); free(dev);
            return PARSEC_ERR_DEVICE;
        }
        B200_CUDA(cudaSetDevice(dev_id), "cudaSetDevice", {});
        B200_CUDA(cudaStreamCreateWithFlags(&dev->dma_stream, cudaStreamNonBlocking), "cudaStreamCreate", {});
    }
    /* one exec stream: what submit / stage / complete_stage callbacks receive (device_gpu.h:283-298) */
    gpu->max_exec_streams = 1;
    gpu->exec_stream = (parsec_gpu_exec_stream_t**)malloc(sizeof(parsec_gpu_exec_stream_t*));
    dev->lane = (parsec_cuda_exec_stream_t*)calloc(1, sizeof(parsec_cuda_exec_stream_t));
    gpu->exec_stream[0] = &dev->lane->super;
    gpu->num_exec_streams = 1;
    if( !dev->dry_run ) B200_CUDA(cudaStreamCreateWithFlags(&dev->lane->cuda_stream, cudaStreamNonBlocking), "cudaStreamCreate", {});
    PARSEC_OBJ_CONSTRUCT(&dev->lane->super.infos, parsec_info_object_array_t);
    parsec_info_object_array_init(&dev->lane->super.infos, &parsec_per_stream_infos, &dev->lane->super);
    dev->lane->super.fifo_pending = (parsec_list_t*)PARSEC_OBJ_NEW(parsec_list_t);
    if( -1 == asprintf(&dev->lane->super.name, "b200(%d)", dev_id) ) dev->lane->super.name = NULL;

    device->type                 = PARSEC_DEV_CUDA;      /* BODY [type=CUDA] chores match unchanged (device.c:123-148) */
    device->attach               = parsec_device_attach;
    device->detach               = parsec_device_detach;
    device->taskpool_register    = parsec_device_taskpool_register;
    device->taskpool_unregister  = parsec_device_taskpool_unregister;
    device->memory_register      = b200_memory_register;
    device->memory_unregister    = b200_memory_unregister;
    device->memory_release       = b200_memory_release;
    device->data_advise          = b200_data_advise;
    device->kernel_scheduler     = b200_kernel_scheduler;
    device->all_devices_attached = b200_all_devices_attached;
    gpu->set_device       = b200_set_device;
    gpu->memory_info      = b200_memory_info;
    gpu->memory_allocate  = b200_memory_allocate;
    gpu->memory_free      = b200_memory_free;
    gpu->find_incarnation = b200_find_incarnation;
    /* sm_100 rates, GFLOP/s (the reference's table stops before Blackwell, device_cuda_module.c:45-142):
     * dense bf16/fp16 2250 T, tf32 1100 T, fp32 80 T, fp64 40 T */
    device->gflops_fp16 = 2250000; device->gflops_tf32 = 1100000; device->gflops_fp32 = 80000; device->gflops_fp64 = 40000;
    device->gflops_guess = 0;
    device->device_load = 0;

    PARSEC_OBJ_CONSTRUCT(&gpu->gpu_mem_lru, parsec_list_t);
    PARSEC_OBJ_CONSTRUCT(&gpu->gpu_mem_owned_lru, parsec_list_t);
    PARSEC_OBJ_CONSTRUCT(&gpu->pending, parsec_fifo_t);
    PARSEC_OBJ_CONSTRUCT(&dev->stalled, parsec_list_t);
    PARSEC_OBJ_CONSTRUCT(&dev->settled, parsec_list_t);
    PARSEC_OBJ_CONSTRUCT(&dev->waiting_out, parsec_list_t);
    PARSEC_OBJ_CONSTRUCT(&dev->cold_q, parsec_list_t);
    PARSEC_OBJ_CONSTRUCT(&dev->waiting_event, parsec_list_t);
    memset(&dev->lru_lock, 0, sizeof dev->lru_lock);
    dev->inbox_ring = (b200_task_t * volatile *)calloc(B200_INBOX_SLOTS, sizeof(b200_task_t*));

    int nblocks = parsec_b200_memory_number_of_blocks;
    if( dev->dry_run && -1 == nblocks ) nblocks = 4096;
    if( PARSEC_SUCCESS != parsec_device_memory_reserve(gpu, parsec_b200_memory_percentage, nblocks, (size_t)parsec_b200_memory_block_size) ) goto failed;

    dev->tile_described = (uint8_t*)calloc((size_t)gpu->mem_nb_blocks + 1, 1);
    pb2_stream_params_t sp;
    memset(&sp, 0, sizeof sp);
    sp.cmd_slots = parsec_b200_cmd_slots;
    sp.max_tiles = (int32_t)gpu->mem_nb_blocks;
    sp.idle_us = parsec_b200_idle_us;
    sp.dry_run = dev->dry_run;
    sp.max_workers = parsec_b200_max_workers;
    sp.trace = (NULL != parsec_b200_trace && '\0' != parsec_b200_trace[0]);
    if( parsec_b200_nvtx && NULL == b200_nvtx_domain ) b200_nvtx_domain = nvtxDomainCreateA("parsec_b200");
    if( PB2_SUCCESS != pb2_stream_create(dev->engine, &sp, &dev->stream) ) goto failed;
    *module = device;
    return PARSEC_SUCCESS;
failed:
    parsec_warning("device_b200: initialisation of device %d failed", dev_id);
    if( NULL != dev->engine ) pb2_engine_destroy(dev->engine);
    free(device->name); free(dev);
    return PARSEC_ERROR;
}

int parsec_b200_module_fini(parsec_device_module_t *device)
{
    parsec_device_b200_module_t *dev = (parsec_device_b200_module_t*)device;
    parsec_device_gpu_module_t *gpu = &dev->super.super;
    if( NULL != dev->stream ) { (void)pb2_stream_quiesce(dev->stream); }
    b200_profile_print(dev);
    b200_trace_write(dev);
    free(dev->trace_ev); dev->trace_ev = NULL; dev->trace_n = dev->trace_cap = 0;
    while( dev->epilogs_done < dev->epilogs_started ) { parsec_atomic_rmb(); }
    while( b200_write_back_some(dev, 64) > 0 ) { }
    parsec_device_memory_release(gpu);
    b200_registration_cache_drop(dev);
    if( NULL != dev->stream ) { pb2_stream_destroy(dev->stream); dev->stream = NULL; }
    free((void*)dev->inbox_ring); dev->inbox_ring = NULL;
    PARSEC_OBJ_DESTRUCT(&gpu->pending);
    PARSEC_OBJ_DESTRUCT(&dev->lane->super.infos);
    free(dev->lane->super.name);
    PARSEC_OBJ_RELEASE(dev->lane->super.fifo_pending);
    if( !dev->dry_run ) {
        (void)cudaStreamDestroy(dev->lane->cuda_stream);
        (void)cudaStreamDestroy(dev->dma_stream);
    }
    free(dev->tile_described);
    free(dev->lane); free(gpu->exec_stream);
    if( NULL != dev->engine ) { pb2_engine_destroy(dev->engine); dev->engine = NULL; }
    free(device->name); device->name = NULL;
    return PARSEC_SUCCESS;
}
