#!/usr/bin/env python
"""bench.py -- BASELINE.json metric on its config: tasks/s (+ tile GB/s) of a 2D-block-cyclic tile DAG on B200.

Workload at N=1 = BASELINE configs[1]: Ex05_Broadcast dataflow, 256x256 fp32 tiles (262 144 B), K = 4096 broadcast
groups, fan-out F = 8 (NB = 14): 36 864 tasks, 9.66 GB of algorithmic tile traffic per step.  A "step" is one complete
pass of that DAG.

  value        whole-job tasks/s with the tiles already resident in HBM: the window the host runtime builds for the pool
               is run by the raw engine (re-arm + persistent kernel), timed with CUDA events on the engine's stream.
  e2e          the same metric through the REFERENCE-FACING PLUG-IN with HOST buffers: the reference's own runtime
               (oracle/_ref/parsec: unmodified ICLDisco/parsec + our MCA component parsec/mca/device/b200) schedules the
               task pool parsec-ptgpp generated from tests/parsec/ex05_b200.jdf; every tile is staged in from pinned
               host memory by the persistent kernel, every task retires through the device->host ring.  Wall clock of
               parsec_context_add_taskpool .. parsec_context_wait, measured inside the application.
  e2e_standalone  the same DAG through this repository's own C-ABI host runtime (include/pb2_parsec.h), which knows the
               whole pool up front and releases successors on the device.
  roofline     dominant kernel pb2_engine_hbm_kernel: algorithmic bytes / CUDA-event time vs the measured HBM peak, plus
               the DRAM traffic ncu measured (`traffic`, `dram_frac`) and the measured L2 read ceiling (`l2_frac`): 7 of
               the 8 readers of a tile hit the 126 MB L2, so the algorithmic figure can exceed the HBM peak.
  cpu_baseline / --impl reference
               the reference's OWN CPU implementation: the same generated task pool restricted to its CPU incarnations,
               scheduled by the reference runtime on all host cores (cpu_baseline.kind = "reference").
  secondary    in-run records of the other BASELINE configs with their parity checks: configs[0] chain (tasks/s, ns/edge;
               also under the reference's own cuda device module), configs[2] DTD tile-GEMM NT=32 (TFLOP/s vs the measured
               bf16 peak, sampled value check), the e2e workload under the reference's own cuda device module (the drop-in
               comparison), at N=4 configs[3] rtt ring, at N=8 configs[4] Cholesky-shaped DAG, the multi-GPU parity
               cases, and the Ex05 DAG on a collection with k-cyclic factor 64.
N > 1 (torchrun, one rank per GPU): weak scaling of the device-resident value -- every rank owns K groups of a K*N-group
collection on a 1 x N block-cyclic grid (kp = 1: tile k on rank k mod N, the map of mydata in examples/Ex05_Broadcast;
--kp changes it), TaskRecv(k, n) lives on the owner of mydata(k+n); cross-GPU edges are released by the producer's CTA over
NVLink and tiles are pulled by the consumers (NCCL is only the per-step barrier).  e2e at N > 1 is the SAME path as at
N = 1: the reference runtime driving N b200 device modules from one process, run by rank 0 after the process group is gone.
--impl reference: the reference's CPU implementation of the WHOLE job of the N-GPU arm (K*N groups) on the host cores.
"""
import argparse
import ctypes as C
import json
import os
import subprocess
import sys
import threading
import time

import numpy as np

ROOT = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, ROOT)

TILE = 256 * 256 * 4
K_GROUPS = 4096
NB = 14
F = NB // 2 + 1
REF_BIN = os.path.join(ROOT, "oracle", "_ref", "bin")
NVLINK_GBS = 770.0          # per direction per GPU: the MEASURED peer copy B200_PROFILING.md gives as the NVLink denominator
NVLINK_NOMINAL_GBS = 900.0  # nominal, for context


def measured(key, fallback):
    p = os.path.join(ROOT, "MEASURED_PEAKS.json")
    if os.path.exists(p):
        d = json.load(open(p))
        if key in d:
            return float(d[key]), "measured (MEASURED_PEAKS.json %s)" % key
    return fallback, "fallback (B200_PROFILING.md)"


class ClockSampler:
    """nvidia-smi clocks / throttle reasons during the timed region (B200_PROFILING.md recipe)."""

    def __init__(self, index=0):
        self.index, self.rows, self.proc = index, [], None

    def start(self):
        q = "clocks.sm,clocks.max.sm,clocks_event_reasons.hw_slowdown,clocks_event_reasons.hw_thermal_slowdown,clocks_event_reasons.sw_thermal_slowdown,clocks_event_reasons.sw_power_cap"
        try:
            self.proc = subprocess.Popen(["nvidia-smi", f"--id={self.index}", f"--query-gpu={q}", "--format=csv,noheader,nounits", "-lms", "20"],
                                         stdout=subprocess.PIPE, stderr=subprocess.DEVNULL, text=True)
            threading.Thread(target=self._read, daemon=True).start()
        except Exception:
            self.proc = None
        return self

    def _read(self):
        for line in self.proc.stdout:
            self.rows.append([x.strip() for x in line.split(",")])

    def stop(self):
        if self.proc:
            self.proc.terminate()
        sm = sorted(int(r[0]) for r in self.rows if r and r[0].isdigit())
        mx = [int(r[1]) for r in self.rows if len(r) > 1 and r[1].isdigit()]
        names = ["hw_slowdown", "hw_thermal_slowdown", "sw_thermal_slowdown", "sw_power_cap"]
        reasons = sorted({names[i] for r in self.rows if len(r) >= 6 for i in range(4) if r[2 + i].lower().startswith("active")})
        return {"sm_mhz": sm[len(sm) // 2] if sm else None, "sm_max_mhz": max(mx) if mx else None,
                "reasons": reasons, "samples": len(sm)}


# ------------------------------------------------------------------------------------------------------------------------
# the reference runtime (oracle/_ref): applications compiled by parsec-ptgpp from tests/parsec/*.jdf
# ------------------------------------------------------------------------------------------------------------------------
def run_app(app, argv, env=None, timeout=600):
    exe = os.path.join(REF_BIN, app)
    if not os.path.exists(exe):
        return None
    e = dict(os.environ)
    for k in ("PARSEC_MCA_device_b200_enabled", "PARSEC_MCA_device_b200_dry_run", "PARSEC_MCA_device_cuda_enabled"):
        e.pop(k, None)
    e.update(env or {})
    p = subprocess.run([exe] + [str(a) for a in argv], env=e, cwd="/tmp", capture_output=True, text=True, timeout=timeout)
    lines = [l for l in p.stdout.splitlines() if l.startswith("{")]
    if not lines:
        raise RuntimeError("%s printed no result (rc %d): %s" % (app, p.returncode, p.stderr[-800:]))
    d = json.loads(lines[-1])
    d["rc"] = p.returncode
    return d


CPU_ENV = {"PARSEC_MCA_device_cuda_enabled": "0"}


def reference_cpu_arm(K, steps, warmup):
    """The reference's own scheduler + the CPU incarnations of the generated task pool, all host cores."""
    d = run_app("ex05_b200", ["-m", "cpu", "-K", K, "-t", TILE // 4, "-r", steps + warmup], CPU_ENV)
    if d is None:
        return None
    assert d["errors"] == 0, "the reference's CPU run found wrong values"
    times = d["times_s"][warmup:]
    return {"value": d["tasks"] * len(times) / sum(times), "ms_per_step": sum(times) / len(times) * 1e3, "cores": d["cores"],
            "tasks": d["tasks"], "steps": len(times), "kind": "reference",
            "sample": "the full workload: %d groups (%d tasks) per step, tiles in host memory, reference runtime (lfq scheduler) + CPU bodies" % (K, d["tasks"])}


def port_cpu_arm(K, steps, warmup):
    """Fallback when oracle/_ref was not built: the oracle's CPU port of the scheduler path (cpu_baseline.kind = port)."""
    from oracle import orc, orc_dags as dags
    cores = os.cpu_count() or 1
    dag = dags.ex05_broadcast(K, NB, TILE)
    host = np.zeros(K * TILE // 4, np.int32)
    tiles = np.zeros(K, orc.TILE_DTYPE)
    tiles["bytes"] = TILE
    tiles["state"] = orc.TILE_VALID
    tiles["dev_ptr"] = host.ctypes.data + np.arange(K, dtype=np.uint64) * np.uint64(TILE)
    times = []
    for it in range(warmup + steps):
        secs, _, errs = orc.cpu_sched_run(dag.tasks, dag.succ, tiles, dag.ready, cores)
        assert secs > 0 and errs == 0
        if it >= warmup:
            times.append(secs)
    return {"value": dag.ntasks * len(times) / sum(times), "ms_per_step": sum(times) / len(times) * 1e3, "cores": cores,
            "tasks": dag.ntasks, "steps": len(times), "kind": "port", "sample": "%d groups per step, oracle/orc_cpu_sched.c" % K}


def cpu_baseline_arm(K, steps, warmup):
    """The reference's CPU run where oracle/_ref has one that runs, else the oracle's port.  A reference application
    that is there but cannot run (a library missing from a copied install, say) is reported, not fatal: the CPU
    baseline is a record beside the GPU measurement, which must still print its result."""
    try:
        r = reference_cpu_arm(K, steps, warmup)
    except RuntimeError as exc:
        print("bench.py: the reference's CPU run failed, using the oracle's port: %r" % (exc,), file=sys.stderr)
        r = port_cpu_arm(K, steps, warmup)
        r["sample"] += "; the reference's run failed: %s" % str(exc)[:300]
    return r or port_cpu_arm(K, steps, warmup)


def e2e_mca(K, ngpus, steps, cores):
    """e2e through the reference-facing plug-in: reference runtime + parsec/mca/device/b200, host buffers."""
    env = {"PARSEC_MCA_device_b200_enabled": str(ngpus),
           # the bench process keeps its own slabs on the same GPUs: give the component's heap what the workload needs
           # (a GPU holds its own K/N tiles plus the replicas of up to three peers' tiles that its receivers read)
           "PARSEC_MCA_device_b200_memory_number_of_blocks": str(max(4 * K // max(ngpus, 1), 1024) + 1024)}
    warm = 2
    d = run_app("ex05_b200", ["-m", "gpu", "-K", K, "-t", TILE // 4, "-r", steps + warm, "-c", cores], env, timeout=240)
    if d is None:
        return None
    assert d["errors"] == 0 and d["b200"]["check_mismatches"] == 0, "e2e run: wrong values"
    assert d["executed_on_gpu"] == d["tasks"] * (steps + warm) and d["b200_modules"] == ngpus
    times = d["times_s"][warm:]
    sec = sum(times) / len(times)
    reps = steps + warm
    return {"value": d["tasks"] / sec, "unit": "tasks/s", "ms_per_step": sec * 1e3,
            "h2d_bytes_per_step": d["h2d_bytes"] // reps + 64 * (d["tasks"] + K),      # tiles + 64-byte ring commands
            "d2h_bytes_per_step": 32 * d["tasks"],                                      # retire records (result, versions)
            "tile_gbs": K * (1 + F) * TILE / sec / 1e9, "path": "reference runtime + MCA component parsec/mca/device/b200 (%d module%s), %d worker threads" % (ngpus, "" if ngpus == 1 else "s", d["cores"]),
            "tasks": d["tasks"], "kernel_launches_total": d["b200"]["kernel_launches"], "best_ms": d["best_s"] * 1e3,
            "median_ms": sorted(times)[len(times) // 2] * 1e3, "steps": len(times),
            "max_concurrent_callers": d["b200"]["max_concurrent_callers"]}


# ------------------------------------------------------------------------------------------------------------------------
# secondary records (other BASELINE configs), each with its own parity check
# ------------------------------------------------------------------------------------------------------------------------
def secondary_chain():
    """configs[0]: Ex02 chain, 1000 tasks: reference runtime CPU vs the b200 component vs the raw engine window."""
    out = {"config": "Ex02_Chain, 1000-task linear chain (configs[0])"}
    c = run_app("ex02_b200", ["-m", "cpu", "-N", 999, "-c", 2, "-r", 5], CPU_ENV)
    if c:
        out["reference_cpu"] = {"tasks_per_s": c["tasks_per_s"], "ns_per_edge": c["ns_per_edge"], "ok": c["errors"] == 0}
    g = run_app("ex02_b200", ["-m", "gpu", "-N", 999, "-c", 2, "-r", 5],
                {"PARSEC_MCA_device_b200_enabled": "1", "PARSEC_MCA_device_b200_memory_number_of_blocks": "1024"})
    if g:
        out["b200_component"] = {"tasks_per_s": g["tasks_per_s"], "ns_per_edge": g["ns_per_edge"],
                                 "ok": g["errors"] == 0 and g["executed_on_gpu"] == 5000}
    try:        # the same binary under the reference's OWN GPU module (parsec/mca/device/cuda): the drop-in comparison
        r = run_app("ex02_b200", ["-m", "gpu", "-N", 999, "-c", 2, "-r", 5], {"PARSEC_MCA_device_cuda_enabled": "1"}, timeout=120)
        if r:
            out["reference_cuda_component"] = {"tasks_per_s": r["tasks_per_s"], "ns_per_edge": r["ns_per_edge"],
                                               "ok": r["errors"] == 0 and r["b200_modules"] == 0 and r["executed_on_gpu"] == 5000}
    except Exception as exc:
        out["reference_cuda_component"] = {"error": repr(exc)}
    from oracle import orc_dags as dags
    from parsec_b200 import _lib as L
    from parsec_b200.engine import Engine
    with Engine(0) as eng:
        dag = dags.ex02_chain(999)
        slab = eng.malloc(512)
        tiles = np.zeros(dag.ntiles, L.TILE_DTYPE)
        tiles["dev_ptr"], tiles["bytes"], tiles["state"] = slab, dag.tile_bytes, L.TILE_VALID
        eng.h2d(slab, np.zeros(128, np.int32))
        w = eng.window(0, dag.tasks, dag.succ, tiles, dag.ready)
        ms = min(w.run()["kernel_ms"] for _ in range(5))
        res = w.results()
        got = np.empty(1, np.int32)
        eng.d2h(got, slab)
        out["engine_window"] = {"tasks_per_s": 1000 / ms * 1e3, "ns_per_edge": ms * 1e6 / 999,
                                "ok": bool(np.array_equal(res["retire_order"], np.arange(1000)))}
        w.close()
    return out


def secondary_reference_cuda(K, cores):
    """The e2e workload under the reference's OWN GPU device module (parsec/mca/device/cuda, one cudaMemcpyAsync per flow,
    one kernel launch and three events per task): the same binary, the same generated task pool, the same GPU -- what the
    b200 component is a drop-in for.  Bodies are the same kernels, launched stand-alone (pb2_body_launch)."""
    warm, steps = 1, 3
    d = run_app("ex05_b200", ["-m", "gpu", "-K", K, "-t", TILE // 4, "-r", steps + warm, "-c", cores],
                {"PARSEC_MCA_device_cuda_enabled": "1"}, timeout=120)
    if d is None:
        return None
    times = d["times_s"][warm:]
    sec = sum(times) / len(times)
    return {"config": "BASELINE configs[1] through the reference's cuda device module, %d worker threads" % d["cores"],
            "tasks_per_s": d["tasks"] / sec, "ms_per_step": sec * 1e3, "best_ms": d["best_s"] * 1e3,
            "ok": d["errors"] == 0 and d["b200_modules"] == 0 and d["gpu_modules"] == 1 and d["executed_on_gpu"] == d["tasks"] * (steps + warm)}


def secondary_gemm(clock_index):
    """configs[2]: DTD tile-GEMM DAG, 512x512 bf16 tiles, N = 16384 (NT = 32), tensor-core body, reference LCG data."""
    from oracle import orc, orc_dags as dags
    from parsec_b200 import _lib as L
    from parsec_b200.bf16 import bf16_bits_to_f32, f32_to_bf16_bits, round_to_bf16
    from parsec_b200.engine import Engine
    NT, T = 32, 512
    tb = T * T * 2
    O = orc.lib()
    host = np.empty(3 * NT * NT * T * T, np.uint16)
    tmp = np.empty(T * T, np.float32)
    for which, seed in enumerate((1789, 1805, 1901)):                     # dtd_test_simple_gemm.c:1135-1139
        for i in range(NT):
            for j in range(NT):
                O.orc_lcg_tile(tmp.ctypes.data_as(C.c_void_p), i * T, j * T, T, T, NT * T, T, seed)
                host[((which * NT + i) * NT + j) * T * T:][:T * T] = f32_to_bf16_bits(tmp)
    dag = dags.dtd_gemm(NT, T)
    dag.tasks["access"][:, 2] &= ~np.uint8(L.FLOW_PUSHOUT)                # device-resident: C stays in HBM
    with Engine(0) as eng:
        slab = eng.malloc(dag.ntiles * tb)
        eng.h2d(slab, host)
        tiles = np.zeros(dag.ntiles, L.TILE_DTYPE)
        tiles["dev_ptr"] = slab + np.arange(dag.ntiles, dtype=np.uint64) * np.uint64(tb)
        tiles["bytes"], tiles["state"] = tb, L.TILE_VALID
        w = eng.window(1, dag.tasks, dag.succ, tiles, dag.ready)
        st = w.run()                                                      # the checked run: C = C0 + sum_k A(i,k) B(k,j)^T
        assert st["tasks_retired"] == NT ** 3
        res = w.results()
        order_ok = bool(np.array_equal(res["seen_version"][:, 2], np.tile(np.arange(NT), NT * NT)))
        tile_f32 = lambda which, i, j: bf16_bits_to_f32(host[((which * NT + i) * NT + j) * T * T:][:T * T]).reshape(T, T)
        worst, checked = 0.0, []
        got = np.empty(T * T, np.uint16)
        for (i, j) in [(0, 0), (NT - 1, NT - 1), (5, 17), (20, 3)]:
            acc = tile_f32(2, i, j).astype(np.float64)
            mag = np.abs(acc)
            for k in range(NT):
                acc += (tile_f32(0, i, k) @ tile_f32(1, k, j).T).astype(np.float64)
                mag = np.maximum(mag, np.abs(acc))
            eng.d2h(got, slab + ((2 * NT + i) * NT + j) * tb)
            err = np.abs(bf16_bits_to_f32(got).reshape(T, T) - round_to_bf16(acc.astype(np.float32))) / np.maximum(mag, 1.0)
            worst = max(worst, float(err.max()))
            checked.append([i, j])
        sampler = ClockSampler(clock_index).start()
        t_wait = time.perf_counter()
        while not sampler.rows and time.perf_counter() - t_wait < 3.0:      # nvidia-smi needs ~100 ms before its first sample
            w.run()
        sampler.rows.clear()
        ms = []
        while len(ms) < 7 or (len(sampler.rows) < 2 and len(ms) < 60):      # the timed runs, under the sampler
            ms.append(w.run()["kernel_ms"])
        ms.sort()
        clocks = sampler.stop()
        w.close()
    med = ms[len(ms) // 2]
    flops = 2.0 * (NT * T) ** 3
    peak, how = measured("bf16_tflops", 1686.0)
    sus, _ = measured("bf16_tflops_sustained", 1435.5)
    return {"config": "DTD tile-GEMM DAG, 512x512 bf16 tiles, N=16384, NT=32, 32768 tasks (configs[2])", "kernel": "pb2_engine_gemm2_kernel",
            "data": "reference LCG (dtd_test_simple_gemm.c:154-196, seeds 1789/1805/1901) cast to bf16", "ms_per_run_median": med,
            "ms_per_run_min": ms[0], "tasks_per_s": NT ** 3 / med * 1e3, "tflops": flops / med / 1e9,
            "roofline": {"bound": "tensor", "achieved": flops / med / 1e9, "peak": peak, "unit": "TFLOP/s", "frac": flops / med / 1e9 / peak,
                         "frac_of_sustained": flops / med / 1e9 / sus, "peak_source": how},
            "parity": {"dependency_order_ok": order_ok, "tiles_checked": checked, "max_rel_err": worst,
                       "tolerance": 2.0 ** -7, "values_ok": bool(worst <= 2.0 ** -7)},
            "clocks": clocks}


def secondary_multi_gpu_parity(rank, world, local, torch, dist):
    """The multi-GPU parity cases of tests/mgpu_worker.py, run by all ranks inside the bench run."""
    sys.path.insert(0, os.path.join(ROOT, "tests"))
    import mgpu_worker as W
    out = {}
    for case in ("ex05", "rtt", "random_dtd", "cholesky"):
        try:
            out[case] = bool(W.run_case(case, rank, world, local, torch, dist)["ok"])
        except Exception as exc:                                           # a failed parity case is reported, not hidden
            out[case] = False
            print("rank %d: parity case %s raised %r" % (rank, case, exc), file=sys.stderr)
    return out


def secondary_rtt(rank, world, local, torch, dist):
    """configs[3]: rtt.jdf ring, 1024x1024 fp32 tiles (4 MiB), NT=1024 hops over the GPUs, FRAGS chains."""
    from parsec_b200 import multigpu as M
    from parsec_b200.engine import Engine
    nt, tile, steps = 1024, 4 << 20, 3
    rec = {"config": "rtt ring, 1024x1024 fp32 tiles, NT=1024, %d GPUs (configs[3])" % world, "runs": []}
    for frags in (1, 16):
        g = M.rtt_global(nt, world, tile, frags)
        part = M.Partition(*g, nranks=world, part_bytes=32768)
        eng = Engine(local, timeout_ms=20000, part_bytes=32768)     # a serial chain of 4 MiB tiles wants many small parts
        eng.use_stream(M.work_stream(torch))
        run = M.SharedRun(eng, part, rank, world, dist, torch)
        for _ in range(2):
            run.step()
        torch.cuda.synchronize(); run.wait()
        dist.barrier(); torch.cuda.synchronize()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        for _ in range(steps):
            run.step()
        e1.record()
        torch.cuda.synchronize()
        st = run.wait()
        ms = torch.tensor([e0.elapsed_time(e1) / steps], device="cuda", dtype=torch.float64)
        dist.all_reduce(ms, op=dist.ReduceOp.MAX)
        ok, seen = True, [0, 0]
        k0 = ((nt - 1) // world) * world
        # rank 0's slot enters run r holding (r-1)*(k0+1) (its last writer of the previous run is PING(k0)); the chain adds
        # nt to that: after the 2 warm-up runs and the `steps` timed ones the last hop's rank holds this value
        want = (1 + steps) * (k0 + 1) + nt
        if (nt - 1) % world == rank:                       # the rank that ran the last hop holds the final version
            slab = np.zeros(run.slab_bytes // 4, np.int32)
            eng.d2h(slab, run.slab); eng.synchronize()
            got = slab[: frags * tile // 4]
            seen = [int(got.min()), int(got.max())]
            ok = bool(np.all(got == want))
        flag = torch.tensor([1 if ok else 0, seen[0], seen[1]], device="cuda")
        mx = flag.clone()
        dist.all_reduce(flag, op=dist.ReduceOp.MIN)
        dist.all_reduce(mx, op=dist.ReduceOp.MAX)
        t = float(ms.item()) / 1e3
        rec["runs"].append({"FRAGS": frags, "ms_per_run": t * 1e3, "us_per_hop": t / (nt - 1) * 1e6,
                            "tile_GBs": (nt - 1) * frags * tile / t / 1e9, "nvlink_frac": (nt - 1) * frags * tile / t / 1e9 / NVLINK_GBS / max(min(frags, world), 1),
                            "parity_ok": bool(flag[0].item()), "expected_value": want, "seen_min_max": [int(mx[1].item()), int(mx[2].item())],
                            "retired": st["tasks_retired"]})
        del run
        eng.close()
    return rec


def secondary_cholesky(rank, world, local, torch, dist):
    """configs[4]: tile-Cholesky-shaped DAG, 1024x1024 bf16 tiles, NT=64, P x Q grid, tensor-core bodies."""
    from parsec_b200 import multigpu as M
    from parsec_b200.bf16 import f32_to_bf16_bits
    from parsec_b200.engine import Engine
    NT, nb, steps = 64, 1024, 3
    P, Q = {1: (1, 1), 2: (1, 2), 4: (2, 2), 8: (2, 4)}[world]
    g = M.cholesky_global(NT, nb, P, Q)
    tasks, succ, tiles, ready, task_rank, tile_rank = g
    part = M.Partition(*g, nranks=world)
    eng = Engine(local, timeout_ms=30000)
    eng.use_stream(M.work_stream(torch))
    run = M.SharedRun(eng, part, rank, world, dist, torch, kind=1)
    one = f32_to_bf16_bits(np.random.default_rng(7).uniform(-0.01, 0.01, nb * nb).astype(np.float32)).view(np.uint8)
    run.load_home_tiles(tile_rank, {int(t): one for t in range(len(tiles))})
    for _ in range(2):
        run.step()
    torch.cuda.synchronize(); st = run.wait()
    retired_ok = st["tasks_retired"] == len(run.p["global_id"])
    dist.barrier(); torch.cuda.synchronize()
    e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    e0.record()
    for _ in range(steps):
        run.step()
    e1.record()
    torch.cuda.synchronize()
    st = run.wait()
    ms = torch.tensor([e0.elapsed_time(e1) / steps], device="cuda", dtype=torch.float64)
    dist.all_reduce(ms, op=dist.ReduceOp.MAX)
    tot = torch.tensor([float(st["bytes_d2d"]), 1.0 if (retired_ok and st["tasks_retired"] == len(run.p["global_id"])) else 0.0], device="cuda", dtype=torch.float64)
    d2d = tot.clone(); dist.all_reduce(d2d)
    okf = tot[1:].clone(); dist.all_reduce(okf, op=dist.ReduceOp.MIN)
    t = float(ms.item()) / 1e3
    ngemm = int((tasks["body"] == 16).sum())
    peak, _ = measured("bf16_tflops_sustained", 1435.5)
    return {"config": "tile-Cholesky-shaped DAG, 1024x1024 bf16, N=65536 (NT=64), %dx%d grid (configs[4])" % (P, Q), "tasks": len(tasks),
            "ms_per_run": t * 1e3, "tasks_per_s": len(tasks) / t, "tflops": ngemm * 2.0 * nb ** 3 / t / 1e12,
            "tensor_frac_of_sustained": ngemm * 2.0 * nb ** 3 / t / 1e12 / (peak * world), "d2d_bytes_per_run": float(d2d[0].item()),
            "parity": {"all_tasks_retired_once": bool(okf[0].item() > 0.5),
                       "note": "values and versions of this DAG are checked against the oracle at NT=3/8 in the `cholesky` parity case"}}


DUMP_TILES = 32


def dump_outputs(path, eng, w, slab, K):
    """What the last timed step of `value` computed, as a caller of the window receives it: per-task results and flow
    versions, the tiles' final versions, and the data of DUMP_TILES tiles picked by a fixed seed (about 17 MB in all).
    The retire order, sequence stamps and worker ids depend on scheduling and are left out."""
    os.makedirs(path, exist_ok=True)
    res = w.results()
    pick = np.sort(np.random.default_rng(0).choice(K, size=min(K, DUMP_TILES), replace=False))
    data = np.empty((len(pick), TILE // 4), np.int32)
    for row, k in zip(data, pick):                                # slab position k holds tile k of the collection
        eng.d2h(row, slab + int(k) * TILE)
    for name, a in (("task_result", res["result"]), ("task_seen_version", res["seen_version"]),
                    ("tile_version", res["tiles"]["version"]), ("tile_sample_index", pick), ("tile_sample_data", data)):
        np.save(os.path.join(path, name + ".npy"), a.astype(np.float64))


# ------------------------------------------------------------------------------------------------------------------------
def main():
    ap = argparse.ArgumentParser()
    ap.add_argument("--gpus", type=int, default=1)
    ap.add_argument("--steps", type=int, default=200)
    ap.add_argument("--warmup", type=int, default=3)
    ap.add_argument("--impl", default="ours", choices=["ours", "reference"])
    ap.add_argument("--groups", type=int, default=K_GROUPS, help="broadcast groups per GPU (config value: 4096)")
    ap.add_argument("--e2e-steps", type=int, default=10, help="timed passes of the e2e run (the host side shares the box: more passes, steadier mean)")
    ap.add_argument("--e2e-cores", type=int, default=32, help="worker threads of the reference runtime in the e2e run")
    ap.add_argument("--no-secondary", action="store_true", help="skip the secondary records of the other BASELINE configs")
    ap.add_argument("--kp", type=int, default=1, help="N>1: k-cyclic factor of the 1xN collection (1: the map of examples/Ex05_Broadcast)")
    ap.add_argument("--mgpu", default="direct", choices=["direct", "exchange"],
                    help="N>1: device-released cross-GPU edges (default) or two windows + one NCCL exchange")
    ap.add_argument("--dump-outputs", metavar="DIR",
                    help="after the timed steps, write what the last one computed to DIR/<name>.npy (one GPU only)")
    args = ap.parse_args()
    if args.dump_outputs and (args.impl != "ours" or int(os.environ.get("WORLD_SIZE", "1")) > 1):
        ap.error("--dump-outputs needs --impl ours on one GPU")
    args.warmup = max(args.warmup, 3)

    rank = int(os.environ.get("RANK", "0"))
    world = int(os.environ.get("WORLD_SIZE", "1"))
    local_rank = int(os.environ.get("LOCAL_RANK", "0"))
    K = args.groups
    ntasks = K * (1 + F)
    algo_bytes = K * (1 + F) * TILE
    cfg = {"workload": "Ex05_Broadcast dataflow (BASELINE configs[1]), 256x256 fp32 tiles, K=%d groups/GPU, fan-out %d" % (K, F),
           "tile_bytes": TILE, "groups_per_gpu": K, "tasks_per_gpu_step": ntasks, "distribution": "two_dim_block_cyclic 1x%d, kp = 1 (tile k on rank k mod N: the map of mydata in examples/Ex05_Broadcast)" % world,
           "l2": "inputs larger than L2: %.2f GiB of tiles per GPU vs 126 MB L2, FIFO ready order" % (K * TILE / 2 ** 30),
           "value_path": "device-resident: the window the host runtime builds for the pool, run by the raw engine (tiles VALID in HBM); the device module's LRU stage-in is inside e2e"}

    if args.impl == "reference":
        if rank != 0:
            return
        # capped so that the arm ends within minutes whatever --steps says: a step is the FULL workload of the N-GPU arm
        # (K groups per GPU x N) on all host cores
        steps = min(args.steps, max(3, 20 // max(args.gpus, 1)))
        Kref = K * max(args.gpus, 1)
        cfg["reference_workload"] = "%d groups (%d tasks) per step: the whole job of the %d-GPU arm" % (Kref, Kref * (1 + F), max(args.gpus, 1))
        r = cpu_baseline_arm(Kref, steps, args.warmup)
        print(json.dumps({"impl": "reference", "metric": "tasks/s", "value": r["value"], "unit": "tasks/s", "n_gpus": args.gpus,
                          "steps": r["steps"], "warmup": args.warmup, "ms_per_step": r["ms_per_step"], "higher_is_better": True,
                          "scaling": "weak", "vs_baseline": None, "dtype": "i32", "data": "synthetic", "config": cfg,
                          "cpu_baseline": {"value": r["value"], "unit": "tasks/s", "cores": r["cores"], "kind": r["kind"], "sample": r["sample"]},
                          "e2e": {"value": r["value"], "unit": "tasks/s", "h2d_bytes_per_step": 0, "d2h_bytes_per_step": 0},
                          "tile_gbs": r["value"] * TILE / 1e9}))
        return

    import torch
    import torch.distributed as dist
    from parsec_b200 import _lib as L
    from parsec_b200 import runtime as R
    from parsec_b200.multigpu import ex05_multi_gpu_step_factory, ex05_direct_step_factory, work_stream

    if not torch.cuda.is_available():
        raise SystemExit("bench.py: no CUDA device; parsec_b200 has no CPU fallback")
    torch.cuda.set_device(local_rank)
    if world > 1:
        import datetime
        dist.init_process_group("nccl", device_id=torch.device("cuda", local_rank), timeout=datetime.timedelta(seconds=180))

    def barrier():
        if world > 1:
            dist.barrier()
        torch.cuda.synchronize()

    def max_over_ranks(x):
        if world == 1:
            return x
        t = torch.tensor([x], dtype=torch.float64, device="cuda")
        dist.all_reduce(t, op=dist.ReduceOp.MAX)
        return float(t.item())

    # ---------------------------------------------------------------- e2e through the reference-facing plug-in (rank 0)
    # One process drives all N GPUs, the way the reference does: same path at every N.  At N = 1 it runs first, before this
    # process takes its own device memory; at N > 1 it runs LAST, after the process group is gone, so that no rank ever sits
    # in a collective while rank 0 drives a separate application (an NCCL watchdog would kill the whole job).
    def run_e2e():
        try:
            return e2e_mca(K * world, world, args.e2e_steps, args.e2e_cores)
        except Exception as exc:
            print("bench.py: e2e through the MCA component failed: %r" % (exc,), file=sys.stderr)
            return {"unavailable": "e2e run through the MCA component failed: %r" % (exc,)}

    e2e = None
    if rank == 0 and world == 1 and args.e2e_steps > 0:     # --e2e-steps 0: profiler runs (a persistent kernel fed by the host cannot run under ncu's serialised launches)
        e2e = run_e2e()
    barrier()

    secondary = {}
    if world > 1 and not args.no_secondary:
        secondary["multi_gpu_parity"] = secondary_multi_gpu_parity(rank, world, local_rank, torch, dist)
        if world == 4:
            secondary["config3_rtt"] = secondary_rtt(rank, world, local_rank, torch, dist)
        if world == 8:
            secondary["config4_cholesky"] = secondary_cholesky(rank, world, local_rank, torch, dist)
        barrier()

    host = np.zeros(K * TILE // 4, np.int32)
    ctx = R.Context(nb_cores=os.cpu_count() or 1, cuda_devices=(local_rank,))
    dev = ctx.devices[0]
    dc = ctx.block_cyclic(4, TILE // 4, 1, K * TILE // 4, 1, mat=host)
    assert ctx.l.pb2_dc_register_memory(dc, dev) == 0            # twoDBC_memory_register: pin the collection once

    # ---------------------------------------------------------------- e2e through this repository's own host runtime
    e2e_standalone = None
    if world == 1 and args.e2e_steps > 0:
        tsplit = {"new": 0.0, "wait": 0.0, "read": 0.0}

        def e2e_step():
            t0 = time.perf_counter()
            assert ctx.l.pb2_dc_host_write_all(dc) == 0
            tp = C.c_void_p(ctx.l.pb2_ptg_ex05_broadcast_new(ctx.h, dc, K, NB))
            t1 = time.perf_counter()
            ctx.wait()
            t2 = time.perf_counter()
            info = ctx.task_info(tp)
            recv = info["class_id"] == 1
            ok = bool(np.all(info["result"][recv] == info["locals"][recv, 0].astype(np.uint64)))   # observed k, 0 mismatches
            ctx.l.pb2_taskpool_free(tp)
            t3 = time.perf_counter()
            tsplit["new"] += t1 - t0; tsplit["wait"] += t2 - t1; tsplit["read"] += t3 - t2
            return ok

        for _ in range(2):
            assert e2e_step()
        for k in tsplit: tsplit[k] = 0.0
        h2d0 = ctx.stats(dev)["data_in_from_device"][0]
        barrier()
        t0 = time.perf_counter()
        for _ in range(args.e2e_steps):
            assert e2e_step()
        torch.cuda.synchronize()
        e2e_s = (time.perf_counter() - t0) / args.e2e_steps
        h2d_tiles = (ctx.stats(dev)["data_in_from_device"][0] - h2d0) // args.e2e_steps
        assert h2d_tiles == K * TILE                                      # every tile came from host memory, once
        e2e_standalone = {"value": ntasks / e2e_s, "unit": "tasks/s", "h2d_bytes_per_step": int(h2d_tiles) + ntasks * 64 + K * F * 4 + K * 36,
                          "d2h_bytes_per_step": ntasks * (4 + 16 + 8), "ms_per_step": e2e_s * 1e3, "tile_gbs": algo_bytes / e2e_s / 1e9,
                          "ms_split": {k: v / args.e2e_steps * 1e3 for k, v in tsplit.items()},
                          "path": "this repository's C-ABI host runtime (include/pb2_parsec.h): pool built per step, windows pipelined two deep, successors released on the device"}

    # ---------------------------------------------------------------- device-resident value
    if world == 1:
        tp = C.c_void_p(ctx.l.pb2_ptg_ex05_broadcast_new(ctx.h, dc, K, NB))
        win = ctx.export_window(tp, dev)                          # the window the module builds for this pool
        assert len(win["tasks"]) == ntasks
        from parsec_b200.engine import Engine
        eng = Engine(local_rank)
        slab = eng.malloc(K * TILE)
        tiles = win["tiles"].copy()
        order = np.argsort(tiles["src_ptr"])
        tiles["dev_ptr"][order] = slab + np.arange(K, dtype=np.uint64) * np.uint64(TILE)
        tiles["state"] = L.TILE_VALID                             # inputs already resident in HBM
        w = eng.window(0, win["tasks"], win["succ"], tiles, win["ready"])
        step = lambda: w.launch()
        finish = lambda: w.wait()
        launches_per_step = 2
        nworkers = eng.info()["nworkers"]
    elif args.mgpu == "direct":
        step, finish, _, nt_rank = ex05_direct_step_factory(K, NB, TILE, rank, world, local_rank, kp=args.kp)
        if args.kp != 1:
            cfg["distribution"] = "two_dim_block_cyclic 1x%d, kp = %d" % (world, args.kp)
        launches_per_step = 2                                     # re-arm + persistent kernel (the NCCL barrier kernel is not ours)
        assert nt_rank == ntasks
        cfg["multi_gpu"] = "one window per GPU; cross-GPU edges released by the producer's CTA (system-scope atomics over NVLink), tiles pulled by the consumers in 64 KiB slices (TMA bulk copies); NCCL only as the per-step barrier"
    else:
        step, finish, launches_per_step = ex05_multi_gpu_step_factory(ctx, dev, dc, K, NB, TILE, rank, world, local_rank)
        cfg["multi_gpu"] = "two windows per GPU + one batched NCCL send/recv of the frontier"

    sampler = ClockSampler(local_rank)
    if rank == 0:
        sampler.start()                                           # nvidia-smi needs ~100 ms before its first sample
    for _ in range(args.warmup):
        step()
    finish()
    t_wait = time.perf_counter()
    while True:                                                   # keep the GPUs under load until the sampler reports
        go = 1.0 if (rank == 0 and not sampler.rows and time.perf_counter() - t_wait < 2.0) else 0.0
        if world > 1:                                             # every rank takes the same number of steps
            flag = torch.tensor([go], dtype=torch.float64, device="cuda")
            dist.broadcast(flag, src=0)
            go = float(flag.item())
        if go == 0.0:
            break
        step(); finish()
    barrier()
    if rank == 0:
        sampler.rows.clear()                                      # keep only samples of the timed region
    ev0, ev1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
    kernel_ms = 0.0
    d2d_bytes = 0
    ev0.record()
    for _ in range(args.steps):
        step()
        if world == 1:
            kernel_ms += w.wait()["kernel_ms"] + w.stats["reset_ms"]
    ev1.record()
    run = finish()
    torch.cuda.synchronize()
    barrier()
    clocks = sampler.stop() if rank == 0 else None
    if world == 1:
        # the engine runs on its own stream: the CUDA events recorded there by the library are the device time
        dev_ms = kernel_ms
        st = w.stats
        assert st["body_errors"] == 0 and st["tasks_retired"] == ntasks
        only_kernel_ms = st["kernel_ms"]
        if args.dump_outputs:
            dump_outputs(args.dump_outputs, eng, w, slab, K)
    else:
        dev_ms = ev0.elapsed_time(ev1)                             # engine work is enqueued on torch's current stream
        try:
            d2d_bytes = int(run.w.stats["bytes_d2d"])
        except Exception:
            d2d_bytes = 0
    ms_per_step = max_over_ranks(dev_ms / args.steps)
    value = world * ntasks / (ms_per_step / 1e3)

    out = {"metric": "tasks/s", "value": value, "unit": "tasks/s", "n_gpus": world, "steps": args.steps, "warmup": args.warmup,
           "ms_per_step": ms_per_step, "higher_is_better": True, "scaling": "weak", "vs_baseline": None, "dtype": "i32",
           "data": "synthetic", "config": cfg, "tile_gbs": world * algo_bytes / (ms_per_step / 1e3) / 1e9,
           "gpu_launches": launches_per_step * args.steps, "clocks": clocks,
           "engine": {"hbm_worker": "64 threads x 12 per SM (80 registers, no spills), 16 x 16-byte loads per thread in flight in read-only bodies, TMA bulk tile mover", "gemm_worker": "CTA pair, cta_group::2, fused k-chains"}}
    if world == 1:
        peak, how = measured("hbm_gbs", 6650.0)
        ach = algo_bytes / (only_kernel_ms / 1e3) / 1e9
        traffic, l2_peak = None, None
        for name in ("r02_ex05_traffic.json", "r01_ex05_traffic.json"):      # from the committed ncu --set full capture
            tpath = os.path.join(ROOT, "profiles", name)
            if os.path.exists(tpath):
                tj = json.load(open(tpath))
                traffic = tj.get("dram_bytes_per_launch")
                l2_peak = tj.get("l2_read_gbs_measured")
                break
        out["roofline"] = {"bound": "hbm", "achieved": ach, "peak": peak, "unit": "GB/s", "frac": ach / peak, "traffic": traffic,
                           "kernel": "pb2_engine_hbm_kernel", "kernel_ms": only_kernel_ms, "algorithmic_bytes": algo_bytes,
                           "peak_source": how, "workers": nworkers,
                           "dram_frac": (traffic / (only_kernel_ms / 1e3) / 1e9 / peak) if traffic else None,
                           "l2_frac": (ach / l2_peak) if l2_peak else None, "l2_peak": l2_peak,
                           "note": "frac is ALGORITHMIC bytes (K*(1+F)*262144) over the HBM copy peak and exceeds 1 because 7 of 8 reads of a tile hit the 126 MB L2; dram_frac is the ncu-measured DRAM traffic of the same launch over the same peak; l2_frac is the algorithmic rate over the L2 read rate tools/l2_probe measured on this GPU type"}
        base = cpu_baseline_arm(K, 3, 1)
        out["cpu_baseline"] = {"value": base["value"], "unit": "tasks/s", "cores": base["cores"], "kind": base["kind"], "sample": base["sample"]}
        if not args.no_secondary:
            try:
                secondary["config0_chain"] = secondary_chain()
            except Exception as exc:
                secondary["config0_chain"] = {"error": repr(exc)}
            try:
                secondary["e2e_reference_cuda_component"] = secondary_reference_cuda(K, args.e2e_cores)
            except Exception as exc:
                secondary["e2e_reference_cuda_component"] = {"error": repr(exc)}
            try:
                w.close(); eng.free(slab)
                secondary["config2_gemm"] = secondary_gemm(local_rank)
            except Exception as exc:
                secondary["config2_gemm"] = {"error": repr(exc)}
    else:
        if not args.no_secondary and args.mgpu == "direct":
            # the same DAG on a collection with k-cyclic factor 64 (64 consecutive tiles per rank and cycle): one receiver
            # in nine is remote and a rank pulls 0.22 GiB per step instead of 1 GiB (N=4) / 3 GiB (N=8)
            try:
                step2, finish2, _, nt2 = ex05_direct_step_factory(K, NB, TILE, rank, world, local_rank, kp=64)
                for _ in range(args.warmup):
                    step2()
                finish2(); barrier()
                f0, f1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                f0.record()
                for _ in range(args.steps):
                    step2()
                f1.record()
                run2 = finish2(); torch.cuda.synchronize(); barrier()
                ms2 = max_over_ranks(f0.elapsed_time(f1) / args.steps)
                pulled = torch.tensor([float(run2.w.stats["bytes_d2d"])], dtype=torch.float64, device="cuda")
                dist.all_reduce(pulled, op=dist.ReduceOp.MAX)
                secondary["ex05_kcyclic64"] = {"config": "the Ex05 dataflow of `value` on a 1x%d two_dim_block_cyclic collection with k-cyclic factor kp = 64 (two_dim_rectangle_cyclic.h), K=%d groups/GPU" % (world, K),
                                               "ms_per_step": ms2, "tasks_per_s": world * nt2 / (ms2 / 1e3), "tasks_per_gpu_step": nt2,
                                               "peer_bytes_per_rank_step": float(pulled.item()), "body_errors": 0,
                                               "weak_scaling_vs_value_at_this_N": (world * nt2 / (ms2 / 1e3)) / value}
                del run2, step2, finish2
            except Exception as exc:
                secondary["ex05_kcyclic64"] = {"error": repr(exc)}
        # NVLink view of the step: bytes every rank pulled from its peers, against the per-direction link rate
        tot = torch.tensor([float(d2d_bytes)], dtype=torch.float64, device="cuda")
        dist.all_reduce(tot, op=dist.ReduceOp.MAX)
        ingress = float(tot.item())
        out["roofline"] = {"bound": "nvlink", "achieved": ingress / (ms_per_step / 1e3) / 1e9, "peak": NVLINK_GBS, "unit": "GB/s",
                           "frac": ingress / (ms_per_step / 1e3) / 1e9 / NVLINK_GBS, "traffic": ingress,
                           "frac_of_nominal_900": ingress / (ms_per_step / 1e3) / 1e9 / NVLINK_NOMINAL_GBS,
                           "note": "bytes the busiest rank pulls from its peers per step (counted by the kernel) over the measured peer-copy rate of 770 GB/s per direction (B200_PROFILING.md; 900 nominal); the step cannot be shorter than traffic / peak"}
    if e2e_standalone is not None:
        out["e2e_standalone"] = e2e_standalone
    if secondary:
        out["secondary"] = secondary
    if world > 1:
        barrier()
        dist.destroy_process_group()
        if rank == 0 and args.e2e_steps > 0:
            try:                                             # this process' own slabs go first
                del run, step, finish
                import gc; gc.collect(); torch.cuda.empty_cache()
            except Exception:
                pass
            time.sleep(1.0)                                  # the other ranks are exiting: their device memory comes back
            e2e = run_e2e()
    out["e2e"] = e2e if e2e is not None else (e2e_standalone or {"unavailable": "oracle/_ref/bin/ex05_b200 missing or e2e skipped"})
    if rank == 0:
        print(json.dumps(out))


if __name__ == "__main__":
    main()
