"""Pins the CPU oracle (oracle/) against the reference: known answers of the reference's own tests and
examples, and the answers of the reference's own compiled code (zone_malloc.c, data.c, two_dim_rectangle_cyclic.c,
device.c) to the inputs below, stored in tests/golden/reference_builds.npz by tests/golden/make_reference_builds.py.
Where oracle/Makefile.ref has built those reference sources into oracle/_ref, the build must still give the stored
answers.  No GPU needed."""
import ctypes as C
import os
import random

import numpy as np
import pytest

from oracle import orc, orc_dags as dags

HAVE_REF_ZONE = os.path.exists(orc.REF_ZONE_PATH)
HAVE_REF_DATA = os.path.exists(orc.REF_DATA_PATH)
HAVE_REF_TWODBC = os.path.exists(orc.REF_TWODBC_PATH)
HAVE_REF_SELECT = os.path.exists(orc.REF_SELECT_PATH)
GOLDEN_REF = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_builds.npz")


def reference_answers(name, have_build, answers):
    """The stored answers of the reference build for one test; `answers()` recomputes them from the build."""
    want = np.load(GOLDEN_REF)[name]
    if have_build:
        assert np.array_equal(answers(), want), f"the reference build no longer gives the answers stored for {name}"
    return want


def tiles_for(dag, valid=False):
    t = np.zeros(dag.ntiles, orc.TILE_DTYPE)
    t["bytes"] = dag.tile_bytes
    t["src_ptr"] = np.arange(dag.ntiles, dtype=np.uint64) * np.uint64(dag.tile_bytes)   # offsets into host
    t["state"] = orc.TILE_VALID if valid else orc.TILE_INVALID
    return t


# ------------------------------------------------------------------ DAG execution known answers
@pytest.mark.parametrize("NB", [0, 1, 10, 999])
def test_ex02_chain_known_answer(NB):
    """Ex02_Chain.jdf:44-50: 'I am element k in the chain' -- task k observes k, final value NB (config 1)."""
    dag = dags.ex02_chain(NB)
    out = orc.run_window(dag.tasks, dag.succ, tiles_for(dag), dag.ready, np.zeros(1, np.int32))
    assert out["rc"] == 0 and out["stats"]["tasks_retired"] == NB + 1
    assert np.array_equal(out["retire_order"], np.arange(NB + 1))
    assert np.array_equal(out["seen_version"][:, 0], np.arange(NB + 1))
    assert out["device"][0].view(np.int32)[0] == NB
    assert out["stats"]["bytes_h2d"] == 0                  # NEW data is never pulled in (device_gpu.c:2049)


@pytest.mark.parametrize("K,NB", [(1, 0), (4, 6), (37, 14)])
def test_ex05_broadcast_known_answer(K, NB):
    """Ex05_Broadcast.jdf:33-39,53-57: every TaskRecv(k, n) prints k."""
    dag = dags.ex05_broadcast(K, NB, 64)
    host = np.full(K * 16, -1, np.int32)
    out = orc.run_window(dag.tasks, dag.succ, tiles_for(dag), dag.ready, host)
    F = NB // 2 + 1
    assert out["rc"] == 0 and out["stats"]["body_errors"] == 0
    assert np.array_equal(out["result"][K:] & np.uint64(0xFFFFFFFF), np.repeat(np.arange(K), F).astype(np.uint64))
    assert out["stats"]["bytes_h2d"] == K * 64 and out["stats"]["stage_ins"] == K


@pytest.mark.parametrize("NB_TOKEN", [1, 3, 16])
def test_ptg_pingpong_known_answer(NB_TOKEN):
    """ptg_pingpong.jdf:144-149: after INIT(i) + CPU(+i) + GPU(+i) every element is 3*i."""
    dag = dags.ptg_pingpong(NB_TOKEN)
    host = np.zeros(2 * NB_TOKEN, np.int32)
    out = orc.run_window(dag.tasks, dag.succ, tiles_for(dag), dag.ready, host)
    assert out["rc"] == 0
    assert np.array_equal(host, 3 * np.arange(2 * NB_TOKEN))


def test_dtd_new_tile_known_answer():
    """dtd_test_new_tile_cuda_kernels.cu:17,30,47-49: init i, times two => 2*i, and the accumulated sum."""
    dag = dags.dtd_new_tile(5, 100)
    out = orc.run_window(dag.tasks, dag.succ, tiles_for(dag), dag.ready, np.zeros(500, np.int32))
    assert out["rc"] == 0
    for d in out["device"]:
        assert np.array_equal(d.view(np.int32), 2 * np.arange(100))
    assert sum(int(d.view(np.int32).sum()) for d in out["device"]) == 5 * 2 * (99 * 100 // 2)


def test_rtt_chain_known_answer():
    """rtt.jdf:26-47 with body T += 1: after NT hops T == T0 + NT; the last hop writes back to A(f, k%WS)."""
    dag = dags.rtt_chain(17, 3, 64)
    host = np.arange(48, dtype=np.float32)
    expect = host + 17
    out = orc.run_window(dag.tasks, dag.succ, tiles_for(dag), dag.ready, host)
    assert out["rc"] == 0 and np.array_equal(host, expect)
    assert np.all(out["tiles"]["version"] == 17)


def test_deadlock_is_reported():
    dag = dags.ex02_chain(4)
    dag.tasks["dep_goal"][2] = 0x3
    out = orc.run_window(dag.tasks, dag.succ, tiles_for(dag), dag.ready, np.zeros(1, np.int32))
    assert out["rc"] == -1 and out["stats"]["tasks_retired"] == 2


def test_gemm_body_matches_numpy():
    from parsec_b200.bf16 import bf16_bits_to_f32, f32_to_bf16_bits, round_to_bf16
    rng = np.random.default_rng(3)
    T, NT = 32, 2
    A, B, Cm = (round_to_bf16(rng.uniform(-.5, .5, (NT, NT, T, T)).astype(np.float32)) for _ in range(3))
    dag = dags.dtd_gemm(NT, T)
    host = np.concatenate([f32_to_bf16_bits(x).ravel() for x in (A, B, Cm)])
    out = orc.run_window(dag.tasks, dag.succ, tiles_for(dag), dag.ready, host)
    assert out["rc"] == 0
    got = bf16_bits_to_f32(host[2 * NT * NT * T * T:]).reshape(NT, NT, T, T)
    for i in range(NT):
        for j in range(NT):
            c = Cm[i, j].copy()
            for k in range(NT):
                c = round_to_bf16(c + A[i, k] @ B[k, j].T)
            assert np.allclose(got[i, j], c, rtol=2 ** -7, atol=2 ** -7)


# ------------------------------------------------------------------ DTD ordering rule
def test_dtd_rule_gemm_matches_builder():
    """The per-tile last-writer / readers rule applied to dtd_test_simple_gemm.c:675-696's insertion order
    gives exactly the C(i,j) chains of the numpy builder."""
    NT = 4
    dag = dags.dtd_gemm(NT)
    n = dag.ntasks
    nbf = np.full(n, 3, np.int32)
    ft = np.full((n, 4), -1, np.int32)
    ft[:, :3] = dag.tasks["tile"][:, :3]
    fo = np.zeros((n, 4), np.int32)
    fo[:, 0] = fo[:, 1] = orc.DTD_INPUT
    fo[:, 2] = orc.DTD_INOUT
    src, dst, fl, dep = orc.dtd_build(nbf, ft, fo, dag.ntiles)
    es, ed, ef = dag.edges()
    assert sorted(zip(src.tolist(), dst.tolist(), fl.tolist())) == sorted(zip(es.tolist(), ed.tolist(), ef.tolist()))
    assert np.array_equal(dep, dag.tasks["dep_goal"])


def test_dtd_rule_war_and_reader_runs():
    """W0 R1 R2 R3 W4 R5 on one tile: readers wait for W0 only; W4 waits for W0 and R1..R3 (WAR gate,
    insert_function.c:2102-2118); R5 waits for W4."""
    ops = [orc.DTD_INOUT, orc.DTD_INPUT, orc.DTD_INPUT, orc.DTD_INPUT, orc.DTD_INOUT, orc.DTD_INPUT]
    n = len(ops)
    ft = np.full((n, 4), -1, np.int32); ft[:, 0] = 0
    fo = np.zeros((n, 4), np.int32); fo[:, 0] = ops
    src, dst, fl, dep = orc.dtd_build(np.ones(n, np.int32), ft, fo, 1)
    edges = sorted(zip(src.tolist(), dst.tolist()))
    assert edges == [(0, 1), (0, 2), (0, 3), (0, 4), (1, 4), (2, 4), (3, 4), (4, 5)]
    assert dep.tolist() == [0, 1, 1, 1, 4, 1]


# ------------------------------------------------------------------ 2D block cyclic map
@pytest.mark.parametrize("P,Q,kp,kq,ip,jq", [(1, 1, 1, 1, 0, 0), (2, 2, 1, 1, 0, 0), (2, 4, 1, 1, 1, 3), (1, 4, 1, 1, 0, 0),
                                              (2, 3, 2, 3, 0, 0), (3, 2, 2, 2, 1, 1)])
def test_twodbc_owner_and_slots(P, Q, kp, kq, ip, jq):
    """two_dim_rectangle_cyclic.c:258-286, 351-412: every tile has exactly one owner, the owner's local slots
    are a bijection onto [0, nb_local_tiles), key = n*lmt + m round-trips (key2coords)."""
    L = orc.lib()
    mb = nb = 4
    lm, ln = 4 * 11, 4 * 7
    ds = [orc.twodbc(r, mb, nb, lm, ln, P=P, Q=Q, kp=kp, kq=kq, ip=ip, jq=jq) for r in range(P * Q)]
    total = 0
    for r, d in enumerate(ds):
        slots = set()
        for m in range(d.mt):
            for n in range(d.nt):
                owner = L.orc_twodbc_rank_of(C.byref(d), m, n)
                pos = L.orc_twodbc_position(C.byref(d), m, n)
                assert (pos >= 0) == (owner == r)
                if owner == r:
                    assert pos not in slots and 0 <= pos < d.nb_local_tiles
                    slots.add(pos)
                    assert L.orc_twodbc_tile_offset_elems(C.byref(d), m, n) == pos * mb * nb
                key = L.orc_twodbc_key(C.byref(d), m, n)
                assert key == n * d.lmt + m
                mm, nn = C.c_int(), C.c_int()
                L.orc_twodbc_key2coords(C.byref(d), key, C.byref(mm), C.byref(nn))
                assert (mm.value, nn.value) == (m, n)
        assert len(slots) == d.nb_local_tiles
        total += len(slots)
    assert total == ds[0].mt * ds[0].nt
    if kp == kq == 1 and ip == jq == 0:
        d = ds[0]
        for m in range(d.mt):
            for n in range(d.nt):
                assert L.orc_twodbc_rank_of(C.byref(d), m, n) == (m % P) * Q + (n % Q)   # SURVEY 8(e)


def _twodbc_cases():
    """Plain, k-cyclic and offset grids, full and sub-matrices, every rank: (case, pb2_matrix_block_cyclic_new args)."""
    rng = random.Random(2026)
    for case in range(60):
        P, Q = rng.choice([(1, 1), (1, 4), (2, 2), (2, 4), (3, 2), (4, 1)])
        kp, kq = rng.choice([(1, 1), (1, 1), (2, 1), (2, 3), (3, 2)])
        ip, jq = rng.randrange(P), rng.randrange(Q)
        mb, nb = rng.choice([(4, 4), (3, 5), (8, 2)])
        lm, ln = mb * rng.randrange(3, 14) + rng.randrange(mb), nb * rng.randrange(3, 12) + rng.randrange(nb)
        i, j = (0, 0) if case % 3 else (rng.randrange(lm // 2), rng.randrange(ln // 2))
        m, n = lm - i - rng.randrange(0, (lm - i) // 3 + 1), ln - j - rng.randrange(0, (ln - j) // 3 + 1)
        for rank in range(P * Q):
            yield case, (rank, mb, nb, lm, ln, i, j, m, n, P, Q, kp, kq, ip, jq)


def twodbc_reference_answers():
    """Per case: the 12 derived sizes of ref_twodbc_info, then rank_of, data_key and rank_of_key(data_key) of every
    tile (m, n) in row-major order."""
    ref = orc.ref_twodbc()
    out = []
    for _, args in _twodbc_cases():
        rd = ref.ref_twodbc_new(*args)
        info = (C.c_int64 * 12)()
        ref.ref_twodbc_info(rd, info)
        out += list(info)
        for mm in range(info[2]):
            for nn in range(info[3]):
                k = ref.ref_twodbc_key(rd, mm, nn)
                out += [ref.ref_twodbc_rank_of(rd, mm, nn), k, ref.ref_twodbc_rank_of_key(rd, k)]
        ref.ref_twodbc_free(rd)
    return np.array(out, np.int64)


def test_twodbc_oracle_and_product_equal_reference_build():
    """The reference's own two_dim_rectangle_cyclic.c vs the oracle's restatement vs the product's
    pb2_matrix_block_cyclic_new: owner, key, derived sizes."""
    from parsec_b200 import runtime as R
    want = iter(reference_answers("twodbc", HAVE_REF_TWODBC, twodbc_reference_answers).tolist())
    L = orc.lib()
    rl = R.lib()
    ctxp = C.c_void_p()
    assert rl.pb2_init(C.byref(ctxp), 1) == 0
    try:
        for case, args in _twodbc_cases():
            od = orc.twodbc(*args)
            pd = C.c_void_p(rl.pb2_matrix_block_cyclic_new(ctxp, 4, *args))
            assert pd.value
            info = tuple(next(want) for _ in range(12))
            assert (od.lmt, od.lnt, od.mt, od.nt, od.nb_elem_r, od.nb_elem_c, od.nb_local_tiles, od.bsiz, od.llm, od.lln,
                    od.rrank, od.crank) == info, (case, args)
            pinfo = (C.c_int64 * 8)()
            assert rl.pb2_dc_info(pd, pinfo) == 0
            assert tuple(pinfo)[:7] == info[:7], (case, args)
            for mm in range(od.mt):
                for nn in range(od.nt):
                    r_ref, k_ref, r_of_k_ref = next(want), next(want), next(want)
                    assert L.orc_twodbc_rank_of(C.byref(od), mm, nn) == r_ref, (case, args, mm, nn)
                    assert rl.pb2_dc_rank_of(pd, mm, nn) == r_ref, (case, args, mm, nn)
                    assert L.orc_twodbc_key(C.byref(od), mm, nn) == k_ref == rl.pb2_dc_data_key(pd, mm, nn)
                    assert r_of_k_ref == r_ref
            rl.pb2_data_collection_free(pd)
        assert next(want, None) is None
    finally:
        rl.pb2_fini(C.byref(ctxp))


def test_twodbc_rtt_placement():
    """rtt_main.c:191-198 / rtt.jdf:30: PING(k, f) lives on A(f, k % WS) of a 1 x WS grid => owner k % WS."""
    WS, FRAGS = 4, 3
    d = orc.twodbc(0, 8, 8, 8 * FRAGS, 8 * WS, P=1, Q=WS)
    for k in range(20):
        for f in range(FRAGS):
            assert orc.lib().orc_twodbc_rank_of(C.byref(d), f, k % WS) == k % WS


# ------------------------------------------------------------------ LCG generator
def test_lcg_jump_equals_stepping():
    """dtd_test_simple_gemm.c:154-172: Rnd64_jump(n, seed) is n steps of x <- A*x + C."""
    L = orc.lib()
    for seed in (1789, 1805, 1901):
        x = seed
        for n in range(0, 70):
            assert L.orc_rnd64_jump(n, seed) == x
            x = L.orc_rnd64_step(x)
        assert L.orc_rnd64_jump(12345 + 678, seed) == L.orc_rnd64_jump(678, L.orc_rnd64_jump(12345, seed))


def test_lcg_tile_is_a_window_of_the_global_matrix():
    """A tile generated at (m, n) equals the same window of the matrix generated as one tile (jump-ahead)."""
    L = orc.lib()
    M, mb = 24, 8
    full = np.zeros((M, M), np.float32, order="F")
    L.orc_lcg_tile(full.ctypes.data_as(C.c_void_p), 0, 0, M, M, M, M, 1789)
    t = np.zeros((mb, mb), np.float32, order="F")
    L.orc_lcg_tile(t.ctypes.data_as(C.c_void_p), 8, 16, mb, mb, M, mb, 1789)
    assert np.array_equal(t, full[8:16, 16:24])
    assert np.all(np.abs(full) <= 0.5)


# ------------------------------------------------------------------ device selection
def _sel(devs, access, present, pref, owner, skew=20, allow_cpu=0):
    arr = (orc.SelDev * len(devs))(*[orc.SelDev(*d) for d in devs])
    a = [np.array(x, np.int32) for x in (access, present, pref, owner)]
    return orc.lib().orc_select_best_device(arr, len(devs), len(access), *[x.ctypes.data_as(C.c_void_p) for x in a], skew, allow_cpu)


SEL_CPU, SEL_REC, SEL_CUDA = 1, 2, 4
SEL_TYPES = [SEL_CPU, SEL_REC, SEL_CUDA, SEL_CUDA, SEL_CUDA, SEL_CUDA]


def _select_cases():
    """4200 random tasks over a CPU, the recursive device and four GPUs: affinity by preferred/owner device, ETA with
    several skews, taskpool device masks, CPU incarnations with and without load_balance_allow_cpu."""
    rng = random.Random(77)
    for allow_cpu in (0, 1):
        for skew in (20, 0, 50):
            for case in range(700):
                loads = [rng.choice([0, 0, rng.randrange(0, 5000)]) for _ in SEL_TYPES]
                ests = [rng.randrange(1, 400) for _ in SEL_TYPES]
                nb = rng.randrange(1, 5)
                access = [rng.choice([0x04, 0x08, 0x0C]) for _ in range(nb)]
                present = [rng.choice([1, 1, 1, 0]) for _ in range(nb)]
                pref = [rng.choice([-1, -1, -1, 0, 2, 3, 4, 5]) for _ in range(nb)]
                owner = [rng.choice([-1, 0, 0, 2, 3, 4, 5]) for _ in range(nb)]
                chore = SEL_CUDA | (SEL_CPU if rng.random() < 0.4 else 0)
                mask = rng.choice([0x3f, 0x3f, 0x3d, 0x0f, 0x35, 0x31, 0x03])
                yield allow_cpu, skew, case, loads, ests, access, present, pref, owner, chore, mask


def select_reference_answers():
    """Per task: the device parsec_select_best_device picks and the load it reports."""
    ref = orc.ref_select()
    ref.ref_sel_init(20, 0)
    for t in SEL_TYPES:
        assert ref.ref_sel_add_device(t, 0, 1) >= 0
    out, mode = [], None
    for allow_cpu, skew, case, loads, ests, access, present, pref, owner, chore, mask in _select_cases():
        if mode != (skew, allow_cpu):
            mode = (skew, allow_cpu)
            ref.ref_sel_init(skew, allow_cpu)
        for d in range(len(SEL_TYPES)):
            ref.ref_sel_set_load(d, loads[d], ests[d])
        a = [np.array(x, np.int32) for x in (access, present, pref, owner)]
        load = C.c_int64()
        got = ref.ref_sel_select(len(access), *[x.ctypes.data_as(C.c_void_p) for x in a], chore, mask, C.byref(load))
        out += [got, load.value if got >= 0 else 0]
    return np.array(out, np.int64)


def test_select_oracle_equals_reference_build():
    """The reference's own parsec_select_best_device (device.c:100-310, driven with fake device modules and tasks)
    vs the oracle."""
    want = reference_answers("select", HAVE_REF_SELECT, select_reference_answers).reshape(-1, 2)
    cases = list(_select_cases())
    assert len(cases) == len(want)
    for (allow_cpu, skew, case, loads, ests, access, present, pref, owner, chore, mask), (got, load) in zip(cases, want.tolist()):
        devs = [(1 if SEL_TYPES[d] == SEL_CUDA else 0, 1 if SEL_TYPES[d] == SEL_REC else 0,
                 1 if ((mask >> d) & 1) and (SEL_TYPES[d] & chore) else 0, loads[d], ests[d]) for d in range(len(SEL_TYPES))]
        assert _sel(devs, access, present, pref, owner, skew, allow_cpu) == got, \
            (case, allow_cpu, skew, devs, access, present, pref, owner, chore, hex(mask))
        if got >= 0:
            assert load == ests[got]


def test_select_best_device_rules():
    # devices: 0 cpu, 1 recursive, 2..5 gpus; (is_gpu, is_recursive, enabled, load, estimate)
    devs = [(0, 0, 1, 0, 10), (0, 1, 1, 0, 10), (1, 0, 1, 0, 10), (1, 0, 1, 0, 10), (1, 0, 1, 0, 10), (1, 0, 1, 0, 10)]
    RW, R = 0x0C, 0x04
    # get_best_device_check.jdf:68-83: preferred_device of the written tile decides: gpu (n*nt+m) % ngpu
    nt, ngpu = 5, 4
    for m in range(nt):
        for n in range(nt):
            g = 2 + (n * nt + m) % ngpu
            assert _sel(devs, [RW], [1], [g], [0]) == g
    assert _sel(devs, [RW, R], [1, 1], [-1, -1], [3, 4]) == 3           # written data already on gpu 3
    assert _sel(devs, [R, RW], [1, 1], [-1, -1], [4, 0]) == 4           # read data on gpu 4 -> rdata_dev, idle
    assert _sel(devs, [R], [1], [-1], [0]) == 5                          # no affinity: least ETA, highest index first
    loaded = [list(d) for d in devs]
    loaded[4][3] = 100                                                   # gpu 4 busy: (100+10)/1.2 > 10 => move
    assert _sel(loaded, [R], [1], [-1], [4]) == 5
    loaded[4][3] = 1                                                     # (1+10)/1.2 < 10 => stay (20 % skew)
    assert _sel(loaded, [R], [1], [-1], [4]) == 4
    only_cpu = [(0, 0, 1, 0, 10)] + [(1, 0, 0, 0, 10)] * 3
    assert _sel(only_cpu, [R], [1], [-1], [0]) == 0
    assert _sel([(0, 0, 0, 0, 1)], [R], [1], [-1], [0]) == -1


# ------------------------------------------------------------------ zone allocator
def _zone_scenario(zm, zf):
    """tests/runtime/cuda/zonemalloc.c:32-80 (128 segments of 512 B)."""
    N = 128
    seg = [zm(512) for _ in range(N)]
    assert all(s is not None for s in seg) and sorted(seg) == list(range(N))
    assert zm(512) is None
    for s in seg: zf(s)
    seg = [zm(512) for _ in range(N)]
    assert all(s is not None for s in seg)
    for i in range(0, N, 2): zf(seg[i])
    for i in range(1, N, 2): zf(seg[i])
    seg = [zm(512 // ((i % 2) + 1)) for i in range(N)]
    assert all(s is not None for s in seg)
    for i in range(N - 1, 0, -1): zf(seg[i])
    return seg[0]


def test_zone_reference_scenario():
    L = orc.lib()
    z = L.orc_zone_init(128, 512)
    def zm(sz):
        r = L.orc_zone_malloc(z, sz)
        return None if r < 0 else r
    first = _zone_scenario(zm, lambda s: L.orc_zone_free(z, s))
    assert L.orc_zone_in_use(z) == 512
    assert L.orc_zone_free(z, first) == 0 and L.orc_zone_free(z, first) == -2    # double free is reported
    nfree, largest = C.c_int(), C.c_int()
    L.orc_zone_free_profile(z, C.byref(nfree), C.byref(largest))
    assert (nfree.value, largest.value) == (1, 128)                              # fully coalesced again
    assert L.orc_zone_malloc(z, 0) == -1
    L.orc_zone_fini(z)


ZONE_SEEDS, ZONE_OPS, ZONE_NSEG, ZONE_UNIT = 25, 1500, 96, 512


def _zone_run(seed, malloc, free, in_use):
    """One random malloc/free sequence over ZONE_NSEG segments of ZONE_UNIT bytes.  Per operation: the first segment
    malloc returned (-1: none; -2: the operation was a free), then the bytes in use."""
    rnd = random.Random(seed)
    live, out = [], []
    for _ in range(ZONE_OPS):
        if live and rnd.random() < 0.45:
            free(live.pop(rnd.randrange(len(live))))
            out.append(-2)
        else:
            seg = malloc(rnd.choice([1, 256, 512, 513, 1024, 2000, 4096, 8192]))
            if seg >= 0:
                live.append(seg)
            out.append(seg)
        out.append(in_use())
    return out


def zone_reference_answers():
    ref = C.CDLL(orc.REF_ZONE_PATH)
    ref.zone_malloc_init.restype = C.c_void_p; ref.zone_malloc_init.argtypes = [C.c_void_p, C.c_int, C.c_size_t]
    ref.zone_malloc.restype = C.c_void_p; ref.zone_malloc.argtypes = [C.c_void_p, C.c_size_t]
    ref.zone_free.argtypes = [C.c_void_p, C.c_void_p]
    ref.zone_in_use.restype = C.c_size_t; ref.zone_in_use.argtypes = [C.c_void_p]
    buf = (C.c_char * (ZONE_NSEG * ZONE_UNIT))()
    base = C.addressof(buf)
    out = []
    for seed in range(ZONE_SEEDS):
        zr = ref.zone_malloc_init(base, ZONE_NSEG, ZONE_UNIT)
        malloc = lambda size: (lambda p: -1 if not p else (p - base) // ZONE_UNIT)(ref.zone_malloc(zr, size))
        out += _zone_run(seed, malloc, lambda seg: ref.zone_free(zr, base + seg * ZONE_UNIT), lambda: ref.zone_in_use(zr))
    return np.array(out, np.int64)


def test_zone_oracle_equals_reference_build():
    """Same malloc/free sequences through the reference's own parsec/utils/zone_malloc.c and through the restatement:
    identical addresses and in-use bytes at every step."""
    want = reference_answers("zone", HAVE_REF_ZONE, zone_reference_answers).reshape(ZONE_SEEDS, ZONE_OPS, 2)
    L = orc.lib()
    for seed in range(ZONE_SEEDS):
        zo = L.orc_zone_init(ZONE_NSEG, ZONE_UNIT)

        def free(seg):
            assert L.orc_zone_free(zo, seg) == 0
        got = np.array(_zone_run(seed, lambda size: L.orc_zone_malloc(zo, size), free, lambda: L.orc_zone_in_use(zo))).reshape(-1, 2)
        L.orc_zone_fini(zo)
        bad = np.flatnonzero((got != want[seed]).any(axis=1))
        assert not len(bad), (seed, int(bad[0]), got[bad[0]].tolist(), want[seed][bad[0]].tolist())


# ------------------------------------------------------------------ coherency protocol
COH_SEEDS, COH_STEPS, COH_NDEV = 200, 12, 6


def _coherency_run(seed, add_copy, get, owner, start, end, set_version):
    """Random start/end_transfer_ownership sequences on one datum over COH_NDEV devices.  `get(dev)` returns
    (present, coherency state, readers, version).  One row per access: seed, step, the device start returned, the
    owner, then the four fields of every copy (zeros for an absent one)."""
    R, W = 0x04, 0x08
    rnd = random.Random(seed)
    rows = []
    for step in range(COH_STEPS):
        dev = rnd.randrange(2, COH_NDEV)
        acc = rnd.choice([R, W, R | W, R, R | W])
        if not get(dev)[0]:
            add_copy(dev)
        # a sane program never has two owners: skip accesses the reference asserts against
        if get(dev)[1] == 0x1 and owner() != dev:
            continue
        r = start(dev, acc)
        end(dev, acc)
        if acc & W:   # what stage_in does next: the written replica gets a newer version
            set_version(dev, get(r if r >= 0 else dev)[3] + 1)
        elif r >= 0:
            set_version(dev, get(r)[3])
        row = [seed, step, r, owner()]
        for d in range(COH_NDEV):
            c = get(d)
            row += list(c) if c[0] else [0, 0, 0, 0]
        rows.append(row)
    return rows


def coherency_reference_answers():
    ref = C.CDLL(orc.REF_DATA_PATH)
    ref.ref_data_new.restype = C.c_void_p
    for fn in (ref.ref_data_add_copy, ref.ref_data_set, ref.ref_data_get, ref.ref_data_owner, ref.ref_start_transfer,
               ref.ref_end_transfer, ref.ref_data_set_owner):
        fn.argtypes = None
    assert ref.ref_data_setup(COH_NDEV) == 0
    rows = []
    for seed in range(COH_SEEDS):
        rd = C.c_void_p(ref.ref_data_new())

        def get_all(dev):
            out = (C.c_int * 5)()            # present, coherency, status, readers, version
            ref.ref_data_get(rd, dev, out)
            return list(out)

        def set_version(dev, v):
            _, coh, status, readers, _ = get_all(dev)
            ref.ref_data_set(rd, dev, coh, status, v, readers)
        rows += _coherency_run(seed, lambda dev: ref.ref_data_add_copy(rd, dev), lambda dev: [get_all(dev)[i] for i in (0, 1, 3, 4)],
                               lambda: ref.ref_data_owner(rd), lambda dev, acc: ref.ref_start_transfer(rd, dev, acc),
                               lambda dev, acc: ref.ref_end_transfer(rd, dev, acc), set_version)
    return np.array(rows, np.int64)


def test_coherency_oracle_equals_reference_build():
    """Random start/end_transfer_ownership sequences through the reference's own parsec/data.c and the restatement
    leave identical host-visible state and return values."""
    want = reference_answers("coherency", HAVE_REF_DATA, coherency_reference_answers)
    L = orc.lib()
    rows = []
    for seed in range(COH_SEEDS):
        od = orc.OrcData()
        L.orc_data_create(C.byref(od), COH_NDEV, 0)

        def add_copy(dev):
            od.copy[dev].present = 1

        def set_version(dev, v):
            od.copy[dev].version = v
        rows += _coherency_run(seed, add_copy,
                               lambda dev: [od.copy[dev].present, od.copy[dev].coherency_state, od.copy[dev].readers, od.copy[dev].version],
                               lambda: od.owner_device, lambda dev, acc: L.orc_data_start_transfer_ownership(C.byref(od), dev, acc),
                               lambda dev, acc: L.orc_data_end_transfer_ownership(C.byref(od), dev, acc), set_version)
    got = np.array(rows, np.int64)
    assert got.shape == want.shape
    bad = np.flatnonzero((got != want).any(axis=1))
    assert not len(bad), ("seed, step, start, owner, then per copy: present, state, readers, version",
                          got[bad[0]].tolist(), want[bad[0]].tolist())


def test_gpu_task_protocol_versions():
    """RW on a GPU: H2D from the host, version+1, OWNED; a second GPU reading the same version pulls D2D from the
    first (device_gpu.c:1892-2008); pushout brings the host copy to the GPU's version (device_gpu.c:3247-3255)."""
    L = orc.lib()
    R, W = 0x04, 0x08
    d = orc.OrcData()
    L.orc_data_create(C.byref(d), 4, 0)
    req = C.c_int()
    peer = 0b1100
    assert L.orc_gpu_stage_in(C.byref(d), 2, 0, R | W, peer, C.byref(req)) == 0       # H2D from the host
    assert d.copy[2].version == 1 and d.copy[2].data_transfer_status == 1
    L.orc_gpu_stage_in_complete(C.byref(d), 2, R | W)
    assert d.copy[2].coherency_state == 0x1 and d.owner_device == 2 and d.copy[0].coherency_state == 0x4
    L.orc_gpu_task_complete(C.byref(d), 2, R | W, 0)
    assert d.copy[2].readers == 0
    # successor on GPU 3 reads the GPU-2 replica (its data_in): D2D
    assert L.orc_gpu_stage_in(C.byref(d), 3, 2, R, peer, C.byref(req)) == 2
    assert d.copy[3].version == 1
    L.orc_gpu_stage_in_complete(C.byref(d), 3, R)
    assert d.copy[3].coherency_state == 0x4
    L.orc_gpu_task_complete(C.byref(d), 3, R, 0)
    # another RW on GPU 2 with pushout: already there, version 2, host follows
    assert L.orc_gpu_stage_in(C.byref(d), 2, 2, R | W, peer, C.byref(req)) == -1
    assert d.copy[2].version == 2
    L.orc_gpu_task_complete(C.byref(d), 2, R | W, 1)
    assert d.copy[0].version == 2 and d.copy[0].coherency_state == 0x4 and d.copy[2].coherency_state == 0x4
    # NEW data is never transferred
    n = orc.OrcData()
    L.orc_data_create(C.byref(n), 4, 1)
    assert L.orc_gpu_stage_in(C.byref(n), 2, 0, R | W, peer, C.byref(req)) == -1
    assert n.copy[2].version == 1 and n.copy[2].data_transfer_status == 2


# ------------------------------------------------------------------ CPU scheduler port == sequential oracle
@pytest.mark.parametrize("nthreads", [1, 4])
def test_cpu_scheduler_port_results(nthreads):
    dag = dags.ex05_broadcast(64, 14, 256)
    host = np.zeros(64 * 64, np.int32)
    t = tiles_for(dag, valid=True)
    t["dev_ptr"] = host.ctypes.data + np.arange(64, dtype=np.uint64) * np.uint64(256)
    secs, per_thread, errs = orc.cpu_sched_run(dag.tasks, dag.succ, t, dag.ready, nthreads)
    assert secs > 0 and errs == 0 and per_thread.sum() == dag.ntasks
    assert np.array_equal(host.reshape(64, 64)[:, 0], np.arange(64))
