"""The third-generation fused leaf-tile scan (zebra_b200/csrc/zb_scan3_kernel.cuh) run ON THE CPU from its own source
(tests/scan3_emu.cpp: one std::thread per CUDA thread; mbarriers, the TMA copy engine, shuffles and ballots emulated) and
compared with the oracle: every (key, ordinal) entry of every visit's top-n' list, bit for bit -- the leaf branch of
tree_result (/root/reference/src/database/index/lsh.rs:299-331) with Metric::distance of distance.rs:19-49, :103-114.

What this covers without a GPU: the ring protocol (full / empty / tile-info / query barriers: a missing wait reads stale
data because copies land late, an extra arrival aborts), the 16-lane fold over the half-warp and which thread ends up with
which row, the transposition through shared memory, list insertion with ties and tombstones, partial row blocks, partial
query tiles (QH = 1 .. 8), dim % 48 != 0 and dim % 16 != 0, and the shared per-query bound; the shared-memory layout and
the tile capacity (16, 8 or 4 queries) the launch code picks as rows grow, and the kernel body run at each capacity."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

from oracle import zb_oracle as zo

HERE = os.path.dirname(os.path.abspath(__file__))
F32 = np.float32
SENT = np.uint64(0xFFFFFFFFFFFFFFFF)


@pytest.fixture(scope="module", params=[(3, 0, 4), (3, 0, 8), (3, 1, 4), (2, 0, 4)], ids=["kc3", "kc3-8warps", "kc3-epilogue-warp", "kc2"])
def emu(tmp_path_factory, request):
    """The build variants of the kernel body: T3_KC = 3 (the default: a stage's chunks straight-line) and 2 (operands
    software-pipelined across stage boundaries); T3_EPW = 1 (a dedicated epilogue warp per team keeps the lists of n' <= 32);
    TW = 8 (eight math warps per team, 8 rows of a block each: 640 threads; what the library launches for n' > 32)."""
    kc, epw, tw = request.param
    out = str(tmp_path_factory.mktemp("s3") / f"libscan3_emu_kc{kc}_epw{epw}_tw{tw}.so")
    build_emu(out, kc, epw)
    return load_emu(out, kc, epw, tw)


def build_emu(out, kc=3, epw=0):
    subprocess.check_call(["g++", "-O1", "-std=c++20", "-ffp-contract=off", "-fno-fast-math", "-fPIC", "-shared", "-pthread",
                           f"-DT3_KC={kc}", f"-DT3_EPW={epw}", "-g", "-rdynamic", "-fvisibility=hidden", "-Wl,-Bsymbolic", "-o", out,
                           os.path.join(HERE, "scan3_emu.cpp")])


def load_emu(path, kc=3, epw=0, tw=4):
    L = C.CDLL(path)
    assert L.emu_scan3_set_team_warps(tw) == 0               # the kernel body's TW (a template parameter: both shapes are in every build)
    L.variant = (kc, epw, tw)
    L.emu_scan3.restype = C.c_int
    L.emu_scan3.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint32, C.c_uint64] + [C.c_void_p] * 7 + \
                           [C.c_uint32] + [C.c_void_p] * 12
    L.emu_scan3_layout.restype = None
    L.emu_scan3_layout.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_void_p]
    return L


# ---- shared-memory layout and the (query capacity, ring depth) the launch code picks -------------------------------------
OPTIN_B200 = 232_448          # cudaDevAttrMaxSharedMemoryPerBlockOptin of a B200 (227 KB)
LAYOUT_FIELDS = ("stage", "queries", "sums", "lists", "meta", "info", "bars", "total")


def scan3_layout(emu, nst, dim, qcap, kr):
    out = np.zeros(8, np.uint32)
    emu.emu_scan3_layout(nst, dim, qcap, kr, out.ctypes.data)
    return dict(zip(LAYOUT_FIELDS, (int(x) for x in out)))


def t3_config(emu, dim, kr, optin=OPTIN_B200):
    """zb_scan.cu t3_config over the header's t3_layout: the largest tile (16, 8, then 4 queries) that leaves at least 3 ring
    stages for two teams + 1024 B, with the deepest ring that fits; None where the fused kernel does not fit at all."""
    for qcap in (16, 8, 4):
        for nst in range(8, 2, -1):
            if 2 * scan3_layout(emu, nst, dim, qcap, kr)["total"] + 1024 <= optin:
                return qcap, nst
    return None


def canonical_sq_norm(x):
    """|x|^2 as the kernels accumulate it (16-lane order): the dot product of x with itself through the oracle."""
    return np.array([zo.dot(v, v) for v in x], dtype=F32)


def build_case(rng, dim, leaf_lens, nq, visits_per_leaf, np_max, tomb_frac, dup=True):
    dimp = (dim + 15) // 16 * 16
    P = int(sum(leaf_lens))
    rows = rng.standard_normal((P, dim)).astype(F32)
    if dup and P > 40:
        rows[P // 2:P // 2 + 10] = rows[:10]              # equal keys: order by position
    queries = rng.standard_normal((nq, dim)).astype(F32)
    if dup:
        queries[0] = rows[3]                                # distance exactly 0
    leaf_off = np.concatenate([[0], np.cumsum(leaf_lens)]).astype(np.int64)
    tomb_bits = rng.random(P) < tomb_frac
    ordv = (rng.permutation(P).astype(np.uint64) + np.uint64(1000))   # ordinal of every position (any injective map)
    # visits: for every leaf a random subset of queries, each with its own n'
    v_leaf, v_q, v_np = [], [], []
    for l, c in enumerate(visits_per_leaf):
        for q in rng.choice(nq, size=min(c, nq), replace=False):
            v_leaf.append(l); v_q.append(int(q)); v_np.append(int(rng.integers(1, np_max + 1)))
    perm = rng.permutation(len(v_leaf))                     # visits arrive in walker order, not grouped by leaf
    v_leaf = np.array(v_leaf, np.uint32)[perm]; v_q = np.array(v_q, np.uint32)[perm]; v_np = np.array(v_np, np.uint32)[perm]
    return dict(dim=dim, dimp=dimp, P=P, rows=rows, queries=queries, leaf_off=leaf_off, leaf_len=np.array(leaf_lens, np.uint32),
                tomb=tomb_bits, ord=ordv, v_leaf=v_leaf, v_q=v_q, v_np=v_np)


def run_emu(emu, case, metric, top_k, tq, qcap=16, nst=4, blocks=2, same_np=None, kr=1, l2_filter=False, info=None):
    """l2_filter: METRIC 3 of the kernel (the dot-product filter for L2 / L2 squared) followed by the exact second pass
    (t3_refine_warp); the entries must be what the exact kernel writes.  info (a dict) receives flags, candidates, stats."""
    dim, dimp, P = case["dim"], case["dimp"], case["P"]
    rows_p = np.zeros((P + 1, dimp), F32); rows_p[:P, :dim] = case["rows"]
    q_p = np.zeros((case["queries"].shape[0], dimp), F32); q_p[:, :dim] = case["queries"]
    tomb_words = np.zeros(P // 32 + 8, np.uint32)
    for p in np.nonzero(case["tomb"])[0]:
        tomb_words[p >> 5] |= np.uint32(1 << (p & 31))
    with np.errstate(divide="ignore"):
        bm_rinv = 1.0 / np.sqrt(canonical_sq_norm(case["rows"]).astype(np.float64))
        q_rinv = 1.0 / np.sqrt(canonical_sq_norm(case["queries"]).astype(np.float64))
    v_leaf, v_q = case["v_leaf"], case["v_q"]
    v_np = case["v_np"] if same_np is None else np.full_like(case["v_np"], same_np)
    nv = v_leaf.size
    live_len = np.array([int((~case["tomb"][case["leaf_off"][l]:case["leaf_off"][l + 1]]).sum()) for l in range(case["leaf_len"].size)])
    ent_len = np.minimum(live_len[v_leaf], v_np).astype(np.uint32)
    v_ent_off = np.concatenate([[0], np.cumsum(ent_len)]).astype(np.uint32)
    # group visits by leaf, cut tiles of <= tq queries (full tiles first), as ts_scatter / ts_filltiles do
    order = np.argsort(v_leaf, kind="stable").astype(np.uint32)
    tile_leaf, tile_first, tile_count = [], [], []
    pos = 0
    for l in range(case["leaf_len"].size):
        c = int((v_leaf == l).sum())
        done = 0
        while done < c:
            n = min(tq, c - done)
            tile_leaf.append(l); tile_first.append(pos + done); tile_count.append(n)
            done += n
        pos += c
    tile_leaf = np.array(tile_leaf, np.uint32); tile_first = np.array(tile_first, np.uint32); tile_count = np.array(tile_count, np.uint32)
    members = np.arange(P + 1, dtype=np.uint32)
    gthr = np.full(case["queries"].shape[0], SENT, np.uint64)
    entries = np.zeros((int(v_ent_off[-1]) + 1, 2), np.uint64)
    stats = np.zeros(8, np.uint64)
    if l2_filter:
        assert metric in (zo.L2SQ, zo.L2) and kr == 1
        chunks = dimp // 16
        with np.errstate(over="ignore", invalid="ignore"):
            bm_n2 = np.concatenate([canonical_sq_norm(case["rows"]), np.zeros(1, F32)])
            q_n2 = canonical_sq_norm(case["queries"])
        leaf_n2max = np.zeros(case["leaf_len"].size, F32)
        for l in range(case["leaf_len"].size):
            x = bm_n2[case["leaf_off"][l]:case["leaf_off"][l + 1]]
            x = x[x <= F32(1e37)]                            # NaN and inf compare false
            leaf_n2max[l] = x.max() if x.size else 0
        ecoef = F32(F32(4 * chunks + 32) * F32(2.0 ** -24) * F32(1.01))
        cand = np.full(nv * 32 + 1, 0xDEADBEEFDEADBEEF, np.uint64)
        cut = np.full(nv + 1, np.nan, F32)
        flag = np.full(nv + 1, 7, np.uint8)
        emu.emu_scan3_set_filter.restype = None
        emu.emu_scan3_set_filter.argtypes = [C.c_void_p] * 3 + [C.c_float] + [C.c_void_p] * 3
        emu.emu_scan3_set_filter(bm_n2.ctypes.data, q_n2.ctypes.data, leaf_n2max.ctypes.data, ecoef, cand.ctypes.data, cut.ctypes.data,
                                 flag.ctypes.data)
    done_tiles = emu.emu_scan3(3 if l2_filter else metric, blocks, dim, nst, qcap, kr, top_k, P, rows_p.ctypes.data, bm_rinv.ctypes.data, tomb_words.ctypes.data,
                               case["ord"].ctypes.data, members.ctypes.data, case["leaf_off"].ctypes.data, case["leaf_len"].ctypes.data,
                               tile_leaf.size, tile_leaf.ctypes.data, tile_first.ctypes.data, tile_count.ctypes.data, order.ctypes.data,
                               v_np.ctypes.data, v_q.ctypes.data, v_ent_off.ctypes.data, q_p.ctypes.data, q_rinv.ctypes.data,
                               gthr.ctypes.data, entries.ctypes.data, stats.ctypes.data)
    assert done_tiles >= tile_leaf.size
    assert int(stats[0]) == nv and int(stats[1]) == int(case["leaf_len"][v_leaf].astype(np.int64).sum())
    if l2_filter:
        assert not (entries != 0).any()                     # the first pass writes candidates, not entries
        assert set(np.unique(flag[:nv])) <= {0, 1}
        emu.emu_refine.restype = C.c_int
        emu.emu_refine.argtypes = [C.c_int, C.c_int, C.c_int] + [C.c_void_p] * 8 + [C.c_uint32] + [C.c_void_p] * 7
        pulled = emu.emu_refine(metric, 2, dim, rows_p.ctypes.data, tomb_words.ctypes.data, case["ord"].ctypes.data, members.ctypes.data,
                                case["leaf_off"].ctypes.data, case["leaf_len"].ctypes.data, q_p.ctypes.data, order.ctypes.data, nv,
                                v_leaf.ctypes.data, v_np.ctypes.data, v_q.ctypes.data, v_ent_off.ctypes.data, gthr.ctypes.data,
                                entries.ctypes.data, stats.ctypes.data)
        assert pulled >= nv
        assert int(stats[4]) == int(flag[:nv].sum())
        if info is not None:
            info.update(flag=flag[:nv].copy(), cut=cut[:nv].copy(), cand=cand[:nv * 32].reshape(nv, 32).copy(), exact_rows=int(stats[5]),
                        flagged=int(stats[4]))
    return entries, v_ent_off, v_np, gthr


def expected_visit(case, metric, v, np_v):
    l, q = int(case["v_leaf"][v]), int(case["v_q"][v])
    lo, hi = int(case["leaf_off"][l]), int(case["leaf_off"][l + 1])
    pos = np.arange(lo, hi)
    pos = pos[~case["tomb"][lo:hi]]
    if pos.size == 0:
        return np.zeros((0, 2), np.uint64)
    keys = zo.distance_bits_batch(metric, case["rows"][pos], np.broadcast_to(case["queries"][q], (pos.size, case["dim"])).copy())
    idx = np.lexsort((pos, keys))[:np_v]                    # (key, position): position order == ordinal order inside a leaf (D3)
    return np.stack([keys[idx], case["ord"][pos[idx]]], axis=1)


@pytest.mark.parametrize("metric", [zo.COSINE, zo.L2SQ, zo.L2])
@pytest.mark.parametrize("dim,tq", [(48, 16), (100, 16), (40, 7), (200, 11)])
def test_per_visit_lists_equal_oracle(emu, metric, dim, tq):
    rng = np.random.default_rng(dim * 7 + metric)
    leaf_lens = [1, 63, 64, 65, 130, 17, 200, 128, 5]
    visits = [1, 2, 5, 9, 16, 3, 21, 13, 4]                 # tiles of 1..16 queries: every QH variant, several tiles per leaf
    case = build_case(rng, dim, leaf_lens, 24, visits, np_max=32, tomb_frac=0.15)
    # top_k no visit's n' equals: the shared per-query bound is never published, every list is the exact per-visit top-n'
    entries, ent_off, v_np, _ = run_emu(emu, case, metric, top_k=0xFFFFFFFF, tq=tq)
    for v in range(case["v_leaf"].size):
        exp = expected_visit(case, metric, v, int(v_np[v]))
        got = entries[ent_off[v]:ent_off[v + 1]]
        assert got.shape[0] == exp.shape[0], v
        assert np.array_equal(got, exp), (v, int(case["v_leaf"][v]), int(case["v_q"][v]), int(v_np[v]))


def test_shared_bound_keeps_the_per_query_answer(emu):
    """All visits ask for n' = top_k, so full lists publish their k-th key and later visits of the same query drop candidates
    above it: per-visit lists may be shorter, the per-query top-k over all visits (dedup by ordinal) must not change."""
    rng = np.random.default_rng(99)
    leaf_lens = [150, 90, 200, 64, 70, 129]
    visits = [12, 12, 12, 12, 12, 12]
    case = build_case(rng, 64, leaf_lens, 12, visits, np_max=8, tomb_frac=0.1)
    k = 8
    entries, ent_off, _, gthr = run_emu(emu, case, zo.L2SQ, top_k=k, tq=16, same_np=k, blocks=3)
    assert (gthr != SENT).any()
    for q in range(12):
        got, exp = [], []
        for v in np.nonzero(case["v_q"] == q)[0]:
            e = entries[ent_off[v]:ent_off[v + 1]]
            got += [tuple(x) for x in e if x[1] != SENT]
            exp += [tuple(x) for x in expected_visit(case, zo.L2SQ, v, k)]
        got_k = sorted(set(got))[:k]
        exp_k = sorted(set(exp))[:k]
        assert got_k == exp_k, q


def test_small_query_capacity_and_deep_ring(emu):
    """qcap = 8 (long rows: the query block leaves room for 8 queries only) with a 6-stage ring, one block."""
    rng = np.random.default_rng(5)
    case = build_case(rng, 96, [70, 131, 64], 10, [8, 10, 3], np_max=20, tomb_frac=0.0)
    entries, ent_off, v_np, _ = run_emu(emu, case, zo.COSINE, top_k=0xFFFFFFFF, tq=8, qcap=8, nst=6, blocks=1)
    for v in range(case["v_leaf"].size):
        assert np.array_equal(entries[ent_off[v]:ent_off[v + 1]], expected_visit(case, zo.COSINE, v, int(v_np[v]))), v


def test_tile_config_regimes(emu):
    """Which tile shape the launch code picks as rows grow, and that every shape it can pick is a sound layout: regions in
    order without overlap, each as large as the kernel addresses it, TMA / bulk-copy destinations on 128 B, the tile info on
    16 B, mbarriers on 8 B, and two teams + 1024 B of alignment slack within the 227 KB a block may opt into."""
    picked = {}
    for kr in (1, 4):
        for dimp in range(16, 6001, 16):
            picked[kr, dimp] = cfg = t3_config(emu, dimp, kr)
            if cfg is None:
                continue
            qcap, nst = cfg
            lay = scan3_layout(emu, nst, dimp, qcap, kr)
            need = dict(stage=nst * 64 * emu.variant[0] * 16 * 4,
                        queries=(qcap * dimp + 16) * 4,              # two regions of qcap / 2 queries, the second 64 B further
                        sums=2 * qcap * 64 * 4, lists=qcap * 3 * kr * 32 * 4, meta=5 * qcap * 4,
                        info=2 * 32, bars=(2 * 8 + 8) * 8)
            names = LAYOUT_FIELDS[:-1]
            assert lay["stage"] == 0
            for a, b in zip(names, names[1:] + ("total",)):
                assert lay[b] - lay[a] >= need[a], (kr, dimp, cfg, a, lay)
            for f in ("stage", "queries", "sums", "total"):
                assert lay[f] % 128 == 0, (kr, dimp, cfg, f, lay)
            assert lay["info"] % 16 == 0 and lay["bars"] % 8 == 0, (kr, dimp, cfg, lay)
            assert 2 * lay["total"] + 1024 <= OPTIN_B200
    for kr in (1, 4):                                   # the ring only grows shallower inside a capacity
        seq = [picked[kr, d] for d in range(16, 6001, 16) if picked[kr, d]]
        assert all(a[0] > b[0] or (a[0] == b[0] and a[1] >= b[1]) for a, b in zip(seq, seq[1:])), kr
    if emu.variant[0] != 3:
        return                                                  # the regimes below are those of the 12 KB stage the library ships
    cap = lambda kr, d: picked[kr, d] and picked[kr, d][0]
    assert picked[1, 16] == (16, 8) and picked[1, 992] == (16, 3)
    assert cap(1, 992) == 16 and cap(1, 1008) == 8              # n' <= 32: 16-query tiles up to 992 floats per row
    assert cap(1, 2208) == 8 and cap(1, 2224) == 4
    assert cap(1, 4672) == 4 and picked[1, 4688] is None        # beyond: quad_tile / score_pairs
    assert cap(4, 704) == 16 and cap(4, 720) == 8               # n' <= 128
    assert cap(4, 1920) == 8 and cap(4, 1936) == 4
    assert cap(4, 4384) == 4 and picked[4, 4400] is None
    for dim, qcap, nst1, nst4 in SMALL_TILES:
        assert picked[1, dim] == (qcap, nst1) and picked[4, dim] == (qcap, nst4)


# (dim, qcap, ring depth for n' <= 32, ring depth for n' <= 128): what the launch code picks at these row lengths
SMALL_TILES = [(1040, 8, 6, 5), (2240, 4, 6, 5)]


def check_small_tiles(emu, dim, qcap, nst, kr):
    """The kernel body at a tile capacity below 16 with the ring depth picked for that row length: tiles of every size 1 .. qcap
    (one leaf per size, one with two full tiles and a single query), tombstones, exact duplicate rows, a query equal to a
    stored row, partial row blocks; every visit's list exact for the three exact metrics and (n' <= 32) for L2 / L2 squared
    through the dot-product filter and its second pass; then n' = top_k everywhere, so the shared per-query bound is
    published and read, and the per-query answer must not change."""
    rng = np.random.default_rng(dim + 10 * qcap + kr)
    visits = list(range(1, qcap + 1)) + [2 * qcap + 1]
    leaf_lens = [1, 63, 64, 65, 130, 17, 70, 128, 129][:len(visits) - 1] + [150]
    np_max = 32 if kr == 1 else 128
    case = build_case(rng, dim, leaf_lens, 2 * qcap + 3, visits, np_max=np_max, tomb_frac=0.15)
    if kr != 1:
        case["v_np"][:4] = [128, 127, 100, 33]
    lo = int(case["leaf_off"][-2])                              # last leaf: a group of near copies of one row (the filter's cancellation)
    for i in range(1, 25):
        case["rows"][lo + i] = case["rows"][lo]
        case["rows"][lo + i, i] = np.nextafter(case["rows"][lo, i], F32(np.inf) if i % 2 else F32(-np.inf), dtype=F32)
    case["queries"][1] = case["rows"][lo]
    for metric in (zo.COSINE, zo.L2SQ, zo.L2):
        entries, ent_off, v_np, _ = run_emu(emu, case, metric, top_k=0xFFFFFFFF, tq=qcap, qcap=qcap, nst=nst, kr=kr)
        check_every_visit(case, metric, entries, ent_off, v_np)
    if kr == 1:                                                 # the filter takes n' <= 16
        fcase = dict(case, v_np=np.minimum(case["v_np"], 16))
        entries, ent_off, v_np, _ = run_emu(emu, fcase, zo.L2SQ, top_k=0xFFFFFFFF, tq=qcap, qcap=qcap, nst=nst, l2_filter=True)
        check_every_visit(fcase, zo.L2SQ, entries, ent_off, v_np)
    k = 10 if kr == 1 else 100
    for filt in ((False, True) if kr == 1 else (False,)):
        entries, ent_off, _, gthr = run_emu(emu, case, zo.L2, top_k=k, tq=qcap, qcap=qcap, nst=nst, kr=kr, same_np=k, blocks=2,
                                            l2_filter=filt)
        assert (gthr != SENT).any()
        for q in range(case["queries"].shape[0]):
            got, exp = [], []
            for v in np.nonzero(case["v_q"] == q)[0]:
                got += [tuple(x) for x in entries[ent_off[v]:ent_off[v + 1]] if x[1] != SENT]
                exp += [tuple(x) for x in expected_visit(case, zo.L2, v, k)]
            assert sorted(set(got))[:k] == sorted(set(exp))[:k], (filt, q)


@pytest.mark.parametrize("kr", [1, 4])
@pytest.mark.parametrize("dim,qcap,nst1,nst4", SMALL_TILES, ids=[f"{d}d-{q}q" for d, q, _, _ in SMALL_TILES])
def test_small_tile_capacities(emu, dim, qcap, nst1, nst4, kr):
    check_small_tiles(emu, dim, qcap, nst1 if kr == 1 else nst4, kr)


@pytest.mark.parametrize("dim,H,n,tq", [(48, 16, 200, 16), (100, 37, 333, 16), (64, 5, 70, 16), (200, 24, 150, 8)])
def test_projection_mode_signs_equal_point_is_above(emu, dim, H, n, tq):
    """MODE 1 of the same kernel body (flat-table hashing): sign[row][plane] = Hyperplane::point_is_above (lsh.rs:39-43) for
    every (row, plane), planes in tiles of <= 16, rows in ranges that are not multiples of the 64-row stage."""
    rng = np.random.default_rng(dim + H)
    dimp = (dim + 15) // 16 * 16
    rows = rng.standard_normal((n, dim)).astype(F32)
    coef = rng.standard_normal((H, dim)).astype(F32)
    cst = rng.standard_normal(H).astype(F32)
    coef[0] = 0; cst[0] = -0.0                              # dot = +0, constant -0: above
    rows[5] = 0
    rows_p = np.zeros((n + 1, dimp), F32); rows_p[:n, :dim] = rows
    coef_p = np.zeros((H, dimp), F32); coef_p[:, :dim] = coef
    Hp = (H + 15) // 16 * 16
    sign = np.full((n, Hp), 7, np.uint8)
    stats = np.zeros(8, np.uint64)
    emu.emu_project3.restype = C.c_int
    emu.emu_project3.argtypes = [C.c_int, C.c_int, C.c_int, C.c_int, C.c_uint64, C.c_void_p, C.c_int, C.c_void_p, C.c_void_p,
                                 C.c_uint32, C.c_uint32, C.c_void_p, C.c_int, C.c_void_p]
    emu.emu_project3(2, dim, 4, 16, n, rows_p.ctypes.data, H, coef_p.ctypes.data, cst.ctypes.data, 100, tq, sign.ctypes.data, Hp,
                     stats.ctypes.data)
    exp = np.stack([zo.above_batch(np.broadcast_to(coef[h], rows.shape).copy(), np.full(n, cst[h], F32), rows) for h in range(H)], axis=1)
    assert np.array_equal(sign[:, :H], exp.astype(np.uint8))
    assert np.all(sign[:, H:] == 7)                        # nothing written beyond the planes


@pytest.mark.parametrize("metric", [zo.COSINE, zo.L2SQ])
def test_lists_of_up_to_128_entries(emu, metric):
    """KR = 4 (n' up to 128, BASELINE config 5's top-100): entry i of a list lives in lane i / 4, register i % 4; every
    visit's list against the oracle, with n' from 1 to 128, ties, tombstones and leaves shorter than n'."""
    rng = np.random.default_rng(4 + metric)
    leaf_lens = [300, 64, 129, 40, 257]
    visits = [9, 16, 5, 3, 12]
    case = build_case(rng, 48, leaf_lens, 16, visits, np_max=128, tomb_frac=0.2)
    case["v_np"][:4] = [128, 127, 100, 33]
    entries, ent_off, v_np, _ = run_emu(emu, case, metric, top_k=0xFFFFFFFF, tq=16, kr=4)
    for v in range(case["v_leaf"].size):
        exp = expected_visit(case, metric, v, int(v_np[v]))
        got = entries[ent_off[v]:ent_off[v + 1]]
        assert got.shape[0] == exp.shape[0], v
        assert np.array_equal(got, exp), (v, int(case["v_leaf"][v]), int(case["v_q"][v]), int(v_np[v]))


def test_shared_bound_with_long_lists(emu):
    """KR = 4 with every visit asking for n' = top_k = 100: published bounds may shorten later lists, the per-query top-100
    over all visits must not change."""
    rng = np.random.default_rng(123)
    leaf_lens = [260, 190, 300, 150]
    case = build_case(rng, 32, leaf_lens, 6, [6, 6, 6, 6], np_max=100, tomb_frac=0.1)
    k = 100
    entries, ent_off, _, gthr = run_emu(emu, case, zo.L2SQ, top_k=k, tq=16, same_np=k, blocks=2, kr=4)
    assert (gthr != SENT).any()
    for q in range(6):
        got, exp = [], []
        for v in np.nonzero(case["v_q"] == q)[0]:
            e = entries[ent_off[v]:ent_off[v + 1]]
            got += [tuple(x) for x in e if x[1] != SENT]
            exp += [tuple(x) for x in expected_visit(case, zo.L2SQ, v, k)]
        assert sorted(set(got))[:k] == sorted(set(exp))[:k], q


def test_fold_row_is_a_bijection():
    rows = sorted(((t >> 1) & 1) | ((t & 1) << 1) | (t & 4) | (t & 8) for t in range(16))
    assert rows == list(range(16))
    rows8 = sorted((t & 1) | ((t >> 1) & 2) | ((t >> 1) & 4) for t in range(16))   # 8 rows per warp: every row on threads t and t ^ 2
    assert rows8 == sorted(list(range(8)) * 2)


# ---- METRIC 3: L2 / L2 squared through the dot-product filter + exact second pass ---------------------------------------
def check_every_visit(case, metric, entries, ent_off, v_np):
    for v in range(case["v_leaf"].size):
        exp = expected_visit(case, metric, v, int(v_np[v]))
        got = entries[ent_off[v]:ent_off[v + 1]]
        assert got.shape[0] == exp.shape[0], v
        assert np.array_equal(got, exp), (v, int(case["v_leaf"][v]), int(case["v_q"][v]), int(v_np[v]))


@pytest.mark.parametrize("metric", [zo.L2SQ, zo.L2])
@pytest.mark.parametrize("dim,tq", [(48, 16), (100, 16), (200, 11)])
def test_l2_filter_per_visit_lists_equal_oracle(emu, metric, dim, tq):
    """Every visit's list after the two passes is the exact top-n' (n' up to 16: what the launch code admits), with ties,
    tombstones, a distance of exactly zero, partial blocks and every QH."""
    rng = np.random.default_rng(dim * 11 + metric)
    leaf_lens = [1, 63, 64, 65, 130, 17, 200, 128, 5]
    visits = [1, 2, 5, 9, 16, 3, 21, 13, 4]
    case = build_case(rng, dim, leaf_lens, 24, visits, np_max=16, tomb_frac=0.15)
    info = {}
    entries, ent_off, v_np, _ = run_emu(emu, case, metric, top_k=0xFFFFFFFF, tq=tq, l2_filter=True, info=info)
    check_every_visit(case, metric, entries, ent_off, v_np)
    assert info["flagged"] == 0                             # well-separated random data: the filter alone decides
    live = sum(min(int(n), 32) for n in case["leaf_len"][case["v_leaf"]])
    assert info["exact_rows"] < live                        # ... and the second pass looked at a fraction of the listed rows


def test_l2_filter_crowded_keys_flag_the_visit(emu):
    """More than 32 rows within the error band of the n'-th best (here: 50 copies of one row, and rows a few ulps apart):
    the 32-entry list cannot hold every candidate, the visit is flagged and its leaf scanned exactly -- ties by position."""
    rng = np.random.default_rng(77)
    case = build_case(rng, 64, [150, 90, 64], 6, [6, 6, 6], np_max=12, tomb_frac=0.1, dup=False)
    case["rows"][20:70] = case["rows"][5]                   # leaf 0: 51 equal rows
    near = case["rows"][160].copy()
    for i in range(40):                                      # leaf 1: 40 rows that differ in the last bits of one coordinate
        case["rows"][170 + i] = near
        case["rows"][170 + i, 3] = np.nextafter(near[3], F32(np.inf) if i % 2 else F32(-np.inf), dtype=F32)
    case["queries"][0] = case["rows"][5]
    case["queries"][1] = near
    info = {}
    entries, ent_off, v_np, _ = run_emu(emu, case, zo.L2SQ, top_k=0xFFFFFFFF, tq=16, l2_filter=True, info=info)
    check_every_visit(case, zo.L2SQ, entries, ent_off, v_np)
    assert info["flagged"] >= 2


def test_l2_filter_unusable_norms_fall_back_to_the_exact_scan(emu):
    """Rows and queries whose squared norms overflow, are infinite or NaN, and subnormal / zero vectors."""
    rng = np.random.default_rng(78)
    case = build_case(rng, 48, [100, 70, 40, 64], 8, [8, 8, 8, 8], np_max=10, tomb_frac=0.05, dup=False)
    case["rows"][3, 0] = F32(3e19)                          # |row|^2 = 9e38: inf
    case["rows"][7, 5] = F32(np.nan)
    case["rows"][110, 2] = F32(np.inf)
    case["rows"][120] *= F32(1e18)                          # |row|^2 ~ 5e37: above the limit, finite
    case["rows"][175] = 0
    case["rows"][176] = F32(1e-30)                          # squares underflow to subnormals / zero
    case["rows"][177] = F32(1e-22)
    case["queries"][2] = 0
    case["queries"][3] = F32(1e-25)
    case["queries"][4, 1] = F32(np.nan)
    case["queries"][5] *= F32(2e18)
    info = {}
    with np.errstate(over="ignore", invalid="ignore"):
        entries, ent_off, v_np, _ = run_emu(emu, case, zo.L2, top_k=0xFFFFFFFF, tq=16, l2_filter=True, info=info)
        check_every_visit(case, zo.L2, entries, ent_off, v_np)
    assert info["flagged"] >= 8


def test_l2_filter_wide_norm_range_inside_a_leaf(emu):
    """The error bound of a leaf follows its largest row: small rows next to rows 10^4 times longer stay exact (more candidates,
    possibly flagged visits, never a wrong list)."""
    rng = np.random.default_rng(79)
    case = build_case(rng, 80, [120, 200], 10, [10, 10], np_max=8, tomb_frac=0.0, dup=False)
    case["rows"][:120:3] *= F32(1e4)
    case["rows"][130:200] *= F32(1e-3)
    case["queries"][:5] *= F32(1e-3)
    entries, ent_off, v_np, _ = run_emu(emu, case, zo.L2SQ, top_k=0xFFFFFFFF, tq=16, l2_filter=True)
    check_every_visit(case, zo.L2SQ, entries, ent_off, v_np)


@pytest.mark.parametrize("metric", [zo.L2SQ, zo.L2])
def test_l2_filter_shared_bound_keeps_the_per_query_answer(emu, metric):
    """n' = top_k everywhere: full lists publish G = A_(n') + Eq, later visits (and the second pass) drop rows above it; the
    per-query top-k over all visits must be the exact one."""
    rng = np.random.default_rng(101 + metric)
    leaf_lens = [150, 90, 200, 64, 70, 129]
    case = build_case(rng, 64, leaf_lens, 12, [12] * 6, np_max=8, tomb_frac=0.1)
    k = 8
    entries, ent_off, _, gthr = run_emu(emu, case, metric, top_k=k, tq=16, same_np=k, blocks=3, l2_filter=True)
    assert (gthr != SENT).any()
    for q in range(12):
        got, exp = [], []
        for v in np.nonzero(case["v_q"] == q)[0]:
            e = entries[ent_off[v]:ent_off[v + 1]]
            got += [tuple(x) for x in e if x[1] != SENT]
            exp += [tuple(x) for x in expected_visit(case, metric, v, k)]
        assert sorted(set(got))[:k] == sorted(set(exp))[:k], q


@pytest.mark.parametrize("seed", [1, 2, 3, 4])
def test_l2_filter_randomised_cases(emu, seed):
    """Random shapes around the filter's edges: groups of equal and nearly equal rows whose sizes straddle the 32-entry candidate
    list, scales from 1e-3 to 1e3, n' from 1 to 16, tombstones, queries equal to stored rows -- every visit's list exact, with
    and without the shared per-query bound."""
    if emu.variant[0] != 3 or emu.variant[1]:
        pytest.skip("the filter ships with the default stage shape; the other build variants run the fixed cases above")
    rng = np.random.default_rng(1000 + seed)
    dim = int(rng.choice([16, 40, 64, 100, 130]))
    nleaf = int(rng.integers(3, 7))
    leaf_lens = [int(x) for x in rng.integers(20, 220, nleaf)]
    nq = int(rng.integers(6, 20))
    visits = [int(x) for x in rng.integers(1, min(nq, 16) + 1, nleaf)]
    case = build_case(rng, dim, leaf_lens, nq, visits, np_max=16, tomb_frac=float(rng.choice([0.0, 0.1, 0.3])), dup=False)
    scale = F32(10.0 ** rng.uniform(-3, 3))
    case["rows"] = (case["rows"] * scale).astype(F32)
    case["queries"] = (case["queries"] * scale).astype(F32)
    P = case["P"]
    for _ in range(int(rng.integers(2, 6))):                       # groups of copies / near copies of one row, 2 .. 40 strong
        g = int(rng.integers(2, 41))
        idx = rng.choice(P, size=min(g, P), replace=False)
        src = case["rows"][idx[0]].copy()
        for j, i in enumerate(idx):
            case["rows"][i] = src
            if j % 3 == 1:                                          # a few ulps away in one coordinate
                c = int(rng.integers(0, dim))
                case["rows"][i, c] = np.nextafter(src[c], F32(np.inf) if j % 2 else F32(-np.inf), dtype=F32)
        case["queries"][int(rng.integers(0, nq))] = src             # and a query sitting exactly on the group
    metric = zo.L2SQ if seed % 2 else zo.L2
    entries, ent_off, v_np, _ = run_emu(emu, case, metric, top_k=0xFFFFFFFF, tq=16, l2_filter=True)
    check_every_visit(case, metric, entries, ent_off, v_np)
    k = int(rng.integers(1, 17))                                    # the same data with n' = top_k everywhere: bounds are published
    entries, ent_off, _, _ = run_emu(emu, case, metric, top_k=k, tq=16, same_np=k, blocks=2, l2_filter=True)
    for q in range(nq):
        got, exp = [], []
        for v in np.nonzero(case["v_q"] == q)[0]:
            e = entries[ent_off[v]:ent_off[v + 1]]
            got += [tuple(x) for x in e if x[1] != SENT]
            exp += [tuple(x) for x in expected_visit(case, metric, v, k)]
        assert sorted(set(got))[:k] == sorted(set(exp))[:k], (seed, q)
