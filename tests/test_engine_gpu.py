"""GPU parity of the CSR-level engine (through the C ABI) against the oracle."""
import numpy as np
import pytest

from holo_b200 import synth
from holo_b200.capi import (COST_DISABLED, Csr, DIST_INF, HSPF_E_JOB_STATUS, HSPF_E_NEEDS_ORACLE,
                            HspfError, JS_SATURATED, VF_HOP, VF_LEAF, VF_LEAF_UNLESS_ROOT)
from oracle import pyoracle

pytestmark = pytest.mark.gpu

PLANES = ["dist", "hops", "first_parent", "n_parents", "nh_mask"]


def check(res, j, ref, nh_words=1):
    for k in PLANES:
        got = getattr(res, k)[j]
        exp = ref[k]
        if not np.array_equal(got, exp):
            bad = np.nonzero((got != exp).reshape(len(exp), -1).any(axis=1))[0]
            raise AssertionError(f"job {j} plane {k}: {len(bad)} mismatches, first v={bad[0]} "
                                 f"got={got[bad[0]]} exp={exp[bad[0]]}")
    assert res.job_status[j] == ref["status"]


@pytest.mark.parametrize("V,E,seed,kw", [
    (2, 2, 1, {}),
    (5, 12, 2, {}),
    (100, 400, 3, {}),
    (100, 400, 4, dict(cost_choices=[10, 20])),
    (300, 1400, 5, dict(lan_fraction=0.1)),
    (300, 1400, 6, dict(cost_choices=[10, 20], lan_fraction=0.1)),
    (2000, 8000, 7, dict(cost_lo=1, cost_hi=1000)),
])
@pytest.mark.parametrize("isis", [False, True])
def test_small_all_roots_vs_faithful(ctx, V, E, seed, kw, isis):
    t = synth.random_topology(V, E, synth.SEED_BASE + seed, **kw)
    csr = synth.topology_csr(t, isis=isis)
    g = ctx.upload(csr)
    nv = csr.n_vertices
    roots = np.arange(nv, dtype=np.uint32) if nv <= 300 else np.arange(0, nv, 97, dtype=np.uint32)
    res = ctx.run(g, roots, nh_words=2)
    for j, r in enumerate(roots):
        ref = pyoracle.csr_spf(csr, int(r), vec_mode=int(isis), nh_words=2)
        check(res, j, ref)
    g.free()


def test_c2_shape_1k_roots_vs_heap_and_sample_faithful(ctx):
    t = synth.random_topology(10000, 40000, synth.SEED_BASE + 2)
    csr = synth.topology_csr(t)
    g = ctx.upload(csr)
    roots = np.arange(1000, dtype=np.uint32)
    res = ctx.run(g, roots)
    assert res.status == 0
    for j, r in enumerate(roots):
        check(res, j, pyoracle.csr_spf_heap(csr, int(r)))
    for j in (0, 499, 999):
        check(res, j, pyoracle.csr_spf(csr, int(roots[j])))
    # size-independent properties on every job
    assert (res.dist[np.arange(1000), roots] == 0).all()
    row, col, cost = csr.row_ptr, csr.col, csr.cost
    src = np.repeat(np.arange(csr.n_vertices), np.diff(row))
    for j in range(0, 1000, 50):
        d = res.dist[j].astype(np.int64)
        assert (d[col] <= d[src] + cost).all()          # triangle inequality on every edge
        fp = res.first_parent[j]
        ok = fp != 0xFFFFFFFF
        assert ok.sum() == csr.n_vertices - 1
    g.free()


def test_c5_shape_ecmp_lans(ctx):
    t = synth.random_topology(10000, 40000, synth.SEED_BASE + 5, cost_choices=[10, 20], lan_fraction=0.05)
    csr = synth.topology_csr(t)
    g = ctx.upload(csr)
    L = len(t.lans)
    roots = np.concatenate([np.arange(L, L + 64), np.asarray([m[0] + L for m, _ in t.lans[:64]])]).astype(np.uint32)
    res = ctx.run(g, roots, nh_words=2)
    for j, r in enumerate(roots):
        check(res, j, pyoracle.csr_spf_heap(csr, int(r), nh_words=2))
    for j in (0, 64, 100):
        check(res, j, pyoracle.csr_spf(csr, int(roots[j]), nh_words=2))
    g.free()


def test_perturbations_isis_shape(ctx):
    t = synth.random_topology(3000, 12000, synth.SEED_BASE + 3, cost_lo=1, cost_hi=1000)
    csr = synth.topology_csr(t, isis=True, reject_above=0xFE000000)
    g = ctx.upload(csr)
    # adjacency k = forward edges (a->b, b->a): find CSR edge indices
    row, col = csr.row_ptr, csr.col
    L = len(t.lans)

    def edge_index(u, v, nth):
        idx = [e for e in range(row[u], row[u + 1]) if col[e] == v]
        return idx[nth]

    n_jobs = 200
    overrides, seen = [], {}
    for k in range(n_jobs):
        a, b = int(t.p2p_a[k]) + L, int(t.p2p_b[k]) + L
        # parallel adjacencies share endpoints: the n-th adjacency between {a, b}
        # owns the n-th a->b and the n-th b->a CSR edge (edges keep adjacency order)
        key = (min(a, b), max(a, b))
        nth = seen.get(key, 0)
        seen[key] = nth + 1
        e1, e2 = edge_index(a, b, nth), edge_index(b, a, nth)
        overrides.append([(e1, COST_DISABLED), (e2, COST_DISABLED)] if k % 3 else [(e1, 7), (e2, 9)])
    roots = np.full(n_jobs, L, dtype=np.uint32)
    res = ctx.run(g, roots, overrides=overrides)
    for j in range(n_jobs):
        check(res, j, pyoracle.csr_spf(csr, int(roots[j]), overrides=overrides[j], vec_mode=1))
    g.free()


def test_leaf_flags_and_reject(ctx):
    t = synth.random_topology(400, 1800, synth.SEED_BASE + 9, cost_lo=1, cost_hi=63, lan_fraction=0.05)
    csr = synth.topology_csr(t, isis=True, reject_above=90)
    L = len(t.lans)
    csr.vflags[L + 5] |= VF_LEAF
    csr.vflags[L + 9] |= VF_LEAF_UNLESS_ROOT
    csr.vflags[L + 17] |= VF_LEAF_UNLESS_ROOT
    csr.vflags[L + 30] |= VF_LEAF
    g = ctx.upload(csr)
    roots = np.asarray([L, L + 5, L + 9, L + 17, L + 100], dtype=np.uint32)
    res = ctx.run(g, roots)
    for j, r in enumerate(roots):
        ref = pyoracle.csr_spf(csr, int(r), vec_mode=1)
        check(res, j, ref)
    assert (res.dist[0] == DIST_INF).any()     # reject_above=90 leaves some vertices unreached
    g.free()


def test_disconnected_and_tiny(ctx):
    # two components + an isolated vertex
    row = np.asarray([0, 1, 2, 3, 4, 4], dtype=np.uint32)
    col = np.asarray([1, 0, 3, 2], dtype=np.uint32)
    cost = np.asarray([5, 6, 7, 8], dtype=np.uint32)
    csr = Csr(row, col, cost, np.full(5, VF_HOP, np.uint8), saturate_at=0xFFFF)
    g = ctx.upload(csr)
    res = ctx.run(g, np.arange(5, dtype=np.uint32))
    for j in range(5):
        check(res, j, pyoracle.csr_spf(csr, j))
    g.free()


def test_zero_cost_router_link_is_refused(ctx):
    row = np.asarray([0, 1, 2], dtype=np.uint32)
    csr = Csr(row, np.asarray([1, 0], np.uint32), np.asarray([0, 3], np.uint32), np.full(2, VF_HOP, np.uint8))
    with pytest.raises(HspfError) as ei:
        ctx.upload(csr)
    assert ei.value.code == HSPF_E_NEEDS_ORACLE


def test_saturation_is_flagged(ctx):
    # a chain whose far end exceeds 65535 in OSPF u16 arithmetic
    n = 6
    src = np.arange(n - 1)
    row = np.zeros(n + 1, np.uint32)
    col, cost = [], []
    for v in range(n):
        if v > 0:
            col.append(v - 1); cost.append(20000)
        if v < n - 1:
            col.append(v + 1); cost.append(20000)
        row[v + 1] = len(col)
    csr = Csr(row, np.asarray(col, np.uint32), np.asarray(cost, np.uint32), np.full(n, VF_HOP, np.uint8),
              saturate_at=0xFFFF)
    g = ctx.upload(csr)
    res = ctx.run(g, np.asarray([0], np.uint32))
    assert res.status == HSPF_E_JOB_STATUS
    assert res.job_status[0] & JS_SATURATED
    ref = pyoracle.csr_spf(csr, 0)
    assert ref["status"] & JS_SATURATED
    g.free()


def test_large_vertex_count_uses_global_state(ctx):
    t = synth.random_topology(70000, 280000, synth.SEED_BASE + 4, cost_lo=1, cost_hi=100)
    csr = synth.topology_csr(t)
    g = ctx.upload(csr)
    roots = np.asarray([0, 12345, 69999], dtype=np.uint32)
    res = ctx.run(g, roots)
    for j, r in enumerate(roots):
        check(res, j, pyoracle.csr_spf_heap(csr, int(r)))
    g.free()


def test_quad_image_beyond_shared_memory_runs_the_general_kernel(ctx):
    """40 000 routers have a quad image, but its per-job state (~280 KB) exceeds shared memory: the
    graph is not on the fast path, and a host-pointer batch big enough for the pipelined copy-back
    (>= 256 jobs) runs the general kernel and returns."""
    from holo_b200.capi import quad_image
    t = synth.random_topology(40000, 80000, synth.SEED_BASE + 41)
    csr = synth.topology_csr(t)
    assert quad_image(csr).eligible
    g = ctx.upload(csr)
    assert not ctx.graph_info(g)["fast_path"]
    roots = np.arange(0, 40000, 156, dtype=np.uint32)[:256]
    assert len(roots) == 256
    res = ctx.run(g, roots)
    for j in (0, 128, 255):
        check(res, j, pyoracle.csr_spf(csr, int(roots[j])))
    g.free()


def test_edge_cases_through_the_abi(ctx):
    # single isolated vertex
    csr = Csr(np.asarray([0, 0], np.uint32), np.zeros(0, np.uint32), np.zeros(0, np.uint32),
              np.full(1, VF_HOP, np.uint8), saturate_at=0xFFFF)
    g = ctx.upload(csr)
    res = ctx.run(g, np.asarray([0], np.uint32))
    assert res.dist[0, 0] == 0 and res.hops[0, 0] == 0 and res.first_parent[0, 0] == 0xFFFFFFFF
    # empty job list is a no-op
    res = ctx.run(g, np.zeros(0, np.uint32))
    assert res.dist.shape == (0, 1) and res.status == 0
    # root out of range is rejected on the host
    with pytest.raises(HspfError):
        ctx.run(g, np.asarray([5], np.uint32))
    g.free()


def test_override_limits(ctx):
    t = synth.random_topology(50, 220, synth.SEED_BASE + 31)
    csr = synth.topology_csr(t)
    g = ctx.upload(csr)
    # 8 overrides in one job is the maximum, 9 is refused; results with 8 match the oracle
    ov8 = [(e, 3 + e) for e in range(8)]
    res = ctx.run(g, np.asarray([0], np.uint32), overrides=[ov8])
    check(res, 0, pyoracle.csr_spf(csr, 0, overrides=ov8))
    with pytest.raises(HspfError):
        ctx.run(g, np.asarray([0], np.uint32), overrides=[[(e, 1) for e in range(9)]])
    # a zero-cost override out of a router is order dependent: flagged, not computed silently
    res = ctx.run(g, np.asarray([0], np.uint32), overrides=[[(0, 0)]])
    assert res.status == HSPF_E_JOB_STATUS and res.job_status[0] & 0x4
    g.free()


def test_many_first_hop_atoms_need_more_words(ctx):
    # a root on several large LANs has > 64 first-hop atoms
    lans = [([0] + list(range(1 + 30 * k, 1 + 30 * (k + 1))), [10] * 31) for k in range(3)]
    R = 100
    a = np.arange(1, R, dtype=np.uint32)
    t = synth.Topology(R, a, a - 1, np.full(R - 1, 7, np.uint32), np.full(R - 1, 9, np.uint32), lans)
    csr = synth.topology_csr(t)
    g = ctx.upload(csr)
    root = len(lans) + 0
    from holo_b200.capi import atom_count, JS_TOO_MANY_ATOMS
    n_atoms = atom_count(csr, root)
    assert n_atoms > 64
    res = ctx.run(g, np.asarray([root], np.uint32), nh_words=1)
    assert res.job_status[0] & JS_TOO_MANY_ATOMS
    res = ctx.run(g, np.asarray([root], np.uint32), nh_words=4)
    assert res.status == 0
    check(res, 0, pyoracle.csr_spf(csr, root, nh_words=4))
    g.free()


@pytest.mark.parametrize("V,E,seed,kw,isis", [
    (100, 400, 3, {}, False),
    (100, 400, 4, dict(cost_choices=[10, 20]), False),          # heavy ECMP
    (300, 1400, 5, dict(lan_fraction=0.1), False),              # non-HOP vertices at hops 0
    (300, 1400, 6, dict(cost_choices=[10, 20], lan_fraction=0.1), True),
    (400, 1200, 8, dict(cost_choices=[5]), False),              # all-equal costs: ECMP under ECMP
    (3000, 12000, 9, dict(cost_choices=[10, 20, 30], lan_fraction=0.05), False),
])
def test_jump_and_kahn_next_hop_phases_agree_with_oracle(ctx, V, E, seed, kw, isis):
    """One next-hop word, no overrides: the engine propagates next hops by pointer jumping
    when the root has at most 32 first-hop atoms and by the Kahn push otherwise (or on the
    "general_kahn" path).  Both must give the oracle's planes."""
    t = synth.random_topology(V, E, synth.SEED_BASE + seed, **kw)
    csr = synth.topology_csr(t, isis=isis)
    g = ctx.upload(csr)
    nv = csr.n_vertices
    roots = np.arange(nv, dtype=np.uint32) if nv <= 400 else np.arange(0, nv, 41, dtype=np.uint32)
    refs = [pyoracle.csr_spf(csr, int(r), vec_mode=int(isis), nh_words=1) for r in roots]
    ok = [j for j, ref in enumerate(refs) if ref["status"] == 0]
    assert len(ok) > len(roots) // 2
    # three device paths: the quad-space kernel (default), and spf_batch_kernel with the
    # pointer-jumping and the Kahn next-hop phase
    for path in ("auto", "general", "general_kahn"):
        with ctx.path(path):
            res = ctx.run(g, roots, nh_words=1)   # a root that ran out of atoms only flags its own job
        for j in ok:
            check(res, j, refs[j])
        for j, ref in enumerate(refs):
            assert res.job_status[j] == ref["status"]
    g.free()


def test_atom_count_selects_the_next_hop_phase_per_job(ctx):
    """One batch mixes roots below and above the 32-atom limit of the jump phase: a root on
    two 20-router LANs (43 atoms, Kahn push) and ordinary routers (jump)."""
    lans = [([0] + list(range(1 + 20 * k, 1 + 20 * (k + 1))), [10] * 21) for k in range(2)]
    R = 120
    a = np.arange(1, R, dtype=np.uint32)
    t = synth.Topology(R, a, a - 1, np.full(R - 1, 7, np.uint32), np.full(R - 1, 9, np.uint32), lans)
    csr = synth.topology_csr(t)
    from holo_b200.capi import atom_count
    L = len(lans)
    roots = np.asarray([L + 0, L + 5, L + 60, L + 119, 0, 1], np.uint32)   # router 0, others, both LAN vertices
    counts = [atom_count(csr, int(r)) for r in roots]
    assert max(counts) > 32 and min(counts) <= 32 and max(counts) <= 64
    g = ctx.upload(csr)
    res = ctx.run(g, roots, nh_words=1)
    assert res.status == 0
    for j, r in enumerate(roots):
        check(res, j, pyoracle.csr_spf(csr, int(r), nh_words=1))
    g.free()


@pytest.mark.parametrize("V,E,seed,kw,isis", [
    (100, 400, 3, {}, False),
    (300, 1400, 6, dict(cost_choices=[10, 20], lan_fraction=0.1), False),
    (3000, 12000, 9, dict(cost_choices=[10, 20, 30], lan_fraction=0.05), True),
])
def test_narrow_planes_equal_the_wide_ones(ctx, V, E, seed, kw, isis):
    """hspf_run_batch16: the same results in 16-bit planes, skipped planes stay untouched."""
    from holo_b200.capi import JS_NARROW
    t = synth.random_topology(V, E, synth.SEED_BASE + seed, **kw)
    csr = synth.topology_csr(t, isis=isis)
    g = ctx.upload(csr)
    assert ctx.graph_info(g)["fast_path"]
    nv = csr.n_vertices
    roots = np.arange(nv, dtype=np.uint32) if nv <= 300 else np.arange(0, nv, 37, dtype=np.uint32)
    wide = ctx.run(g, roots, nh_words=1)
    nar = ctx.run16(g, roots)
    for j in range(len(roots)):
        st = int(nar["job_status"][j])
        if wide.job_status[j] == 0 and (wide.nh_mask[j] >> np.uint64(16)).any():
            assert st & JS_NARROW          # more than 16 first-hop atoms in use: does not fit
            continue
        assert (st & ~JS_NARROW) == wide.job_status[j]
        if st:
            continue
        d = wide.dist[j]
        assert np.array_equal(nar["dist"][j], np.where(d == DIST_INF, 0xFFFF, d).astype(np.uint16))
        assert np.array_equal(nar["hops"][j], wide.hops[j])
        fp = wide.first_parent[j]
        assert np.array_equal(nar["first_parent"][j], np.where(fp == 0xFFFFFFFF, 0xFFFF, fp).astype(np.uint16))
        assert np.array_equal(nar["n_parents"][j], wide.n_parents[j])
        assert np.array_equal(nar["nh_mask"][j], wide.nh_mask[j, :, 0].astype(np.uint16))
    # OSPF caller: three planes only
    part = ctx.run16(g, roots, planes=("dist", "hops", "nh_mask"))
    assert np.array_equal(part["dist"], nar["dist"]) and np.array_equal(part["nh_mask"], nar["nh_mask"])
    g.free()


def test_narrow_planes_refused_off_the_fast_path(ctx):
    t = synth.random_topology(60, 240, synth.SEED_BASE + 21, cost_lo=70000, cost_hi=70100)
    csr = synth.topology_csr(t, isis=True)
    g = ctx.upload(csr)
    assert not ctx.graph_info(g)["fast_path"]
    with pytest.raises(HspfError) as ei:
        ctx.run16(g, np.asarray([0], np.uint32))
    assert ei.value.code == -5
    g.free()


def test_device_pointer_jobs_are_validated_on_the_device(ctx):
    """HSPF_RUN_DEVICE_PTRS: the host cannot see the job arrays; a bad root or override edge
    flags its own job HSPF_JS_INVALID and the other jobs of the batch are unaffected."""
    import ctypes as C
    import torch
    from holo_b200 import capi
    t = synth.random_topology(200, 900, synth.SEED_BASE + 22)
    csr = synth.topology_csr(t)
    V = csr.n_vertices
    for path in ("auto", "general"):
        with ctx.path(path):
            g = ctx.upload(csr)
            roots = torch.tensor([0, V + 7, 5, 0xFFFFFFF], dtype=torch.int32, device="cuda")
            n = 4
            bufs = dict(dist=torch.full((n, V), -7, dtype=torch.int32, device="cuda"),
                        hops=torch.zeros((n, V), dtype=torch.int16, device="cuda"),
                        fp=torch.zeros((n, V), dtype=torch.int32, device="cuda"),
                        npar=torch.zeros((n, V), dtype=torch.int16, device="cuda"),
                        nh=torch.zeros((n, V), dtype=torch.int64, device="cuda"),
                        st=torch.zeros((n,), dtype=torch.int32, device="cuda"))
            js = capi.JobsStruct()
            js.n_jobs = n
            js.roots = C.cast(roots.data_ptr(), C.POINTER(C.c_uint32))
            rs = capi.ResultStruct()
            rs.dist = C.cast(bufs["dist"].data_ptr(), C.POINTER(C.c_uint32))
            rs.hops = C.cast(bufs["hops"].data_ptr(), C.POINTER(C.c_uint16))
            rs.first_parent = C.cast(bufs["fp"].data_ptr(), C.POINTER(C.c_uint32))
            rs.n_parents = C.cast(bufs["npar"].data_ptr(), C.POINTER(C.c_uint16))
            rs.nh_mask = C.cast(bufs["nh"].data_ptr(), C.POINTER(C.c_uint64))
            rs.nh_words = 1
            rs.job_status = C.cast(bufs["st"].data_ptr(), C.POINTER(C.c_uint32))
            ctx.run_device(g, js, rs)
            st = bufs["st"].cpu().numpy()
            assert list(st) == [0, capi.JS_INVALID, 0, capi.JS_INVALID]
            d = bufs["dist"].cpu().numpy().astype(np.uint32)
            assert np.array_equal(d[0], pyoracle.csr_spf(csr, 0)["dist"])
            assert np.array_equal(d[2], pyoracle.csr_spf(csr, 5)["dist"])
            assert (bufs["dist"][1] == -7).all()          # skipped job: planes untouched
            g.free()


def test_reserved_sms_shrink_the_grid_and_small_batches_still_run(ctx):
    """hspf_ctx_reserve_sms leaves SMs to a concurrent kernel by launching fewer persistent CTAs;
    batches of 1..4 jobs must still be computed (ADVICE r1)."""
    t = synth.random_topology(300, 1300, synth.SEED_BASE + 23)
    csr = synth.topology_csr(t)
    g = ctx.upload(csr)
    ctx.reserve_sms(40)
    try:
        for n in (1, 2, 3, 4, 300):
            roots = np.arange(n, dtype=np.uint32)
            res = ctx.run(g, roots)
            for j in (0, n - 1):
                check(res, j, pyoracle.csr_spf(csr, int(roots[j])))
    finally:
        ctx.reserve_sms(0)
    g.free()


@pytest.mark.parametrize("shape", ["fast", "wide_costs", "lans"])
def test_update_costs_in_place_equals_a_fresh_upload(ctx, shape):
    """hspf_graph_update_costs patches every cost-bearing array of the device image (CSR, transpose, packed
    twins, quad-space records): a batch on the patched graph gives the planes of a fresh upload of the
    modified CSR, on the fast path, on the general path (u32 costs) and with transit networks."""
    from holo_b200 import capi
    kw = dict(lans=dict(lan_fraction=0.1)).get(shape, {})
    t = synth.random_topology(400, 1800, synth.SEED_BASE + 61, **kw)
    # wide_costs: IS-IS-style u32 arithmetic (no OSPF saturation), costs that do not pack: general kernel
    csr = synth.topology_csr(t, isis=(shape == "wide_costs"), saturate_at=0 if shape == "wide_costs" else 0xFFFF)
    hop = (csr.vflags & 1).astype(bool)
    tails = np.repeat(np.arange(csr.n_vertices), np.diff(csr.row_ptr.astype(np.int64)))
    cand = np.nonzero(hop[tails])[0]                            # edges out of routers carry the costs
    if shape == "wide_costs":
        csr.cost[cand[::7]] = 70000 + (csr.cost[cand[::7]] % 50)
    rng = np.random.default_rng(5)
    L = len(t.lans)
    roots = rng.choice(np.arange(L, csr.n_vertices), 40, replace=False).astype(np.uint32)
    g = ctx.upload(csr)
    assert ctx.graph_info(g)["fast_path"] == (shape != "wide_costs")
    edges = rng.choice(cand, 60, replace=False).astype(np.uint32)
    new = rng.integers(1, 250 if shape != "wide_costs" else 90000, len(edges)).astype(np.uint32)
    ctx.update_costs(g, edges, new)
    csr2 = capi.Csr(csr.row_ptr.copy(), csr.col.copy(), csr.cost.copy(), csr.vflags.copy(), reject_above=csr.reject_above,
                    saturate_at=csr.saturate_at, flags=csr.flags, delta=csr.delta)
    csr2.cost[edges] = new
    got = ctx.run(g, roots)
    g2 = ctx.upload(csr2)
    want = ctx.run(g2, roots)
    for name in ("dist", "hops", "first_parent", "n_parents", "nh_mask", "job_status"):
        assert np.array_equal(getattr(got, name), getattr(want, name)), name
    for j in (0, 17, 39):
        ref = pyoracle.csr_spf_heap(csr2, int(roots[j]), nh_words=1)
        assert np.array_equal(got.dist[j], ref["dist"]) and np.array_equal(got.nh_mask[j].reshape(-1), ref["nh_mask"].reshape(-1))
    with ctx.path("general"):                                   # the general kernel reads the other copies
        alt = ctx.run(g, roots)
    for name in ("dist", "hops", "first_parent", "n_parents", "nh_mask"):
        assert np.array_equal(getattr(alt, name), getattr(want, name)), name
    # refusals leave the graph as it is
    if shape == "fast":
        with pytest.raises(capi.HspfError):
            ctx.update_costs(g, edges[:1], [70000])             # does not fit the packed image
        with pytest.raises(capi.HspfError):
            ctx.update_costs(g, edges[:1], [0])                 # zero cost out of a router
        with pytest.raises(capi.HspfError):
            ctx.update_costs(g, [csr.n_edges], [5])
        again = ctx.run(g, roots)
        assert np.array_equal(again.dist, want.dist)
    g.free(); g2.free()
