"""The GPU-resident keypoint map (csrc/gmap.cu) at its edges, against the oracle's Map and a Python replica of the map
(gmap_replica.py, which also keeps the entry tags and the export order).

CPU: the replica equals the oracle on random frames and on every case below, and hand cases pin both.
GPU: every case is compared after every update on gmap_get_keypoints, gmap_export, gmap_scans tags and gmap_size:
ballot-round and chunk edges inside one deep block, rejections and overwrites inside one update, more than 1024 blocks in
one update, positions on lattice and block boundaries, the gather cube's edges and budgets, export / import of a map
larger than one radix tile, full entry / chunk / table pools, and non-finite or unstorable input."""
import ctypes as C

import numpy as np
import pytest

import gmap_replica as rep

f32 = np.float32
GRID = (np.arange(11) * 850.0 - 4250.0).astype(f32)            # 11 positions 850 mm apart inside one 10 m block
CELL = np.stack(np.meshgrid(GRID, GRID, GRID, indexing="ij"), -1).reshape(-1, 3)   # 1331 points, none within 800 mm
PERM = np.array([[0, -1, 0, 0], [1, 0, 0, 0], [0, 0, 1, 0]], f32)  # a rotation whose products and sums are exact


def bits(a):
    return np.ascontiguousarray(a, f32).view(np.uint32)


def desc_of(n, seed):
    rng = np.random.default_rng(seed)
    return rng.integers(0, 2 ** 63, (n, 6), dtype=np.uint64) * np.uint64(2) + rng.integers(0, 2, (n, 6), dtype=np.uint64)


def pose_T(yaw, t):
    c, s = np.cos(yaw), np.sin(yaw)
    return np.array([[c, -s, 0, t[0]], [s, c, 0, t[1]], [0, 0, 1, t[2]]], f32)


# ---- the cases: lists of updates (xyz, ratio, desc, pose) and the cubes to gather ------------------------------------------
def random_frames(seed=3, frames=5):
    rng = np.random.default_rng(seed)
    out = []
    for k in range(frames):
        n = int(rng.integers(300, 1500))
        xyz = rng.uniform(-30000, 30000, (n, 3)).astype(f32)
        xyz[:, 2] *= 0.3
        m = n // 6                                              # neighbours within 800 mm and exact re-observations
        xyz[rng.integers(0, n, m)] = xyz[rng.integers(0, n, m)] + rng.uniform(-600, 600, (m, 3)).astype(f32)
        xyz[rng.integers(0, n, m)] = xyz[rng.integers(0, n, m)]
        ratio = rng.choice(np.linspace(0.1, 1.0, 30).astype(f32), n)
        out.append((xyz, ratio, desc_of(n, 100 + k), None if k == 0 else pose_T(0.07 * k, (650.0 * k, -45.5, 12.25))))
    return out


def deep_block_frames():
    """block (0, 0, 0) grows to 135 entries (5 chunks) over three updates; its members sit at keypoint indices 31, 32,
    63, 64 and n-1 of every frame, the rest of a frame lies in four other blocks.  Entries 31, 32, 63 and 64 of the block
    are salient (0.9), the others 0.3.  The fourth update overwrites entries 31 and 64 in place, is rejected by 32 and 63
    alone (10 mm away, saliency 0.6 or an equal position at 0.5), and appends a keypoint 10 mm from entry 33"""
    rng = np.random.default_rng(11)
    n, per = 150, 45
    order = rng.permutation(len(CELL))
    frames, used = [], 0
    for u in range(3):
        members = np.sort(np.concatenate([[31, 32, 63, 64, n - 1], rng.choice(np.setdiff1d(np.arange(n - 1), [31, 32, 63, 64]), per - 5, replace=False)]))
        xyz = (CELL[rng.integers(0, len(CELL), n)] + f32([20000.0, 0, 0]) * rng.choice([-2, -1, 1, 2], (n, 1))).astype(f32)
        xyz[members] = CELL[order[used:used + per]]
        ratio = rng.choice(np.float32([0.2, 0.4, 0.6]), n).astype(f32)
        ratio[members] = np.where(np.isin(np.arange(used, used + per), [31, 32, 63, 64]), f32(0.9), f32(0.3))
        used += per
        frames.append((xyz, ratio, desc_of(n, 200 + u), None))
    entry = CELL[order[:used]]                                  # entry j of the block, in insertion order
    xyz = (CELL[rng.integers(0, len(CELL), n)] + f32(20000.0) * np.array([1, 0, 0], f32)).astype(f32)
    ratio = np.full(n, 0.5, f32)
    plan = {31: (entry[31], 0.95), 32: (entry[32] + f32([0, 0, 10]), 0.6), 63: (entry[63] + f32([0, 0, 10]), 0.6),
            64: (entry[64], 0.95), 100: (entry[32], 0.5), n - 1: (entry[33] + f32([0, 0, 10]), 0.6)}
    for i, (p, r) in plan.items():
        xyz[i], ratio[i] = p, r
    frames.append((xyz, ratio, desc_of(n, 204), None))
    return frames


def interplay_frames():
    """keypoints of one update reject and overwrite each other, in 40 blocks; a second update overwrites entries of the
    first (same slot, new tag) and is rejected by others"""
    rng = np.random.default_rng(5)
    # per block: insert, rejected, overwrite (same slot), rejected, insert, overwrite, insert, rejected (equal saliency)
    pattern = np.array([[0, 0, 0], [100, 0, 0], [0, 0, 0], [300, 0, 0], [900, 0, 0], [900, 0, 0], [0, 2000, 0], [0, 2400, 0]], f32)
    pratio = np.float32([0.5, 0.4, 0.7, 0.6, 0.1, 0.2, 0.3, 0.3])
    cells = np.stack(np.meshgrid(np.arange(-3, 4), np.arange(-3, 4), indexing="ij"), -1).reshape(-1, 2)[rng.choice(49, 40, replace=False)]
    base = np.concatenate([cells * 10000.0 - 2000.0, np.zeros((40, 1))], 1).astype(f32)
    xyz = (base[:, None, :] + pattern[None]).reshape(-1, 3)
    ratio = np.tile(pratio, 40)
    rows, seen = [], np.zeros(40, int)                          # blocks interleaved, each block's keypoints in pattern order
    for b in rng.permutation(np.repeat(np.arange(40), 8)):
        rows.append(8 * b + seen[b])
        seen[b] += 1
    first = (xyz[rows], ratio[rows], desc_of(320, 300), None)
    again = np.concatenate([base, base + f32([900, 1000, 0]), base + f32([0, 2400, 0])])
    aratio = np.concatenate([np.full(40, 0.8, f32), np.full(40, 0.15, f32), np.full(40, 0.3, f32)])
    return [first, (again, aratio, desc_of(120, 301), None)]


def many_block_frames(per=4, seed=9):
    """12^3 = 1728 blocks, lattice coordinates -6..5 on every axis, `per` keypoints each, in one update"""
    rng = np.random.default_rng(seed)
    b = np.stack(np.meshgrid(*[np.arange(-6, 6)] * 3, indexing="ij"), -1).reshape(-1, 3)
    xyz = (np.repeat(b, per, 0) * 10000.0 + rng.uniform(-4900, 4900, (len(b) * per, 3))).astype(f32)
    p = rng.permutation(len(xyz))
    return [(xyz[p], rng.choice(np.linspace(0.1, 1, 10).astype(f32), len(xyz)), desc_of(len(xyz), 400), None)]


def boundary_values(extra=True):
    """block boundaries 5000 k, the lattice points 10 mm beside them, their float32 neighbours (and a few snap cases)"""
    v = [f32(5000.0 * k) for k in range(-2, 3)] + [f32(5000.0 * k + d) for k in (-2, -1, 1, 2) for d in (-10.0, 10.0)]
    out = set()
    for a in v:
        out.add(float(a))
        if a != 0:
            out.update([float(np.nextafter(a, f32(np.inf))), float(np.nextafter(a, f32(-np.inf)))])
    if extra:
        out.update([-0.0, 4999.99, -15.9, -5.0])
    return np.array(sorted(out), f32)


def boundary_frames():
    """positions that land on the boundaries after the pose: exactly with PERM + T (the sums are exact), and with a small
    rotation, which rounds them somewhere next to the boundaries"""
    rng = np.random.default_rng(13)
    vals = boundary_values()
    tgt = np.stack([rng.choice(vals, 900), rng.choice(vals, 900), rng.choice(vals, 900)], 1).astype(f32)
    T = f32([2500.0, -2500.0, 1250.0])
    P = PERM.copy()
    P[:, 3] = T
    # world = (-y + T0, x + T1, z + T2)
    src = np.stack([tgt[:, 1] - T[1], -(tgt[:, 0] - T[0]), tgt[:, 2] - T[2]], 1).astype(f32)
    ratio = rng.choice(np.linspace(0.1, 1, 7).astype(f32), 900)
    frames = [(src, ratio, desc_of(900, 500), P)]
    frames.append((tgt, ratio[::-1].copy(), desc_of(900, 501), pose_T(1e-6, (0.0, 0.0, 0.0))))
    frames.append((tgt, ratio, desc_of(900, 502), None))
    return frames


CASES = {"random": random_frames, "deep": deep_block_frames, "interplay": interplay_frames, "many_blocks": many_block_frames,
         "boundaries": boundary_frames}
COVER = {"random": ([0, 0, 0], 80000.0), "deep": ([0, 0, 0], 60000.0), "interplay": ([0, 0, 0], 50000.0),
         "many_blocks": ([-5000, -5000, -5000], 60000.0), "boundaries": ([0, 0, 0], 30000.0)}
CUBES = [([0, 0, 0], 0.0), ([5000, -5000, 5000], 0.0), ([2500, 2500, -2500], 2500.0), ([5000, -5000, 15000], 10000.0),
         ([-15000, 4999.99, 0], 5000.0), ([12000, -3000, 500], 15000.0)]


def assert_same_get(a, b, where):
    assert len(a[0]) == len(b[0]), (where, len(a[0]), len(b[0]))
    assert np.array_equal(bits(a[0]), bits(b[0])) and np.array_equal(a[1], b[1]), where


# ---- CPU -------------------------------------------------------------------------------------------------------------------
def test_hand_cases(oracle):
    d = desc_of(8, 1)
    for m in (oracle.Map(), rep.Map()):
        m.add([[1234.9, -15.9, -0.0]], [0.5], d[:1])            # truncation toward zero: (1230, -10, +0)
        xyz = m.get([0, 0, 0], 0.0)[0]
        assert np.array_equal(bits(xyz), bits([[1230.0, -10.0, 0.0]])), type(m)
        # block edges round half away from zero: 5000 -> block 1, -5000 -> block -1, 4999.99 -> 4990 -> block 0
        m.add([[5000.0, 0, 0], [4999.99, 0, 0], [-5000.0, 0, 0], [-4999.99, 0, 0]], [0.5] * 4, d[1:5])
        assert np.array_equal(m.get([10000.0, 0, 0], 0.0)[0], [[5000.0, 0, 0]]), type(m)
        assert np.array_equal(m.get([-10000.0, 0, 0], 0.0)[0], [[-5000.0, 0, 0]]), type(m)
        assert np.array_equal(m.get([0, 0, 0], 0.0)[0], [[1230.0, -10.0, 0.0], [4990.0, 0, 0], [-4990.0, 0, 0]]), type(m)
        m.add([[-5.0, -0.0, 9.99]], [0.9], d[5:6])              # (-5, -0, 9.99) -> (+0, +0, +0)
        assert np.array_equal(bits(m.get([0, 0, 0], 0.0)[0][3]), bits([0.0, 0.0, 0.0])), type(m)
    r = rep.Map()
    r.add([[0.0, 0, 0]], [0.5], d[:1])
    r.add([[9.0, 0, 0], [0.0, 500, 0]], [0.7, 0.5], d[1:3])     # overwrite (same lattice position), then rejected
    x, dd, t = r.export()
    assert np.array_equal(t, [1]) and np.array_equal(dd, d[1:2]) and len(r) == 1


@pytest.mark.parametrize("case", sorted(CASES))
def test_replica_equals_oracle(oracle, case):
    om, rm = oracle.Map(), rep.Map()
    for u, (xyz, ratio, desc, pose) in enumerate(CASES[case]()):
        om.add(xyz, ratio, desc, pose)
        assert rm.add(xyz, ratio, desc, pose) == 0
        assert len(rm) == len(om), (case, u)
        pos, r = COVER[case]
        assert_same_get(rm.get(pos, r), om.get(pos, r), (case, u, "cover"))
        assert len(rm.get(pos, r)[0]) == len(om)
        x, d, _ = rm.export()
        assert_same_get((x[:, :3], d), om.get(pos, r), (case, u, "export"))   # one covering cube visits blocks in map order
        for pos, r in CUBES:
            assert_same_get(rm.get(pos, r), om.get(pos, r), (case, u, pos, r))


def test_cases_hit_their_edges():
    """the cases do what their docstrings say"""
    m = rep.Map()
    for u, f in enumerate(deep_block_frames()):
        m.add(*f)
        blk = m.blocks[rep.block_id(0, 0, 0)]
        assert len(blk) == 45 * (u + 1) if u < 3 else len(blk) == 136
    assert [e[5] for e in blk[30:34]] == [0, 3, 0, 0] and [e[5] for e in blk[63:66]] == [1, 3, 1] and blk[-1][5] == 3
    w = rep.transform(boundary_frames()[0][0], boundary_frames()[0][3])
    assert np.isin(boundary_values(extra=False), w).all()
    m = rep.Map()
    for f in interplay_frames():
        m.add(*f)
    for blk in m.blocks.values():
        assert [e[5] for e in blk] == [1, 0, 0, 1] and blk[0][3] == f32(0.8)


# ---- GPU -------------------------------------------------------------------------------------------------------------------
def snapshot(ctx):
    x, d = ctx.gmap_export()
    tags, traj = ctx.gmap_scans()
    return x, d, tags, traj, ctx.gmap_size()


def assert_same_snapshot(a, b, where=""):
    assert np.array_equal(bits(a[0]), bits(b[0])) and np.array_equal(a[1], b[1]), (where, "export")
    assert np.array_equal(a[2], b[2]), (where, "tags")
    assert np.array_equal(bits(a[3]), bits(b[3])), (where, "trajectory")
    assert tuple(a[4]) == tuple(b[4]), (where, "size", a[4], b[4])


def assert_map(ctx, rm, where, dropped=0, om=None, cubes=()):
    """size, export, tags and gathers of the device map against the replica (and the oracle)"""
    x, d = ctx.gmap_export()
    rx, rd, rt = rm.export()
    size = ctx.gmap_size()
    assert size == (len(rm), dropped) and len(x) == len(rm), (where, "size/export mismatch", size, len(x), len(rm))
    assert np.array_equal(bits(x), bits(rx)) and np.array_equal(d, rd), (where, "export")
    assert np.array_equal(ctx.gmap_scans()[0], rt), (where, "tags")
    for pos, r in cubes:
        g = ctx.gmap_get_keypoints(pos, r)
        assert_same_get(g, rm.get(pos, r)[:2], (where, pos, r))
        if om is not None:
            assert_same_get(g, om.get(pos, r), (where, "oracle", pos, r))


def lib_get(bshot, ctx, pos, r, cap=0):
    """bshot_gmap_get_keypoints -> (return code, *n_out)"""
    pos = np.ascontiguousarray(pos, f32)
    n = C.c_size_t()
    rc = bshot.lib().bshot_gmap_get_keypoints(ctx.h, pos.ctypes.data_as(C.c_void_p), r, None, None, cap, C.byref(n))
    return rc, n.value


def after_case_invariants(bshot, ctx, cover):
    """export == the gather of a covering cube; import(export()) is the identity (with every tag 0); a re-anchor with the
    current trajectory changes nothing"""
    x, d = ctx.gmap_export()
    g = ctx.gmap_get_keypoints(*cover)
    assert np.array_equal(bits(g[0]), bits(x[:, :3])) and np.array_equal(g[1], d), "export != covering gather"
    before = snapshot(ctx)
    ctx.gmap_reanchor(before[3])
    assert_same_snapshot(snapshot(ctx), before, "re-anchor no-op")
    ctx.gmap_import(x, d)
    xi, di = ctx.gmap_export()
    assert np.array_equal(bits(xi), bits(x)) and np.array_equal(di, d), "import round trip"
    assert ctx.gmap_size() == (len(x), 0) and not ctx.gmap_scans()[0].any()


@pytest.mark.gpu
@pytest.mark.parametrize("case", sorted(CASES))
def test_cases_match_oracle_and_replica(bshot, oracle, case):
    with bshot.Context(0, 16384, 8192, 1 << 16) as ctx:
        ctx.gmap_create(1 << 16, 4096)
        om, rm = oracle.Map(), rep.Map()
        for u, (xyz, ratio, desc, pose) in enumerate(CASES[case]()):
            ctx.gmap_add(xyz, ratio, desc, pose)
            om.add(xyz, ratio, desc, pose)
            rm.add(xyz, ratio, desc, pose)
            assert len(rm) == len(om)
            assert_map(ctx, rm, (case, u), om=om, cubes=[COVER[case]] + CUBES)
        assert len(ctx.gmap_scans()[1]) == len(CASES[case]())
        after_case_invariants(bshot, ctx, COVER[case])


@pytest.mark.gpu
def test_gather_cube_budgets(bshot, oracle):
    """exactly 32^3 probed blocks succeed, 33 x 32 x 32 return BSHOT_E_CAPACITY; exactly max_targets entries in range
    succeed, one more returns BSHOT_E_CAPACITY with the true count"""
    full, over = [-155000.0, 5000.0, 5000.0], [-155000.0, 0.0, 5000.0]   # both cubes hold block 0 and not block 1
    rm = rep.Map()
    assert rm.probes(full, 155000.0) == 32 ** 3 and rm.probes(over, 155000.0) == 32 * 33 * 32
    with bshot.Context(0, 16384, 1000, 1000) as ctx:           # max_targets is at least max_keypoints
        ctx.gmap_create(1 << 14, 4096)
        om = oracle.Map()
        xyz = np.concatenate([CELL[:1000], [[10000.0, 0, 0]]]).astype(f32)   # 1000 entries in block 0, one in block 1
        ratio, desc = np.full(1001, 0.5, f32), desc_of(1001, 600)
        for s in (slice(0, 1000), slice(1000, 1001)):
            ctx.gmap_add(xyz[s], ratio[s], desc[s])
            om.add(xyz[s], ratio[s], desc[s])
            rm.add(xyz[s], ratio[s], desc[s])
        assert_map(ctx, rm, "budgets", om=om, cubes=[([0, 0, 0], 0.0), ([10000.0, 0, 0], 0.0), (full, 155000.0)])
        assert lib_get(bshot, ctx, full, 155000.0) == (0, 1000)
        assert lib_get(bshot, ctx, over, 155000.0)[0] == bshot.E_CAPACITY
        rc, n = lib_get(bshot, ctx, [0, 0, 0], 0.0)
        assert (rc, n) == (0, 1000)
        rc, n = lib_get(bshot, ctx, [2500, 0, 0], 2500.0)      # blocks 0 and 1: 1001 > max_targets
        assert (rc, n) == (bshot.E_CAPACITY, 1001)
        with pytest.raises(bshot.BshotError) as e:
            ctx.gmap_get_keypoints([2500, 0, 0], 2500.0)
        assert e.value.code == bshot.E_CAPACITY


@pytest.mark.gpu
def test_pool_full_in_one_block(bshot):
    """1331 keypoints in one block, max_entries 1024: the first 1024 in keypoint order are stored, 307 are dropped"""
    ratio, desc = np.full(len(CELL), 0.5, f32), desc_of(len(CELL), 700)
    with bshot.Context(0, 16384, 2048, 1 << 14) as ctx:
        ctx.gmap_create(1024, 64)
        ctx.gmap_add(CELL, ratio, desc)
        rm = rep.Map()
        rm.add(CELL[:1024], ratio[:1024], desc[:1024])
        assert_map(ctx, rm, "pool full", dropped=307, cubes=[([0, 0, 0], 0.0)])
        after_case_invariants(bshot, ctx, ([0, 0, 0], 0.0))


def block_lattice(n):
    """n distinct blocks (lattice coordinates from a cube around the origin), keypoint at each block's centre"""
    k = int(np.ceil(n ** (1 / 3)))
    b = np.stack(np.meshgrid(*[np.arange(k) - k // 2] * 3, indexing="ij"), -1).reshape(-1, 3)[:n]
    return (b * 10000.0).astype(f32), ([-5000.0] * 3, 10000.0 * (k // 2 + 2))


@pytest.mark.gpu
def test_chunk_pool_full(bshot):
    """gmap_create(1024, 1) holds 97 chunks.  200 keypoints in 200 blocks: 97 stored, 103 dropped, and the size is the
    export's length.  Then the stored blocks are filled without new chunks until the entry pool is full: 1024 stored"""
    xyz, cover = block_lattice(200)
    ratio, desc = np.full(200, 0.5, f32), desc_of(200, 800)
    with bshot.Context(0, 16384, 2048, 1 << 14) as ctx:
        ctx.gmap_create(1024, 1)
        ctx.gmap_add(xyz, ratio, desc)
        x, d = ctx.gmap_export()
        size = ctx.gmap_size()
        assert size == (97, 103) and len(x) == 97, ("size/export mismatch", size, len(x))
        src = {tuple(p): i for i, p in enumerate(xyz)}
        idx = [src[tuple(p)] for p in x[:, :3]]
        assert len(set(idx)) == 97 and np.array_equal(d, desc[idx]) and np.all(x[:, 3] == 0.5)
        assert not ctx.gmap_scans()[0].any()
        # 10 more keypoints in each stored block, 850 mm or more from its entry: 970 candidates for 927 free entries
        off = CELL[np.any(CELL != 0, axis=1)][:10]
        fill = (x[:, None, :3] + off[None]).reshape(-1, 3).astype(f32)
        fdesc = desc_of(len(fill), 801)
        ctx.gmap_add(fill, np.full(len(fill), 0.5, f32), fdesc)
        x2, d2 = ctx.gmap_export()
        size = ctx.gmap_size()
        assert len(x2) == size[0] == 1024 and size[1] == 103 + 970 - 927, ("size/export mismatch", size, len(x2))
        tags = ctx.gmap_scans()[0]
        every = {tuple(p): (dd.tobytes(), 0) for p, dd in zip(xyz, desc)}
        every.update({tuple(p): (dd.tobytes(), 1) for p, dd in zip(fill, fdesc)})
        assert all(every[tuple(p)] == (dd.tobytes(), int(t)) for p, dd, t in zip(x2[:, :3], d2, tags))
        after_case_invariants(bshot, ctx, cover)


@pytest.mark.gpu
def test_table_full(bshot):
    """a 1024-slot table (max_blocks 512) with chunks to spare: 1100 blocks, 1024 stored and 76 dropped"""
    xyz, cover = block_lattice(1100)
    ratio, desc = np.full(1100, 0.5, f32), desc_of(1100, 900)
    with bshot.Context(0, 16384, 2048, 1 << 14) as ctx:
        ctx.gmap_create(1 << 15, 512)
        ctx.gmap_add(xyz, ratio, desc)
        x, d = ctx.gmap_export()
        assert ctx.gmap_size() == (1024, 76) and len(x) == 1024
        src = {tuple(p): i for i, p in enumerate(xyz)}
        idx = [src[tuple(p)] for p in x[:, :3]]
        assert len(set(idx)) == 1024 and np.array_equal(d, desc[idx])
        after_case_invariants(bshot, ctx, cover)


@pytest.mark.gpu
def test_non_finite_and_unstorable_keypoints_are_skipped(bshot, oracle):
    """NaN, +-Inf and beyond +-2.1e9 mm rows (before or after the pose) are skipped and not dropped: the map is what the
    oracle stores from the other rows.  Rows at exactly +-2.1e9 mm are stored"""
    rng = np.random.default_rng(17)
    n = 600
    xyz = rng.uniform(-20000, 20000, (n, 3)).astype(f32)
    bad = rng.choice(n, 120, replace=False)
    xyz[bad, rng.integers(0, 3, 120)] = rng.choice(np.float32([np.nan, np.inf, -np.inf, 2.2e9, -1e30, 3e38]), 120)
    edge = rng.choice(np.setdiff1d(np.arange(n), bad), 4, replace=False)
    xyz[edge] = [[2.1e9, 0, 0], [-2.1e9, 0, 0], [0, 2.1e9, -2.1e9], [2.1e9, 2.1e9, 2.1e9]]
    ratio, desc = rng.uniform(0, 1, n).astype(f32), desc_of(n, 1000)
    with bshot.Context(0, 16384, 2048, 1 << 14) as ctx:
        ctx.gmap_create(1 << 14, 4096)
        om, rm = oracle.Map(), rep.Map()
        for u, pose in enumerate([None, pose_T(0.3, (1000.0, -2000.0, 30.0))]):
            good = rep.storable(rep.transform(xyz, pose))
            ctx.gmap_add(xyz, ratio, desc, pose)
            om.add(xyz[good], ratio[good], desc[good], pose)
            assert rm.add(xyz, ratio, desc, pose) == (~good).sum() >= 120
            x, _ = ctx.gmap_export()
            near0 = lambda a: int(np.any((a == 0) | (a == -10), axis=1).sum())   # NaN snapped to 0, a wrapped int to -10
            assert ctx.gmap_size() == (len(rm), 0) and len(x) == len(om), \
                ("entries at the origin", near0(x[:, :3]) - near0(rm.export()[0][:, :3]), ctx.gmap_size(), len(om))
            assert_map(ctx, rm, ("skipped", u), om=om, cubes=[([0, 0, 0], 60000.0), ([2.1e9, 0, 0], 0.0)])
        # a transform that carries finite rows beyond the storable range
        far = pose_T(0.0, (2.0e9, 0.0, 0.0))
        ctx.gmap_add(xyz[good], ratio[good], desc[good], far)
        assert rm.add(xyz[good], ratio[good], desc[good], far) > 0
        assert_map(ctx, rm, "far")


@pytest.mark.gpu
def test_non_finite_pose_changes_nothing(bshot, synth):
    """gmap_add and gmap_update_from_frame with a non-finite pose return BSHOT_E_INVALID; map, tags, trajectory, size
    and the update count are unchanged"""
    rng = np.random.default_rng(19)
    xyz = rng.uniform(-20000, 20000, (300, 3)).astype(f32)
    ratio, desc = rng.uniform(0, 1, 300).astype(f32), desc_of(300, 1100)
    with bshot.Context(0, 65536, 1024, 1 << 14) as ctx:
        ctx.gmap_create(1 << 14, 4096)
        ctx.gmap_add(xyz, ratio, desc)
        ctx.extract_frame(synth.make_scan("hdl32e", 0)[::2].copy(), bshot.default_params(top_k=400))
        before = snapshot(ctx)
        for v in (np.nan, np.inf, -np.inf):
            for k in (0, 3, 11):
                P = pose_T(0.1, (10.0, 20.0, 30.0))
                P.reshape(-1)[k] = v
                for call in (lambda: ctx.gmap_add(xyz, ratio, desc, P), lambda: ctx.gmap_update_from_frame(P)):
                    with pytest.raises(bshot.BshotError) as e:
                        call()
                    assert e.value.code == bshot.E_INVALID
                    assert_same_snapshot(snapshot(ctx), before, (v, k))
        ctx.gmap_update_from_frame(pose_T(0.1, (10.0, 20.0, 30.0)))
        assert len(ctx.gmap_scans()[1]) == 2


@pytest.mark.gpu
def test_reanchor_out_of_range_changes_nothing(bshot):
    """a rigid, finite correction that moves entries beyond +-2.1e9 mm returns BSHOT_E_INVALID; export, tags, trajectory,
    size and pose are bit for bit unchanged"""
    rng = np.random.default_rng(23)
    with bshot.Context(0, 16384, 1024, 1 << 14) as ctx:
        ctx.gmap_create(1 << 14, 4096)
        for u in range(3):
            ctx.gmap_add(rng.uniform(-20000, 20000, (200, 3)).astype(f32), rng.uniform(0, 1, 200).astype(f32), desc_of(200, 1200 + u),
                         pose_T(0.1 * u, (1000.0 * u, 0.0, 0.0)))
        before = snapshot(ctx)
        pose0 = ctx.gmap_reanchor(before[3])
        for t in (1e30, 2.2e9, -3e9):
            moved = before[3].copy()
            moved[1, 0, 3] = t
            with pytest.raises(bshot.BshotError) as e:
                ctx.gmap_reanchor(moved)
            assert e.value.code == bshot.E_INVALID, t
            assert_same_snapshot(snapshot(ctx), before, t)
            assert np.array_equal(bits(ctx.gmap_reanchor(before[3])), bits(pose0))
        moved = before[3].copy()
        moved[2, 1, 3] += f32(1.5e9)                            # still storable: moves
        ctx.gmap_reanchor(moved)
        x, _ = ctx.gmap_export()
        assert len(x) == len(before[0]) and (x[:, 1] > 1.4e9).sum() == (before[2] == 2).sum()
