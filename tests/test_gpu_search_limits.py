"""The exact top-k search at the edges of its contract: data built to defeat the fp16 tensor-core pass, every
k-dependent code path up to k = 1024, the shared-memory limit of the merge, and alpha-QE at its largest k.

The search promises the exact top-k by fp64 score (ties -> lower index) or DIRB200_EOVERFLOW.  The tensor-core pass
may drop a row only when a band of 2*eps16 below the (fp16-path) k-th score proves it cannot be in the top-k.  The
adversarial pair below sits just inside that band: with eps16 large enough the result must be exact, with eps16 a
little smaller it must visibly lose the row - so a kernel that applies a narrower band than intended fails here.
GPU tests are marked `gpu`; the check of the construction itself runs on the CPU."""
import functools

import numpy as np
import pytest
import torch

import search_model as M
from oracle import dir_oracle as O
from conftest import rel_l2

gpu = pytest.mark.gpu
DEV = "cuda:0"

# ------------------------------------------------------------------------------------------ adversarial rounding pair
# D = 1024, b = 2^-5, m = b + 2^-16 (an fp16 rounding midpoint), t = 2^-26.  q rounds DOWN on [0, 510) and UP on
# [510, 1020); row A lives where q rounds down, row B where it rounds up.  All values are exact in fp32 and the fp16-path
# products are exact in fp32, so the reversal does not depend on the accumulation order.
ADV_D = 1024
EPS_NARROW = 4e-4     # band 8e-4  < the 9.65e-4 fp16-path reversal: the pass MUST lose A (proves the test sees the band)
EPS_TIGHT = 5e-4      # band 1e-3  > the reversal, and still >= |fp16-path - exact| of A and B: the result must be exact
EPS_DEFAULT = 1.2e-3  # the library default
EPS_ALL = [EPS_NARROW, EPS_TIGHT, EPS_DEFAULT]


def adversarial_pair():
    b, t = 2.0 ** -5, 2.0 ** -26
    m = b + 2.0 ** -16
    q = np.zeros(ADV_D, np.float32)
    q[:510], q[510:1020], q[1020] = m - t, m + t, b
    a = np.zeros(ADV_D, np.float32)
    a[:510], a[1020] = m - t, 2.0 ** -12          # 2^-12 is on the fp16 grid: a small, exact lead of A over B
    bb = np.zeros(ADV_D, np.float32)
    bb[510:1020] = m + t
    return q, a, bb


def test_adversarial_pair_reverses_the_order_inside_the_band():
    """CPU: the construction keeps its edge.  Exact scores rank A first by 6.7e-6; the fp16 path ranks B first by
    9.65e-4 - between the narrow band (8e-4) and the tight one (1e-3).  Each fp16-path score is off by 4.86e-4 <
    EPS_TIGHT, so eps16 = 5e-4 is still a valid error bound and the search must be exact with it.  For the rank
    counts: B's fp16-path score lies 4.8e-4 above s_A, outside +-EPS_NARROW but inside +-EPS_TIGHT."""
    q, a, b = adversarial_pair()
    m, t = 2.0 ** -5 + 2.0 ** -16, 2.0 ** -26
    assert float(q[0]) == m - t and float(q[510]) == m + t and float(b[1019]) == m + t    # exact in fp32
    assert 0.998 < np.linalg.norm(q.astype(np.float64)) <= 1.0
    q16 = q.astype(np.float16).astype(np.float64)
    assert np.all(q16[:510] == 2.0 ** -5) and np.all(q16[510:1020] == 2.0 ** -5 + 2.0 ** -15)   # down / up
    ex = M.exact_scores(q[None], np.stack([a, b]))[0]
    fa, fb = M.fast_scores(q[None], np.stack([a, b]))[0].astype(np.float64)
    assert 6.0e-6 < ex[0] - ex[1] < 7.5e-6                                                # exact: A before B
    rev = fb - fa                                                                         # fp16 path: B before A
    assert 2 * EPS_NARROW + 1e-4 < rev < 2 * EPS_TIGHT - 2e-5, rev
    assert max(abs(fa - ex[0]), abs(fb - ex[1])) < EPS_TIGHT - 1e-5
    assert EPS_NARROW + 5e-5 < fb - ex[0] < EPS_TIGHT - 1e-5
    # the model of the algorithm shows the same split: narrow band -> B replaces A, tight band -> exact
    rng = np.random.default_rng(0)
    db = _unit(rng.standard_normal((200, ADV_D), dtype=np.float32))
    strong = _near(rng, q, np.linspace(0.95, 0.7, 4))
    db[[10, 50, 90, 130]], db[170], db[180] = strong, a, b
    ref_s, ref_i = M.exact_topk(q[None], db, 5)
    assert ref_i[0, 4] == 170
    band0 = M.BAND
    try:
        for eps, want_a in ((EPS_NARROW, False), (EPS_TIGHT, True), (EPS_DEFAULT, True)):
            M.BAND = np.float32(2 * eps)
            _, got_i, _ = M.sharded_search(q[None], db, 5, [(0, 200)], sample_rows=4096)
            assert (got_i[0, 4] == 170) == want_a and (want_a or got_i[0, 4] == 180)
    finally:
        M.BAND = band0


# ------------------------------------------------------------------------------------------------------- helpers
def _ops():
    from dirb200 import ops
    ops.require_gpu(0)
    return ops


def _unit(x):
    x = np.asarray(x, np.float64)
    return (x / np.linalg.norm(x, axis=-1, keepdims=True)).astype(np.float32)


def _near(rng, q, cos):
    """Unit rows at the given cosines to q (random directions orthogonal to it for the rest)."""
    u = q.astype(np.float64) / np.linalg.norm(q.astype(np.float64))
    cos = np.asarray(cos, np.float64)
    noise = rng.standard_normal((cos.shape[0], u.shape[0]))
    noise -= (noise @ u)[:, None] * u
    noise /= np.linalg.norm(noise, axis=1, keepdims=True)
    return _unit(cos[:, None] * u + np.sqrt(1 - cos * cos)[:, None] * noise)


def _exact_topk(q, db, k):
    """search_model.exact_topk in row chunks: one fp64 reduction per (query, row) whose bits depend only on the two
    vectors, so exact duplicates tie exactly (the GPU's exact scores have the same property)."""
    n = db.shape[0]
    ex = np.empty((q.shape[0], n))
    step = max(1, (1 << 22) // max(1, q.shape[0] * db.shape[1]))
    for a in range(0, n, step):
        ex[:, a:a + step] = M.exact_scores(q, db[a:a + step])
    out_s = np.full((q.shape[0], k), -np.inf)
    out_i = np.full((q.shape[0], k), -1, np.int64)
    for i in range(q.shape[0]):
        order = np.lexsort((np.arange(n), -ex[i]))[:k]
        out_s[i, :order.shape[0]] = ex[i][order]
        out_i[i, :order.shape[0]] = order
    return out_s, out_i


def _ref(q, db, k):
    """Oracle top-k padded to k columns with (-inf, -1) when k > N."""
    rs, ri = O.topk(q, db, k)
    out_s = np.full((q.shape[0], k), -np.inf)
    out_i = np.full((q.shape[0], k), -1, np.int64)
    out_s[:, :rs.shape[1]], out_i[:, :ri.shape[1]] = rs, ri
    return out_s, out_i


def _assert_exact(s, i, ref_s, ref_i):
    s, i = (s.cpu().numpy(), i.cpu().numpy()) if isinstance(s, torch.Tensor) else (s, i)
    np.testing.assert_array_equal(i, ref_i)                                # indices bit-exact, -1 tails included
    fin = ref_i >= 0
    np.testing.assert_allclose(s[fin], ref_s[fin], rtol=0, atol=1e-12)
    assert np.all(np.isneginf(s[~fin]))


def _set_options(index, opts):
    for key, v in opts.items():
        index.set_option(key, v)


def _bounds(sizes):
    b = np.concatenate([[0], np.cumsum(sizes)]).astype(np.int64)
    return list(zip(b[:-1].tolist(), b[1:].tolist()))


def _two_phase(ops, shards, qd, k, c, packed=False):
    """dist.ShardedIndex.search with the collectives done in-process: phase 1 per shard, MIN of the selection
    thresholds, phase 2 per shard, merge of the lists (topk_merge, or topk_merge_packed on the all-gather layout)."""
    sel = torch.stack([sh.search_begin(qd, k, c) for sh in shards]).min(dim=0).values.contiguous()
    if packed:
        buf = torch.empty((len(shards), 2, qd.shape[0], k), dtype=torch.int64, device=DEV)
        for j, sh in enumerate(shards):
            sh.search_finish(qd, k, sel, out=buf[j])
        return ops.topk_merge_packed(buf, k)
    outs = [sh.search_finish(qd, k, sel) for sh in shards]
    return ops.topk_merge(torch.stack([o[0] for o in outs]).contiguous(), torch.stack([o[1] for o in outs]).contiguous(), k)


def _peer_search(shards, xs, qd, k, c):
    """One sharded search over the peer-memory exchange, all ranks driven phase by phase from this process.  Every
    shard's status is collected (an uncollected error would make that shard refuse the next search); the first error
    is raised after all of them were read."""
    for ph in (1, 2, 3):
        for sh, x in zip(shards, xs):
            sh.search_sharded(x, qd, k, c, phase=ph)
    res = [sh.search_sharded(x, qd, k, c, phase=4) for sh, x in zip(shards, xs)]
    err = None
    for sh in shards:
        try:
            sh.check()
        except Exception as e:          # noqa: BLE001 - re-raised below
            err = err or e
    if err is not None:
        raise err
    return res


def _peer_group(ops, shards, nq, k, eps=None):
    G = len(shards)
    xs = [ops.Exchange(0, G, r, nq, k) for r in range(G)]
    ops.Exchange.open_local(xs)
    for sh in shards:
        sh.set_option("deferred_check", 1)
        if eps is not None:
            sh.set_option("eps16", eps)
    return xs


def _close(xs):
    torch.cuda.synchronize()
    for x in xs:
        x.close()


# ---------------------------------------------------------------------------------- a. the band, on every path
@functools.lru_cache(maxsize=None)
def _adv_case(n, k, layout, seed=0):
    """q[0] = the adversarial query (+ 2 random queries); a random unit-norm database with k-1 rows far above A and B
    (cosines 0.6 .. 0.95), A and B at ranks k and k+1 of the exact order, B at rank k of the fp16-path order.
    layout 'spread': the k+1 planted rows evenly over the rows; 'groups': one per group of 32 rows from row 0 (the
    group-max seed then sees each of them as its own group maximum); 'tail': all after row 2048 (outside a small
    seed sample, so that the seed threshold is loose and the candidate lists overflow).
    -> (q, db, row of A, row of B)."""
    rng = np.random.default_rng(seed)
    qa, a, b = adversarial_pair()
    db = _unit(rng.standard_normal((n, ADV_D), dtype=np.float32))
    if layout == "groups":
        pos = 32 * np.arange(k + 1) + (5 * np.arange(k + 1)) % 32
    elif layout == "tail":
        pos = np.linspace(2048, n - 1, k + 1).astype(np.int64)
    else:
        pos = np.linspace(0, n - 1, k + 1).astype(np.int64)
    assert len(set(pos.tolist())) == k + 1 and pos.max() < n
    perm = rng.permutation(k + 1)
    i_a, i_b, strong = int(pos[perm[0]]), int(pos[perm[1]]), pos[perm[2:]]
    db[strong] = _near(rng, qa, np.linspace(0.95, 0.6, k - 1))
    db[i_a], db[i_b] = a, b
    q = np.concatenate([qa[None], _unit(rng.standard_normal((2, ADV_D), dtype=np.float32))])
    return q, db, i_a, i_b


def _check_band(s, i, ref_s, ref_i, k, i_a, i_b, eps):
    assert ref_i[0, k - 1] == i_a and i_b not in ref_i[0]                 # the construction: A is the k-th row
    s, i = s.cpu().numpy(), i.cpu().numpy()
    _assert_exact(s[1:], i[1:], ref_s[1:], ref_i[1:])                     # the random queries are exact at any eps
    if eps == EPS_NARROW:
        # a band narrower than the reversal loses A and returns B in its place: the test can see the band
        _assert_exact(s[:1, :k - 1], i[:1, :k - 1], ref_s[:1, :k - 1], ref_i[:1, :k - 1])
        assert i[0, k - 1] == i_b, "a band of %g should have dropped row A (%d): got %d" % (2 * eps, i_a, i[0, k - 1])
    else:
        _assert_exact(s[:1], i[:1], ref_s[:1], ref_i[:1])


# name -> (N, k, layout, options, expected seed rows (dense_rows) or None)
BAND_PATHS = {
    "small": (3000, 10, "spread", {}, 3000),                     # N <= S: dense scores of every row
    "group_max_seed": (40000, 100, "groups", {}, 8192),          # S = 8192 rows, S/32 >= k: seed from group maxima
    "dense_seed": (20000, 1024, "spread", {}, 20000),            # 256 < k, 8192 < N < 32k: S = N, dense seed + filter
    "overflow_retry": (60000, 50, "tail", {"sample_rows": 256, "cand_cap": 512, "retries": 3}, None),
}


@gpu
@pytest.mark.parametrize("eps", EPS_ALL)
@pytest.mark.parametrize("path", list(BAND_PATHS))
def test_band_single_index(path, eps):
    ops = _ops()
    n, k, layout, opts, dense_rows = BAND_PATHS[path]
    q, db, i_a, i_b = _adv_case(n, k, layout)
    ref_s, ref_i = O.topk(q, db, k)
    index = ops.Index(torch.from_numpy(db).to(DEV))
    _set_options(index, opts)
    index.set_option("eps16", eps)
    s, i = index.search(torch.from_numpy(q).to(DEV), k)
    st = index.stats()
    if dense_rows is not None:
        assert st["dense_rows"] == dense_rows, st
    if path == "overflow_retry":
        assert st["retries"] >= 1, st                                    # the gated retry passes did run
    _check_band(s, i, ref_s, ref_i, k, i_a, i_b, eps)


@functools.lru_cache(maxsize=None)
def _adv_sharded_case(k=20, sizes=(5000, 7000)):
    """Two shards, A in shard 0 and B in shard 1.  With c = shard_quota(k, sizes) = k/2: shard 0 holds c strong rows
    (its c-th best is far above B), shard 1 holds c-1 strong rows + B (its c-th best IS B's fp16-path score), so the
    MIN over the shards is B's score and shard 0 must keep A within the band of a threshold set by another shard."""
    rng = np.random.default_rng(1)
    qa, a, b = adversarial_pair()
    n0, n1 = sizes
    db = _unit(rng.standard_normal((n0 + n1, ADV_D), dtype=np.float32))
    c = k // 2
    strong = _near(rng, qa, np.linspace(0.95, 0.6, k - 1))
    p0 = np.linspace(0, n0 - 1, c + 1).astype(np.int64)
    p1 = n0 + np.linspace(0, n1 - 1, c).astype(np.int64)
    db[p0[:-1]], db[p1[:-1]] = strong[:c], strong[c:]
    i_a, i_b = int(p0[-1]), int(p1[-1])
    db[i_a], db[i_b] = a, b
    q = np.concatenate([qa[None], _unit(rng.standard_normal((2, ADV_D), dtype=np.float32))])
    return q, db, i_a, i_b


@gpu
@pytest.mark.parametrize("eps", EPS_ALL)
@pytest.mark.parametrize("proto", ["two_phase", "peer_exchange"])
def test_band_sharded(proto, eps):
    ops = _ops()
    from dirb200.dist import shard_quota
    k, sizes = 20, (5000, 7000)
    q, db, i_a, i_b = _adv_sharded_case(k, sizes)
    c = shard_quota(k, list(sizes))
    assert c == k // 2
    ref_s, ref_i = O.topk(q, db, k)
    dbt, qd = torch.from_numpy(db).to(DEV), torch.from_numpy(q).to(DEV)
    shards = [ops.Index(dbt[a:b].contiguous(), index_offset=a) for a, b in _bounds(sizes)]
    if proto == "two_phase":
        for sh in shards:
            sh.set_option("eps16", eps)
        s, i = _two_phase(ops, shards, qd, k, c)
        _check_band(s, i, ref_s, ref_i, k, i_a, i_b, eps)
        return
    xs = _peer_group(ops, shards, q.shape[0], k, eps)
    try:
        for _ in range(2):                                             # both parities of the exchange slots
            for s, i in _peer_search(shards, xs, qd, k, c):
                _check_band(s, i, ref_s, ref_i, k, i_a, i_b, eps)
    finally:
        _close(xs)


@gpu
@pytest.mark.parametrize("eps", EPS_ALL)
def test_band_rank_counts(eps):
    """rank_counts with A as a positive: B's fp16-path score is above s_A but its exact score is below - it must be
    re-scored, not counted as ranking before A."""
    ops = _ops()
    k = 10
    q, db, i_a, i_b = _adv_case(3000, k, "spread")
    strong = int(O.topk(q[:1], db, 1)[1][0, 0])
    rows_q = [sorted([strong, i_a, i_b]), [5, 17, 2999], [0, 1234]]
    offs = np.array([0] + list(np.cumsum([len(r) for r in rows_q])), np.int32)
    rows = np.array(sum(rows_q, []), np.int64)
    flags = np.array([0 if r == i_b else 1 for r in rows_q[0]] + [1, 1, 1, 1, 0], np.uint8)
    ref_s, ref_a = O.rank_counts(q, db, offs, rows)
    index = ops.Index(torch.from_numpy(db).to(DEV))
    index.set_option("eps16", eps)
    sc, above = index.rank_counts(torch.from_numpy(q).to(DEV), offs, rows, flags)
    sc, above = sc.cpu().numpy(), above.cpu().numpy()
    np.testing.assert_allclose(sc, ref_s, rtol=0, atol=1e-12)
    m = flags == 1
    t_a = int(np.nonzero(rows[:3] == i_a)[0][0])
    assert ref_a[t_a] == k - 1                                          # the k-1 strong rows, not B
    if eps == EPS_NARROW:
        assert above[t_a] == ref_a[t_a] + 1                             # B counted from its fp16-path score alone
        keep = m.copy()
        keep[t_a] = False
        np.testing.assert_array_equal(above[keep], ref_a[keep])
    else:
        np.testing.assert_array_equal(above[m], ref_a[m])


# ------------------------------------------------------------------ b. kernels against the model's data kinds
@functools.lru_cache(maxsize=None)
def _kind_case(kind, n, dim, seed=0):
    """The data families of tests/test_properties.py at sizes the kernels tile."""
    rng = np.random.RandomState(seed + 1000 * n + dim)
    nq = 5
    q = _unit(rng.standard_normal((nq, dim)))
    if kind in ("random", "skewed"):
        db = _unit(rng.standard_normal((n, dim)))
        if kind == "skewed":                                            # the first rows (one shard) are all good matches
            m = max(1, n // 6)
            db[:m] = _unit(q[rng.randint(0, nq, m)] + 0.2 * rng.standard_normal((m, dim)))
    elif kind == "duplicates":                                          # few distinct rows, many exact copies
        base = _unit(rng.standard_normal((max(1, n // 20), dim)))
        db = base[rng.randint(0, base.shape[0], n)]
    elif kind == "clustered":                                           # scores packed within a fraction of the band
        db = _unit(q[0][None, :] + 2e-3 * rng.standard_normal((n, dim)))
    else:                                                               # planted: a few strong matches in a random crowd
        db = _unit(rng.standard_normal((n, dim)))
        for j in rng.randint(0, n, min(n, 8)):
            db[j] = _unit((q[rng.randint(nq)] + 0.3 * rng.standard_normal(dim))[None])[0]
    return q, np.ascontiguousarray(db)


KINDS = ["random", "planted", "duplicates", "clustered", "skewed"]
KIND_SHAPES = [(255, 64), (256, 192), (257, 1024), (513, 64), (4097, 192), (9000, 64)]


def _exact_or_overflow(kind, fn, ref_s, ref_i):
    """The contract: the exact list, or DIRB200_EOVERFLOW (-4) - which random and planted data never need."""
    from dirb200.lib import DirbError
    try:
        res = fn()
    except DirbError as e:
        assert e.status == -4, e
        assert kind not in ("random", "planted"), "%s data must never overflow: %s" % (kind, e)
        return False
    for s, i in (res if isinstance(res, list) else [res]):
        _assert_exact(s, i, ref_s, ref_i)
    return True


@gpu
@pytest.mark.parametrize("n,dim", KIND_SHAPES, ids=lambda v: str(v))
@pytest.mark.parametrize("kind", KINDS)
def test_kernels_match_model_data(kind, n, dim):
    ops = _ops()
    from dirb200.dist import shard_quota
    k = 40
    q, db = _kind_case(kind, n, dim)
    ref_s, ref_i = _exact_topk(q, db, k)
    dbt, qd = torch.from_numpy(db).to(DEV), torch.from_numpy(q).to(DEV)
    for sample in (0, 256):                                             # default (N <= S: small path) / group-max seed
        index = ops.Index(dbt)
        if sample:
            index.set_option("sample_rows", sample)
        _exact_or_overflow(kind, lambda: index.search(qd, k), ref_s, ref_i)
    sizes = [n // 3, 0, n - n // 3 - 7, 7]                              # uneven, empty, smaller than k
    c = shard_quota(k, sizes)
    shards = [ops.Index(dbt[a:b].contiguous(), index_offset=a) for a, b in _bounds(sizes)]
    for sh in shards:
        sh.set_option("sample_rows", 256)
    _exact_or_overflow(kind, lambda: _two_phase(ops, shards, qd, k, c), ref_s, ref_i)
    shards = [ops.Index(dbt[a:b].contiguous(), index_offset=a) for a, b in _bounds(sizes)]
    for sh in shards:
        sh.set_option("sample_rows", 256)
    xs = _peer_group(ops, shards, q.shape[0], k)
    try:
        for _ in range(3):
            if not _exact_or_overflow(kind, lambda: _peer_search(shards, xs, qd, k, c), ref_s, ref_i):
                break
    finally:
        _close(xs)


# ---------------------------------------------------------------------------------------- c. k, Q and dim limits
def _random_case(n, nq, dim, seed):
    rng = np.random.default_rng(seed)
    db = _unit(rng.standard_normal((n, dim), dtype=np.float32))
    q = _unit(rng.standard_normal((nq, dim), dtype=np.float32))
    hit = rng.integers(0, n, nq)
    q[: nq // 2] = _unit(db[hit[: nq // 2]] + 0.5 * q[: nq // 2])     # half the queries have a close neighbour
    return q, db


# (k, N, Q, dim, seed rows S the search must pick): S = N and N <= 8192 -> small path; S/32 >= k -> group-max seed;
# otherwise dense seed over S rows + filter pass over all N
K_CASES = [
    (1, 3000, 129, 64, 3000),
    (255, 3000, 128, 192, 3000),
    (256, 3000, 127, 64, 3000),
    (257, 9000, 1, 1024, 8224),          # group-max seed with exactly k groups (S = 32 k)
    (1000, 600, 3, 64, 600),             # k > N: (-inf, -1) tail
    (1024, 1024, 2, 128, 1024),          # k = N
    (1024, 20000, 4, 64, 20000),         # dense seed, S = N > 8192
    (1024, 9000, 129, 64, 9000),         # dense seed, Q > one 128-row query tile
    (1000, 100000, 2, 64, 32000),        # group-max seed, S = 32 k
]


@gpu
@pytest.mark.parametrize("k,n,nq,dim,S", K_CASES, ids=lambda v: str(v))
def test_k_q_dim_limits(k, n, nq, dim, S):
    ops = _ops()
    q, db = _random_case(n, nq, dim, seed=k + n)
    ref_s, ref_i = _ref(q, db, k)
    index = ops.Index(torch.from_numpy(db).to(DEV))
    s, i = index.search(torch.from_numpy(q).to(DEV), k)
    assert index.stats()["dense_rows"] == S, index.stats()
    _assert_exact(s, i, ref_s, ref_i)


@gpu
@pytest.mark.parametrize("k,sizes", [(1000, (300, 0, 6000, 2000)), (1024, (2500, 2500, 2500, 2500)), (257, (100, 9000))],
                         ids=lambda v: str(v))
def test_large_k_sharded(k, sizes):
    """k up to 1024 over shards smaller than k (and empty): two-phase protocol with both merge entry points and the
    peer exchange - merges of G*k = 4000 / 4096 entries."""
    ops = _ops()
    from dirb200.dist import shard_quota
    q, db = _random_case(sum(sizes), 5, 64, seed=k)
    ref_s, ref_i = _ref(q, db, k)
    dbt, qd = torch.from_numpy(db).to(DEV), torch.from_numpy(q).to(DEV)
    c = shard_quota(k, list(sizes))
    shards = [ops.Index(dbt[a:b].contiguous(), index_offset=a) for a, b in _bounds(sizes)]
    for packed in (False, True):
        s, i = _two_phase(ops, shards, qd, k, c, packed=packed)
        _assert_exact(s, i, ref_s, ref_i)
    xs = _peer_group(ops, shards, q.shape[0], k)
    try:
        for _ in range(3):
            for s, i in _peer_search(shards, xs, qd, k, c):
                _assert_exact(s, i, ref_s, ref_i)
    finally:
        _close(xs)


def _tied_case(k, n_tied, n=8000, dim=64):
    """k-1 strong rows (distinct, cosines 0.98 .. 0.85) and n_tied exact copies of one row at cosine 0.75 in a random
    crowd: rank k is a tie of n_tied rows, all of which survive the band."""
    rng = np.random.default_rng(k)
    q = _unit(rng.standard_normal((2, dim), dtype=np.float32))
    db = _unit(rng.standard_normal((n, dim), dtype=np.float32))
    pos = rng.permutation(n)[: k - 1 + n_tied]
    db[pos[: k - 1]] = _near(rng, q[0], np.linspace(0.98, 0.85, k - 1))
    db[pos[k - 1:]] = _near(rng, q[0], [0.75])[0]
    return q, db


@gpu
@pytest.mark.parametrize("k,n_tied,fits", [(256, 1100, False), (257, 1100, True), (1024, 2100, False)])
def test_survivor_capacity_switch_at_k_256(k, n_tied, fits):
    """The re-scoring keeps 1024 survivors per query for k <= 256 and 2048 above.  More tied rows than that must end in
    DIRB200_EOVERFLOW; fewer must give the exact list, ties broken by index."""
    ops = _ops()
    from dirb200.lib import DirbError
    q, db = _tied_case(k, n_tied)
    index = ops.Index(torch.from_numpy(db).to(DEV))
    qd = torch.from_numpy(q).to(DEV)
    if not fits:
        with pytest.raises(DirbError) as e:
            index.search(qd, k)
        assert e.value.status == -4 and "eps16" in str(e.value)
        return
    s, i = index.search(qd, k)
    ref_s, ref_i = _exact_topk(q, db, k)
    tied = np.nonzero((db == db[ref_i[0, k - 1]]).all(axis=1))[0]
    assert tied.shape[0] == n_tied and ref_i[0, k - 1] == tied.min()      # the lowest-index copy wins the tie
    _assert_exact(s, i, ref_s, ref_i)


# ----------------------------------------------------------------------------------------------- d. merge limits
def _shard_lists(G, nq, k, seed):
    """G ordered per-shard lists (score desc, index asc) per query with ties across shards (scores on a 1/64 grid),
    distinct global indices and (-inf, -1) tails of random length (some lists empty, some full)."""
    rng = np.random.default_rng(seed)
    sc = np.full((G, nq, k), -np.inf)
    ix = np.full((G, nq, k), -1, np.int64)
    for qi in range(nq):
        ids = rng.permutation(G * k * 4)[: G * k]
        for g in range(G):
            nv = int(rng.choice([0, k, int(rng.integers(0, k + 1))]))
            s = np.round(rng.uniform(-1, 1, nv) * 64) / 64
            i = ids[g * k: g * k + nv]
            o = np.lexsort((i, -s))
            sc[g, qi, :nv], ix[g, qi, :nv] = s[o], i[o]
    return sc, ix


@gpu
@pytest.mark.parametrize("G,k", [(3, 1024), (7, 439), (4, 1024), (8, 512), (64, 64), (1, 1024)], ids=lambda v: str(v))
def test_merge_at_the_shared_memory_limit(G, k):
    """topk_merge / topk_merge_packed hold G*k 16-byte entries per query in shared memory; the entry points accept
    G*k <= 4096.  3072 entries fill the 48 KiB a launch gets by default (with the kernel's static shared variable: more
    than that), 3073 is one above, 4096 the maximum."""
    ops = _ops()
    nq = 6
    sc, ix = _shard_lists(G, nq, k, seed=G * k)
    ref_s, ref_i = O.merge_topk(list(sc), list(ix), k)
    ms, mi = ops.topk_merge(torch.from_numpy(sc).to(DEV), torch.from_numpy(ix).to(DEV), k)
    _assert_exact(ms, mi, ref_s, ref_i)
    packed = np.stack([sc.view(np.int64), ix], axis=1)                 # (G, 2, Q, k): score bits, indices
    ms, mi = ops.topk_merge_packed(torch.from_numpy(np.ascontiguousarray(packed)).to(DEV), k)
    _assert_exact(ms, mi, ref_s, ref_i)


@gpu
def test_merge_refuses_more_than_4096_entries():
    ops = _ops()
    from dirb200.lib import DirbError
    sc, ix = _shard_lists(2, 2, 2049, seed=0)
    with pytest.raises(DirbError) as e:
        ops.topk_merge(torch.from_numpy(sc).to(DEV), torch.from_numpy(ix).to(DEV), 2049)
    assert e.value.status == -2
    with pytest.raises(DirbError):
        ops.Exchange(0, 8, 0, 4, 513)                                   # world * max_k > 4096


@gpu
def test_peer_exchange_world8_k512():
    """The largest merge of the peer path (8 x 512 entries) on one GPU, several searches in a row so that both slot
    parities are used after it - a merge that failed to launch would leave the epoch behind and the next search would
    read stale tables."""
    ops = _ops()
    from dirb200.dist import shard_quota
    G, k, n_per = 8, 512, 2000
    rng = np.random.default_rng(8)
    db = _unit(rng.standard_normal((G * n_per, 64), dtype=np.float32))
    qs = [_unit(rng.standard_normal((9, 64), dtype=np.float32)) for _ in range(2)]
    refs = [_ref(q, db, k) for q in qs]
    dbt = torch.from_numpy(db).to(DEV)
    sizes = [n_per] * G
    c = shard_quota(k, sizes)
    shards = [ops.Index(dbt[a:b].contiguous(), index_offset=a) for a, b in _bounds(sizes)]
    xs = _peer_group(ops, shards, 9, k)
    try:
        for j in (0, 1, 0, 1):
            qd = torch.from_numpy(qs[j]).to(DEV)
            for s, i in _peer_search(shards, xs, qd, k, c):
                _assert_exact(s, i, *refs[j])
    finally:
        _close(xs)


# ------------------------------------------------------------------------------------------- e. alpha-QE, large k
@gpu
@pytest.mark.parametrize("k", [1024, 2048])
@pytest.mark.parametrize("alpha", [0.5, 3.0])
def test_aqe_expand_large_k(k, alpha):
    """aqe_expand at k = 1024 and at its maximum 2048, with -1 entries (a fully empty list, a -1 tail, scattered -1):
    normalize(q + sum_j db[idx_j] * s_j^alpha) in fp64; the per-shard partial sums add up to the same expansion."""
    ops = _ops()
    rng = np.random.default_rng(k)
    n, dim, nq = 5000, 256, 6
    db = _unit(rng.standard_normal((n, dim), dtype=np.float32))
    q = _unit(rng.standard_normal((nq, dim), dtype=np.float32))
    idx = np.stack([rng.permutation(n)[:k] for _ in range(nq)]).astype(np.int64)
    sc = rng.uniform(0.05, 1.0, (nq, k))
    idx[0] = -1                                                         # no neighbour at all: the normalised query
    idx[1, k // 3:] = -1                                                # a -1 tail
    idx[2, rng.random(k) < 0.2] = -1                                    # scattered -1
    ref = q.astype(np.float64).copy()
    for r in range(nq):
        ok = idx[r] >= 0
        ref[r] += (db[idx[r][ok]].astype(np.float64) * (sc[r][ok] ** alpha)[:, None]).sum(axis=0)
    ref /= np.linalg.norm(ref, axis=1, keepdims=True)
    dbt, qd = torch.from_numpy(db).to(DEV), torch.from_numpy(q).to(DEV)
    it, st = torch.from_numpy(idx).to(DEV), torch.from_numpy(sc).to(DEV)
    out = ops.aqe_expand(qd, dbt, it, st, alpha)
    assert rel_l2(out.cpu().numpy(), ref) < 1e-5
    np.testing.assert_allclose(out.cpu().numpy()[0], q[0], rtol=0, atol=1e-6)
    cut = 1777
    part = torch.zeros_like(qd)
    for a, b in ((0, cut), (cut, n)):
        part += ops.aqe_expand(qd, dbt[a:b].contiguous(), it, st, alpha, partial=True, row_offset=a, n_rows=b - a)
    both = ops.pool_scales([part, qd], "mean", l2=True)
    assert rel_l2(both.cpu().numpy(), ref) < 1e-5
