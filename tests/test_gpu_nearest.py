"""fks_nearest_configurations on the device against the nearest reference (tests/nearest_reference.py), fed the distances
fks_end_states_pairwise_distance returns over records that hold the candidates and then the queries (entry [i][m + j]).
Ids and distance bits must match exactly, on both kernel paths, for every k, on repeated calls and on another stream."""
import numpy as np
import pytest
import torch

from fast_kinematic_simulator_b200 import capi, workloads as W

import device_records as DR
import nearest_reference as NR

pytestmark = pytest.mark.gpu

MAX_K = 64
MIN_CHUNK = 2048  # fewest candidates per chunk of a split (fks_consumers.cu)
PAIRWISE_MAX = 16384  # records per pairwise call here: a 2 GiB matrix


def _split_switch():
    """Fewest queries that take the query-tiled path whatever m: more than 2 * 8 queries per SM (fks_consumers.cu)."""
    return 16 * torch.cuda.get_device_properties(0).multi_processor_count + 1


def gpu_distances(sim, cand, queries, query_rows=None):
    """The m x len(query_rows) block [i][m + j] of the pairwise matrix over records (candidates, then queries), in calls
    over subsets of the records: candidate chunks together with the chosen queries."""
    m, n_q = len(cand), len(queries)
    rows = np.arange(n_q) if query_rows is None else np.asarray(query_rows)
    dr, _ = DR.records(sim, np.concatenate([cand, queries]) if m else queries)
    chunk = max(1, PAIRWISE_MAX - len(rows))
    out = np.empty((m, len(rows)))
    for c0 in range(0, m, chunk):
        c = min(chunk, m - c0)
        ids = np.concatenate([np.arange(c0, c0 + c), m + rows])
        mat = torch.empty(len(ids), len(ids), dtype=torch.float64, device="cuda")
        sim.end_states_pairwise_distance(dr, len(ids), mat, DR.u32(ids), stream=DR.stream())
        out[c0:c0 + c] = mat[:c, c:].cpu().numpy()
    torch.cuda.synchronize()
    return out


def run_nearest(sim, d_cand, m, d_q, n_q, k, stream=None):
    ids = torch.full((max(n_q * k, 1),), -7, dtype=torch.int32, device="cuda")
    dist = torch.full((max(n_q * k, 1),), -7.0, dtype=torch.float64, device="cuda")
    sim.nearest_configurations(d_cand, m, d_q, n_q, k, ids, dist, stream=stream if stream is not None else DR.stream())
    return ids, dist


def host(ids, dist, n_q, k):
    torch.cuda.synchronize()
    return ids.cpu().numpy().view(np.uint32)[:n_q * k].reshape(n_q, k), dist.cpu().numpy()[:n_q * k].reshape(n_q, k)


def check(sim, cand, queries, k, dist_matrix=None, query_rows=None, expect_launches=None):
    """GPU answer against the reference fed the GPU pairwise distances; returns the GPU ids and distances."""
    cand = np.ascontiguousarray(cand, dtype=np.float64).reshape(-1, sim.config_stride)
    queries = np.ascontiguousarray(queries, dtype=np.float64).reshape(-1, sim.config_stride)
    m, n_q = len(cand), len(queries)
    d_cand = torch.from_numpy(cand).cuda() if m else None
    d_q = torch.from_numpy(queries).cuda()
    before = sim.launch_count
    got = host(*run_nearest(sim, d_cand, m, d_q, n_q, k), n_q, k)
    if expect_launches is not None:
        assert sim.launch_count - before == expect_launches
    if dist_matrix is None:
        dist_matrix = gpu_distances(sim, cand, queries, query_rows)
    want = NR.nearest(dist_matrix, k)
    rows = slice(None) if query_rows is None else np.asarray(query_rows)
    assert np.array_equal(got[0][rows], want[0]), int(np.sum(got[0][rows] != want[0]))
    assert got[1][rows].tobytes() == want[1].tobytes()
    return got, dist_matrix


def _end_states(name, n):
    w = W.make(name, n_particles=n)
    sim = w.make_simulator()
    out = sim.forward_simulate_robots(w.starts, w.targets, True, capi.NOISE_PHILOX)
    return sim, np.ascontiguousarray(out.records["cfg"]).reshape(n, sim.config_stride)


@pytest.mark.parametrize("name", ["se2_arena", "se3_narrow_passage", "arm_table"])
def test_workload_end_states_as_candidates(name):
    n = 3000
    sim, cfg = _end_states(name, n + 400)
    cand = cfg[:n]
    # queries: other end states, candidates themselves (distance 0, duplicates of one another) and the first end state
    queries_all = np.concatenate([cfg[n:], cand[::7][:40], np.repeat(cand[:1], 3, axis=0)])
    switch = _split_switch()
    dist_all = gpu_distances(sim, cand, queries_all)
    for n_q in (1, 5, 300, len(queries_all)):
        for k in (1, 7, 32, MAX_K):
            check(sim, cand, queries_all[:n_q], k, dist_matrix=dist_all[:, :n_q], expect_launches=1 if n_q >= switch else 2)
    # the query-tiled path on the same candidates
    many = np.concatenate([queries_all] * (switch // len(queries_all) + 1))[:switch]
    dist_many = np.concatenate([dist_all] * (switch // len(queries_all) + 1), axis=1)[:, :switch]
    for k in (1, 7, 32, MAX_K):
        check(sim, cand, many, k, dist_matrix=dist_many, expect_launches=1)
    sim.close()


def _se2(n, rng, scale=10.0):
    return np.stack([rng.uniform(0, scale, n), rng.uniform(0, scale, n), rng.uniform(-np.pi, np.pi, n)], axis=1)


def _synthetic_sim():
    return W.make("se2_arena", n_particles=4).make_simulator()


def test_sizes_across_the_switch_between_the_paths():
    rng = np.random.default_rng(3)
    sim = _synthetic_sim()
    switch = _split_switch()
    queries = _se2(switch + 8, rng)
    for m in (1, 63, 64, MIN_CHUNK, MIN_CHUNK + 1, 3 * MIN_CHUNK + 5, 20000):
        cand = _se2(m, rng)
        dist = gpu_distances(sim, cand, queries)
        for n_q in (1, 2, 7, 8, 9, 100, switch - 1, switch):
            split = m > MIN_CHUNK and n_q < switch
            for k in (1, 33):
                check(sim, cand, queries[:n_q], k, dist_matrix=dist[:, :n_q], expect_launches=2 if split else 1)
    sim.close()


def test_one_query_against_2_20_candidates():
    rng = np.random.default_rng(20)
    sim = _synthetic_sim()
    m = 1 << 20
    cand = _se2(m, rng, scale=100.0)
    cand[rng.integers(0, m, 1000)] = cand[17]  # duplicates of one candidate
    queries = np.concatenate([cand[17:18], _se2(2, rng, scale=100.0)])
    dist = gpu_distances(sim, cand, queries)
    for n_q in (1, 3):
        for k in (1, 7, 32, MAX_K):
            got, _ = check(sim, cand, queries[:n_q], k, dist_matrix=dist[:, :n_q], expect_launches=2)
    assert got[1][0, 0] == 0.0 and got[0][0, 0] == np.flatnonzero(np.all(cand == cand[17], axis=1))[0]
    sim.close()


def test_4096_queries_against_65536_candidates_on_a_sample():
    rng = np.random.default_rng(4096)
    w = W.make("arm_table", n_particles=4)
    sim = w.make_simulator()
    stride = sim.config_stride
    m, n_q = 65536, 4096
    cand = rng.uniform(-np.pi, np.pi, (m, stride))
    queries = rng.uniform(-np.pi, np.pi, (n_q, stride))
    rows = np.sort(rng.choice(n_q, 96, replace=False))
    rows[0], rows[-1] = 0, n_q - 1
    for k in (1, 64):
        check(sim, cand, queries, k, query_rows=rows, expect_launches=1)
    sim.close()


def test_ties_duplicates_and_nan_configurations():
    rng = np.random.default_rng(21)
    sim = _synthetic_sim()
    m = 6000
    # SE(2) configurations on a small integer grid: most distances tie; some NaN
    cand = np.stack([rng.integers(0, 3, m), rng.integers(0, 3, m), rng.integers(-1, 2, m) * (np.pi / 2)], axis=1).astype(np.float64)
    cand[rng.random(m) < 0.05] = np.nan
    cand[rng.random(m) < 0.01, 2] = np.nan
    queries = np.stack([rng.integers(0, 3, 40), rng.integers(0, 3, 40), rng.integers(-1, 2, 40) * (np.pi / 2)], axis=1).astype(np.float64)
    queries[3] = np.nan  # every distance NaN: the first k candidates at +inf
    dist = gpu_distances(sim, cand, queries)
    for n_q in (1, 4, 40):
        for k in (1, 7, 32, MAX_K):
            got, _ = check(sim, cand, queries[:n_q], k, dist_matrix=dist[:, :n_q], expect_launches=2)
    assert got[0][3].tolist() == list(range(MAX_K)) and np.all(got[1][3] == np.inf)
    # the query-tiled path on the same candidates
    switch = _split_switch()
    reps = switch // len(queries) + 1
    many, dist_many = np.concatenate([queries] * reps)[:switch], np.concatenate([dist] * reps, axis=1)[:, :switch]
    for k in (7, MAX_K):
        check(sim, cand, many, k, dist_matrix=dist_many, expect_launches=1)
    # fewer candidates than k, all NaN among them: padding after the ranked +inf
    few = np.full((5, 3), np.nan)
    got, _ = check(sim, few, queries[:2], 7)
    assert got[0][0].tolist() == [0, 1, 2, 3, 4, 0xFFFFFFFF, 0xFFFFFFFF] and np.all(got[1] == np.inf)
    sim.close()


def test_repeated_calls_and_a_side_stream_agree():
    rng = np.random.default_rng(5)
    sim = _synthetic_sim()
    m = 50000
    cand = torch.from_numpy(_se2(m, rng, scale=4.0)).cuda()
    switch = _split_switch()
    qa = torch.from_numpy(_se2(switch, rng, scale=4.0)).cuda()
    qb = torch.from_numpy(_se2(3, rng, scale=4.0)).cuda()
    for n_q in (1, 16, switch):  # split (2 launches) and query-tiled (1)
        first = host(*run_nearest(sim, cand, m, qa, n_q, 40), n_q, 40)
        for _ in range(3):
            again = host(*run_nearest(sim, cand, m, qa, n_q, 40), n_q, 40)
            assert first[0].tobytes() == again[0].tobytes() and first[1].tobytes() == again[1].tobytes()
        side = torch.cuda.Stream()
        with torch.cuda.stream(side):
            on_side = host(*run_nearest(sim, cand, m, qa, n_q, 40, stream=side.cuda_stream), n_q, 40)
        assert first[0].tobytes() == on_side[0].tobytes() and first[1].tobytes() == on_side[1].tobytes()
    # two split calls in flight on two streams share the simulator's workspace
    want_a = host(*run_nearest(sim, cand, m, qa, 16, 64), 16, 64)
    want_b = host(*run_nearest(sim, cand, m, qb, 3, 64), 3, 64)
    s1, s2 = torch.cuda.Stream(), torch.cuda.Stream()
    torch.cuda.synchronize()
    with torch.cuda.stream(s1):
        a = run_nearest(sim, cand, m, qa, 16, 64, stream=s1.cuda_stream)
    with torch.cuda.stream(s2):
        b = run_nearest(sim, cand, m, qb, 3, 64, stream=s2.cuda_stream)
    got_a, got_b = host(*a, 16, 64), host(*b, 3, 64)
    for got, want in ((got_a, want_a), (got_b, want_b)):
        assert got[0].tobytes() == want[0].tobytes() and got[1].tobytes() == want[1].tobytes()
    sim.close()


def test_invalid_arguments_and_empty_calls():
    rng = np.random.default_rng(6)
    sim = _synthetic_sim()
    cand = torch.from_numpy(_se2(100, rng)).cuda()
    q = torch.from_numpy(_se2(4, rng)).cuda()
    ids = torch.empty(4 * MAX_K, dtype=torch.int32, device="cuda")
    dist = torch.empty(4 * MAX_K, dtype=torch.float64, device="cuda")

    def refused(**kw):
        args = dict(d_candidates=cand, m=100, d_queries=q, n_queries=4, k=3, d_ids=ids, d_distances=dist)
        args.update(kw)
        with pytest.raises(capi.FksError) as e:
            sim.nearest_configurations(**args)
        assert e.value.code == capi.ERR_INVALID_ARGUMENT

    refused(k=0)
    refused(k=MAX_K + 1)
    refused(k=0, n_queries=0)
    refused(m=2 ** 32)
    refused(n_queries=2 ** 26, k=MAX_K)  # n_queries * k = 2^32
    refused(n_queries=2 ** 32 // 3 + 1)
    for name in ("d_candidates", "d_queries", "d_ids", "d_distances"):
        refused(**{name: None})
    before = sim.launch_count
    # no queries: nothing to write, no launch, buffers may be null
    sim.nearest_configurations(None, 0, None, 0, 5, None, None)
    sim.nearest_configurations(cand, 100, None, 0, MAX_K, None, None)
    assert sim.launch_count == before
    # no candidates: one launch writes the padding, d_candidates may be null
    ids.fill_(-7)
    dist.fill_(-7.0)
    sim.nearest_configurations(None, 0, q, 4, 5, ids, dist)
    assert sim.launch_count == before + 1
    h_ids, h_dist = host(ids, dist, 4, 5)
    assert np.all(h_ids == 0xFFFFFFFF) and np.all(h_dist == np.inf)
    assert np.all(ids.cpu().numpy()[20:] == -7)  # nothing past n_queries * k
    # n_queries * k just below 2^32 passes the size checks and is refused for the null buffer alone
    refused(n_queries=(2 ** 32 - 1) // MAX_K, k=MAX_K, d_ids=None)
    # after refusals a valid call works
    check(sim, _se2(100, rng), _se2(4, rng), 3)
    sim.close()
