"""The three objective kernels that promise the reference's values bit for bit, against their numpy oracles at every
task count the ABI accepts:

* ``gnnpn_pn_reward_f32``   (modelPN ``calc`` / ``reward``, fp32)  vs ``po.composition_objective`` / ``po.reward``
* ``gnnpn_woa_fitness_f64`` (``ESWOA.calc``, f64)                 vs ``wo.calc``
* ``gnnpn_ml2pn_score_f64`` (``ML2PN.calc``, f64)                 vs ``mo.calc`` / ``mo.scores``

plus the device ESWOA search at its limits against the host engine on the CPU oracle, and the shape refusals.

Every comparison is exact (bit patterns; NaN matches NaN where the oracle gives NaN).  The inputs are built so that a
wrong operation order shows: q0 spans seven decades with negatives and zeros, so a sequential sum and numpy's pairwise
sum differ on them; the product factors lie in (0.9, 1); the ML2PN sets hold compositions that violate both constraints
and whose score rounds differently when the two violations are added at once.  ``test_inputs_tell_orders_apart`` checks
on the CPU that the inputs have that power, so the GPU tests cannot pass because the inputs are too easy."""
import math

import numpy as np
import pytest

from conftest import record_parity
from oracle import ml2pn_oracle as mo
from oracle import pn_oracle as po
from oracle import woa_oracle as wo

KMAX = 512               # kMaxTasks (pn.cu) and kMaxTasksWoa (woa.cu)
N_REWARD = 300           # instances per reward launch: not a multiple of the 128-thread block
P_FIT = 40               # random compositions per fitness / score launch
N_DOUBLE = 6             # ML2PN compositions per launch that violate both constraints and round apart
GNNPN_ESHAPE = -2


def _mixed_q0(g, shape, dtype=np.float64):
    """q0 with magnitudes 1e-4 .. 1e3, ~15 % negative, ~5 % zero."""
    v = 10.0 ** g.uniform(-4, 3, shape)
    v = np.where(g.random(shape) < 0.15, -v, v)
    return np.where(g.random(shape) < 0.05, 0.0, v).astype(dtype)


def _calm_rows(g, k):
    return np.stack([g.uniform(0, 0.2, k), g.uniform(0.5, 1, k), g.uniform(0.9, 1, k), g.uniform(0.9, 1, k)], 1)


def _median_product(K):
    """exp(K * E[log u]) for u ~ U(0.9, 1): bounds drawn around it give both verdicts at every K."""
    return math.exp(-0.05175 * K)


def _bits_differ(a, b):
    """Mask of elements whose bit patterns differ, NaN matching NaN."""
    a, b = np.asarray(a), np.asarray(b)
    assert a.dtype == b.dtype and a.shape == b.shape, (a.dtype, b.dtype, a.shape, b.shape)
    u = {4: np.uint32, 8: np.uint64}[a.dtype.itemsize]
    return ~((a.view(u) == b.view(u)) | (np.isnan(a) & np.isnan(b)))


def _seq_sum(v):
    """A plain left-to-right sum in the dtype of v."""
    return np.cumsum(v, dtype=v.dtype)[-1]


# ------------------------------------------------------------------------------------------------------ reward inputs
N_EDGE = 13     # instances 0 .. N_EDGE-1 of every reward launch are the edge cases below


def reward_case(K, tag):
    """inputs fp32 [n, L, F], picks int32 [K, n]; L = K + 3 rows per instance, F = tag + 9 columns."""
    g = np.random.default_rng(7_000 + 2 * K + tag)
    n, L, F = N_REWARD, K + 3, tag + 9
    x = g.uniform(-1, 1, (n, L, F)).astype(np.float32)       # the columns the objective does not read are noise
    q = x[:, :, tag:tag + 8]                                  # a view: q0 q1 q2 q3 lo1 hi1 lo2 hi2
    q[..., 0] = _mixed_q0(g, (n, L), np.float32)
    q[..., 1] = g.uniform(0, 1, (n, L))
    q[..., 2:4] = g.uniform(0.9, 1, (n, L, 2))
    med = _median_product(K)
    for i in range(2):
        lo = med * g.uniform(0.2, 1.2, (n, L))
        q[..., 4 + 2 * i] = lo
        q[..., 5 + 2 * i] = lo * g.uniform(1, 5, (n, L))
    idx = g.integers(0, L, (K, n)).astype(np.int32)
    for b in range(N_EDGE):
        idx[:, b] = g.permutation(L)[:K]
    r0 = idx[0]                                              # the step-0 row of every instance: it holds the bounds

    def prod(b, i):
        return np.cumprod(q[b, idx[:, b], 2 + i], dtype=np.float32)[-1]

    # 0 / 1: no q0 > 0 -- s / 0 is -inf (some q0 < 0) or NaN (all zero), as numpy gives it
    q[0, :, 0] = -np.abs(q[0, :, 0]) - np.float32(1e-4)
    q[1, :, 0] = 0.0
    # 2: products exactly on lo (first) and on hi (second): strict comparisons, no violation
    q[2, r0[2], 4], q[2, r0[2], 5] = prod(2, 0), np.float32(1.0)
    q[2, r0[2], 6], q[2, r0[2], 7] = np.float32(0.0), prod(2, 1)
    # 3: one ulp inside the other way: both violated
    q[3, r0[3], 4], q[3, r0[3], 5] = np.nextafter(prod(3, 0), np.float32(np.inf)), np.float32(1.0)
    q[3, r0[3], 6], q[3, r0[3], 7] = np.float32(0.0), np.nextafter(prod(3, 1), np.float32(-np.inf))
    # 4 / 5: only the step-0 row's bounds count -- every other row says the opposite
    for b, (ok, bad) in ((4, ((0.0, 1.0), (2.0, 3.0))), (5, ((2.0, 3.0), (0.0, 1.0)))):
        q[b, :, 4:8] = bad * 2
        q[b, r0[b], 4:8] = ok * 2
    # 6 .. 12: viol + obj on or next to a 5-decimal half point.  One positive q0 = 0.5 and zeros make s = 0.5 exactly,
    # #(q0 > 0) = 1, so obj = (1.5 - m) / 2 exactly for the min q1 = m in [0.75, 1.5]
    j = int(g.integers(0, 37_000))
    m_half = np.float32(1.5 - 2 * (j + 0.5) * 1e-5)
    ms = [np.float32(1.46875)] * 3 + [m_half, np.nextafter(m_half, np.float32(2)), np.nextafter(m_half, np.float32(0)),
                                      np.float32(1.5 - 2 * 0.000125)]
    for b, m in zip(range(6, 13), ms):          # 1.46875: obj = 2^-6 = 0.015625, a tie at the 5th decimal
        q[b, :, 0] = 0.0
        q[b, idx[0, b], 0] = 0.5
        q[b, :, 1] = m
        viol = (b - 6) % 3                       # 0, 1 or 2 violated constraints
        q[b, :, 4:8] = (0.0, 1.0, 0.0, 1.0)
        if viol >= 1:
            q[b, :, 4] = 2.0
        if viol == 2:
            q[b, :, 6] = 2.0
    return x, idx


def reward_reference(x, idx, tag):
    """(viol int32, obj fp32, reward fp32) of ``po.composition_objective`` / ``po.reward``."""
    import torch
    n = x.shape[0]
    acts = x[np.arange(n)[None, :], idx]                                   # [K, n, F]
    with np.errstate(all="ignore"):
        viol, obj = po.composition_objective(acts, tag)
        rew = po.reward(list(torch.from_numpy(acts)), None, idx.shape[0], "High", 0 if tag == 0 else 20)
    return viol.astype(np.int32), obj, rew.numpy()


# ---------------------------------------------------------------------------------------- fitness / score inputs
def composition_case(Kmax, ml2pn):
    """qos f64 [T, 4], idx int32 [P, idx_ld] (idx_ld > Kmax), klen int32 [P], bounds f64 [P, 4].

    Rows 0 and 1 take 1 and Kmax picks.  Entries past klen[p] name the last row of qos, whose values would change any
    result they entered.  With ``ml2pn``, the last N_DOUBLE compositions violate both constraints and are chosen so
    that (obj + 1) + 1 != obj + 2."""
    g = np.random.default_rng(9_000 + 2 * Kmax + ml2pn)
    T = 4 * Kmax + 16
    qos = np.stack([_mixed_q0(g, T), g.uniform(0, 1, T), g.uniform(0.9, 1, T), g.uniform(0.9, 1, T)], 1)
    P = P_FIT
    klen = g.integers(1, Kmax + 1, P).astype(np.int32)
    klen[0], klen[1] = 1, Kmax
    idx_ld = Kmax + 5
    poison = T                                    # appended below
    idx = np.full((P, idx_ld), poison, np.int32)
    for p in range(P):
        idx[p, :klen[p]] = g.integers(0, T, klen[p])
    bounds = np.empty((P, 4))
    for p in range(P):
        med = _median_product(int(klen[p]))
        for i in range(2):
            bounds[p, 2 * i] = med * g.uniform(0.2, 1.2)
            bounds[p, 2 * i + 1] = bounds[p, 2 * i] * g.uniform(1, 5)
    rows = [qos]
    if ml2pn:
        # calm rows (q0 in (0, 0.2), q1 in (0.5, 1)) keep obj in (0, 0.5), where its low bits fall off when 1 is
        # added; a composition is kept when the two ways of adding the violations round apart (~5 % of draws)
        extra_idx, extra_len = [], []
        base = T
        while len(extra_idx) < N_DOUBLE:
            k = int(g.integers(1, Kmax + 1)) if len(extra_idx) else Kmax
            r = _calm_rows(g, k)
            obj = mo.calc([r[:, c] for c in range(4)], [[-np.inf, np.inf], [-np.inf, np.inf]])
            if (obj + 1) + 1 == obj + 2:
                continue
            rows.append(r)
            extra_idx.append(np.arange(base, base + k))
            extra_len.append(k)
            base += k
        poison = base
        idx[idx == T] = poison
        ex = np.full((N_DOUBLE, idx_ld), poison, np.int32)
        for d, (e, k) in enumerate(zip(extra_idx, extra_len)):
            ex[d, :k] = e
        idx = np.concatenate([idx, ex])
        klen = np.concatenate([klen, np.asarray(extra_len, np.int32)])
        bounds = np.concatenate([bounds, np.tile([2.0, 3.0, 2.0, 3.0], (N_DOUBLE, 1))])   # products < 1 < lo
    rows.append(np.asarray([[1e300, -1e300, 1e-300, 1e300]]))     # the poison row
    return np.concatenate(rows), idx, klen, bounds


def composition_reference(qos, idx, klen, bounds, ml2pn):
    """(viol, obj, fitness-or-score) per composition from ``wo.calc`` / ``mo.calc``."""
    P = len(klen)
    viol, obj, fit = np.empty(P, np.int32), np.empty(P), np.empty(P)
    with np.errstate(all="ignore"):
        for p in range(P):
            rows = qos[idx[p, :klen[p]]]
            cons = [[bounds[p, 0], bounds[p, 1]], [bounds[p, 2], bounds[p, 3]]]
            if ml2pn:
                cols = [rows[:, c] for c in range(4)]
                fit[p] = mo.calc(cols, cons)
                obj[p] = mo.calc(cols, [[-np.inf, np.inf], [-np.inf, np.inf]])     # the objective before violations
                viol[p] = sum(int(not (c[0] <= np.cumprod(cols[2 + j])[-1] <= c[1])) for j, c in enumerate(cons))
            else:
                v, o = wo.calc([tuple(r) for r in rows], [[c] for c in cons])
                viol[p], obj[p], fit[p] = v, o, v + o
    return viol, obj, fit


NEVER = [-np.inf, np.inf, -np.inf, np.inf]       # bounds no product violates: mo.calc gives the bare objective


def scores_case():
    """(allActions, constraints) for ``ML2PN.composition_scores``: K lists of [n][8] python floats, ~30 % neutral
    [0, 1, 1, 1] picks (instance 3 keeps a single real pick), mixed q0 on even instances and calm rows on odd ones;
    the second half of the instances violates both constraints."""
    g = np.random.default_rng(31)
    K, n, h = 20, 400, 200
    acts = g.uniform(0, 1, (K, n, 8))
    acts[:, 0::2, :4] = np.stack([_mixed_q0(g, (K, h)), g.uniform(0, 1, (K, h)), g.uniform(0.9, 1, (K, h)),
                                  g.uniform(0.9, 1, (K, h))], -1)
    acts[:, 1::2, :4] = _calm_rows(g, K * h).reshape(K, h, 4)
    neutral = g.random((K, n)) < 0.3
    neutral[0] = False                                         # every instance keeps at least one real pick
    neutral[1:, 3] = True
    acts[neutral, :4] = (0.0, 1.0, 1.0, 1.0)
    cons = np.empty((n, 4))
    med = _median_product(K)
    for i in range(2):
        cons[:, 2 * i] = med * g.uniform(0.2, 1.2, n)
        cons[:, 2 * i + 1] = cons[:, 2 * i] * g.uniform(1, 5, n)
    cons[h:] = (2.0, 3.0, 2.0, 3.0)                            # products < 1 < lo: both violated
    return [[[float(v) for v in acts[k, j]] for j in range(n)] for k in range(K)], cons


# ------------------------------------------------------------------------------------------------------- CPU
def test_inputs_tell_orders_apart():
    """At every task count >= 9 the inputs hold a composition whose plain sequential sum differs from np.sum (fp32 for
    the reward, f64 for fitness and score); every ML2PN set holds compositions with (obj + 1) + 1 != obj + 2."""
    for K in range(9, KMAX + 1):
        for tag in (0, 1):
            x, idx = reward_case(K, tag)
            q0 = x[np.arange(x.shape[0])[None, :], idx, tag]                 # [K, n]
            assert any(_seq_sum(q0[:, b]) != np.sum(np.ascontiguousarray(q0[:, b])) for b in range(q0.shape[1])), K
        for ml2pn in (False, True):
            qos, idx, klen, _ = composition_case(K, ml2pn)
            assert any(_seq_sum(qos[idx[p, :klen[p]], 0]) != np.sum(qos[idx[p, :klen[p]], 0])
                       for p in range(len(klen)) if klen[p] >= 9), (K, ml2pn)
    for K in range(1, KMAX + 1):
        qos, idx, klen, bounds = composition_case(K, True)
        _, obj, score = composition_reference(qos, idx, klen, bounds, True)
        d = slice(len(klen) - N_DOUBLE, None)
        assert (score[d] == obj[d] + 2).sum() == 0 and ((obj[d] + 1) + 1 == score[d]).all(), K
    acts, cons = scores_case()
    pre = mo.scores(acts, len(acts), [NEVER] * len(cons))
    score = mo.scores(acts, len(acts), cons.tolist())
    h = len(cons) // 2
    assert ((pre[h:] + 1) + 1 != pre[h:] + 2).any() and np.array_equal(score[h:], (pre[h:] + 1) + 1)
    assert sum(sum(r[:4]) == 3 for a in acts for r in a) > 0

def test_reward_edge_instances_cover_their_cases():
    """The hand-built reward instances are what they claim to be, according to the oracle."""
    for K in (1, 8, 129, 512):
        x, idx = reward_case(K, 0)
        viol, obj, rew = reward_reference(x, idx, 0)
        assert obj[0] == -np.inf and np.isnan(obj[1])
        assert viol[2] == 0 and viol[3] == 2 and viol[4] == 0 and viol[5] == 2
        assert [int(v) for v in viol[6:12]] == [0, 1, 2, 0, 1, 2] and obj[6] == 0.015625
        assert rew[6] == np.float32(0.01562) and rew[7] == np.float32(1.01562)      # ties go to the even digit
        assert len({float(o) for o in obj[9:12]}) == 3


# ------------------------------------------------------------------------------------------------------- GPU
def _cuda(a):
    import torch
    return torch.from_numpy(np.ascontiguousarray(a)).cuda()


@pytest.mark.gpu
def test_reward_every_task_count_bitwise():
    import torch
    from gnnpn_sc_b200 import ops
    bad = {}
    for K in range(1, KMAX + 1):
        for tag in (0, 1):
            x, idx = reward_case(K, tag)
            viol, obj, rew = (t.cpu().numpy() for t in ops.pn_reward(_cuda(x), _cuda(idx), tag))
            rv, ro, rr = reward_reference(x, idx, tag)
            miss = (viol != rv) | _bits_differ(obj, ro) | _bits_differ(rew, rr)
            if miss.any():
                bad[(K, tag)] = np.nonzero(miss)[0].tolist()
    torch.cuda.synchronize()
    record_parity("objective_exact_reward_K1_512", mismatched_launches=len(bad),
                  mismatched_instances=sum(len(v) for v in bad.values()))
    assert not bad, sorted(bad)


def _composition_launch(fn, qos, idx, klen, bounds, Kmax):
    """One call of gnnpn_woa_fitness_f64 / gnnpn_ml2pn_score_f64 with idx's own leading dimension (> Kmax)."""
    import torch
    from gnnpn_sc_b200 import _lib, ops
    P = len(klen)
    d_qos, d_idx, d_klen, d_bounds = _cuda(qos), _cuda(idx), _cuda(klen), _cuda(bounds)
    viol = torch.empty(P, dtype=torch.int32, device="cuda")
    obj = torch.empty(P, dtype=torch.float64, device="cuda")
    fit = torch.empty(P, dtype=torch.float64, device="cuda")
    _lib.check(getattr(_lib.lib(), fn)(d_qos.data_ptr(), qos.shape[0], d_idx.data_ptr(), idx.shape[1], d_klen.data_ptr(),
                                       d_bounds.data_ptr(), P, Kmax, viol.data_ptr(), obj.data_ptr(), fit.data_ptr(),
                                       ops._stream()), fn)
    return viol.cpu().numpy(), obj.cpu().numpy(), fit.cpu().numpy()


@pytest.mark.gpu
@pytest.mark.parametrize("ml2pn", [False, True], ids=["eswoa_fitness", "ml2pn_score"])
def test_fitness_and_score_every_task_count_bitwise(ml2pn):
    fn = "gnnpn_ml2pn_score_f64" if ml2pn else "gnnpn_woa_fitness_f64"
    bad = {}
    for Kmax in range(1, KMAX + 1):
        qos, idx, klen, bounds = composition_case(Kmax, ml2pn)
        got = _composition_launch(fn, qos, idx, klen, bounds, Kmax)
        ref = composition_reference(qos, idx, klen, bounds, ml2pn)
        miss = (got[0] != ref[0]) | _bits_differ(got[1], ref[1]) | _bits_differ(got[2], ref[2])
        if miss.any():
            bad[Kmax] = np.nonzero(miss)[0].tolist()
    record_parity(f"objective_exact_{'ml2pn_score' if ml2pn else 'woa_fitness'}_K1_512", mismatched_launches=len(bad),
                  mismatched_compositions=sum(len(v) for v in bad.values()))
    assert not bad, bad


@pytest.mark.gpu
def test_ml2pn_composition_scores_bitwise():
    """``ML2PN.composition_scores`` (neutral rows dropped through the index table) == ``mo.scores``, with neutral
    [0, 1, 1, 1] picks and with compositions that violate both constraints."""
    from gnnpn_sc_b200.ML2PN import composition_scores
    acts, cons = scores_case()
    ref = mo.scores(acts, len(acts), cons.tolist())
    got = composition_scores(acts, len(acts), cons)
    miss = _bits_differ(got, ref)
    record_parity("objective_exact_ml2pn_composition_scores", instances=len(ref), mismatches=int(miss.sum()))
    assert not miss.any(), np.nonzero(miss)[0]


def _search_problem(g, K, size1=0.0):
    """ESWOA instance of K tasks: lists of 1 .. 12 candidates (a share ``size1`` of size 1), q0 of magnitudes
    1e-4 .. 1 (so every fitness is below the initial best of 3), bounds around the median product."""
    services = []
    for _ in range(K):
        m = 1 if g.random() < size1 else int(g.integers(2, 13))
        services.append([(float(10 ** g.uniform(-4, 0)), float(g.uniform(0, 1)), float(g.uniform(0.9, 1)),
                          float(g.uniform(0.9, 1))) for _ in range(m)])
    med = _median_product(K)
    lo1, lo2 = med * g.uniform(0.2, 1.2), med * g.uniform(0.2, 1.2)
    return services, [[[lo1, lo1 * g.uniform(1, 5)]], [[lo2, lo2 * g.uniform(1, 5)]]], None


@pytest.mark.gpu
@pytest.mark.parametrize("name,ks,size1,pop,iters", [
    ("one_task", [1, 1, 1], 0.0, 16, 12),
    ("kmax128_pop128", [128, 128], 0.1, 128, 10),          # the largest shared-memory request
    ("ragged", [1, 7, 128, 40, 2], 0.2, 33, 10),
    ("single_candidates", [5, 30], 1.0, 8, 10),
])
def test_device_search_at_limits_equals_cpu_host_chain(name, ks, size1, pop, iters):
    """``run_many_device`` == ``run_many`` on the CPU oracle with the same Philox draws: best-so-far trajectory, best
    fitness and best position, bit for bit (no GPU fitness on the host side)."""
    import copy
    from gnnpn_sc_b200.WOA import PhiloxRng, run_many, run_many_device
    g = np.random.default_rng(sum(ks) + pop)
    probs = [_search_problem(g, k, size1) for k in ks]
    seeds = [50 + 3 * k for k in range(len(ks))]
    dev = run_many_device(copy.deepcopy(probs), popSize=pop, MAX_Iter=iters, seeds=seeds)
    host = run_many(copy.deepcopy(probs), popSize=pop, MAX_Iter=iters, fitness=wo.CpuFitness,
                    rngs=[PhiloxRng(s) for s in seeds])
    diff = 0
    for k, (d, h) in enumerate(zip(dev, host)):
        diff += d[2] != h[2] or d[0] != h[0] or [tuple(r) for r in d[1]] != [tuple(r) for r in h[1]]
    record_parity(f"objective_exact_device_search_{name}", mismatched_instances=diff)
    for k, (d, h) in enumerate(zip(dev, host)):
        assert d[2] == h[2], (name, k)
        assert d[0] == h[0] and [tuple(r) for r in d[1]] == [tuple(r) for r in h[1]], (name, k)


@pytest.mark.gpu
def test_refusals_launch_nothing():
    import torch
    from gnnpn_sc_b200 import _lib, ops
    lib, st = _lib.lib(), ops._stream()
    buf = torch.zeros(1 << 20, dtype=torch.float64, device="cuda")
    p = buf.data_ptr()
    reward = lambda K=4, tag=0, F=10: lib.gnnpn_pn_reward_f32(p, p, 3, 600, F, K, tag, p, p, p, st)
    before = _lib.launch_count()
    assert reward(K=0) == GNNPN_ESHAPE and reward(K=KMAX + 1) == GNNPN_ESHAPE
    assert reward(tag=2) == GNNPN_ESHAPE and reward(tag=-1) == GNNPN_ESHAPE
    assert reward(F=7) == GNNPN_ESHAPE and reward(tag=1, F=8) == GNNPN_ESHAPE
    for fn in (lib.gnnpn_woa_fitness_f64, lib.gnnpn_ml2pn_score_f64):
        assert fn(p, 16, p, KMAX + 1, None, p, 4, KMAX + 1, p, p, p, st) == GNNPN_ESHAPE
        assert fn(p, 16, p, KMAX, None, p, 4, 0, p, p, p, st) == GNNPN_ESHAPE
    search = lambda P=8, KM=4: lib.gnnpn_woa_search_f64(p, 16, p, p, p, p, p, p, p, p, p, p, 2, P, KM, 3, st)
    assert search(KM=129) == GNNPN_ESHAPE and search(P=129) == GNNPN_ESHAPE
    assert search(KM=0) == GNNPN_ESHAPE and search(P=0) == GNNPN_ESHAPE
    assert _lib.launch_count() == before
