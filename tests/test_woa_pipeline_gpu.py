"""The ESWOA stage of the ML+2PN pipeline on the device (``gnnpn_woa_prepare_f64`` + the unchanged search) against the host
path it replaces, bit for bit: ``loadDataOther`` + ``_add_s`` for the candidate lists, the seed preparation of
``WOA.start``, ``_Instance`` and ``_Engine._init_population`` for the initial state, ``run_many_device`` and
``WOA(..., engine="device").start()`` for the results."""
import copy
import json
import os

import numpy as np
import pytest
import torch

from oracle import pn_oracle as po

NEUTRAL = np.array([0, 1, 1, 1], dtype=np.float32)


# ----------------------------------------------------------------------------------------------- CPU: the host helper
def test_woa_arrays_match_load_data_other(tmp_path, golden_dir):
    """woa_arrays parses nodefeatures as loadDataOther does: the plain candidate lists rebuilt from its request order and
    float64 local bounds, and its global bounds, equal loadDataOther's on the reference loader fixture."""
    from gnnpn_sc_b200.WOA import loadDataOther
    from gnnpn_sc_b200.pipeline import woa_arrays
    with open(os.path.join(golden_dir, "woa_loader.json")) as f:
        d = json.load(f)
    root = str(tmp_path)
    os.makedirs(os.path.join(root, "data", "toy"))
    for name, obj in d["data"].items():
        with open(os.path.join(root, "data", "toy", name), "w") as f:
            json.dump(obj, f)
    feats, cons, _ = loadDataOther("toy", False, None, False, root)
    nodef, sf = d["data"]["nodefeatures.data"], d["data"]["serviceFeature.data"]
    K = len(sf)
    req, n_req, local, glob = woa_arrays(nodef, K)
    lo = len(nodef) // 4 * 3
    assert req.dtype == np.int32 and local.dtype == np.float64 and glob.dtype == np.float64
    for k, b in enumerate(range(lo, len(nodef))):
        assert cons[k] == [[list(glob[b, :2])], [list(glob[b, 2:])]]
        lists = []
        for cat in req[b, :n_req[b]]:
            lc, hc, lq, hq = local[b, cat]
            rows = [tuple(r[-4:]) for r in sf[str(cat + 1)]]
            lists.append([r for r in rows if lc <= r[2] <= hc and lq <= r[3] <= hq])
        assert [c for c in lists if c] == feats[k]
        assert (req[b, n_req[b]:] == -1).all()


# ----------------------------------------------------------------------------------------------- GPU helpers
def _write(root, name, ds):
    from gnnpn_sc_b200 import synth
    synth.write_dataset(root, name, ds)


def _solutions(seed_rows):
    """WOA.start's seed rows (WOA.py:591-594) from fp32 [n, K, 4] picks: float64 values, neutral rows dropped."""
    sols = []
    for inst in seed_rows:
        rows = [[float(v) for v in r] for r in inst]
        sols.append([r for r in rows if sum(r) != 3])
    return sols


def _seed_ids(seed_rows, seed_ids):
    """Service id of every seed row (the categories whose pick is not neutral, in category order)."""
    return [[int(i) for r, i in zip(rows, ids) if sum(float(v) for v in r) != 3] for rows, ids in zip(seed_rows, seed_ids)]


def _sset(sols):
    return [{tuple(round(v, 5) for v in r) for r in s} for s in sols]


def _host_init(feats, cons, sols, P, seeds):
    """_Instance + _Engine._init_population, as run_many_device runs them before its launch."""
    from gnnpn_sc_b200 import WOA as W
    inst = [W._Instance(copy.deepcopy(f), copy.deepcopy(c), copy.deepcopy(s) if s else None, P, 1, W.PhiloxRng(sd))
            for f, c, s, sd in zip(feats, cons, sols, seeds)]
    W._Engine(inst, None)
    return inst


def _prepare(svc_raw, ptr, woa, seed_rows, seed_ids, seeds, P, reduct):
    from gnnpn_sc_b200 import ops
    from gnnpn_sc_b200.WOA import _round5
    req, n_req, local, glob = woa
    t = lambda a: torch.from_numpy(np.ascontiguousarray(a)).cuda()
    return ops.woa_prepare(t(svc_raw), t(_round5(svc_raw)), t(ptr), t(req), t(n_req), t(local), t(glob), t(seed_rows),
                           t(seed_ids.astype(np.int32)), t(np.asarray(seeds, np.int64)), P, reduct)


def _check_prepared(p, inst, feats, svc_raw, sol_ids, sols):
    """Device lists, sizes, order, appended seed rows, population and best state == the host's, value for value."""
    from gnnpn_sc_b200.WOA import _round5
    p = {k: v.cpu().numpy() for k, v in p.items()}
    assert not p["flags"].any()
    svc_round = _round5(svc_raw)
    for w, it in enumerate(inst):
        k = len(it.services)
        assert p["klen"][w] == k
        seeded = bool(sols[w])
        table = svc_round if seeded else svc_raw
        for l in range(k):
            b, n = p["base"][w, l], p["size"][w, l]
            got = [tuple(float(v) for v in r) for r in p["qos"][b:b + n]]
            assert got == [tuple(float(v) for v in r) for r in it.services[l]], (w, l)
            n0 = len(feats[w][l])
            ids = p["ids"][b:b + n]
            assert (table[ids[:n0]] == p["qos"][b:b + n0]).all()
            assert ((ids >= 0) & (ids < len(svc_raw))).all()
            if n > n0:                                                         # seed row l appended to list l
                assert n == n0 + 1 and ids[n0] == sol_ids[w][l]
        assert (p["pops"][w, :, :k] == it._pops).all() and (p["pops"][w, :, k:] == 0).all()
        assert p["best_fit"][w] == it.bestFitness and p["best_ref"][w] == it.best_ref
        if it.best_vec is not None:
            assert (p["best_vec"][w, :k] == it.best_vec).all()


def _pn_nets(K, N):
    from gnnpn_sc_b200 import modelPN as M
    cfg = po.PNConfig(seq_len=K * N, s_number=N, s_category=K)
    nets = []
    for level, seed in (("Low", 1), ("High", 2)):
        m = M.CombinatorialRL(0, 256, K * N, 0, 10, 1, M.reward, "Dot", N, K, level=level)
        m.load_state_dict(po.make_state_dict(cfg, seed))
        nets.append(m.cuda().eval())
    return nets


SHAPES = {"qws": dict(K=47, S=2507, N=5, dist="qws", reduct=0, P=50, iters=20, gcn=2),
          "normal": dict(K=50, S=2500, N=10, dist="normal", reduct=0.55, P=60, iters=20, gcn=2)}


def _pipeline(shape, n=64, seed=11):
    """A synthetic dataset, ML2PN with the ESWOA stage, and compose() on its test split (instance ids lo..n-1)."""
    from gnnpn_sc_b200 import synth, loadData, trainML, modelML
    from gnnpn_sc_b200.pipeline import ML2PN, constraint_arrays, service_arrays, woa_arrays
    c = SHAPES[shape]
    K, S = c["K"], c["S"]
    ds = synth.ml_dataset(n_instances=n, K=K, S=S, seed=seed, dist=c["dist"], min_tasks=10)
    samples = trainML.build_samples(loadData.ml_arrays(ds))
    torch.manual_seed(seed)
    net = modelML.Net(128, S, 20, 2, c["gcn"], isServices=True)
    net.reset_parameters()
    net = net.cuda().eval()
    low, high = _pn_nets(K, c["N"])
    dev_sample = type(samples[0])(**{k: (v.cuda() if torch.is_tensor(v) else v) for k, v in vars(samples[0]).items()})
    pipe = ML2PN(net, low, high, dev_sample, ds["serviceFeature"], "cuda",
                 woa={"popSize": c["P"], "MAX_Iter": c["iters"], "reduct": c["reduct"]})
    lo = n // 4 * 3
    nodef = ds["nodefeatures"][lo:]
    woa = woa_arrays(nodef, K)
    ids = np.arange(lo, n, dtype=np.int64)
    rb = trainML.collate_requests(samples[lo:], device="cuda")
    cons = [torch.from_numpy(a).cuda() for a in constraint_arrays(nodef, K)]
    out = pipe.compose(rb, *cons, woa=[torch.from_numpy(a).cuda() for a in (*woa, ids)])
    torch.cuda.synchronize()
    raw, ptr = service_arrays(ds["serviceFeature"], dtype=np.float64)
    idx = out["idx_high"].cpu().numpy()                                                  # [K, n_test]
    rows = out["rows"].cpu().numpy()
    seed_rows = np.stack([rows[b, idx[:, b], :4] for b in range(len(nodef))])          # [n_test, K, 4]
    seed_ids = out["services"].cpu().numpy().astype(np.int32)
    return dict(ds=ds, samples=samples, pipe=pipe, out=out, woa=woa, ids=ids, lo=lo, raw=raw, ptr=ptr,
                seed_rows=seed_rows, seed_ids=seed_ids, c=c, K=K)


# ----------------------------------------------------------------------------------------------- GPU: dataset shapes
@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["qws", "normal"])
def test_prepare_equals_host_lists_seed_and_initial_state(shape, tmp_path):
    from gnnpn_sc_b200.WOA import loadDataOther
    r = _pipeline(shape)
    c, root = r["c"], str(tmp_path)
    _write(root, "ds", r["ds"])
    sols = _solutions(r["seed_rows"])
    assert sum(1 for s in sols if s) > len(sols) // 2                     # real PNHigh picks seed most instances
    feats, cons, _ = loadDataOther("ds", c["reduct"], _sset(sols), False, root)
    if c["reduct"]:
        plain, _, _ = loadDataOther("ds", 0, None, False, root)
        assert feats != plain                                             # the running front thins the lists
    p = _prepare(r["raw"], r["ptr"], r["woa"], r["seed_rows"], r["seed_ids"], r["ids"], c["P"], c["reduct"])
    inst = _host_init(feats, cons, sols, c["P"], r["ids"])
    _check_prepared(p, inst, feats, r["raw"], _seed_ids(r["seed_rows"], r["seed_ids"]), sols)


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["qws", "normal"])
def test_compose_woa_equals_run_many_device_and_file_driver(shape, tmp_path):
    from gnnpn_sc_b200 import WOA as W
    r = _pipeline(shape)
    c, root, out, K = r["c"], str(tmp_path), r["out"], r["K"]
    _write(root, "ds", r["ds"])
    sols = _solutions(r["seed_rows"])
    feats, cons, mc = W.loadDataOther("ds", c["reduct"], _sset(sols), False, root)
    probs = [(f, cn, s if s else None) for f, cn, s in zip(feats, cons, sols)]
    host = W.run_many_device(copy.deepcopy(probs), popSize=c["P"], MAX_Iter=c["iters"], seeds=list(r["ids"]))
    fit, traj, svc = (out[k].cpu().numpy() for k in ("woa_fitness", "woa_traj", "woa_services"))
    assert [h[0] for h in host] == fit.tolist()
    assert [h[2] for h in host] == traj.tolist()
    # best composition: list l's best row (host) is a row of device list l carrying the reported service id
    p = {k: v.cpu().numpy() for k, v in _prepare(r["raw"], r["ptr"], r["woa"], r["seed_rows"], r["seed_ids"], r["ids"],
                                                   c["P"], c["reduct"]).items()}
    for w, (_, best_rows, _) in enumerate(host):
        k = p["klen"][w]
        assert len(best_rows) == k and sorted(np.nonzero(svc[w] >= 0)[0]) == sorted(p["list_cat"][w, :k])
        for l in range(k):
            b, n = p["base"][w, l], p["size"][w, l]
            sid = svc[w, p["list_cat"][w, l]]
            hits = [j for j in range(n) if p["ids"][b + j] == sid and tuple(p["qos"][b + j]) == tuple(best_rows[l])]
            assert hits, (w, l)
    # the same picks as allActions files through the file-level driver
    ptr = r["ptr"]
    n_test = len(sols)
    actions = [[[float(v) for v in r["seed_rows"][i, k]] + [0, 0, 0, 0] for i in range(n_test)] for k in range(K)]
    os.makedirs(os.path.join(root, "solutions", "PNHigh", "ds"))
    with open(os.path.join(root, "solutions", "PNHigh", "ds", "allActions3.txt"), "w") as f:
        json.dump(actions, f)
    res = W.WOA("ds", K, 0, 1, 0, 0, int(ptr[1] - ptr[0]), c["reduct"], 3, c["iters"], c["P"], root=root,
                engine="device").start()
    assert res["quality"] == [m / q for m, q in zip(mc[r["lo"]:], fit.tolist())]


@pytest.mark.gpu
def test_run_yields_what_compose_returns():
    """ML2PN.run with the ESWOA arrays in its items == compose on the same batches, a short last batch included."""
    from gnnpn_sc_b200 import trainML
    from gnnpn_sc_b200.pipeline import constraint_arrays, woa_arrays
    r = _pipeline("qws", n=40, seed=5)
    pipe, samples, K = r["pipe"], r["samples"], r["K"]
    nodef = r["ds"]["nodefeatures"]
    cons, woa = constraint_arrays(nodef, K), woa_arrays(nodef, K)
    ids = np.arange(len(nodef), dtype=np.int64)
    parts = [(0, 16), (16, 32), (32, 40)]
    host = [(trainML.collate_requests(samples[a:b], pin=True), *[torch.from_numpy(x[a:b]).pin_memory() for x in cons],
             [torch.from_numpy(x[a:b]).pin_memory() for x in (*woa, ids)]) for a, b in parts]
    got = list(pipe.run(host))
    assert len(got) == len(parts)
    for (a, b), res in zip(parts, got):
        assert len(res) == 5
        rb = trainML.collate_requests(samples[a:b], device="cuda")
        want = pipe.compose(rb, *[torch.from_numpy(x[a:b]).cuda() for x in cons],
                            woa=[torch.from_numpy(x[a:b]).cuda() for x in (*woa, ids)])
        assert torch.equal(res[0], want["services"].to(torch.int32).cpu())
        for g, k in zip(res[2:], ("woa_fitness", "woa_services", "woa_traj")):
            assert torch.equal(g, want[k].cpu()), k
    plain = list(pipe.run(h[:4] for h in host))                             # items without the arrays: two results
    assert all(len(x) == 2 for x in plain) and torch.equal(plain[0][0], got[0][0])


# ----------------------------------------------------------------------------------------------- GPU: hand-built cases
PATCHED = (0.05314, 0.55528, 0.94008, 0.95495)          # one of the six rows WOA.py patches
ROUNDS_APART = 0.123455                                 # round(x, 5) = 0.12345, round(float32(x), 5) = 0.12346


def _toy(tmp_path, reduct):
    """4 categories x 6 services; the test split (instances 24..31) holds the edge cases.  Returns everything the
    device and the host paths take."""
    g = np.random.default_rng(7)
    K, per, n = 4, 6, 32
    svc = {}
    for c in range(K):
        rows = [[0.0] * 5 + [float(g.uniform(0.05, 0.95)), float(g.uniform(0.05, 0.95)), float(g.uniform(0.9, 1)),
                             float(g.uniform(0.9, 1))] for _ in range(per)]
        svc[str(c + 1)] = rows
    svc["1"][0][5] = ROUNDS_APART
    svc["2"][0][5:] = list(PATCHED)
    gnode = [1] + [0] * K + [0, 0.5, 1.0, 0, 0.5, 1.0]
    task = lambda c, lo=0.0: [0] * (c + 1) + [1] + [0] * (K - c - 1) + [0, lo, 1.0, 0, 0.0, 1.0]
    requests = [[task(c) for c in range(K)] for _ in range(24)]            # train split filler
    requests += [
        [task(2), task(0), task(1), task(3)],                               # 0: request order != category order
        [task(0), task(1, lo=2.0), task(2), task(3)],                       # 1: category 1 has no feasible service
        [task(0), task(1), task(2)],                                        # 2: seed row appended (rounds apart)
        [task(1), task(3)],                                                 # 3: a patched seed row
        [task(3), task(0), task(2)],                                        # 4: all picks neutral: unseeded
        [task(0), task(1), task(3), task(2)],                               # 5
        [task(1), task(0)],                                                 # 6
        [task(0), task(2), task(1), task(3)],                               # 7
    ]
    nodef = [[gnode] + r for r in requests]
    root = str(tmp_path)
    os.makedirs(os.path.join(root, "data", "toy"))
    for name, obj in (("nodefeatures.data", nodef), ("serviceFeature.data", svc), ("minCostList.data", [0.4] * n),
                      ("labels.data", [[0] * (per * K)] * n)):
        with open(os.path.join(root, "data", "toy", name), "w") as f:
            json.dump(obj, f)
    # PNHigh-like picks: a feasible service per requested category, neutral rows elsewhere
    lo = n // 4 * 3
    seed_rows = np.tile(NEUTRAL, (n - lo, K, 1))
    seed_ids = np.full((n - lo, K), -1, np.int32)
    for i, req in enumerate(requests[lo:]):
        for node in req:
            c = node.index(1) - 1
            if node[-5] > 1 or i == 4:
                continue
            j = 0 if (i, c) in ((2, 0), (3, 1)) else int(g.integers(0, per))
            seed_rows[i, c] = np.asarray(svc[str(c + 1)][j][-4:], dtype=np.float32)
            seed_ids[i, c] = c * per + j
    assert round(ROUNDS_APART, 5) != round(float(np.float32(ROUNDS_APART)), 5)
    from gnnpn_sc_b200.pipeline import service_arrays, woa_arrays
    raw, ptr = service_arrays(svc, dtype=np.float64)
    return root, nodef[lo:], lo, seed_rows, seed_ids, raw, ptr, K, woa_arrays(nodef[lo:], K)


@pytest.mark.gpu
@pytest.mark.parametrize("reduct", [0, 0.55])
def test_prepare_edge_cases_equal_host(tmp_path, reduct):
    from gnnpn_sc_b200.WOA import loadDataOther, _round5
    root, nodef, lo, seed_rows, seed_ids, raw, ptr, K, woa = _toy(tmp_path, reduct)
    sols = _solutions(seed_rows)
    assert not sols[4] and all(sols[i] for i in range(len(sols)) if i != 4)
    feats, cons, _ = loadDataOther("toy", reduct, _sset(sols), False, root)
    assert len(feats[1]) == 3                                               # the empty list is dropped
    P, seeds = 9, list(range(lo, lo + len(nodef)))
    p = _prepare(raw, ptr, woa, seed_rows, seed_ids, seeds, P, reduct)
    inst = _host_init(feats, cons, sols, P, seeds)
    _check_prepared(p, inst, feats, raw, _seed_ids(seed_rows, seed_ids), sols)
    size = p["size"].cpu().numpy()
    assert size[2, 0] == len(feats[2][0]) + 1                              # instance 2: appended (rounds apart)
    assert size[3, 0] == len(feats[3][0]) + 1                              # instance 3: the patched row is new
    assert tuple(inst[3].services[0][-1]) == (0.05314, 0.55527, 0.94008, 0.95495)
    assert inst[4].solution is None and (_round5(raw) != raw).any()         # unseeded: its rows stay unrounded


@pytest.mark.gpu
def test_seed_longer_than_lists_raises_like_the_host(tmp_path):
    from gnnpn_sc_b200 import ops
    from gnnpn_sc_b200.WOA import loadDataOther
    root, nodef, lo, seed_rows, seed_ids, raw, ptr, K, woa = _toy(tmp_path, 0)
    # instance 1: category 1's task has no feasible service, but the seed carries a pick for it
    seed_rows[1, 1] = raw[ptr[1]].astype(np.float32)
    seed_ids[1, 1] = ptr[1]
    sols = _solutions(seed_rows)
    feats, cons, _ = loadDataOther("toy", 0, _sset(sols), False, root)
    with pytest.raises(IndexError):
        _host_init(feats[1:2], cons[1:2], sols[1:2], 5, [lo + 1])
    p = _prepare(raw, ptr, woa, seed_rows, seed_ids, list(range(lo, lo + len(nodef))), 5, 0)
    flags = p["flags"].cpu().numpy()
    assert flags[1] == 1 and not np.delete(flags, 1).any()
    with pytest.raises(ops.GnnpnError, match=r"more seed rows than candidate lists: instances \[1\]"):
        ops.raise_if_woa_flagged(p["flags"])


@pytest.mark.gpu
def test_seed_shorter_than_lists_raises_like_the_host(tmp_path):
    """A requested category with feasible services but a neutral pick leaves the seed shorter than the lists: the host
    path raises when it evaluates the seed (WOA.py:140), so the device flags the instance."""
    from gnnpn_sc_b200 import ops
    from gnnpn_sc_b200.WOA import loadDataOther
    root, nodef, lo, seed_rows, seed_ids, raw, ptr, K, woa = _toy(tmp_path, 0)
    for i, c in ((0, 1), (3, 3)):                                           # 3 of 4 seed rows; 1 of 2 seed rows
        seed_rows[i, c] = NEUTRAL
        seed_ids[i, c] = -1
    sols = _solutions(seed_rows)
    feats, cons, _ = loadDataOther("toy", 0, _sset(sols), False, root)
    for i in (0, 3):
        assert 0 < len(sols[i]) < len(feats[i])
        with pytest.raises(ValueError):
            _host_init(feats[i:i + 1], cons[i:i + 1], sols[i:i + 1], 5, [lo + i])
    p = _prepare(raw, ptr, woa, seed_rows, seed_ids, list(range(lo, lo + len(nodef))), 5, 0)
    flags = p["flags"].cpu().numpy()
    assert flags[0] == 16 and flags[3] == 16 and not np.delete(flags, [0, 3]).any()
    with pytest.raises(ops.GnnpnError, match=r"fewer seed rows than candidate lists .*: instances \[0, 3\]"):
        ops.raise_if_woa_flagged(p["flags"])


# ----------------------------------------------------------------------------------------------- GPU: ABI
@pytest.mark.gpu
def test_prepare_abi_rejects_null_and_out_of_range_arguments():
    from gnnpn_sc_b200 import _lib
    L = _lib.lib()
    n, S, K, P = 2, 12, 3, 4
    f64 = lambda *s: torch.zeros(s, dtype=torch.float64, device="cuda")
    i32 = lambda *s: torch.zeros(s, dtype=torch.int32, device="cuda")
    rows = L.gnnpn_woa_prepare_rows(n, S, K)
    assert rows == n * (S + K)
    bufs = [f64(S, 4), f64(S, 4), i32(K + 1), S, K, i32(n, K), i32(n), f64(n, K, 4), f64(n, 4),
            torch.zeros(n, K, 4, device="cuda"), i32(n, K), torch.zeros(n, dtype=torch.int64, device="cuda"), n, P, 0.0,
            f64(rows, 4), i32(rows), i32(n, K), i32(n, K), i32(n), i32(n, K), i32(n, P, K), f64(n), i32(n), i32(n, K),
            i32(n)]
    args = lambda b: [x.data_ptr() if torch.is_tensor(x) else x for x in b] + [None]     # NULL stream
    ENULL, ESHAPE = -1, -2
    for j, x in enumerate(bufs):
        if torch.is_tensor(x):
            b = list(bufs); b[j] = None
            assert L.gnnpn_woa_prepare_f64(*args(b)) == ENULL, j
    for j, bad in ((13, 0), (13, 129), (4, 0), (4, 129), (3, 0), (12, -1)):
        b = list(bufs); b[j] = bad
        assert L.gnnpn_woa_prepare_f64(*args(b)) == ESHAPE, (j, bad)
    b = list(bufs); b[12] = (2 ** 31) // (S + K) + 1                       # base would leave the int32 row range
    assert L.gnnpn_woa_prepare_f64(*args(b)) == ESHAPE
