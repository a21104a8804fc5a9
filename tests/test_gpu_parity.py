"""GPU parity tests (run on the B200 box: `pytest -m gpu`).  Everything goes through the
reference-facing overlay (`src.core.*`) or the C ABI; the oracle (NumPy / C ports of the
reference, pinned in test_oracle_golden.py) is the checker.

Tolerances: DSA distances, winners, scores — bit-exact.  KMNC bucket ids and scores, DeepGini
predictions and scores — bit-exact.  LSA — rtol 1e-4 (north_star) with an absolute floor of
2e-4 on the log-density (values cross zero), inf <-> inf.
"""
import ast
import ctypes as C

import numpy as np
import pytest

from oracle import c_oracle, np_oracle
from tests.conftest import case_names

pytestmark = pytest.mark.gpu

LSA_RTOL, LSA_ATOL = 1e-4, 2e-4


def _torch():
    import torch

    return torch


# ------------------------------------------------------------------------------------------
# tensor-core pass: raw accumulator tile vs an fp32 matmul of the packed operands
# ------------------------------------------------------------------------------------------
@pytest.mark.parametrize("d,segments,variant", [(16, 1, 1), (16, 1, 2), (128, 1, 1), (128, 1, 2), (100, 1, 0),
                                                (64, 1, 2), (120, 1, 2), (5, 1, 2), (300, 1, 0), (2048, 1, 0),
                                                (10, 3, 0), (256, 3, 0), (40, 3, 1), (40, 3, 2)])
def test_pair_probe_matches_packed_matmul(d, segments, variant):
    """variant 1 = streaming kernel (128 x 256 tiles), 2 = resident-query kernel (256 x 192 tiles,
    128-byte-swizzled chunks + 32-byte-swizzled tail panels), 0 = whatever tip_nn_filter picks."""
    torch = _torch()
    from simple_tip_b200 import _lib
    from simple_tip_b200 import engine as E

    lib = _lib.load()
    dev = E.require_cuda()
    rng = np.random.default_rng(d * 7 + segments)
    q = torch.from_numpy(rng.normal(size=(256, d)).astype(np.float32)).to(dev)
    t = torch.from_numpy(rng.normal(size=(256, d)).astype(np.float32) * 1.5).to(dev)
    center = torch.from_numpy(rng.normal(size=d).astype(np.float32) * 0.1).to(dev)
    pitch = int(lib.tip_pair_pitch(d, segments))
    k16 = (segments * ((d + 15) // 16 * 16) + 16) // 16
    if variant == 2 and k16 > 9:
        pytest.skip("packed row too wide for the resident-query kernel")
    resident = variant == 2 or (variant == 0 and k16 <= 9)
    rows = 256 if resident else 128
    qp = torch.empty((256, pitch), dtype=torch.bfloat16, device=dev)
    tp = torch.empty((256, pitch), dtype=torch.bfloat16, device=dev)
    qs = torch.empty(256, dtype=torch.float32, device=dev)
    ts = torch.empty(256, dtype=torch.float32, device=dev)
    qe = torch.empty(256, dtype=torch.float32, device=dev)
    scale, coef = (-2.0, 1.0) if segments == 1 else (1.0, -0.5)
    _lib.check(lib.tip_pair_prep(E._p(q), _lib.TIP_F32, 256, d, E._p(center), _lib.ROLE_QUERY, segments, 1.0, 0.0,
                                 E._p(qp), E._p(qs), E._p(qe), E._stream()), "prep q")
    _lib.check(lib.tip_pair_prep(E._p(t), _lib.TIP_F32, 256, d, E._p(center), _lib.ROLE_TRAIN, segments, scale, coef,
                                 E._p(tp), E._p(ts), None, E._stream()), "prep t")
    out_full = torch.zeros((256, 256), dtype=torch.float32, device=dev)
    _lib.check(lib.tip_pair_probe(E._p(qp), 256, E._p(tp), 256, d, segments, pitch, variant, E._p(out_full),
                                  E._stream()), "probe")
    torch.cuda.synchronize()
    out = out_full[:rows]
    qp, qs, q = qp[:rows], qs[:rows], q[:rows]
    want = qp.to(torch.float64) @ tp.to(torch.float64).T
    scale_ref = float((qp.to(torch.float64).abs() @ tp.to(torch.float64).abs().T).max())
    err = float((out.to(torch.float64) - want).abs().max())
    assert err <= 4e-6 * scale_ref + 1e-6, (err, scale_ref)
    # and the packed operands mean what tip_pair_prep documents
    vq = (q - center).to(torch.float64)
    vt = (t - center).to(torch.float64)
    # rounderr = Euclidean norm of what the packed query drops (input to tip_nn_filter's window)
    d16 = (d + 15) // 16 * 16
    v32 = (q - center)
    kept = qp[:, :d].to(torch.float32) if segments == 1 else qp[:, :d].to(torch.float32) + qp[:, d16:d16 + d].to(torch.float32)
    want_err = (v32.to(torch.float64) - kept.to(torch.float64)).norm(dim=1)
    got_err = qe[:rows].to(torch.float64)
    assert bool(((got_err >= want_err * (1 - 1e-6)) & (got_err <= want_err * (1 + 1e-5) + 1e-12)).all())
    if segments == 1:
        d2 = ((vq[:, None, :] - vt[None, :, :]) ** 2).sum(-1)
        approx = out.to(torch.float64) + qs.to(torch.float64)[:, None]
        rel = float(((approx - d2).abs() / d2.clamp(min=1.0)).max())
        assert rel < 3e-2, rel                                   # single bf16 pass
    else:
        a = vq @ vt.T - 0.5 * (vt ** 2).sum(-1)[None, :]
        err3 = float((out.to(torch.float64) - a).abs().max())
        bound = 2e-5 * float(vq.norm(dim=1).max() * vt.norm(dim=1).max()) + 1e-4
        assert err3 < bound, (err3, bound)                       # split-bf16 (3 segments)


# ------------------------------------------------------------------------------------------
# DeepGini / KMNC
# ------------------------------------------------------------------------------------------
def test_deepgini_golden_and_known_answers(golden):
    from src.core.deepgini import DeepGini

    g = golden("gini_apfd_reference.npz")
    for name in ("c1_f32", "c1_f64", "wide"):
        pred, gini = DeepGini.calculate(g[f"{name}.p"])
        assert np.array_equal(pred, g[f"{name}.pred"]), name
        assert gini.dtype == g[f"{name}.gini"].dtype and np.array_equal(gini, g[f"{name}.gini"]), name
    batch = np.array([[0.1, 0.2, 0.3, 0.4], [0.5, 0.1, 0.1, 0.3], [0.25] * 4, [1.0, 0, 0, 0], [0, 1.0, 0, 0]])
    pred, unc = DeepGini.calculate(batch)          # reference tests/test_deepgini.py:15-38
    assert np.all(pred == [3, 0, 0, 0, 1]) and np.all(unc == np.array([0.7, 0.64, 0.75, 0, 0]))
    assert DeepGini.takes_samples() is False and DeepGini.is_confidence() is False
    assert all(a.startswith("custom") for a in DeepGini.aliases())


@pytest.mark.parametrize("n,c,dt", [(10000, 10, np.float32), (3, 1, np.float32), (777, 7, np.float64),
                                    (300, 129, np.float32), (50, 5000, np.float32), (1, 1000, np.float64)])
def test_deepgini_shapes_and_apfd(n, c, dt):
    from src.core.apfd import apfd_from_order
    from src.core.deepgini import DeepGini

    p, truth = np_oracle.synth_softmax(n, c, seed=n + c, dtype=dt)
    pred, gini = DeepGini.calculate(p)
    wp, wg = np_oracle.deepgini_oracle(p)
    assert np.array_equal(pred, wp) and np.array_equal(gini, wg)
    fault = wp != truth
    if fault.any():
        assert apfd_from_order(fault, np.argsort(-gini)) == np_oracle.apfd_oracle(fault, np.argsort(-wg))


def test_kmnc_golden(golden):
    from src.core.neuron_coverage import KMNC

    g = golden("kmnc_reference.npz")
    for name in case_names(g, "score"):
        mins, maxs, act = g[f"{name}.mins"], g[f"{name}.maxs"], g[f"{name}.act"]
        cut, k = int(g[f"{name}.cut"]), int(g[f"{name}.sections"])
        km = KMNC([mins[:cut], mins[cut:]], [maxs[:cut], maxs[cut:]], k)
        score, bucket = km.buckets([act[:, :cut], act[:, cut:]])
        assert np.array_equal(bucket, g[f"{name}.bucket"]), name
        assert np.array_equal(score, g[f"{name}.score"]), name
        s2, prof = km([act[:, :cut], act[:, cut:]])
        assert s2.dtype == g[f"{name}.score"].dtype and np.array_equal(s2, g[f"{name}.score"])
        assert prof.shape == (act.shape[0], act.shape[1], k) and prof.dtype == bool
        assert np.array_equal(prof.sum(axis=2), g[f"{name}.hits"])
        assert np.array_equal(np.where(prof.any(axis=2), prof.argmax(axis=2), -1), g[f"{name}.bucket"])


def test_kmnc_known_answer_from_reference_tests():
    from src.core.neuron_coverage import KMNC

    acts = [np.array([[0.1, 0.4, 0.9, 0.4], [0.1, 0.9, 0.9, 0.4]]),
            np.array([[0.3, 0.2, 0.1, 0.6, 0.8], [0.3, 0.9, 0.1, 0.6, 0.8]]),
            np.array([[0.2, 0.3, 0.4, 0.4], [0.2, 0.9, 0.4, 0.4]])]
    mins = [np.array([0] * 4), np.array([0] * 5), np.array([0.1] * 4)]
    maxs = [np.array([1] * 4), np.array([1] * 5), np.array([0.95] * 4)]
    score, profile = KMNC(mins, maxs, 2)(acts)
    assert np.all(score == np.array([13, 13]))
    assert np.all(profile[0] == np.concatenate([
        [[True, False], [True, False], [False, True], [True, False]],
        [[True, False], [True, False], [True, False], [False, True], [False, True]],
        [[True, False], [True, False], [True, False], [True, False]]]))
    out = [a.copy() for a in acts]
    out[0][0][0], out[1][0][0] = -0.5, 1.5
    assert np.all(KMNC(mins, maxs, 2)(out)[0] == np.array([11, 13]))


@pytest.mark.parametrize("n,d,k", [(2000, 4096, 1000), (513, 1001, 50), (64, 4096, 10000), (301, 1000, 7),
                                   (33, 4, 2)])
def test_kmnc_large_vs_c_oracle(n, d, k):
    from src.core.neuron_coverage import KMNC

    act, mins, maxs = np_oracle.synth_relu(n, d, seed=4)
    km = KMNC([mins], [maxs], k)
    score, bucket = km.buckets([act])
    sub = np.random.default_rng(0).choice(n, size=min(n, 24), replace=False)
    thresh = np.stack(km.thresh)
    cb, cs = c_oracle.kmnc(act[sub], thresh)
    assert np.array_equal(bucket[sub], cb) and np.array_equal(score[sub], cs)
    # size-independent properties on the full output
    assert np.array_equal(score, (bucket >= 0).sum(axis=1))
    inside = (act >= mins) & (act < thresh[-1]) & (km._jumps > 0)
    assert np.array_equal(bucket >= 0, inside)
    lo = mins + km._jumps * np.maximum(bucket, 0)
    hi = mins + km._jumps * (np.maximum(bucket, 0) + 1)
    ok = bucket < 0
    assert np.all(ok | ((lo <= act) & (act < hi)))


@pytest.mark.parametrize("k", [2, 37, 1000])
def test_kmnc_adversarial_statistics_and_values(k):
    """Every neuron kind the fast path folds into constants (regular, negative minimum, constant, inverted, NaN
    statistics, minimum so large that min + jump rounds back to min, underflowing jump) against every value kind
    (NumPy's own thresholds and their float neighbours, the minimum, the maximum, zeros of both signs, NaN, infinities,
    FLT_MAX, denormals), enough rows for the column-strip kernel: dense NumPy restatement of the predicate, bit for bit."""
    from src.core.neuron_coverage import KMNC

    rng = np.random.default_rng(k)
    n, d = 96, 512
    kinds = rng.integers(0, 9, size=d)
    mins = np.zeros(d, dtype=np.float32)
    maxs = rng.uniform(0.5, 3.0, size=d).astype(np.float32)
    mins[kinds == 1] = -2.0
    mins[kinds == 2], maxs[kinds == 2] = 0.7, 0.7                       # constant neuron
    mins[kinds == 3], maxs[kinds == 3] = 1.0, 0.0                       # inverted
    mins[kinds == 4] = np.nan
    mins[kinds == 5], maxs[kinds == 5] = 1e6, 1e6 + 1                   # fl(min + jump) == min for k >= 17
    mins[kinds == 6], maxs[kinds == 6] = 4096.0, 4097.0
    mins[kinds == 7], maxs[kinds == 7] = 0.0, 1e-38                     # jump is denormal, 1/jump overflows
    mins[kinds == 8], maxs[kinds == 8] = -1e-3, 1e-38
    with np.errstate(all="ignore"):
        lo, jumps, thresh = np_oracle.kmnc_thresholds([mins], [maxs], k)
        thresh = np.stack(thresh)
        act = (mins + (maxs - mins) * rng.uniform(-0.1, 1.1, size=(n, d))).astype(np.float32)
        pick = rng.integers(0, k + 1, size=(n, d))
        edge = np.take_along_axis(thresh, pick, axis=0).astype(np.float32)
        how = rng.integers(0, 12, size=(n, d))
        act = np.where(how == 0, edge, act)
        act = np.where(how == 1, np.nextafter(edge, np.float32(-np.inf)), act)
        act = np.where(how == 2, np.nextafter(edge, np.float32(np.inf)), act)
        act = np.where(how == 3, mins, act)
        act = np.where(how == 4, maxs, act).astype(np.float32)
        special = np.array([np.nan, np.inf, -np.inf, 0.0, -0.0, 3.4028235e38, -3.4028235e38, 1e-45, -1e-45, 1e-39],
                           dtype=np.float32)
        act = np.where(how == 5, special[rng.integers(0, special.size, size=(n, d))], act).astype(np.float32)
        want_b, hits = np_oracle.kmnc_buckets_oracle([mins], [maxs], k, act)
    assert hits.max() <= 1
    km = KMNC([mins], [maxs], k)
    score, bucket = km.buckets([act])
    assert np.array_equal(bucket, want_b)
    assert np.array_equal(score, (want_b >= 0).sum(axis=1))
    # and the same rows through the few-samples kernel
    s2, b2 = km.buckets([act[:8]])
    assert np.array_equal(b2, want_b[:8]) and np.array_equal(s2, score[:8])


# ------------------------------------------------------------------------------------------
# DSA
# ------------------------------------------------------------------------------------------
def test_dsa_golden_bit_exact(golden):
    from src.core.surprise import DSA

    g = golden("dsa_reference.npz")
    for name in case_names(g, "dsa"):
        kw = ast.literal_eval(str(g[f"{name}.kw"]))
        xtr, ytr, xte, pte = (g[f"{name}.{k}"] for k in ("xtr", "ytr", "xte", "pte"))
        sa = DSA(xtr, ytr, **kw)
        got = sa(xte, pte)
        assert got.dtype == np.float64 and got.shape == (xte.shape[0],)
        assert np.array_equal(got, g[f"{name}.dsa"], equal_nan=True), name
        assert np.array_equal(sa.last_dist_a, g[f"{name}.dist_a"]), name
        assert np.array_equal(sa.last_dist_b, g[f"{name}.dist_b"]), name
        want = np_oracle.dsa_oracle(xtr, ytr, xte, pte, **kw)
        assert np.array_equal(sa.last_winner_index, want["idx_a"]), name      # argmin indices
        # exhaustive (no tensor-core filter) path gives the same bits
        sa.use_filter = False
        assert np.array_equal(sa(xte, pte), g[f"{name}.dsa"], equal_nan=True), name


def test_dsa_fit_time_table_gives_the_same_bits(golden):
    """Extension: DSA.fit_other_class_table() tabulates dist_b per train row at fit time; calls then run stage 1 only.
    Same score, dist_a, dist_b and winner bits as the reference's golden vectors and as the two-stage call (eager
    first call, captured second, replayed third), float32 and float64, including a class without other classes'
    rows missing (every class present) and labels the reference never scores."""
    from src.core.surprise import DSA

    g = golden("dsa_reference.npz")
    for name in case_names(g, "dsa"):
        kw = ast.literal_eval(str(g[f"{name}.kw"]))
        xtr, ytr, xte, pte = (g[f"{name}.{k}"] for k in ("xtr", "ytr", "xte", "pte"))
        sa = DSA(xtr, ytr, **kw).fit_other_class_table()
        for _ in range(3):
            got = sa(xte, pte)
            assert np.array_equal(got, g[f"{name}.dsa"], equal_nan=True), name
            assert np.array_equal(sa.last_dist_a, g[f"{name}.dist_a"]), name
            assert np.array_equal(sa.last_dist_b, g[f"{name}.dist_b"]), name
    for dt in (np.float32, np.float64):
        xtr, ytr, xte, pte, _ = np_oracle.synth_clusters(9000, 2500, 96, 7, seed=31)
        xtr, xte = xtr.astype(dt), xte.astype(dt)
        pte = pte.copy()
        pte[::97] = 11                                   # never scored (label outside the training classes)
        sa = DSA(xtr, ytr)
        want = [sa(xte, pte).copy(), sa.last_dist_a.copy(), sa.last_dist_b.copy(), sa.last_winner_index.copy()]
        sa.fit_other_class_table()
        for _ in range(3):
            got = [sa(xte, pte), sa.last_dist_a, sa.last_dist_b, sa.last_winner_index]
            for a, b in zip(got, want):
                assert np.array_equal(a, b, equal_nan=True)
        sa.drop_other_class_table()
        assert np.array_equal(sa(xte, pte), want[0], equal_nan=True)


@pytest.mark.parametrize("n_train,n_test,d,classes,dt,seed", [
    (20000, 1500, 128, 10, np.float32, 2), (5000, 700, 64, 3, np.float32, 3), (3000, 257, 200, 7, np.float32, 4),
    (4000, 300, 128, 10, np.float64, 5), (1500, 100, 1600, 4, np.float32, 6), (900, 130, 9, 2, np.float32, 7)])
def test_dsa_random_vs_c_oracle(n_train, n_test, d, classes, dt, seed):
    from src.core.surprise import DSA

    xtr, ytr, xte, pte, _ = np_oracle.synth_clusters(n_train, n_test, d, classes, seed=seed, dtype=dt)
    want = c_oracle.dsa(xtr, ytr, xte, pte)
    sa = DSA(xtr, ytr)
    got = sa(xte, pte)
    assert np.array_equal(sa.last_winner_index, want["idx_a"])
    assert np.array_equal(sa.last_dist_a, want["dist_a"]) and np.array_equal(sa.last_dist_b, want["dist_b"])
    assert np.array_equal(got, want["dsa"])
    # the filter, not the fallback, did the work
    stats = sa._engine.stats.cpu().numpy()
    assert stats[0] == 0, f"{stats[0]} rows fell back to the exhaustive scan"
    cands = sum(int(cnt.sum().item()) for cnt, _ in sa._engine.last_cand_cnt_by_mode.values())
    assert 2 * n_test <= cands <= 2 * n_test * 40, f"candidate lists unexpectedly long (or empty): {cands}"
    # determinism (reference tests/test_surprise.py:165-171)
    assert np.array_equal(sa(xte, pte), got)


def test_dsa_heavy_ties_and_overflow_fallback():
    """Many exactly tied distances (integer grid, duplicated rows): lowest original index must
    win, also when the candidate list overflows and the exhaustive scan takes over."""
    from src.core.surprise import DSA

    rng = np.random.default_rng(9)
    base = rng.integers(0, 2, size=(40, 16)).astype(np.float32)
    xtr = np.tile(base, (30, 1))                       # every row 30 times
    ytr = np.tile(np.arange(40) % 2, 30).astype(np.int64)
    xte = rng.integers(0, 2, size=(300, 16)).astype(np.float32)
    pte = rng.integers(0, 2, size=300).astype(np.int64)
    want = c_oracle.dsa(xtr, ytr, xte, pte)
    sa = DSA(xtr, ytr)
    got = sa(xte, pte)
    assert np.array_equal(sa.last_winner_index, want["idx_a"])
    assert np.array_equal(got, want["dsa"], equal_nan=True)
    sa._engine.cap = 4                                  # force overflow -> exhaustive rows
    assert np.array_equal(sa(xte, pte), want["dsa"], equal_nan=True)
    assert sa._engine.stats.cpu().numpy()[0] > 0
    # second sighting captures the plan, later calls replay it: the replayed graph carries no exhaustive-scan launches,
    # counts the overflowed lists instead, and the call is repeated on the eager path — same bits every time
    for _ in range(3):
        assert np.array_equal(sa(xte, pte), want["dsa"], equal_nan=True)
        assert np.array_equal(sa.last_winner_index, want["idx_a"])
    plan = next(iter(sa._engine._plans.values()))
    assert plan.speculative and int(plan.overflow.item()) == 0     # detected, cleared, repeated
    sa._engine.cap = 64
    for _ in range(3):                                             # and back to lists that fit: the graph's own result
        assert np.array_equal(sa(xte, pte), want["dsa"], equal_nan=True)


def test_dsa_edge_cases():
    from src.core.surprise import DSA

    xtr, ytr, xte, pte, _ = np_oracle.synth_clusters(400, 50, 24, 4, seed=21)
    sa = DSA(xtr, ytr)
    assert sa(xte[:0], pte[:0]).shape == (0,)
    one = sa(xte[:1], pte[:1])
    assert np.array_equal(one, np_oracle.dsa_oracle(xtr, ytr, xte[:1], pte[:1])["dsa"])
    # labels beyond the training classes are never scored by the reference (np.empty garbage): NaN here
    p2 = pte.copy()
    p2[:5] = 9
    got = sa(xte, p2)
    assert np.isnan(got[:5]).all()
    assert np.array_equal(got[5:], np_oracle.dsa_oracle(xtr, ytr, xte, pte)["dsa"][5:])
    # a class without training rows raises like np.min of an empty array (surprise.py:645)
    y2 = ytr.copy()
    y2[y2 == 1] = 0
    with pytest.raises(ValueError):
        DSA(xtr, y2)(xte, np.ones(50, dtype=np.int64))
    with pytest.raises(AssertionError, match="must be one-dimensional"):
        sa(xte, pte[None, :])
    with pytest.raises(ValueError, match="subsampling"):
        DSA(xtr, ytr, subsampling=-1)


@pytest.mark.parametrize("subsampling", [1.0, 0.3])
def test_dsa_config2_full_size_properties(subsampling):
    """BASELINE config 2 (10k x 60k x 128 fp32): checked on a random row subset against the C
    oracle (exhaustive over all 60k rows) and through size-independent properties."""
    from src.core.surprise import DSA

    xtr, ytr, xte, pte, _ = np_oracle.synth_clusters(60000, 10000, 128, 10, seed=2)
    sa = DSA(xtr, ytr, subsampling=subsampling)
    got = sa(xte, pte)
    assert np.isfinite(got).all() and (got > 0).all()
    rows = np.random.default_rng(0).choice(10000, size=96, replace=False)
    want = c_oracle.dsa(sa.train_activations, sa.train_predictions, xte[rows], pte[rows])
    assert np.array_equal(sa.last_winner_index[rows], want["idx_a"])
    assert np.array_equal(got[rows], want["dsa"])
    # properties: the winner has the predicted class; dist_a is the exact distance to it
    w = sa.last_winner_index
    assert np.array_equal(sa.train_predictions[w], pte)
    sub = rows[:32]
    exact = np.linalg.norm(xte[sub] - sa.train_activations[w[sub]], axis=1)
    assert np.array_equal(exact.astype(np.float32), sa.last_dist_a[sub])
    # train rows as queries: distance 0, winner = lowest index among identical rows
    probe = sa.train_activations[:64]
    z = sa(probe, sa.train_predictions[:64])
    assert (z == 0).all() and np.array_equal(sa.last_winner_index, np.arange(64))
    # idempotence / permutation equivariance
    perm = np.random.default_rng(1).permutation(10000)
    assert np.array_equal(sa(xte[perm], pte[perm]), got[perm])
    assert sa._engine.stats.cpu().numpy()[0] == 0


# ------------------------------------------------------------------------------------------
# LSA
# ------------------------------------------------------------------------------------------
def _close(got, want):
    assert np.array_equal(np.isinf(got), np.isinf(want)), (np.isinf(got).sum(), np.isinf(want).sum())
    assert np.array_equal(np.sign(got[np.isinf(got)]), np.sign(want[np.isinf(want)]))
    f = np.isfinite(want)
    np.testing.assert_allclose(got[f], want[f], rtol=LSA_RTOL, atol=LSA_ATOL)


def test_lsa_golden(golden):
    from src.core.surprise import LSA, MultiModalSA

    g = golden("lsa_reference.npz")
    for name, kw in (("plaus", {}), ("cube", {}), ("mf30", {"max_features": 30}), ("far", {})):
        sa = LSA(g[f"{name}.xtr"], **kw)
        _close(sa(g[f"{name}.xte"]), g[f"{name}.lsa"])
    assert np.array_equal(np.array(LSA(g["mf30.xtr"], max_features=30).removed_neurons), g["mf30.removed"])
    with pytest.warns(UserWarning):
        sing = LSA(g["singular.xtr"])
    assert sing.kde.prepare_failed
    assert np.isinf(sing(g["singular.xte"])).all()
    mm = MultiModalSA.build_by_class(g["mf30.xtr"], g["pclsa.ytr"], lambda x, y: LSA(x))
    _close(mm(g["mf30.xte"], g["pclsa.pte"]), g["pclsa.lsa"])


@pytest.mark.parametrize("n_train,n_test,d,seed,dt", [(6000, 500, 256, 3, np.float32), (3000, 300, 20, 4, np.float32),
                                                      (2500, 129, 300, 5, np.float32), (1000, 64, 10, 6, np.float64)])
def test_lsa_random_vs_oracle(n_train, n_test, d, seed, dt):
    from src.core.surprise import LSA

    xtr, _, xte, _, _ = np_oracle.synth_clusters(n_train, n_test, d, 4, seed=seed, dtype=dt, spread=1.0)
    want = np_oracle.lsa_oracle(xtr, xte)
    got = LSA(xtr)(xte)
    _close(got, want)
    assert np.array_equal(LSA(xtr)(xte), got)            # deterministic across fits and calls


def test_lsa_repeated_batch_shapes_replay_a_graph_with_the_same_bits():
    """A batch shape seen for the second time is captured as one CUDA graph and replayed from then on
    (stable_kde._DensityPlan): eager first call, capturing second call and replays give the same bits, for NumPy and
    device-resident inputs, for other data of the same shape, with and without the one-segment fast pass, and for the
    per-class LSAs of a MultiModalSA (ten plans in flight); a different shape in between does not disturb a plan."""
    torch = _torch()
    from src.core.surprise import LSA, MultiModalSA

    for n_train, n_test, d in ((5000, 1500, 256), (3000, 300, 24)):        # with / without the fast pass
        xtr, ytr, xte, pte, _ = np_oracle.synth_clusters(n_train, n_test, d, 5, seed=41, spread=1.0)
        xte2 = np.ascontiguousarray(xte[::-1])
        sa = LSA(xtr)
        first = sa(xte)
        _close(first, np_oracle.lsa_oracle(xtr, xte))
        for _ in range(3):
            assert np.array_equal(sa(xte), first)
        assert any(k[0] == n_test for k in sa.kde._plans)                   # the graph path is what ran
        assert np.array_equal(sa(torch.from_numpy(xte).cuda()), first)
        other = sa(xte2)                                                    # same shape, other data: same plan
        assert np.array_equal(other, first[::-1])
        part = sa(xte[:77])                                                 # another shape in between (batches under 1024
        _close(part, first[:77])                                            # inputs never try the one-segment pass)
        assert np.array_equal(sa(xte[:77]), part)
        assert np.array_equal(sa(xte), first)
        mm = MultiModalSA.build_by_class(xtr, ytr, lambda x, y: LSA(x))
        want = mm(xte, pte)
        for _ in range(3):
            assert np.array_equal(mm(xte, pte), want, equal_nan=True)


def test_lsa_bf16_stored_traces_config3_shape():
    """BASELINE config 3 shape at reduced N: traces stored in bf16; both sides see the same
    bf16-rounded values (SURVEY.md 8d)."""
    torch = _torch()
    from src.core.surprise import LSA

    xtr, _, xte, _, _ = np_oracle.synth_clusters(8000, 400, 256, 10, seed=3, spread=1.0)
    r = lambda a: torch.from_numpy(a).to(torch.bfloat16).to(torch.float32).numpy()
    xtr, xte = r(xtr), r(xte)
    _close(LSA(xtr)(xte), np_oracle.lsa_oracle(xtr, xte))


def test_lsa_api_edges():
    from src.core.surprise import LSA

    rng = np.random.RandomState(0)
    x = rng.random((500, 12))
    with pytest.raises(AssertionError):
        LSA(x, var_threshold=0.1, max_features=5)
    sa = LSA(x)
    assert sa(x[:0]).shape == (0,)
    assert sa(x[:1]).shape == (1,)
    _close(sa(x[:50].reshape(50, 3, 4)), np_oracle.lsa_oracle(x, x[:50]))


# ------------------------------------------------------------------------------------------
# BASELINE config 5 shape (D = 2048, many classes, ragged class sizes) at reduced N
# ------------------------------------------------------------------------------------------
def test_dsa_config5_shape_streaming_kernel():
    """Exercises the streaming tcgen05 kernel (33 K-chunks), 100 classes with ragged sizes and
    query tiles that are mostly partial; checked against the C oracle on a row subset and against
    the exhaustive GPU scan on every row."""
    from src.core.surprise import DSA

    rng = np.random.default_rng(5)
    classes, d = 100, 2048
    sizes = rng.integers(40, 400, size=classes)
    ytr = np.repeat(np.arange(classes), sizes)
    rng.shuffle(ytr)
    centres = rng.normal(0.0, 0.5, size=(classes, d)).astype(np.float32)
    xtr = (centres[ytr] + rng.normal(size=(ytr.size, d)).astype(np.float32)).astype(np.float32)
    yte = rng.integers(0, classes, size=3000)
    xte = (centres[yte] + rng.normal(size=(3000, d)).astype(np.float32)).astype(np.float32)
    pte = yte.copy()
    flip = rng.random(3000) < 0.1
    pte[flip] = rng.integers(0, classes, size=int(flip.sum()))
    sa = DSA(xtr, ytr)
    got = sa(xte, pte)
    win, da, db = sa.last_winner_index.copy(), sa.last_dist_a.copy(), sa.last_dist_b.copy()
    assert sa._engine.stats.cpu().numpy()[0] == 0
    rows = rng.choice(3000, size=48, replace=False)
    want = c_oracle.dsa(xtr, ytr, xte[rows], pte[rows])
    assert np.array_equal(win[rows], want["idx_a"])
    assert np.array_equal(da[rows], want["dist_a"]) and np.array_equal(db[rows], want["dist_b"])
    assert np.array_equal(got[rows], want["dsa"])
    sa.use_filter = False
    assert np.array_equal(sa(xte, pte), got)
    assert np.array_equal(sa.last_winner_index, win)


# ------------------------------------------------------------------------------------------
# device-resident traces: torch CUDA tensors in, same bits out (no host round trip of the traces)
# ------------------------------------------------------------------------------------------
def test_device_resident_traces_give_the_same_bits():
    torch = _torch()
    from src.core.deepgini import DeepGini
    from src.core.neuron_coverage import KMNC
    from src.core.surprise import DSA, LSA

    dev = torch.device("cuda", 0)
    xtr, ytr, xte, pte, _ = np_oracle.synth_clusters(6000, 700, 128, 6, seed=11)
    want = c_oracle.dsa(xtr, ytr, xte, pte)
    # fit and score from HBM; layers arrive as a list of [N, ...] tensors like a forward hook yields them
    tr_layers = [torch.from_numpy(xtr[:, :48]).to(dev).reshape(-1, 4, 12), torch.from_numpy(xtr[:, 48:]).to(dev)]
    te_layers = [torch.from_numpy(xte[:, :48]).to(dev).reshape(-1, 4, 12), torch.from_numpy(xte[:, 48:]).to(dev)]
    sa = DSA(tr_layers, torch.from_numpy(ytr).to(dev), subsampling=1.0)
    got = sa(te_layers, torch.from_numpy(pte).to(dev))
    assert np.array_equal(got, want["dsa"]) and np.array_equal(sa.last_winner_index, want["idx_a"])
    # seeded sub-sampling picks the same rows on the device as on the host
    a = DSA(xtr, ytr, subsampling=0.3, subsampling_seed=5)(xte, pte)
    b = DSA(torch.from_numpy(xtr).to(dev), ytr, subsampling=0.3, subsampling_seed=5)(torch.from_numpy(xte).to(dev), pte)
    assert np.array_equal(a, b)

    xs, _, xt, _, _ = np_oracle.synth_clusters(2000, 300, 40, 3, seed=12)
    lsa = LSA(xs)
    assert np.array_equal(lsa(xt), lsa(torch.from_numpy(xt).to(dev)))

    act, mins, maxs = np_oracle.synth_relu(300, 1024, seed=13)
    km = KMNC([mins], [maxs], 50)
    score, bucket = km.buckets([act])
    score_d, bucket_d = km.buckets([torch.from_numpy(act).to(dev)], device_out=True)
    assert score_d.is_cuda and np.array_equal(score_d.cpu().numpy(), score) and np.array_equal(bucket_d.cpu().numpy(), bucket)

    rng = np.random.default_rng(14)
    logits = rng.normal(size=(500, 10)).astype(np.float32) * 3
    p = np.exp(logits) / np.exp(logits).sum(1, keepdims=True)
    pred, gini = DeepGini.calculate(p)
    pred_d, gini_d = DeepGini.calculate(torch.from_numpy(p).to(dev))
    assert np.array_equal(pred, pred_d) and np.array_equal(gini, gini_d)


# ------------------------------------------------------------------------------------------
# CAM over compact KMNC profiles (SURVEY.md §8 f1): same order as the reference's generator
# ------------------------------------------------------------------------------------------
def test_cam_from_buckets_matches_reference_order(golden):
    torch = _torch()
    from src.core.neuron_coverage import KMNC
    from src.core.prioritizers import cam_from_buckets

    g = golden("cam_kmnc_reference.npz")
    for i in range(4):
        bucket, score, k = g[f"camk{i}.bucket"], g[f"camk{i}.score"], int(g[f"camk{i}.sections"])
        got = np.array(list(cam_from_buckets(score, bucket, k)), dtype=np.int64)
        assert np.array_equal(got, g[f"camk{i}.order"]), i                 # order of the unmodified reference
        got16 = np.array(list(cam_from_buckets(score, bucket.astype(np.int16), k)), dtype=np.int64)
        assert np.array_equal(got16, got), i
    # larger case, end to end on the device: KMNC bucket ids never leave HBM
    act, mins, maxs = np_oracle.synth_relu(1500, 512, seed=21)
    km = KMNC([mins], [maxs], 100)
    score_d, bucket_d = km.buckets([torch.from_numpy(act).to("cuda")], device_out=True)
    score = score_d.cpu().numpy()
    got = np.array(list(cam_from_buckets(score, bucket_d, 100)), dtype=np.int64)
    want = np_oracle.cam_from_buckets_oracle(score, bucket_d.cpu().numpy(), 100)
    assert np.array_equal(got, want)
    assert sorted(got.tolist()) == list(range(1500))
    # degenerate inputs: nothing coverable -> pure score order; a single sample
    none = np.full((7, 5), -1, dtype=np.int32)
    s = np.array([3, 1, 4, 1, 5, 9, 2])
    assert np.array_equal(np.array(list(cam_from_buckets(s, none, 3))), np_oracle.cam_from_buckets_oracle(s, none, 3))
    one = np.array([[0, 2, -1]], dtype=np.int32)
    assert list(cam_from_buckets(np.array([2]), one, 3)) == [0]


# ------------------------------------------------------------------------------------------
# launch modes of DSA.__call__: first sighting of a batch shape = eager launches, second = CUDA-graph
# capture, later = replay; all give the oracle's bits
# ------------------------------------------------------------------------------------------
def test_dsa_eager_capture_replay_give_the_same_bits():
    from src.core.surprise import DSA

    xtr, ytr, xte, pte, _ = np_oracle.synth_clusters(9000, 1100, 128, 7, seed=31)
    want = c_oracle.dsa(xtr, ytr, xte, pte)
    sa = DSA(xtr, ytr)
    assert len(sa._engine._plans) == 0
    for call in range(4):
        got = sa(xte, pte)
        assert np.array_equal(got, want["dsa"]), call
        assert np.array_equal(sa.last_winner_index, want["idx_a"]), call
        assert np.array_equal(sa.last_dist_b, want["dist_b"]), call
        assert len(sa._engine._plans) == (0 if call == 0 else 1), call      # eager, then one captured plan
    # a different batch in between does not disturb the captured plan
    assert np.array_equal(sa(xte[:300], pte[:300]), want["dsa"][:300])
    assert np.array_equal(sa(xte, pte), want["dsa"])
    # labels beyond the training classes: those rows stay NaN / -1 through the captured plan's fused scatter too
    p2 = pte.copy()
    p2[::50] = 99
    for call in range(3):
        got = sa(xte, p2)
        assert np.isnan(got[::50]).all() and (sa.last_winner_index[::50] == -1).all(), call
        keep = np.ones(pte.shape[0], dtype=bool)
        keep[::50] = False
        assert np.array_equal(got[keep], want["dsa"][keep]), call
    eager_first = DSA(xtr, ytr)
    eager_first.capture_on_first_call = True
    assert np.array_equal(eager_first(xte, pte), want["dsa"]) and len(eager_first._engine._plans) == 1
    # wrong trace width: ValueError like the reference's broadcasting error, never an out-of-bounds read
    with pytest.raises(ValueError):
        sa(xte[:, :100], pte)


# ------------------------------------------------------------------------------------------
# BASELINE configs at their stated sizes (sampled rows against the oracle + size-independent properties)
# ------------------------------------------------------------------------------------------
def test_lsa_config3_full_size():
    """C3: LSA 10k x 60k x 256, traces stored in bf16.  256 sampled inputs against the float64 oracle
    (explicit residuals) with the plain north_star tolerance rtol 1e-4 — no absolute floor — and the APFD
    of the resulting order within 1e-6 of the oracle's on those inputs."""
    torch = _torch()
    from src.core.apfd import apfd_from_order
    from src.core.surprise import LSA

    xtr, _, xte, pte, yte = np_oracle.synth_clusters(60000, 10000, 256, 10, seed=3, spread=1.0)
    r = lambda a: torch.from_numpy(a).to(torch.bfloat16).to(torch.float32).numpy()
    xtr, xte = r(xtr), r(xte)
    sa = LSA(xtr)
    got = sa(xte)
    assert got.shape == (10000,) and np.isfinite(got).all()
    sub = np.sort(np.random.default_rng(0).choice(10000, 256, replace=False))
    want = np_oracle.lsa_oracle(xtr, xte[sub], exact=True)
    rel = np.abs(got[sub] - want) / np.abs(want)
    assert rel.max() <= 1e-4, rel.max()
    fault = (pte != yte)[sub]
    assert fault.any()
    assert abs(apfd_from_order(fault, np.argsort(-got[sub])) - apfd_from_order(fault, np.argsort(-want))) <= 1e-6
    # properties: deterministic; row order does not matter; training points are less surprising than far ones
    perm = np.random.default_rng(1).permutation(10000)
    assert np.array_equal(sa(xte[perm]), got[perm])
    assert sa(xtr[:256]).mean() < got.mean() < sa(xte[:256] + 3.0).mean()


def test_kmnc_config4_full_size():
    """C4: KMNC 10k x 4096, 1000 sections: 48 sampled inputs against the C oracle (thresholds exactly as NumPy
    builds them), every row through the definition of a section."""
    from src.core.neuron_coverage import KMNC

    act, mins, maxs = np_oracle.synth_relu(10000, 4096, seed=4)
    km = KMNC([mins], [maxs], 1000)
    score, bucket = km.buckets([act])
    assert bucket.shape == (10000, 4096) and score.shape == (10000,)
    sub = np.sort(np.random.default_rng(0).choice(10000, size=48, replace=False))
    thresh = np.stack(km.thresh)
    cb, cs = c_oracle.kmnc(act[sub], thresh)
    assert np.array_equal(bucket[sub], cb) and np.array_equal(score[sub], cs)
    assert np.array_equal(score, (bucket >= 0).sum(axis=1))
    inside = (act >= mins) & (act < thresh[-1]) & (km._jumps > 0)
    assert np.array_equal(bucket >= 0, inside)
    b = np.maximum(bucket, 0).astype(np.int64)
    lo = np.take_along_axis(thresh, b, axis=0)
    hi = np.take_along_axis(thresh, b + 1, axis=0)
    assert np.all((bucket < 0) | ((lo <= act) & (act < hi)))


def test_dsa_config5_slice_vs_oracle():
    """C5 shape (2048-d, 1000 classes, bf16-representable traces from the device-side counter RNG) at a
    slice that one GPU scores in a blink: 3000 test x 128k train.  The device RNG equals its host twin bit
    for bit, and 40 sampled inputs equal the CPU ORACLE (brute force over all 128k rows) bit for bit."""
    torch = _torch()
    from oracle import synth_traces as ST
    from src.core.surprise import DSA

    dev = torch.device("cuda", 0)
    n_train, n_test, d, classes, seed = 128000, 3000, 2048, 1000, 5
    xtr = torch.empty((n_train, d), dtype=torch.float32, device=dev)
    ST.fill(xtr, 0, d, classes, seed, 0)
    xte = torch.empty((n_test, d), dtype=torch.float32, device=dev)
    ST.fill(xte, 0, d, classes, seed, 1)
    ytr = np.arange(n_train) % classes
    pte = np.arange(n_test) % classes
    pte[::17] = (pte[::17] + 3) % classes                     # some mispredictions
    rows = np.sort(np.random.default_rng(2).choice(n_train, 50, replace=False))
    assert np.array_equal(ST.traces(torch.from_numpy(rows), d, classes, seed, 0).numpy(), xtr[torch.from_numpy(rows).to(dev)].cpu().numpy())
    assert torch.equal(xtr, xtr.to(torch.bfloat16).to(torch.float32))          # bf16 storage is lossless
    sa = DSA(xtr, ytr)                                       # device tensors in: no host round trip
    got = sa(xte, pte)
    assert np.isfinite(got).all() and sa._engine.stats.cpu().numpy()[0] == 0
    sel = np.sort(np.random.default_rng(3).choice(n_test, 40, replace=False))
    want = c_oracle.dsa(xtr.cpu().numpy(), ytr, ST.traces(torch.from_numpy(sel), d, classes, seed, 1).numpy(), pte[sel])
    assert np.array_equal(sa.last_winner_index[sel], want["idx_a"])
    assert np.array_equal(sa.last_dist_a[sel], want["dist_a"]) and np.array_equal(sa.last_dist_b[sel], want["dist_b"])
    assert np.array_equal(got[sel], want["dsa"])
    assert np.array_equal(sa(xte, pte), got)                 # captured plan, same bits


def test_lsa_orders_give_the_oracles_apfd(golden):
    """APFD parity for the not-bit-exact scorers (BASELINE.md: |dAPFD| <= 1e-6): LSA and per-class LSA."""
    from src.core.apfd import apfd_from_order
    from src.core.surprise import LSA, MultiModalSA

    xtr, ytr, xte, pte, yte = np_oracle.synth_clusters(5000, 1500, 64, 5, seed=41, spread=1.0)
    fault = pte != yte
    got = LSA(xtr)(xte)
    want = np_oracle.lsa_oracle(xtr, xte)
    assert abs(apfd_from_order(fault, np.argsort(-got)) - np_oracle.apfd_oracle(fault, np.argsort(-want))) <= 1e-6
    pc = MultiModalSA.build_by_class(xtr, ytr, lambda x, y: LSA(x))(xte, pte)
    want_pc = np_oracle.pc_lsa_oracle(xtr, ytr, xte, pte)
    assert abs(apfd_from_order(fault, np.argsort(-pc)) - np_oracle.apfd_oracle(fault, np.argsort(-want_pc))) <= 1e-6
    rel = np.abs(got - want) / np.maximum(np.abs(want), 1e-300)
    print(f"LSA max relative error without an absolute floor: {rel.max():.3e}; elements needing the 2e-4 floor: "
          f"{int((rel > 1e-4).sum())} of {rel.size}")


# ------------------------------------------------------------------------------------------
# SURVEY.md §8 f2: NAC / NBC / SNAC / TKNC and the streaming statistics on the GPU, bit for bit against the
# outputs of the reference's own classes; §8 f1: CAM over dense boolean / bit-packed profiles
# ------------------------------------------------------------------------------------------
def _sibling_metrics(nc, mins, maxs, stds):
    m = {"NAC_0": nc.NAC(0.0), "NAC_0.75": nc.NAC(0.75), "TKNC_1": nc.TKNC(1), "TKNC_2": nc.TKNC(2), "TKNC_3": nc.TKNC(3)}
    for sc in (0, 0.5, 1):
        m[f"NBC_{sc}"] = nc.NBC(mins, maxs, stds, sc)
        m[f"SNAC_{sc}"] = nc.SNAC(maxs, stds, sc)
    return m


def test_sibling_coverage_and_statistics_golden(golden):
    torch = _torch()
    import src.core.neuron_coverage as nc
    from src.core.prioritizers import cam, cam_from_bits
    from src.dnn_test_prio.aggregate_statistics import AggregateStatisticsCollector

    s = golden("siblings_reference.npz")
    train = [s[f"sib.train{i}"] for i in range(3)]
    test = [s[f"sib.test{i}"] for i in range(3)]
    cuts = s["sib.cuts"]
    col = AggregateStatisticsCollector()
    for a, b in zip(cuts[:-1], cuts[1:]):
        col.track([l[a:b] for l in train])
    mins, maxs, stds = col.get()
    for i in range(3):
        for got, key in ((mins[i], "min"), (maxs[i], "max"), (stds[i], "std")):
            want = s[f"sib.{key}{i}"]
            assert got.shape == want.shape and got.dtype == want.dtype and np.array_equal(got, want), (key, i)
    # badges straight from HBM (forward-hook tensors) give the same statistics
    col_d = AggregateStatisticsCollector()
    for a, b in zip(cuts[:-1], cuts[1:]):
        col_d.track([torch.from_numpy(l[a:b]).cuda() for l in train])
    for got, want in zip(col_d.get()[2], stds):
        assert np.array_equal(got, want)
    for name, metric in _sibling_metrics(nc, mins, maxs, stds).items():
        score, prof = metric([l.copy() for l in test])
        want_s, want_p = s[f"sib.{name}.score"], s[f"sib.{name}.profile"]
        assert score.dtype == want_s.dtype and np.array_equal(score, want_s), name
        assert prof.dtype == bool and prof.shape == want_p.shape and np.array_equal(prof, want_p), name
        # CAM: dense signature of the reference, and the bit-packed profile that never left HBM
        assert np.array_equal(np.array(list(cam(score, prof))), s[f"sib.{name}.cam"]), name
        sc_d, bits = metric.packed([torch.from_numpy(l).cuda() for l in test])
        assert np.array_equal(sc_d.cpu().numpy(), want_s.astype(np.int32)), name
        assert np.array_equal(np.array(list(cam_from_bits(score, bits))), s[f"sib.{name}.cam"]), name
    # float64 statistics and activations
    tr64 = [l.astype(np.float64) for l in train[:2]]
    col = AggregateStatisticsCollector()
    col.track(tr64)
    mn, mx, sd = col.get()
    for i in range(2):
        assert np.array_equal(mn[i], s[f"sib64.min{i}"]) and np.array_equal(mx[i], s[f"sib64.max{i}"])
        assert sd[i].dtype == np.float64 and np.array_equal(sd[i], s[f"sib64.std{i}"])
    sc64, p64 = nc.NBC(mn, mx, sd, 0.5)([l.astype(np.float64) for l in test[:2]])
    assert np.array_equal(sc64, s["sib64.NBC_0.5.score"]) and np.array_equal(p64, s["sib64.NBC_0.5.profile"])
    # surprise-coverage CAM (handler_surprise.py:101-115): 1000 buckets up to the largest value
    from src.core.surprise import SurpriseCoverageMapper

    prof = SurpriseCoverageMapper(1000, np.max(s["sc.values"])).get_coverage_profile(s["sc.values"])
    assert np.array_equal(prof, s["sc.profile"])
    assert np.array_equal(np.array(list(cam(s["sc.values"], prof))), s["sc.cam"])


def test_sibling_coverage_study_shapes_vs_oracle():
    """The study's layer widths (MNIST: 36 384 neurons over 4 layers, case_study_mnist.py:50-62): scores and profiles of
    every criterion equal the NumPy oracle's; reference known answers (tests/test_coverage_metrics.py)."""
    torch = _torch()
    import src.core.neuron_coverage as nc
    from src.core.prioritizers import cam
    from src.dnn_test_prio.aggregate_statistics import AggregateStatisticsCollector

    rng = np.random.default_rng(81)
    shapes = [(26, 26, 32), (13, 13, 32), (11, 11, 64), (5, 5, 64)]            # 21632 + 5408 + 7744 + 1600 = 36384
    def draw(n, scale):
        return [np.maximum(rng.normal(size=(n,) + sh).astype(np.float32) * scale + 0.1, 0) for sh in shapes]
    train, test = draw(96, 1.0), draw(64, 1.3)
    col = AggregateStatisticsCollector()
    col.track([l[:50] for l in train])
    col.track([l[50:] for l in train])
    mins, maxs, stds = col.get()
    o_min, o_max, o_std = np_oracle.stats_oracle([[l[:50] for l in train], [l[50:] for l in train]])
    for i in range(4):
        assert np.array_equal(mins[i], o_min[i]) and np.array_equal(maxs[i], o_max[i]) and np.array_equal(stds[i], o_std[i]), i
    want = {"NAC_0.75": np_oracle.nac_oracle(0.75, test), "NBC_0.5": np_oracle.nbc_oracle(mins, maxs, stds, 0.5, test),
            "SNAC_0": np_oracle.snac_oracle(maxs, stds, 0, test)}
    got = _sibling_metrics(nc, mins, maxs, stds)
    for name, (ws, wp) in want.items():
        gs, gp = got[name](test)
        assert gs.dtype == ws.dtype and np.array_equal(gs, ws) and np.array_equal(gp, wp), name
    # TKNC on tie-free layers (positive part only has ties at 0, never among the top 3 of these layers)
    dense = [rng.normal(size=(64, 500)).astype(np.float32), rng.normal(size=(64, 7, 9)).astype(np.float32)]
    for k in (1, 2, 3, 10):
        ws, wp = np_oracle.tknc_oracle(k, dense)
        gs, gp = nc.TKNC(k)(dense)
        assert np.array_equal(gs, ws) and np.array_equal(gp, wp), k
    # reference known answers: tests/test_coverage_metrics.py:67-168
    acts = [np.array([[0.1, 0.4, 0.9, 0.4], [0.1, 0.9, 0.9, 0.4]]), np.array([[0.3, 0.2, 0.1, 0.6, 0.8], [0.3, 0.9, 0.1, 0.6, 0.8]]),
            np.array([[0.2, 0.3, 0.4, 0.4], [0.2, 0.9, 0.4, 0.4]])]
    mn = [np.array([0] * 4), np.array([0] * 5), np.array([0.1] * 4)]
    mx = [np.array([1] * 4), np.array([1] * 5), np.array([0.95] * 4)]
    zero = [np.array([0] * 4), np.array([0] * 5), np.array([0] * 4)]
    pt2 = [np.array([0.2] * 4), np.array([0.2] * 5), np.array([0.2] * 4)]
    out = [a.copy() for a in acts]
    out[0][0][0], out[1][0][0] = -0.1, 1.5
    assert np.all(nc.NBC(mn, mx, zero, scaler=1)(acts)[0] == [0, 0])
    assert np.all(nc.NBC(mn, mx, zero, scaler=1)(out)[0] == [2, 0])
    assert np.all(nc.NBC(mn, mx, pt2, scaler=1)(out)[0] == [1, 0])
    assert np.all(nc.NBC(mn, mx, pt2, scaler=6)(out)[0] == [0, 0])
    assert np.all(nc.SNAC(mx, zero, scaler=1)(out)[0] == [1, 0]) and np.all(nc.SNAC(mx, pt2, scaler=6)(out)[0] == [0, 0])
    score, profile = nc.TKNC(2)(acts)
    assert np.all(score == [6, 6])
    assert np.all(profile[0][4:9] == [False, False, False, True, True]) and np.all(profile[0][9:] == [False, False, True, True])
    assert np.all(profile[0][:4] == [False, True, True, False]) or np.all(profile[0][:4] == [False, False, True, True])
    nac_score, nac_prof = nc.NAC(0.5)(acts)
    assert np.array_equal(nac_prof, np.concatenate(acts, axis=1) > 0.5) and np.all(nac_score == nac_prof.sum(axis=1))
    # dense CAM at a realistic size against the restated reference loop
    prof = rng.random((700, 3000)) < 0.02
    sc = prof.sum(axis=1)
    assert np.array_equal(np.array(list(cam(sc, prof))), np_oracle.cam_oracle(sc, prof))
    sc2 = rng.random(700)                                  # float scores: the tail is by score, the greedy part by coverage
    assert np.array_equal(np.array(list(cam(sc2, prof[:, :40]))), np_oracle.cam_oracle(sc2, prof[:, :40]))


# ------------------------------------------------------------------------------------------
# SURVEY.md §8 f3: MDSA / MLSA scored on the GPU (fits = the reference's sklearn calls)
# ------------------------------------------------------------------------------------------
def test_mdsa_mlsa_golden_and_live_sklearn(golden):
    from src.core.surprise import MDSA, MLSA, MultiModalSA

    g = golden("mdsa_mlsa_reference.npz")
    xtr, ytr, xte, pte = g["x.xtr"], g["x.ytr"], g["x.xte"], g["x.pte"]
    m = MDSA(xtr)
    np.testing.assert_allclose(m(xte), g["mdsa.out"], rtol=1e-4)
    np.testing.assert_allclose(m(xte), m.covariance_matrix.mahalanobis(xte), rtol=1e-4)      # the live third-party arithmetic
    pc = MultiModalSA.build_by_class(xtr, ytr, lambda x, y: MDSA(x))
    np.testing.assert_allclose(pc(xte, pte), g["pcmdsa.out"], rtol=1e-4)
    # float32 traces in, float64 distances out (sklearn validates to float and scipy's cdist returns float64)
    out32 = MDSA(xtr.astype(np.float32))(xte.astype(np.float32))
    assert out32.dtype == np.float64
    np.testing.assert_allclose(out32, g["mdsa.out"], rtol=2e-4)
    # singular covariance: sklearn's pinvh precision, eigen-factor whitening
    np.testing.assert_allclose(MDSA(g["sing.xtr"])(g["sing.xte"]), g["sing.out"], rtol=1e-4, atol=1e-6)
    # MLSA: the reference's fitted mixture (GaussianMixture's fit draws from NumPy's global RNG) ...
    np.random.seed(1234)
    ml = MLSA(xtr, num_components=3)
    ml.gmm.means_, ml.gmm.precisions_cholesky_, ml.gmm.weights_ = g["mlsa.means"], g["mlsa.prec_chol"], g["mlsa.weights"]
    ml._centres = None
    np.testing.assert_allclose(ml(xte), g["mlsa.out"], rtol=1e-4)
    # ... and a fresh fit against sklearn's own score_samples on this machine
    fresh = MLSA(xtr, num_components=3)
    np.testing.assert_allclose(fresh(xte), -fresh.gmm.score_samples(xte), rtol=1e-4)
    pcm = MultiModalSA.build_by_class(xtr, ytr, lambda x, y: MLSA(x, num_components=3))
    want = np.full(pte.shape, -np.inf)
    for c, sa in pcm.modal_sa.items():
        want[pte == c] = -sa.gmm.score_samples(xte[pte == c])
    np.testing.assert_allclose(pcm(xte, pte), want, rtol=1e-4)
    with pytest.raises(ValueError):
        m(xte[:, :5])


# ------------------------------------------------------------------------------------------
# SURVEY.md §8 f4: traces straight from forward hooks (never leaving HBM) through every scorer, results written in
# the reference's file layout and re-read as APFD
# ------------------------------------------------------------------------------------------
def test_forward_hook_traces_to_scores_to_result_files(tmp_path):
    torch = _torch()
    from simple_tip_b200.core import activations as A
    from simple_tip_b200.core import results as R
    from src.core.apfd import apfd_from_order
    from src.core.deepgini import DeepGini
    from src.core.neuron_coverage import KMNC, NAC
    from src.core.prioritizers import cam_from_bits, cam_from_buckets
    from src.core.surprise import DSA, LSA
    from src.dnn_test_prio.aggregate_statistics import AggregateStatisticsCollector

    torch.manual_seed(0)
    dev = torch.device("cuda", 0)
    model = torch.nn.Sequential(torch.nn.Conv2d(1, 4, 3), torch.nn.ReLU(), torch.nn.MaxPool2d(2), torch.nn.Flatten(),
                                torch.nn.Linear(4 * 5 * 5, 24), torch.nn.ReLU(), torch.nn.Linear(24, 6),
                                torch.nn.Softmax(dim=1)).to(dev)
    tm = A.TransparentModel(model, activation_layers=[1, 5], include_last_layer=True)      # conv ReLU, dense ReLU, softmax
    rng = np.random.default_rng(0)
    xtr = torch.from_numpy(rng.normal(size=(1200, 1, 12, 12)).astype(np.float32)).to(dev)
    xte = torch.from_numpy((rng.normal(size=(300, 1, 12, 12)) * 1.3).astype(np.float32)).to(dev)
    tr = tm.collect(xtr, batch_size=100)
    te = tm.collect(xte, batch_size=100)
    assert all(t.is_cuda for t in tr + te)
    ytr = tr[-1].argmax(dim=1).cpu().numpy()
    pred_d, gini = DeepGini.calculate(te[-1])
    labels = rng.integers(0, 6, size=300)
    mis = pred_d != labels
    # device tensors in == host copies in, for every scorer
    sa_layer_tr, sa_layer_te = tr[1], te[1]
    dsa = DSA(sa_layer_tr, ytr)(sa_layer_te, pred_d)
    want = np_oracle.dsa_oracle(sa_layer_tr.cpu().numpy(), ytr, sa_layer_te.cpu().numpy(), pred_d)
    assert np.array_equal(dsa, want["dsa"], equal_nan=True)
    lsa = LSA(sa_layer_tr.cpu().numpy())(sa_layer_te)
    _close(lsa, np_oracle.lsa_oracle(sa_layer_tr.cpu().numpy(), sa_layer_te.cpu().numpy()))
    col = AggregateStatisticsCollector()
    for badge in tm.walk_activations(xtr[i:i + 100] for i in range(0, 1200, 100)):
        col.track(badge[:2])
    mins, maxs, stds = col.get()
    o_min, o_max, o_std = np_oracle.stats_oracle([[a[i:i + 100].cpu().numpy() for a in tr[:2]] for i in range(0, 1200, 100)])
    assert all(np.array_equal(a, b) for a, b in zip(mins + maxs + stds, o_min + o_max + o_std))
    km = KMNC(mins, maxs, 2)
    k_score, k_bucket = km.buckets(te[:2], device_out=True)
    ws, _ = np_oracle.kmnc_oracle(mins, maxs, 2, [a.cpu().numpy() for a in te[:2]])
    assert np.array_equal(k_score.cpu().numpy(), ws)
    n_score, n_bits = NAC(0.75).packed(te[:2])
    os_, op = np_oracle.nac_oracle(0.75, [a.cpu().numpy() for a in te[:2]])
    assert np.array_equal(n_score.cpu().numpy(), os_)
    out = str(tmp_path)
    R.persist(out, "toy", "nominal", "is_misclassified", 0, mis)
    R.persist(out, "toy", "nominal", "uncertainty_deep_gini", 0, gini)
    R.persist_tip(out, "toy", "nominal", 0, "dsa", dsa)
    # (scores in the reference's dtype: np.argsort's tie order, which decides the tail of cam, depends on it)
    R.persist_tip(out, "toy", "nominal", 0, "KMNC_2", ws, list(cam_from_buckets(k_score.cpu().numpy().astype(ws.dtype), k_bucket, 2)))
    R.persist_tip(out, "toy", "nominal", 0, "NAC_0.75", os_, list(cam_from_bits(os_, n_bits)))
    apfd = R.load_apfd_values(out, "toy", "nominal")
    assert apfd["dsa"][0] == apfd_from_order(mis, np.argsort(-want["dsa"]))
    assert apfd["deep_gini"][0] == apfd_from_order(mis, np.argsort(-np_oracle.deepgini_oracle(te[-1].cpu().numpy())[1]))
    assert apfd["NAC_0.75-cam"][0] == apfd_from_order(mis, np_oracle.cam_oracle(os_, op))
    kprof = np_oracle.kmnc_oracle(mins, maxs, 2, [a.cpu().numpy() for a in te[:2]])[1]
    assert apfd["KMNC_2-cam"][0] == apfd_from_order(mis, np_oracle.cam_oracle(ws, kprof))


# ------------------------------------------------------------------------------------------
# LSA operand tiers: the one-segment fp16 pass is used only where its measured error allows it
# ------------------------------------------------------------------------------------------
def test_lsa_fast_pass_is_verified_and_falls_back():
    torch = _torch()
    from src.core.surprise import LSA

    # high-dimensional traces, large -log densities: the fp16 pass passes its check and meets rtol 1e-4 against the oracle
    xtr, _, xte, _, _ = np_oracle.synth_clusters(9000, 1500, 256, 6, seed=51, spread=1.0)
    sa = LSA(xtr)
    got = sa(xte)
    assert sa.kde.last_fast_check["accepted"], sa.kde.last_fast_check
    assert sa.kde.last_operands.startswith("fp16 x1")
    sub = np.sort(np.random.default_rng(0).choice(1500, 200, replace=False))
    want = np_oracle.lsa_oracle(xtr, xte[sub], exact=True)
    rel = np.abs(got[sub] - want) / np.abs(want)
    assert rel.max() <= 1e-4, rel.max()
    # with the fast pass disabled the same object reproduces the three-segment result (tighter)
    sa.kde._engine.fast_ok = False
    slow = sa(xte)
    assert np.abs(slow[sub] - want).max() / np.abs(want).max() < 5e-6
    assert np.abs(got - slow).max() / np.abs(slow).max() <= 1e-4
    # low-dimensional traces: -log densities are small, the budget is tight -> the check must reject the fast pass
    xs, _, xt, _, _ = np_oracle.synth_clusters(6000, 2048, 6, 3, seed=52, spread=1.0)
    lo = LSA(xs)
    out = lo(xt)
    _close(out, np_oracle.lsa_oracle(xs, xt))
    chk = lo.kde.last_fast_check
    assert lo.kde.last_operands == "split-bf16 x3" or chk["max_rel_diff"] <= 4e-5, chk
    # values beyond fp16's range disable the fast operand at fit time / raise the overflow flag at score time
    big = LSA(xtr * 3.0e4)
    assert big.kde._engine.fast_ok in (False, True)
    far = xte.copy()
    far[:5] *= 1.0e6
    res = LSA(xtr)(far)
    assert np.isinf(res[:5]).all() or np.isfinite(res[5:]).all()
    _close(res[5:][sub[sub >= 5] - 5], np_oracle.lsa_oracle(xtr, far[5:][sub[sub >= 5] - 5]))


def test_dsa_nan_test_trace_is_contained():
    """NaN traces are unsupported inputs (DESIGN.md 9), but one bad row must neither crash the call nor disturb the
    other rows: their scores stay bit-identical to the reference's, on the eager first call, on the captured plan (which
    counts the row's empty candidate list and repeats the call eagerly) and on later calls."""
    from src.core.surprise import DSA

    xtr, ytr, xte, pte, _ = np_oracle.synth_clusters(4000, 300, 64, 4, seed=71)
    bad = xte.copy()
    bad[17, 5] = np.nan
    want = np_oracle.dsa_oracle(xtr, ytr, xte, pte)["dsa"]
    sa = DSA(xtr, ytr)
    keep = np.ones(300, dtype=bool)
    keep[17] = False
    for _ in range(4):
        got = sa(bad, pte)
        assert got.shape == (300,) and np.array_equal(got[keep], want[keep])
    assert np.array_equal(sa(xte, pte), want)            # and a clean batch of the same shape afterwards


def test_dsa_mixed_dtypes_follow_numpy_promotion():
    """float64 test traces against float32 training traces: NumPy promotes the difference to float64
    (surprise.py:638) — same bits here; float16 traces are widened and scored in float32 (documented)."""
    from src.core.surprise import DSA

    xtr, ytr, xte, pte, _ = np_oracle.synth_clusters(3000, 260, 40, 4, seed=61)
    sa = DSA(xtr, ytr)
    x64 = xte.astype(np.float64) + 1e-9
    want = np_oracle.dsa_oracle(xtr, ytr, x64, pte)          # stage 1 in float64, stage 2 (train rows only) in float32
    got = sa(x64, pte)
    assert np.array_equal(got, want["dsa"]) and np.array_equal(sa.last_winner_index, want["idx_a"])
    assert np.array_equal(sa.last_dist_b.astype(np.float32), want["dist_b"])
    f32 = np_oracle.dsa_oracle(xtr, ytr, xte, pte)
    assert not np.array_equal(got, f32["dsa"])                # the promotion is visible in the bits
    assert np.array_equal(sa(xte, pte), np_oracle.dsa_oracle(xtr, ytr, xte, pte)["dsa"])       # float32 path unaffected
    h = xte.astype(np.float16)
    assert np.array_equal(sa(h, pte), np_oracle.dsa_oracle(xtr, ytr, h.astype(np.float32), pte)["dsa"])
