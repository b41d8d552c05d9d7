"""Windows (lh_window_*): percentiles over the last K snapshots, or since the window was configured, against the
oracle.  The expected window is the uint64 sum of the oracle's per-interval dense histograms, reduced with
oracle.process_histogram.  Bar: bucket counts, keys and percentile keys exactly equal, percentile values bit-exact,
sums within 1e-12 of the summed magnitudes."""
import numpy as np
import pytest

pytestmark = pytest.mark.gpu

SEED = 0x10C415C0
PS = [0.0, 0.5, 0.75, 0.9, 0.95, 0.99, 0.999, 0.9999, 1.0]
I32_MIN = np.iinfo(np.int32).min
_decomp = {}


@pytest.fixture(scope="module")
def lh():
    import loghisto_b200
    return loghisto_b200


def dense(sp, H):
    out = np.zeros((H, 65536), dtype=np.uint64)
    out[np.repeat(np.arange(H), np.diff(sp.offsets.astype(np.int64))), sp.keys.view(np.uint16)] = sp.counts
    return out


def assert_matches(oracle, red, sp, want, counters=None, precision=100.0, hs=None):
    """red / sp (a reduction and an export of one window) against the dense uint64[H][65536] sums `want`."""
    H = want.shape[0]
    assert (dense(sp, H) == want).all()
    assert int(sp.offsets[-1]) == int((want != 0).sum())
    if counters is not None:
        assert (sp.counter_deltas == counters).all()
    if precision not in _decomp:
        _decomp[precision] = np.abs(oracle.decompress_table(precision))
    for h in range(H) if hs is None else hs:
        ref = oracle.process_histogram(want[h], PS, precision)
        assert int(red.counts[h]) == ref["total"], h
        if ref["total"] == 0:   # absent from every held interval
            assert np.isnan(red.avgs[h]) and (red.pkeys[h] == I32_MIN).all() and np.isnan(red.pvals[h]).all(), h
            assert sp.offsets[h] == sp.offsets[h + 1], h
            continue
        assert (red.pkeys[h] == ref["pkeys"]).all(), h
        assert (red.pvals[h].view(np.uint64) == ref["pvals"].view(np.uint64)).all(), h
        # the sum is taken in another order than the oracle's: bound the difference by the summed magnitudes, which
        # stays meaningful when large buckets of both signs cancel
        scale = float((_decomp[precision] * want[h].astype(np.float64)).sum())
        assert abs(red.sums[h] - ref["sum"]) <= 1e-12 * scale, h
        assert abs(red.avgs[h] - ref["avg"]) <= 1e-12 * scale / ref["total"], h


def window(e):
    return e.window_reduce(PS), e.window_export()


def test_lifetime_three_streams_with_counters(lh, oracle):
    H, C, n = 3, 4, 300_001
    kinds = (lh.STREAM_U, lh.STREAM_L, lh.STREAM_S)
    want = np.zeros((H, 65536), dtype=np.uint64)
    counters = np.zeros(C, dtype=np.uint64)
    with lh.Engine(device=0, max_histograms=H, max_counters=C) as e:
        e.window_configure(0)
        for i in range(6):
            for h, kind in enumerate(kinds):
                d = e.gen_stream(kind, n, SEED + h, start=i * n)
                e.ingest_f64(h, d, n)
                want[h] += oracle.ingest(oracle.gen_stream(kind, n, SEED + h, start=i * n))
            amounts = np.array([i + 1, 2 ** 63 + i], dtype=np.uint64)
            e.counter_add_u16_host(np.array([0, 3], np.uint16), amounts)
            counters += oracle.counter_add(np.array([0, 3]), amounts, C)
            e.snapshot_begin()
            e.window_fold()
            e.snapshot_end()
            e.sync()
            red, sp = window(e)
            assert_matches(oracle, red, sp, want, counters)
            info = e.window_info()
            assert info["intervals"] == 0 and info["folds"] == i + 1 and info["held"] == i + 1
            assert info["device_bytes"] >= H * 65536 * 8


def test_sliding_three_of_eight(lh, oracle):
    """K = 3 over 8 intervals.  Histogram 1 is touched in interval 1 only; histogram 2 gets |v| >= 2^63, 1e300, NaN
    and infinities in interval 3 only (out-of-window keys: flag 3 while that interval is held); histogram 3 never."""
    H, C, n, K = 4, 2, 200_003, 3
    extreme = np.array([2.0 ** 63, -2.0 ** 63, 9.5e18, 1e300, -1e300, 3e200, np.nan, np.inf, -np.inf, 0.0])
    per = []
    with lh.Engine(device=0, max_histograms=H, max_counters=C) as e:
        e.window_configure(K)
        for i in range(1, 9):
            w = np.zeros((H, 65536), dtype=np.uint64)
            for h in (0, 2):
                vals = oracle.gen_stream(lh.STREAM_S, n, SEED + 7 * i + h)
                e.ingest_f64_host(h, vals)
                w[h] = oracle.ingest(vals)
            if i == 1:
                vals = oracle.gen_stream(lh.STREAM_L, n, SEED)
                e.ingest_f64_host(1, vals)
                w[1] = oracle.ingest(vals)
            if i == 3:
                e.ingest_f64_host(2, extreme)
                w[2] += oracle.ingest(extreme)
            e.counter_add_u16_host(np.array([1], np.uint16), np.array([10 ** i], np.uint64))
            per.append(w)
            e.snapshot_begin()
            e.window_fold()
            e.snapshot_end()
            held = per[-K:]
            want = np.sum(held, axis=0, dtype=np.uint64)
            red, sp = window(e)
            assert_matches(oracle, red, sp, want, np.array([0, sum(10 ** j for j in range(max(1, i - K + 1), i + 1))], np.uint64))
            if i >= 4:
                assert int(red.counts[1]) == 0 and int(sp.offsets[2] - sp.offsets[1]) == 0
            if 3 <= i <= 5:
                assert sp.histogram(2).keys() >= {int(k) for k in oracle.compress_many(extreme)}
            info = e.window_info()
            assert info["held"] == min(i, K) and info["folds"] == i and info["intervals"] == K
            assert info["entries_held"] == sum(int((x != 0).sum()) for x in held)


def test_snapshot_results_unchanged_by_the_window(lh, oracle):
    """Per-snapshot reduce / export are identical with and without a window, and an outstanding async ticket returns
    its own snapshot's numbers after window calls."""
    H, C, n = 5, 3, 400_000
    with lh.Engine(device=0, max_histograms=H, max_counters=C) as a, lh.Engine(device=0, max_histograms=H, max_counters=C) as b:
        a.window_configure(2)
        for i in range(4):
            vals = oracle.gen_stream(lh.STREAM_S, n, SEED + i)
            ids = oracle.gen_ids(0, n, H - 1 - (i % 2), SEED + i).astype(np.uint16)
            for e in (a, b):
                e.ingest_keyed_f64_u16_host(ids, vals)
                e.counter_add_u16_host(np.array([i % C], np.uint16), np.array([i + 1], np.uint64))
            if i % 2 == 0:          # fold first, then the snapshot's own reduce / export
                a.snapshot_begin()
                a.window_fold()
                ra, sa = a.snapshot_reduce(PS), a.snapshot_export()
                a.snapshot_end()
            else:                   # ticket outstanding across fold + window reduce + window export
                a.snapshot_begin()
                t = a.snapshot_reduce_async(PS)
                a.window_fold()
                wr = a.window_reduce([0.25, 0.5])
                a.window_export()
                sa = a.snapshot_export()
                a.snapshot_end()
                a.window_reduce(PS)
                ra = a.snapshot_result(t)
                assert wr.pkeys.shape == (H, 2)
            rb, sb = b.snapshot(PS)
            for f in ("counts", "sums", "avgs", "pkeys", "pvals"):
                assert getattr(ra, f).tobytes() == getattr(rb, f).tobytes(), (i, f)
            for f in ("offsets", "keys", "counts", "counter_deltas"):
                assert getattr(sa, f).tobytes() == getattr(sb, f).tobytes(), (i, f)


def test_state_errors(lh):
    from loghisto_b200 import _lib as L

    def status(fn, *a):
        with pytest.raises(lh.LhError) as ex:
            fn(*a)
        return ex.value.status

    with lh.Engine(device=0, max_histograms=2, max_counters=1) as e:
        for fn, args in ((e.window_reduce, (PS,)), (e.window_export, ()), (e.window_info, ()), (e.window_release, ())):
            assert status(fn, *args) == L.LH_ERR_STATE
        e.snapshot_begin()
        assert status(e.window_fold) == L.LH_ERR_STATE                  # never configured
        assert status(e.window_configure, 2) == L.LH_ERR_STATE          # snapshot open
        e.snapshot_end()
        assert status(e.window_configure, L.LH_MAX_WINDOW_INTERVALS + 1) == L.LH_ERR_INVALID
        e.window_configure(L.LH_MAX_WINDOW_INTERVALS)
        assert status(e.window_fold) == L.LH_ERR_STATE                  # no snapshot open
        e.snapshot_begin()
        e.window_fold()
        assert status(e.window_fold) == L.LH_ERR_STATE                  # second fold of one snapshot
        e.snapshot_end()
        assert e.window_info()["folds"] == 1
        e.window_release()
        for fn, args in ((e.window_reduce, (PS,)), (e.window_export, ()), (e.window_info, ())):
            assert status(fn, *args) == L.LH_ERR_STATE
        e.snapshot_begin()
        assert status(e.window_fold) == L.LH_ERR_STATE
        e.snapshot_end()
        e.window_configure(0)                                            # configure again after a release
        assert e.window_info()["folds"] == 0


def test_keyed_1024_write_combining_k2(lh, oracle):
    """1024 keyed histograms, 4 intervals of 1e8 pairs through the default dispatch (write-combining kernel), K = 2:
    every bucket of every histogram against the oracle's streaming keyed checker summed over the held intervals."""
    H, n, K = 1024, 100_000_000, 2
    with lh.Engine(device=0, max_histograms=H, max_counters=1) as e:
        e.tune("keyed_mode", 0)
        e.window_configure(K)
        d_v = e.alloc(n, np.float64)
        d_i = e.alloc(n, np.uint16)
        prev = None
        for i in range(4):
            e.gen_stream(lh.STREAM_U, n, SEED, start=i * n, out=d_v)
            e.gen_ids_u16(0, n, H, SEED, start=i * n, out=d_i)
            e.ingest_keyed_f64_u16(d_i, d_v, n)
            e.snapshot_begin()
            e.window_fold()
            e.snapshot_end()
            cur = oracle.stream_ingest_keyed(lh.STREAM_U, n, H, SEED, val_start=i * n, ids_start=i * n)
            want = cur if prev is None else cur + prev
            red, sp = window(e)
            assert_matches(oracle, red, sp, want, hs=(0, 1, 511, 1023))
            assert (red.counts == want.sum(axis=1)).all()
            prev = cur


@pytest.mark.parametrize("H", [1, 1024])     # one-shot and two-shot forms of the peer all-reduce
def test_two_ranks_hold_the_global_window(lh, oracle, H):
    """Two contexts in one process (lh_comm_import): each ingests its shard, all-reduce, fold.  Both ranks' windows
    are identical to each other and to one context that ingested the whole stream."""
    import torch
    from loghisto_b200.distributed import shard_range
    world, C, n_total, K = 2, 4, 2_000_001, 2
    devs = [0, 1] if torch.cuda.device_count() >= 2 else [0, 0]
    engs = [lh.Engine(device=d, max_histograms=H, max_counters=C) for d in devs]
    single = lh.Engine(device=0, max_histograms=H, max_counters=C)
    try:
        handles = b"".join(e.comm_export() for e in engs)
        for r, e in enumerate(engs):
            e.comm_import(r, world, handles)
        for e in engs + [single]:
            e.window_configure(K)
        per = []
        for i in range(3):
            vals = oracle.gen_stream(lh.STREAM_S, n_total, SEED + i)
            ids = oracle.gen_ids(0, n_total, H, SEED + i).astype(np.uint16)
            per.append(oracle.ingest_keyed(ids, vals, H))
            for r, e in enumerate(engs):
                a, b = shard_range(r, world, n_total)
                e.ingest_keyed_f64_u16_host(ids[a:b].copy(), vals[a:b].copy())
                e.counter_add_u16_host(np.array([r], np.uint16), np.array([2 ** 63 + i], np.uint64))
            single.ingest_keyed_f64_u16_host(ids, vals)
            single.counter_add_u16_host(np.array([0, 1], np.uint16), np.array([2 ** 63 + i] * 2, np.uint64))
            for e in engs:
                e.snapshot_begin()
                e.snapshot_allreduce(counters=True)
            single.snapshot_begin()
            for e in engs + [single]:
                e.window_fold()
                e.snapshot_end()
            exports = [e.window_export() for e in engs + [single]]
            for sp in exports[:2]:
                for f in ("offsets", "keys", "counts", "counter_deltas"):
                    assert getattr(sp, f).tobytes() == getattr(exports[2], f).tobytes(), (i, f)
            want = np.sum(per[-K:], axis=0, dtype=np.uint64)
            red = engs[1].window_reduce(PS)
            assert_matches(oracle, red, exports[1], want, hs=range(min(H, 8)))
            for e in engs:
                assert e.comm_info()["status"] == 0
    finally:
        for e in engs + [single]:
            e.close()


def test_precision_200_and_wrapping_counter_sums(lh, oracle):
    H, C, n, K = 2, 2, 300_000, 2
    per, cs = [], []
    with lh.Engine(device=0, max_histograms=H, max_counters=C, precision=200) as e:
        e.window_configure(K)
        for i in range(4):
            vals = oracle.gen_stream(lh.STREAM_S, n, SEED + i)
            e.ingest_f64_host(1, vals)
            per.append(np.stack([np.zeros(65536, np.uint64), oracle.ingest(vals, precision=200.0)]))
            amounts = np.array([2 ** 63 + 3 + i, 2 ** 64 - 1], dtype=np.uint64)
            e.counter_add_u16_host(np.array([0, 1], np.uint16), amounts)
            cs.append(amounts)
            e.snapshot_begin()
            e.window_fold()
            e.snapshot_end()
            want_c = np.sum(cs[-K:], axis=0, dtype=np.uint64)
            if i >= 1:   # two held intervals: 2^64 + 5 + 2i and 2^65 - 2 wrap
                assert want_c.tolist() == [5 + 2 * i, 2 ** 64 - 2]
            red, sp = window(e)
            assert_matches(oracle, red, sp, np.sum(per[-K:], axis=0, dtype=np.uint64), want_c, precision=200.0)


def test_sharded_engine_folds_once_per_snapshot(lh, oracle):
    from loghisto_b200.distributed import ShardedEngine
    H, n = 2, 100_000
    with lh.Engine(device=0, max_histograms=H, max_counters=1) as e:
        se = ShardedEngine(e, 0)
        assert se.world == 1
        e.window_configure(0)
        want = np.zeros((H, 65536), dtype=np.uint64)
        for i in range(3):
            vals = oracle.gen_stream(lh.STREAM_L, n, SEED + i)
            e.ingest_f64_host(0, vals)
            want[0] += oracle.ingest(vals)
            red, _ = se.snapshot(PS, window=True)
            assert int(red.counts[0]) == n
            assert e.window_info()["folds"] == i + 1
        se.snapshot(PS)
        h = se.snapshot_async(PS, window=True)
        se.result(h)
        assert e.window_info()["folds"] == 4
        red, sp = window(e)
        assert_matches(oracle, red, sp, want)
