"""Mixed-company batches without a GPU: the aggregator's match_many_fn mode, recognize_frames against per-frame
recognize with an injected matcher, and the argument checks of Matcher.match_tenants."""
import numpy as np
import pytest

from facerecognition_infrenceengine_b200.aggregator import BatchAggregator


def frame(ident, faces, dim=8):
    e = np.zeros((faces, dim), np.float32)
    e[:, 0] = ident
    e[:, 1] = np.arange(faces)
    return e


def fake_many(calls):
    def fn(Q, companies):
        calls.append((len(Q), list(companies)))
        return Q[:, :1].astype(np.int64), Q[:, 1:2].copy(), np.ones(len(Q), bool)
    return fn


def test_aggregator_mixes_tenants_and_routes_results_back():
    calls = []
    agg = BatchAggregator(None, max_batch=12, max_delay_ms=2000, match_many_fn=fake_many(calls))
    futs = [agg.submit(frame(1, 4), "A"), agg.submit(frame(2, 3), "B"), agg.submit(frame(3, 5), None)]
    res = [f.result(timeout=5) for f in futs]
    assert calls == [(12, ["A"] * 4 + ["B"] * 3 + [None] * 5)]           # one batch, arrival order
    for i, (rows, scores, acc) in enumerate(res):
        assert (rows[:, 0] == i + 1).all() and list(scores[:, 0]) == list(range(len(rows))) and acc.all()
    agg.close()


def test_aggregator_many_respects_max_batch():
    calls = []
    agg = BatchAggregator(None, max_batch=8, max_delay_ms=30, match_many_fn=fake_many(calls))
    futs = [agg.submit(frame(i, 3), "c%d" % i) for i in range(5)]
    for i, f in enumerate(futs):
        assert (f.result(timeout=5)[0] == i).all()
    agg.close()
    assert all(n <= 8 for n, _ in calls) and sum(n for n, _ in calls) == 15
    assert [c for _, cs in calls for c in cs] == [c for i in range(5) for c in ["c%d" % i] * 3]


def test_aggregator_many_failure_fails_only_its_batch():
    seen = []

    def fn(Q, companies):
        seen.append(len(Q))
        if "bad" in companies:
            raise RuntimeError("boom")
        return Q[:, :1].astype(np.int64), Q[:, 1:2].copy(), np.ones(len(Q), bool)

    agg = BatchAggregator(None, max_batch=4, max_delay_ms=20, match_many_fn=fn)
    f1 = agg.submit(frame(1, 4), "bad")
    f1b = agg.submit(frame(2, 4), "A")
    with pytest.raises(RuntimeError):
        f1.result(timeout=5)
    assert (f1b.result(timeout=5)[0] == 2).all()
    agg.close()


class _Store:
    def __init__(self, n):
        self.n = n

    def __len__(self):
        return self.n

    def id_of(self, row):
        return "p%d" % row

    def metadata(self, pid):
        return None


class _Matcher:
    """match / match_tenants over a toy gallery of "company" blocks: row = round(q[0]), accepted when its block is
    the requested company (or no company was given)"""

    def __init__(self):
        self.calls = []

    def _one(self, q, company):
        row = int(round(float(q[0])))
        ok = company is None or row // 10 == int(company[1:])
        return (row if ok else -1), (float(q[1]) if ok else -1.0), ok

    def match(self, Q, k=1, threshold=0.4, company_id=None, with_ids=True):
        from facerecognition_infrenceengine_b200.matcher import MatchResult
        self.calls.append(("match", len(Q)))
        r = [self._one(q, company_id) for q in Q]
        return MatchResult(np.array([[x[0]] for x in r], np.int64).reshape(-1, 1),
                           np.array([[x[1]] for x in r], np.float32).reshape(-1, 1), np.array([x[2] for x in r], bool))

    def match_tenants(self, Q, company_ids, k=1, threshold=0.4, with_ids=True):
        from facerecognition_infrenceengine_b200.matcher import MatchResult
        self.calls.append(("match_tenants", len(Q)))
        r = [self._one(q, c) for q, c in zip(Q, company_ids)]
        return MatchResult(np.array([[x[0]] for x in r], np.int64).reshape(-1, 1),
                           np.array([[x[1]] for x in r], np.float32).reshape(-1, 1), np.array([x[2] for x in r], bool))


def test_recognize_frames_equals_per_frame_recognize():
    import facerecognition_infrenceengine_b200 as frg
    m = _Matcher()
    proc = frg.FaceRecognitionProcessor(_Store(100), matcher=m)

    def faces(rows):
        e = np.zeros((len(rows), 4), np.float32)
        e[:, 0] = rows
        e[:, 1] = 0.5 + np.arange(len(rows)) * 0.01
        return e

    frames = [(faces([12, 31, 15]), "c1"), (faces([]), "c2"), (faces([44, 47]), None), (faces([70]), "c3")]
    got = proc.recognize_frames(frames)
    assert m.calls == [("match_tenants", 6)]
    want = [proc.recognize(e, c) for e, c in frames]
    assert got == want
    assert [len(f) for f in got] == [3, 0, 2, 1]
    assert got[0][1]["person_id"] is None and got[0][0]["person_id"] == "p12"


def test_recognize_frames_needs_match_tenants():
    import facerecognition_infrenceengine_b200 as frg

    class Sharded:
        def match(self, *a, **kw):
            raise AssertionError("not reached")

    proc = frg.FaceRecognitionProcessor(_Store(10), matcher=Sharded())
    with pytest.raises(NotImplementedError, match="Sharded"):
        proc.recognize_frames([(np.zeros((1, 4), np.float32), "c1")])


def test_match_tenants_argument_checks():
    import facerecognition_infrenceengine_b200 as frg

    class Store:
        dim = 4

        def tenant_code(self, c, create=True):
            return 1

    m = frg.Matcher(Store())
    with pytest.raises(ValueError, match="company ids"):
        m.match_tenants(np.zeros((3, 4), np.float32), ["a", "b"])
    with pytest.raises(ValueError, match="Q must be"):
        m.match_tenants(np.zeros(4, np.float32), ["a"])
    with pytest.raises(ValueError, match="Q must be"):
        m.match_tenants(np.zeros((2, 5), np.float32), ["a", "b"])
