"""bench.py --dump-outputs: the dumped arrays are offset-free, float64, within the byte budget, the same from run to run,
and the same for the engine's packed output layout as for the oracle's capacity layout."""
import os

import numpy as np
import pytest

import bench
from oracle.packed import replay_packed
from peritext_b200 import workload


def load(d, prefix=""):
    return {f[len(prefix):-4]: np.load(os.path.join(d, f)) for f in sorted(os.listdir(d)) if f.startswith(prefix) and f.endswith(".npy")}


def canonical_from_dump(dump):
    """Per sampled log: (tokens, spans with their comment lists), rebuilt from the flat sample arrays."""
    out, t, s, c = {}, 0, 0, 0
    for log, n_vis, n_sp, _ in dump["sample_logs"].astype(np.int64):
        spans = []
        for start, flags, link in dump["sample_spans"][s: s + n_sp].astype(np.int64):
            nc = int(flags) >> 8
            spans.append((int(start), int(flags), int(link), tuple(int(x) for x in dump["sample_comments"][c: c + nc])))
            c += nc
        out[int(log)] = (tuple(int(x) for x in dump["sample_tokens"][t: t + n_vis]), tuple(spans))
        t += n_vis; s += n_sp
    assert (t, s, c) == (len(dump["sample_tokens"]), len(dump["sample_spans"]), len(dump["sample_comments"]))
    return out


def check_dump(dump, merged):
    for a in dump.values():
        assert a.dtype == np.float64
    res = dump["results"].astype(np.uint64)
    for row in res:
        i = int(row[0])
        r = merged.results[i]
        assert [int(x) for x in row[1:5]] == [int(r["status"]), int(r["n_elems"]), int(r["n_visible"]), int(r["n_spans"])]
        assert [int(row[5] | row[6] << np.uint64(32)), int(row[7] | row[8] << np.uint64(32))] == [int(x) for x in r["digest"]]
    for i, (toks, spans) in canonical_from_dump(dump).items():
        assert (toks, spans) == merged.canonical(i)[4:6], i


@pytest.mark.parametrize("cfg,n_docs", [("c3", 4), ("c4", 60)])
def test_dump_matches_the_merged_batch_and_respects_the_budget(tmp_path, cfg, n_docs):
    batch = workload.generate(cfg, n_docs=n_docs, ops_per_doc=1500, n_marks=300)
    merged, _ = replay_packed(batch, threads=4)
    assert (merged.results["status"] == 0).all() and len(merged.comment_pool)
    for budget in (bench.DUMP_BYTES, 20_000):
        d = tmp_path / f"{cfg}_{budget}"
        bench.dump_outputs(str(d), merged, budget)
        dump = load(str(d))
        assert sorted(dump) == ["results", "sample_comments", "sample_logs", "sample_spans", "sample_tokens"]
        assert sum(os.path.getsize(d / f) for f in os.listdir(d)) <= budget
        check_dump(dump, merged)
        n = batch.n_logs
        assert len(dump["results"]) == min(n, budget // 2 // 72)
        if budget == bench.DUMP_BYTES:
            assert len(dump["sample_logs"]) == n
        else:
            assert 0 < len(dump["sample_logs"]) < n
        again = tmp_path / f"again_{cfg}_{budget}"
        bench.dump_outputs(str(again), merged, budget, prefix="rank0_")
        for name, a in load(str(again), "rank0_").items():
            assert np.array_equal(a, dump[name]), name


@pytest.mark.gpu
def test_engine_dump_equals_oracle_dump(tmp_path):
    from peritext_b200.engine import BatchEngine
    batch = workload.generate("c4", n_docs=40, ops_per_doc=1000, n_marks=300)
    eng = BatchEngine(0)
    got = eng.run(batch)
    eng.close()
    ref, _ = replay_packed(batch, threads=4)
    for budget in (bench.DUMP_BYTES, 20_000):
        bench.dump_outputs(str(tmp_path / f"engine_{budget}"), got, budget)
        bench.dump_outputs(str(tmp_path / f"oracle_{budget}"), ref, budget)
        a, b = load(str(tmp_path / f"engine_{budget}")), load(str(tmp_path / f"oracle_{budget}"))
        assert sorted(a) == sorted(b)
        for name in a:
            assert np.array_equal(a[name], b[name]), name
        check_dump(a, got)
