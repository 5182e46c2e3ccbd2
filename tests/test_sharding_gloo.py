"""CPU, world_size 2 over gloo: the multi-GPU path's host logic (static window sharding, fixed-stride word-record
packing, the single all_gather, merge) without a GPU.  The per-window work is replaced by a deterministic fake."""
import os

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp


def _fake_words(win: int):
    rng = np.random.default_rng(win)
    out, t = [], 0.0
    for _ in range(int(rng.integers(0, 7))):
        k = int(rng.integers(1, 4))
        d = float(rng.integers(1, 60)) * 0.02
        out.append(dict(start=round(t, 3), end=round(t + d, 3), tokens=rng.integers(256, 50000, k).tolist(),
                        probability=float(np.float32(rng.random()))))
        t += d
    return out


def _worker(rank, world, port, n_windows, q):
    os.environ.update(MASTER_ADDR="127.0.0.1", MASTER_PORT=str(port))
    dist.init_process_group("gloo", rank=rank, world_size=world)
    from stable_ts_b200.sharding import run_sharded, shard_range
    seen = []

    def process(lo, hi):
        seen.append((lo, hi))
        return [_fake_words(w) for w in range(lo, hi)]

    merged = run_sharded(process, n_windows)
    q.put((rank, seen[0], merged))
    dist.barrier()
    dist.destroy_process_group()


def test_shard_ranges_cover_and_balance():
    from stable_ts_b200.sharding import shard_range
    for n in (0, 1, 7, 8, 120, 961):
        for world in (1, 2, 4, 8):
            r = [shard_range(n, k, world) for k in range(world)]
            assert r[0][0] == 0 and r[-1][1] == n
            assert all(a[1] == b[0] for a, b in zip(r, r[1:]))
            sizes = [b - a for a, b in r]
            assert max(sizes) - min(sizes) <= 1


def test_pack_unpack_roundtrip():
    from stable_ts_b200.sharding import capacity, pack_records, unpack_records
    res = [_fake_words(w) for w in range(5)]
    cw, ct = capacity(5, 1)
    back = unpack_records([pack_records(res, 0, cw, ct)], 5, cw)
    for a, b in zip(res, back):
        assert [w["tokens"] for w in a] == [w["tokens"] for w in b]
        assert np.allclose([w["start"] for w in a], [w["start"] for w in b])
        assert [np.float32(w["probability"]) for w in a] == [np.float32(w["probability"]) for w in b]


def test_two_rank_gloo_gather_equals_unsharded():
    n_windows, world = 7, 2
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 29500 + os.getpid() % 2000
    procs = [ctx.Process(target=_worker, args=(r, world, port, n_windows, q)) for r in range(world)]
    [p.start() for p in procs]
    got = [q.get(timeout=120) for _ in range(world)]
    [p.join(timeout=60) for p in procs]
    assert all(p.exitcode == 0 for p in procs)
    expect = [_fake_words(w) for w in range(n_windows)]
    ranges = sorted(g[1] for g in got)
    assert ranges == [(0, 4), (4, 7)]
    for _, _, merged in got:                       # every rank holds the full merged result
        assert len(merged) == n_windows
        for a, b in zip(expect, merged):
            assert [w["tokens"] for w in a] == [w["tokens"] for w in b]
            assert np.allclose([w["end"] for w in a], [w["end"] for w in b], atol=1e-9)


def test_gathered_words_lazy_view_equals_eager_unpack():
    """the lazy view over the gathered rank buffers builds exactly the dicts of the eager unpack (empty windows, ragged
    word counts, negative / slice indexing)"""
    import numpy as np
    from stable_ts_b200 import sharding as S
    rng = np.random.default_rng(3)
    world, per = 3, 7
    res = []
    for w in range(per):
        ws, t = [], 0.0
        for _ in range(int(rng.integers(0, 9))):
            k = int(rng.integers(1, 4))
            ws.append(dict(word="x", start=round(t, 3), end=round(t + 0.14, 3), probability=float(np.float32(rng.random())),
                           tokens=[int(v) for v in rng.integers(0, 50000, size=k)]))
            t += 0.14
        res.append(ws)
    res[2] = []
    cap_w, cap_t = S.capacity(per * world, world)
    bufs = [S.pack_records(res, per * r, cap_w, cap_t) for r in range(world)]
    eager = S.unpack_records(bufs, per * world, cap_w)
    lazy = S.unpack_records(bufs, per * world, cap_w, lazy=True)
    assert len(lazy) == per * world and lazy.n_words == world * sum(len(w) for w in res)
    assert [lazy[i] for i in range(len(lazy))] == eager
    assert lazy[-1] == eager[-1] and lazy[1:4] == eager[1:4]
    for r in range(world):
        for w in range(per):
            assert [d["tokens"] for d in eager[per * r + w]] == [d["tokens"] for d in res[w]]


def gathered_result_dict(world=2, per=3):
    """The result dict rebuilt from the gathered word records of `world` ranks with `per` windows each (-> (dict, n_words))."""
    from stable_ts_b200 import sharding as S
    from stable_ts_b200.tokenizer import Tokenizer
    tk = Tokenizer(True, 99, "en", "transcribe")
    res = []
    for w in range(per):
        ws = _fake_words(100 + w)
        for i, wd in enumerate(ws):
            wd["segment"] = i // 3                      # up to 3 words per segment
        res.append(ws)
    cap_w, cap_t = S.capacity(per * world, world)
    bufs = [S.pack_records([[dict(w, start=w["start"] + 30.0 * (per * r + i), end=w["end"] + 30.0 * (per * r + i)) for w in ws]
                            for i, ws in enumerate(res)], per * r, cap_w, cap_t) for r in range(world)]
    g = S.unpack_records(bufs, per * world, cap_w, lazy=True, tokenizer=tk)
    return S.gathered_to_result(g, tk), world * sum(len(w) for w in res)


def test_gathered_records_rebuild_the_result_wire_format():
    """SURVEY.md section 8f row 4: the gather payload -> dict with WhisperResult.to_dict's keys; loads in the stand-in result
    class exactly as in the reference's own WhisperResult (tests/golden/reference_results.json, written by the unmodified
    reference from the same dict)."""
    import json
    from stable_ts_b200.result import WhisperResult
    from stable_ts_b200.tokenizer import Tokenizer
    tk = Tokenizer(True, 99, "en", "transcribe")
    d, n_words = gathered_result_dict()
    assert d["language"] == "en" and sum(len(s["words"]) for s in d["segments"]) == n_words
    for s in d["segments"]:
        assert s["text"] == "".join(w["word"] for w in s["words"]) == tk.decode(s["tokens"])
        assert s["start"] == s["words"][0]["start"] and s["end"] == s["words"][-1]["end"] and s["seek"] == 30.0 * (s["start"] // 30.0)
    mine = WhisperResult(d)
    assert len(mine.all_words()) == n_words and mine.text == d["text"]
    gold = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", "reference_results.json")
    with open(gold) as f:
        theirs = json.load(f)["sharding_result"]
    assert theirs["text"] == mine.text and len(theirs["words"]) == n_words
    assert theirs["words"] == [w.to_dict() for w in mine.all_words()]
