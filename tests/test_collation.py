"""Host-side batching / collation (SURVEY.md 8(f) rank 3) against the unmodified reference functions (loaded through
oracle/reference_loader.load_reference_collation when the reference tree is mounted) and against hand-written cases that
travel; the pinned staging path on the GPU."""
import json
import os
import random

import pytest
import torch

import conformer_nemo_b200 as cn
from oracle import reference_loader as rl

needs_ref = pytest.mark.skipif(not rl.reference_available(), reason="reference tree not mounted")
GOLDEN = os.path.join(os.path.dirname(__file__), "golden", "collation.json")  # tests/golden/make_golden_collation.py
MANIFEST_KWARGS = [dict(), dict(min_duration=0.1, max_duration=16.7), dict(max_number=7, min_duration=1.0),
                   dict(do_sort_by_duration=True, max_duration=20.0)]
NO_AUDIO = [(None, None, torch.tensor([1, 2, 3]), torch.tensor(3)), (None, None, torch.tensor([4]), torch.tensor(1))]


def _batch(gen, n, with_ids, max_len=50, max_tok=7, dtype=torch.float32):
    out = []
    for i in range(n):
        m, k = int(torch.randint(1, max_len, (1,), generator=gen)), int(torch.randint(0, max_tok, (1,), generator=gen))
        item = (torch.randn(m, generator=gen).to(dtype), torch.tensor(m), torch.randint(0, 20, (k,), generator=gen), torch.tensor(k))
        out.append(item + (100 + i,) if with_ids else item)
    return out


@needs_ref
@pytest.mark.parametrize("with_ids", [False, True])
def test_collate_equals_reference(with_ids):
    a2t, _ = rl.load_reference_collation()
    gen = torch.Generator().manual_seed(3)
    for n in (1, 2, 7):
        batch = _batch(gen, n, with_ids)
        want = a2t._speech_collate_fn(batch, pad_id=28)
        got = cn.speech_collate(batch, pad_id=28)
        assert len(got) == len(want)
        for g, w in zip(got, want):
            assert g.dtype == w.dtype and torch.equal(g, w)
        staged = cn.speech_collate(batch, pad_id=28, audio_out=torch.full((9, 64), 7.0))
        assert torch.equal(staged[0], want[0])  # stale contents of the staging buffer never leak into the padding


@needs_ref
def test_collate_edge_cases_equal_reference():
    a2t, _ = rl.load_reference_collation()
    want, got = a2t._speech_collate_fn(NO_AUDIO, pad_id=0), cn.speech_collate(NO_AUDIO, pad_id=0)
    assert got[0] is None and got[1] is None and want[0] is None
    assert torch.equal(got[2], want[2]) and torch.equal(got[3], want[3])
    for bad in ([(torch.zeros(3), torch.tensor(3), torch.tensor([1]))], ):
        with pytest.raises(ValueError):
            a2t._speech_collate_fn(bad, pad_id=0)
        with pytest.raises(ValueError):
            cn.speech_collate(bad, pad_id=0)
    lying = [(torch.zeros(5), torch.tensor(4), torch.tensor([1]), torch.tensor(1)), (torch.zeros(6), torch.tensor(6), torch.tensor([1]), torch.tensor(1))]
    with pytest.raises(RuntimeError):
        a2t._speech_collate_fn(lying, pad_id=0)
    with pytest.raises(RuntimeError):
        cn.speech_collate(lying, pad_id=0)


def test_collate_hand_cases():
    batch = [(torch.tensor([1., 2., 3.]), torch.tensor(3), torch.tensor([5, 6]), torch.tensor(2), 11),
             (torch.tensor([4.]), torch.tensor(1), torch.tensor([], dtype=torch.int64), torch.tensor(0), 12)]
    sig, lens, tok, tok_lens, ids = cn.speech_collate(batch, pad_id=9)
    assert sig.tolist() == [[1., 2., 3.], [4., 0., 0.]] and lens.tolist() == [3, 1]
    assert tok.tolist() == [[5, 6], [9, 9]] and tok_lens.tolist() == [2, 0]
    assert ids.dtype == torch.int32 and ids.tolist() == [11, 12]


def _write_manifest(path, rng, n):
    with open(path, "w") as f:
        for i in range(n):
            item = {"duration": round(rng.uniform(0.05, 25.0), 3), "text": rng.choice(["hello world", "", "a b c", "skip me"])}
            item["audio_filepath" if i % 3 else "audio_filename"] = f"/data/utt_{i}.wav"
            if i % 5 == 0:
                item["offset"] = 1.5
            f.write(json.dumps(item) + "\n")


def _manifest_parser(text):
    return None if text == "skip me" else [ord(c) - 96 for c in text if c != " "]


@needs_ref
@pytest.mark.parametrize("kw", MANIFEST_KWARGS)
def test_manifest_equals_reference(tmp_path, kw):
    _, coll = rl.load_reference_collation()
    rng = random.Random(5)
    paths = [str(tmp_path / "a.json"), str(tmp_path / "b.json")]
    _write_manifest(paths[0], rng, 23)
    _write_manifest(paths[1], rng, 9)
    want = coll.ASRAudioText(manifests_files=paths, parser=_manifest_parser, **kw)
    got = cn.read_manifest(",".join(paths), parser=_manifest_parser, **kw)
    assert len(got) == len(want) > 0
    for g, w in zip(got, want):
        assert (g.id, g.audio_file, g.duration, g.text_tokens, g.offset, g.text_raw) == \
               (w.id, w.audio_file, w.duration, w.text_tokens, w.offset, w.text_raw)


def test_manifest_errors_and_filters(tmp_path):
    p = tmp_path / "m.json"
    p.write_text(json.dumps({"audio_filepath": "x.wav", "duration": 2.0, "text": "ab"}) + "\n" +
                 json.dumps({"audio_filepath": "y.wav", "duration": 30.0, "text": "cd"}) + "\n" +
                 json.dumps({"audio_filepath": "z.wav", "duration": 3.0, "normalized_text": "ef"}) + "\n")
    got = cn.read_manifest(str(p), max_duration=16.7)
    assert [e.id for e in got] == [0, 2] and got[1].text_raw == "ef"
    bad = tmp_path / "bad.json"
    bad.write_text(json.dumps({"duration": 2.0}) + "\n")
    with pytest.raises(ValueError):
        cn.read_manifest(str(bad))
    bad.write_text(json.dumps({"audio_filepath": "x.wav"}) + "\n")
    with pytest.raises(ValueError):
        cn.read_manifest(str(bad))


@needs_ref
def test_bucketing_iterator_equals_reference():
    a2t, _ = rl.load_reference_collation()
    for n, k in ((10, 4), (8, 4), (3, 5), (0, 2)):
        assert list(cn.BucketingIterator(iter(range(n)), k)) == list(a2t.BucketingIterator(iter(range(n)), k))
    assert list(cn.BucketingIterator(range(5), 2)) == [[0, 1], [2, 3], [4]]


def _golden():
    with open(GOLDEN) as f:
        return json.load(f)


def _tensor(j):
    return None if j is None else torch.tensor(j["data"], dtype=getattr(torch, j["dtype"])).reshape(j["shape"])


@pytest.mark.parametrize("with_ids", [False, True])
def test_collate_equals_golden(with_ids):
    """The same seeded batches as test_collate_equals_reference, against the stored collate outputs."""
    cases = _golden()["collate"][str(with_ids)]
    gen = torch.Generator().manual_seed(3)
    for n, want in zip((1, 2, 7), cases):
        batch = _batch(gen, n, with_ids)
        got = cn.speech_collate(batch, pad_id=28)
        assert len(got) == len(want)
        for g, w in zip(got, want):
            w = _tensor(w)
            assert g.dtype == w.dtype and torch.equal(g, w)
        staged = cn.speech_collate(batch, pad_id=28, audio_out=torch.full((9, 64), 7.0))
        assert torch.equal(staged[0], _tensor(want[0]))
    assert len(cases) == 3


def test_collate_edge_cases_equal_golden():
    z = _golden()
    got = cn.speech_collate(NO_AUDIO, pad_id=0)
    assert got[0] is None and got[1] is None and z["no_audio"][0] is None and z["no_audio"][1] is None
    assert torch.equal(got[2], _tensor(z["no_audio"][2])) and torch.equal(got[3], _tensor(z["no_audio"][3]))
    assert z["errors"] == {"three_tuple": "ValueError", "length_exceeds_signal": "RuntimeError"}
    with pytest.raises(ValueError):
        cn.speech_collate([(torch.zeros(3), torch.tensor(3), torch.tensor([1]))], pad_id=0)
    with pytest.raises(RuntimeError):
        cn.speech_collate([(torch.zeros(5), torch.tensor(4), torch.tensor([1]), torch.tensor(1)),
                           (torch.zeros(6), torch.tensor(6), torch.tensor([1]), torch.tensor(1))], pad_id=0)


@pytest.mark.parametrize("kw", MANIFEST_KWARGS)
def test_manifest_equals_golden(tmp_path, kw):
    """The same two manifests and filter settings as test_manifest_equals_reference, against the stored entries."""
    (want,) = [m["entries"] for m in _golden()["manifest"] if m["kwargs"] == kw]
    rng = random.Random(5)
    paths = [str(tmp_path / "a.json"), str(tmp_path / "b.json")]
    _write_manifest(paths[0], rng, 23)
    _write_manifest(paths[1], rng, 9)
    got = cn.read_manifest(",".join(paths), parser=_manifest_parser, **kw)
    assert len(want) > 0
    assert [[e.id, e.audio_file, e.duration, e.text_tokens, e.offset, e.text_raw] for e in got] == want


def test_bucketing_iterator_equals_golden():
    cases = _golden()["bucketing"]
    assert len(cases) == 4
    for c in cases:
        assert [list(b) for b in cn.BucketingIterator(iter(range(c["n"])), c["k"])] == c["chunks"]


def _service(n_ranks, rank, device=None, n=41, seed=2):
    rng = random.Random(seed)
    lengths = [rng.randint(1600, 16000 * 12) for _ in range(n)]
    gens = {}

    def load(i):
        g = gens.setdefault(i, torch.Generator().manual_seed(1000 + i))
        g.manual_seed(1000 + i)
        return torch.randn(lengths[i], generator=g), torch.arange(i % 4)

    return lengths, load, cn.CollationService(lengths, load, n_ranks=n_ranks, rank=rank, max_batch=8, bucket_frames=100, device=device, pad_id=77)


def test_service_covers_every_utterance_once_and_bounds_padding():
    seen = []
    for rank in range(4):
        lengths, load, svc = _service(4, rank)
        assert svc.padding_fraction() < 0.2  # 100-frame buckets on 10-1200 frame utterances
        for b in svc:
            assert b.audio_signal.shape == (len(b.indices), max(lengths[i] for i in b.indices))
            # the staged batch is a CONTIGUOUS view of its slot: the H2D copy is then one async copy from pinned memory
            assert b.audio_signal.is_contiguous()
            assert b.audio_signal.data_ptr() == svc._audio[b.slot].data_ptr()
            assert b.audio_lengths.tolist() == [lengths[i] for i in b.indices] == b.audio_lengths_host
            assert b.feature_lengths_host(160) == [n // 160 + 1 for n in b.audio_lengths_host]
            assert b.sample_ids.tolist() == b.indices
            for row, i in enumerate(b.indices):
                assert torch.equal(b.audio_signal[row, :lengths[i]], load(i)[0])
                assert float(b.audio_signal[row, lengths[i]:].abs().sum()) == 0.0
                assert b.tokens[row].tolist() == list(range(i % 4)) + [77] * (b.tokens.shape[1] - i % 4)
            seen += b.indices
    assert sorted(seen) == list(range(41))


@pytest.mark.gpu
def test_service_pinned_staging_on_gpu():
    lengths, load, svc = _service(2, 1, device="cuda", n=30)
    assert all(buf.is_pinned() for buf in svc._audio)
    total = 0
    staged = []
    orig = svc._collate

    def spy(idx, slot):  # what goes into .to(device): must be a contiguous view of pinned memory (asynchronous copy)
        out = orig(idx, slot)
        staged.append((out[0].is_contiguous(), out[0].is_pinned()))
        return out

    svc._collate = spy
    for b in svc:
        svc.wait(b)
        assert b.audio_signal.is_cuda and b.audio_lengths.is_cuda
        host = b.audio_signal.cpu()
        for row, i in enumerate(b.indices):
            assert torch.equal(host[row, :lengths[i]], load(i)[0]) and float(host[row, lengths[i]:].abs().sum()) == 0.0
        assert b.audio_lengths.cpu().tolist() == [lengths[i] for i in b.indices]
        total += len(b.indices)
    assert total == len(svc.plan.rank_indices(1)) > 0
    assert staged and all(c and p for c, p in staged), staged


def _gloo_collation_worker(rank, world, port, q):
    import torch.distributed as dist

    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    lengths, load, svc = _service(world, rank, n=23, seed=9)
    # the plan is derived from the lengths alone: no communication on the data path; the gather below is the test's own
    mine = [(i, int(b.audio_lengths[row]), float(b.audio_signal[row].double().sum()))
            for b in svc for row, i in enumerate(b.indices)]
    gathered = [None] * world
    dist.all_gather_object(gathered, mine)
    dist.barrier()
    if rank == 0:
        q.put((gathered, lengths))
    dist.destroy_process_group()


def test_world_size_2_gloo_services_partition_the_manifest():
    import torch.multiprocessing as mp

    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    port = 31500 + os.getpid() % 2000
    procs = [ctx.Process(target=_gloo_collation_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    gathered, lengths = q.get(timeout=180)
    for p in procs:
        p.join(timeout=60)
        assert p.exitcode == 0
    flat = sorted(x for part in gathered for x in part)
    assert [i for i, _, _ in flat] == list(range(23))                       # every utterance exactly once over the ranks
    assert [n for _, n, _ in flat] == lengths
    assert not ({i for i, _, _ in gathered[0]} & {i for i, _, _ in gathered[1]})
    work = [sum(n for _, n, _ in part) for part in gathered]
    assert max(work) <= 1.35 * min(work)                                    # LPT assignment balances the ranks
