"""Generates tests/golden/collation.json: what tests/test_collation.py compares collation against -- the outputs of
``_speech_collate_fn``, ``ASRAudioText`` manifest filtering and ``BucketingIterator`` on the test's own seeded inputs.

    python tests/golden/make_golden_collation.py

With the unmodified reference reachable (oracle/reference_loader.py: $CONFORMER_REF or an install under the repository)
the vectors come from the reference functions; otherwise from this package's restatement of them
(speech_collate / read_manifest / BucketingIterator), which test_collation.py checks against the reference functions
whenever they are reachable.  ``source`` in the file says which produced it.
"""
from __future__ import annotations

import json
import os
import random
import sys
import tempfile

import torch

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)
sys.path.insert(0, os.path.dirname(HERE))

import conformer_nemo_b200 as cn  # noqa: E402
from oracle import reference_loader as rl  # noqa: E402
from test_collation import MANIFEST_KWARGS, NO_AUDIO, _batch, _manifest_parser, _write_manifest  # noqa: E402

OUT = os.path.join(HERE, "collation.json")


def tensor_json(t):
    return None if t is None else {"dtype": str(t.dtype).replace("torch.", ""), "shape": list(t.shape), "data": t.flatten().tolist()}


def raised(fn, *args, **kw):
    try:
        fn(*args, **kw)
    except Exception as e:  # noqa: BLE001 -- the exception class is the datum
        return type(e).__name__
    return None


def main():
    if rl.reference_available():
        a2t, coll = rl.load_reference_collation()
        collate, bucketing = a2t._speech_collate_fn, a2t.BucketingIterator
        read = lambda paths, parser, **kw: list(coll.ASRAudioText(manifests_files=paths, parser=parser, **kw))
        source = f"unmodified reference functions loaded from {os.path.basename(rl.REFERENCE_ROOT.rstrip('/'))}"
    else:
        collate, bucketing = cn.speech_collate, cn.BucketingIterator
        read = lambda paths, parser, **kw: cn.read_manifest(",".join(paths), parser=parser, **kw)
        source = "conformer_nemo_b200 restatement (reference not reachable at generation time)"
    out = {"source": source, "torch": torch.__version__, "collate": {}, "manifest": [], "bucketing": []}
    for with_ids in (False, True):
        gen = torch.Generator().manual_seed(3)
        cases = []
        for n in (1, 2, 7):
            batch = _batch(gen, n, with_ids)
            cases.append([tensor_json(t) for t in collate(batch, pad_id=28)])
        out["collate"][str(with_ids)] = cases
    out["no_audio"] = [tensor_json(t) for t in collate(NO_AUDIO, pad_id=0)]
    out["errors"] = {
        "three_tuple": raised(collate, [(torch.zeros(3), torch.tensor(3), torch.tensor([1]))], pad_id=0),
        "length_exceeds_signal": raised(collate, [(torch.zeros(5), torch.tensor(4), torch.tensor([1]), torch.tensor(1)),
                                                  (torch.zeros(6), torch.tensor(6), torch.tensor([1]), torch.tensor(1))],
                                        pad_id=0),
    }
    with tempfile.TemporaryDirectory() as tmp:
        rng = random.Random(5)
        paths = [os.path.join(tmp, "a.json"), os.path.join(tmp, "b.json")]
        _write_manifest(paths[0], rng, 23)
        _write_manifest(paths[1], rng, 9)
        for kw in MANIFEST_KWARGS:
            entries = read(paths, _manifest_parser, **kw)
            out["manifest"].append({"kwargs": kw, "entries": [[e.id, e.audio_file, e.duration, e.text_tokens, e.offset, e.text_raw]
                                                              for e in entries]})
    for n, k in ((10, 4), (8, 4), (3, 5), (0, 2)):
        out["bucketing"].append({"n": n, "k": k, "chunks": [list(c) for c in bucketing(iter(range(n)), k)]})
    with open(OUT, "w") as f:
        json.dump(out, f, indent=None, separators=(",", ":"))
        f.write("\n")
    print(OUT, source)


if __name__ == "__main__":
    main()
