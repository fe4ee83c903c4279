"""Known-answer vectors the REFERENCE's own tests hold for the hot path's host side, replayed offline.

1. `test_split_tokens` (/root/reference/tests/test_transcribe.py:722-902): token ids -> (words, pieces, ids).  The
   vectors were extracted verbatim by tests/golden/make_split_tokens_vectors.py.  They need the real Whisper
   vocabulary; here a stub tokenizer is rebuilt from the expected pieces themselves (id -> UTF-8 bytes; where the
   reference shows an empty piece followed by a multi-byte one, the bytes are cut inside a code point so that the
   first token alone is an incomplete sequence — exactly the situation the vector documents).  What is tested is
   the product's grouping logic (words.split_on_spaces == T.py:1815-1868), not the vocabulary.
2. The alignment-head table: model_zoo.ALIGNMENT_HEADS (literal (layer, head) pairs) must be the decoded form of
   the reference's base85 masks (T.py:2343-2357, copied as data to tests/golden/alignment_heads_b85.json).
"""
import base64
import gzip
import json
import os

import numpy as np
import pytest

from whisper_timestamped import model_zoo as zoo
from whisper_timestamped import words as W

HERE = os.path.dirname(os.path.abspath(__file__))
VEC = json.load(open(os.path.join(HERE, "golden", "split_tokens_vectors.json")))["vectors"]


class StubTokenizer:
    """decode_with_timestamps / eot / timestamp_begin — all split_on_spaces needs (T.py:1823)."""

    def __init__(self, multilingual, pieces):
        self.eot = 50257 if multilingual else 50256
        self.timestamp_begin = 50364 if multilingual else 50363
        self.pieces = pieces

    def decode_with_timestamps(self, ids):
        out = b""
        for t in ids:
            if t >= self.timestamp_begin:
                out += f"<|{(t - self.timestamp_begin) * 0.02:.2f}|>".encode()
            else:
                out += self.pieces[t]
        return out.decode("utf-8", errors="replace")


def pieces_from_vector(v):
    """id -> bytes, derived from the expected (pieces, ids) of the vector."""
    ts0 = 50364 if v["multilingual"] else 50363
    eot = 50257 if v["multilingual"] else 50256
    table = {}
    for pieces, ids in zip(v["pieces"], v["ids"]):
        k = 0
        while k < len(ids):
            if ids[k] >= eot:                           # timestamps are rendered by the stub; other specials (issue #61's
                if ids[k] < ts0:                        # "<|te|>") are filtered out before decoding: no bytes
                    table.setdefault(ids[k], b"")
                k += 1
                continue
            # a run of empty pieces followed by a non-empty one = one code-point group spread over several tokens
            j = k
            while j < len(ids) and pieces[j] == "" and ids[j] < eot:
                j += 1
            if j == k:
                table.setdefault(ids[k], pieces[k].encode("utf-8"))
                k += 1
                continue
            assert j < len(ids) and ids[j] < eot, (pieces, ids)
            data = pieces[j].encode("utf-8")
            n = j - k + 1
            # cut after the lead byte of the LAST n-1 multi-byte characters... simplest valid choice: every token but
            # the last takes bytes up to (and including) a lead byte, so each prefix is an incomplete sequence
            leads = [i for i, b in enumerate(data) if b >= 0xC0]
            assert len(leads) >= n - 1, (pieces[j], n)
            cuts = [leads[-(n - 1) + i] + 1 for i in range(n - 1)]
            parts = [data[a:b] for a, b in zip([0] + cuts, cuts + [len(data)])]
            for t, p in zip(ids[k:j + 1], parts):
                table.setdefault(t, p)
            k = j + 1
    return table


@pytest.mark.parametrize("v", VEC, ids=[f"line{v['source_line']}" for v in VEC])
def test_split_tokens_vectors_of_the_reference(v):
    tok = StubTokenizer(v["multilingual"], pieces_from_vector(v))
    words, pieces, ids = W.split_on_spaces(v["tokens"], tok)
    assert words == v["words"]
    assert ids == v["ids"]
    assert pieces == v["pieces"]


def test_alignment_heads_table_is_the_reference_masks():
    g = json.load(open(os.path.join(HERE, "golden", "alignment_heads_b85.json")))
    assert set(g["masks"]) <= set(zoo.ALIGNMENT_HEADS)
    for name, dump in g["masks"].items():
        dims = zoo.DIMS[name]
        arr = np.frombuffer(gzip.decompress(base64.b85decode(dump)), dtype=bool)
        mask = arr.reshape(dims.n_text_layer, dims.n_text_head)                  # T.py:2387-2391
        pairs = sorted((int(l), int(h)) for l, h in zip(*np.nonzero(mask)))
        assert pairs == sorted(zoo.ALIGNMENT_HEADS[name]), name
