"""Host BPE tokenizer (tair_b200.tokenizer) — structure on a synthetic merge table, ids against the reference's
tokenizer output (tests/golden/tokenizer_cases.json) when the CLIP merge table is available."""
import gzip
import json
import os

import pytest
import torch

from tair_b200.tokenizer import BPETokenizer

HERE = os.path.dirname(os.path.abspath(__file__))
# OpenAI's CLIP merge table (bpe_simple_vocab_16e6.txt.gz, 1.3 MB) is not redistributed with the project
VOCAB = os.environ.get("TAIR_BPE_VOCAB", "")


def test_missing_vocab_fails_loudly(monkeypatch):
    monkeypatch.delenv("TAIR_BPE_VOCAB", raising=False)
    with pytest.raises(FileNotFoundError):
        BPETokenizer()


def test_synthetic_merge_table(tmp_path):
    p = tmp_path / "merges.txt.gz"
    with gzip.open(p, "wb") as f:
        f.write(b'#version: test\nl l\nh e\nll o</w>\nhe llo</w>\na a\n')
    t = BPETokenizer(str(p))
    assert t.vocab_size == 512 + 5 + 2
    assert t.encode("hello") == [t.encoder["hello</w>"]]
    assert t.encode("Hello  hello") == [t.encoder["hello</w>"]] * 2          # lower-cased, whitespace collapsed
    # every occurrence of the best pair is merged left to right: aaaaa -> aa aa a</w>
    assert t.encode("aaaaa") == [t.encoder["aa"], t.encoder["aa"], t.encoder["a</w>"]]
    assert t.decode(t.encode("hello, hal")) == "hello , hal "
    ids = t(["hello", "a " * 100])
    assert ids.shape == (2, 77) and ids.dtype == torch.long
    assert ids[0].tolist()[:3] == [t.sot_id, t.encoder["hello</w>"], t.eot_id] and ids[0, 3:].sum() == 0
    assert ids[1, 0] == t.sot_id and ids[1, -1] == t.eot_id                  # truncated, last id forced to EOT


@pytest.mark.skipif(not os.path.isfile(VOCAB), reason="CLIP merge table not available (set TAIR_BPE_VOCAB to its path)")
def test_ids_match_reference_tokenizer():
    t = BPETokenizer(VOCAB)
    g = json.load(open(os.path.join(HERE, "golden", "tokenizer_cases.json")))
    ids = t(g["texts"])
    assert ids.tolist() == g["ids"]
    assert t.vocab_size == 49408
