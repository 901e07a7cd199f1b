"""CPU: the router's WordPiece restatement against transformers.BertTokenizer on the same vocabulary; the
router CLI accepts the reference's flags and fails loudly without a GPU (no CPU fallback)."""
import os
import random
import subprocess

import pytest
import torch

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
PKG = os.path.join(ROOT, "modal-examples_b200")

from tei_router.tokenizer import CLS, SEP, VOCAB_SIZE, WordPiece, synthetic_vocab  # noqa: E402

SAMPLES = [
    "Hello, World! This is the in-box B200 runtime.", "  multiple   spaces\tand\nnewlines ", "naïve café résumé über", "don't stop-believing (really)...",
    "数据 mixed 中文 text", "x" * 150 + " tail", "", "UPPER lower MiXeD 12345 3.14159 a_b-c/d", "emoji 🙂 and control\x00chars\x07 here",
    "Show HN: I built a thing that embeds 1M sentences on eight GPUs",
]


def test_synthetic_vocab_shape():
    v = synthetic_vocab()
    assert len(v) == VOCAB_SIZE == len(set(v))
    assert v[0] == "[PAD]" and v[100] == "[UNK]" and v[CLS] == "[CLS]" and v[SEP] == "[SEP]" and v[103] == "[MASK]"


def test_wordpiece_matches_hf_bert_tokenizer(tmp_path):
    from transformers import BertTokenizer

    vocab = synthetic_vocab()
    path = tmp_path / "vocab.txt"
    path.write_text("\n".join(vocab) + "\n", encoding="utf-8")
    hf = BertTokenizer(str(path), do_lower_case=True)
    mine = WordPiece({t: i for i, t in enumerate(vocab)})
    rnd = random.Random(0)
    alphabet = "abcdefghijklmnopqrstuvwxyz  ABC.,!?'-0123456789é中"
    texts = SAMPLES + ["".join(rnd.choice(alphabet) for _ in range(rnd.randint(1, 200))) for _ in range(200)]
    for t in texts:
        assert mine.encode(t, 10_000) == hf.encode(t), t


def test_truncation_and_limit():
    tok = WordPiece()
    long = "ab " * 600
    with pytest.raises(ValueError, match="less than 512 tokens"):
        tok.encode(long, 512, truncate=False)
    ids = tok.encode(long, 512, truncate=True)
    assert len(ids) == 512 and ids[0] == CLS and ids[-1] == SEP and max(ids) < VOCAB_SIZE


@pytest.mark.skipif(torch.cuda.is_available(), reason="GPU present")
def test_router_cli_fails_loudly_without_gpu():
    """Flags as the reference passes them (text_embeddings_inference.py:29-34); without a GPU the process must
    exit non-zero -- the reference's spawn_server poll then raises 'launcher exited unexpectedly' (:44-51)."""
    env = dict(os.environ, PATH=os.path.join(PKG, "bin") + os.pathsep + os.environ["PATH"])
    r = subprocess.run(["text-embeddings-router", "--model-id", "BAAI/bge-base-en-v1.5", "--port", "8000", "--max-client-batch-size", "256"],
                       capture_output=True, text=True, env=env, timeout=300)
    assert r.returncode != 0
    assert "cannot start" in r.stderr
