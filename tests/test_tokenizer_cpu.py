"""The reference's only test, reproduced (src/tokenizer.rs:205-221): the one golden vector the reference holds.

The merge table is the part of the reference's bpe_simple_vocab_16e6.txt the tokenizer reads (header + 48894 merges), stored
xz-compressed under tests/golden (tests/ref_shim/make_ref_fixtures.py)."""
import lzma
import os

import pytest

from stable_diffusion_burn_b200 import tokenizer as T

VOCAB_XZ = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden", T.VOCAB_FILE + ".xz")


@pytest.fixture(scope="module")
def vocab(tmp_path_factory):
    path = tmp_path_factory.mktemp("bpe") / T.VOCAB_FILE
    with lzma.open(VOCAB_XZ, "rt", encoding="utf-8") as f:
        path.write_text(f.read(), encoding="utf-8")
    return str(path)


@pytest.fixture(scope="module")
def tok(vocab):
    return T.SimpleTokenizer(vocab)


def test_reference_kat_encode_decode(tok):
    text = "Hello world! <|startoftext|>asdf<|startoftext|>"
    assert tok.encode(text) == [3306, 1002, 256, 49406, 587, 10468, 49406]
    assert tok.decode(tok.encode(text)) == "hello world ! <|startoftext|>asdf <|startoftext|>"


def test_special_tokens_and_prompt_framing(tok):
    # StableDiffusion::context frames the prompt as <|startoftext|>{text}<|endoftext|> (stablediffusion/mod.rs:200);
    # the unconditional context is the empty prompt -> exactly [49406, 49407] (SURVEY §8a a1)
    assert tok.encode("<|startoftext|><|endoftext|>") == [49406, 49407]
    ids = tok.encode("<|startoftext|>a photo of a cat<|endoftext|>")
    assert ids[0] == 49406 and ids[-1] == 49407 and len(ids) == 7
    assert len(tok.encoder) == 49408


def test_cleaning_quirks(tok):
    assert tok.encode("  Hello   WORLD!\n") == tok.encode("hello world!")
    # no padding / truncation to 77 (SURVEY §2 row 9)
    assert len(tok.encode("cat " * 100)) == 100
    # round trip of non-ASCII bytes through the byte<->unicode table
    assert tok.decode(tok.encode("café ☕")).strip() == "café ☕"


def test_agrees_with_an_independent_clip_tokenizer(tok, vocab, tmp_path):
    """Second opinion on the mirror: transformers.CLIPTokenizer (independently written from the same published BPE) built from the
    same merges file must produce the same ids on plain prompts (no ftfy-specific cleaning involved)."""
    tr = pytest.importorskip("transformers")
    import json
    merges = open(vocab, encoding="utf-8").read().split("\n")[1:49152 - 256 - 2 + 1]
    vocab = [u for _, u in T._byte_unicode_table()]
    vocab = vocab + [v + "</w>" for v in vocab] + ["".join(m.split()) for m in merges] + ["<|startoftext|>", "<|endoftext|>"]
    (tmp_path / "vocab.json").write_text(json.dumps({v: i for i, v in enumerate(vocab)}))
    (tmp_path / "merges.txt").write_text("#version: 0.2\n" + "\n".join(merges) + "\n", encoding="utf-8")
    hf = tr.CLIPTokenizer(str(tmp_path / "vocab.json"), str(tmp_path / "merges.txt"))
    prompts = ["An ancient mossy stone.", "a photograph of an astronaut riding a horse", "Hello world!  multiple   spaces",
               "it's a dog's life, isn't it? 123 4567", "UPPER lower MiXeD", "oil painting, trending on artstation; 4k --hd",
               "café naïve résumé", "a cat\nwith\ttabs", "x" * 40, "don't we'll they've I'm you're he'd"]
    for p in prompts:
        assert tok.encode(p) == hf(p, add_special_tokens=False)["input_ids"], p
