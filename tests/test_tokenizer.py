"""BPE tokenizer: algorithm on a tiny hand-made vocabulary and the reference's known-answer ids
(StableDiffusionTests.swift:43-48) with the part of the reference's CLIP vocabulary / merges that those prompts use
(tests/golden/make_golden_tokenizer.py)."""
import json
import os

import numpy as np

from b200sd.tokenizer import BPETokenizer

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def test_bpe_merges_by_rank_and_pads(tmp_path):
    merges = tmp_path / "merges.txt"
    merges.write_text("#version: 0.2\nl o\nlo w</w>\ne r</w>\nn e\nne w\n")  # ranks 1..5 (line 0 is the comment)
    vocab = {"<|startoftext|>": 0, "<|endoftext|>": 1, "low</w>": 2, "er</w>": 3, "new": 4, "lo": 5, "w": 6, "!": 7}
    (tmp_path / "vocab.json").write_text(json.dumps(vocab))
    tok = BPETokenizer.from_files(merges, tmp_path / "vocab.json", model_max_length=8)
    assert tok.merges[("l", "o")] == 1 and tok.merges[("ne", "w")] == 5
    assert tok.encode_word("low") == ["low</w>"]
    assert tok.encode_word("lower") == ["lo", "w", "er</w>"]
    assert tok.encode_word("newer") == ["new", "er</w>"]
    tokens, ids = tok.tokenize("  Low NEWER  ", min_count=8)
    assert tokens == ["<|startoftext|>", "low</w>", "new", "er</w>", "<|endoftext|>"] + ["<|endoftext|>"] * 3
    assert ids == [0, 2, 4, 3, 1, 1, 1, 1]
    assert tok.decode(tokens[:5]) == "low newer "
    assert tok.tokenize("zz")[1] == [0, 1, 1, 1]  # unknown pieces ("z", "z</w>") map to <|endoftext|>
    out = tok("low " * 20)  # truncation at the encoder's input length
    assert out.shape == (1, 8) and out.dtype == np.float32 and out[0, 0] == 0 and out[0, -1] == 2
    padded = BPETokenizer(tok.merges, vocab, pad_token="!", model_max_length=6)  # second SDXL encoder
    assert padded.input_ids("low") == [0, 2, 1, 7, 7, 7]


def test_reference_known_answer_ids():
    tok = BPETokenizer.from_files(os.path.join(GOLD, "clip_bpe_merges_subset.txt"),
                                  os.path.join(GOLD, "clip_bpe_vocab_subset.json"))
    cases = {
        "a photo of an astronaut riding a horse on mars":
            [49406, 320, 1125, 539, 550, 18376, 6765, 320, 4558, 525, 7496, 49407],
        "Apple CoreML developer tools on a Macbook Air are fast":
            [49406, 3055, 19622, 5780, 10929, 5771, 525, 320, 20617, 1922, 631, 1953, 49407],
    }
    for prompt, expected in cases.items():
        tokens, ids = tok.tokenize(prompt)
        assert ids == expected, (tokens, ids)
    ids77 = tok("a photo of an astronaut riding a horse on mars")
    assert ids77.shape == (1, 77) and list(ids77[0, :12].astype(int)) == cases[
        "a photo of an astronaut riding a horse on mars"] and (ids77[0, 12:] == 49407).all()
