"""Golden fixture for the tokenizer's known-answer test: the part of the CLIP BPE vocabulary and merge list that ship
with the reference (swift/StableDiffusionTests/Resources/{merges.txt,vocab.json}) which tokenizing PROMPTS touches.

    B200SD_REFERENCE=<reference checkout> python tests/golden/make_golden_tokenizer.py

Every merge the BPE loop looks up for these prompts and finds is kept, in the original file order (ranks are
renumbered, their order is not), and every vocabulary entry the result maps to keeps its original id.  With the
subset the tokenizer therefore takes exactly the merges it takes with the full files.
"""
import json
import os
import sys

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)

from b200sd.tokenizer import BPETokenizer  # noqa: E402

OUT = os.path.dirname(os.path.abspath(__file__))
PROMPTS = ["a photo of an astronaut riding a horse on mars",
           "Apple CoreML developer tools on a Macbook Air are fast"]


class _Recording(dict):
    def __init__(self, merges):
        super().__init__(merges)
        self.seen = set()

    def get(self, key, default=None):
        if key in self:
            self.seen.add(key)
        return super().get(key, default)


def main():
    res = os.path.join(os.environ["B200SD_REFERENCE"], "swift", "StableDiffusionTests", "Resources")
    full = BPETokenizer.from_files(os.path.join(res, "merges.txt"), os.path.join(res, "vocab.json"))
    full.merges = _Recording(full.merges)
    tokens = set()
    for p in PROMPTS:
        tokens.update(full.tokenize(p, min_count=full.model_max_length)[0])
    with open(os.path.join(OUT, "clip_bpe_merges_subset.txt"), "w", encoding="utf-8") as f:
        f.write("#version: 0.2\n")
        for a, b in sorted(full.merges.seen, key=full.merges.__getitem__):
            f.write(f"{a} {b}\n")
    vocab = {t: full.vocabulary[t] for t in sorted(tokens | {full.start_token, full.end_token})}
    with open(os.path.join(OUT, "clip_bpe_vocab_subset.json"), "w", encoding="utf-8") as f:
        json.dump(vocab, f, ensure_ascii=False, indent=0, sort_keys=True)
        f.write("\n")
    print(len(full.merges.seen), "merges,", len(vocab), "vocabulary entries")


if __name__ == "__main__":
    main()
