#!/usr/bin/env python
"""Generates tests/golden/e2e_tokens.json: the prompts of the reference's end-to-end suite
(tests/e2e/redis_mock/e2e_test.go:109-244) tokenized with the reference's own checked-in tokenizer
(tests/e2e/redis_mock/testdata/test-model/tokenizer.json, BERT uncased, add_special_tokens=False as in
pkg/tokenization/tokenizer.go:411) by the HF `tokenizers` core -- the library the reference links.
Usage: python tests/golden/make_e2e_tokens.py REFERENCE_CHECKOUT; the tests only read the committed JSON."""
import json
import os
import sys

from tokenizers import Tokenizer

FULL = ("lorem ipsum dolor sit amet, consectetur adipiscing elit. Sed do eiusmod tempor incididunt ut labore et dolore magna aliqua. "
        "Ut enim ad minim veniam, quis nostrud exercitation ullamco laboris nisi ut aliquip ex ea commodo consequat.")
MID = "lorem ipsum dolor sit amet, consectetur adipiscing elit. Sed do eiusmod tempor incididunt ut labore et dolore magna aliqua."
SHORT = "lorem ipsum dolor sit amet, consectetur adipiscing elit."
BASE = "The quick brown fox jumps over the lazy dog"
PROMPTS = {"full": FULL, "mid": MID, "short": SHORT, "miss": "What is the capital of France?",
           "fox2": BASE * 2, "fox100": BASE * 100, "fox500": BASE * 500}


def main():
    tok = Tokenizer.from_file(os.path.join(sys.argv[1], "tests", "e2e", "redis_mock", "testdata", "test-model", "tokenizer.json"))
    out = {"tokenizer": "tests/e2e/redis_mock/testdata/test-model/tokenizer.json (reference @ a378f5b3)", "block_size": 4, "prompts": {}}
    for name, p in PROMPTS.items():
        enc = tok.encode(p, add_special_tokens=False)
        out["prompts"][name] = {"text": p if len(p) < 400 else None, "repeat": None if len(p) < 400 else [BASE, len(p) // len(BASE)],
                                "ids": enc.ids, "offsets": [list(o) for o in enc.offsets]}
    with open(os.path.join(os.path.dirname(os.path.abspath(__file__)), "e2e_tokens.json"), "w") as f:
        json.dump(out, f, separators=(",", ":"))
    print({k: len(v["ids"]) for k, v in out["prompts"].items()})


if __name__ == "__main__":
    main()
