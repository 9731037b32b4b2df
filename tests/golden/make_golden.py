#!/usr/bin/env python
"""Generates the committed golden fixtures in tests/golden/.

Run from the repo root with a checkout of the reference project (for its own fixture) and
python `cbor2` (the independent CBOR implementation):

    python tests/golden/make_golden.py REFERENCE_CHECKOUT

Outputs
  hash_kats.json     request-key known answers.  The expected values are computed with
                     cbor2.dumps(..., canonical=True) + a from-scratch FNV-1a loop, i.e.
                     WITHOUT importing oracle/ -- they pin the oracle's CBOR/FNV restatement
                     against an independent implementation of RFC 7049 canonical form.
                     (The reference's own golden-hash test is skipped upstream,
                     tests/integration/prompt_to_block_test.go:59, and Go is not installed, so
                     hash parity with real Go is "unpinned"; see DESIGN.md.)
  kv_event_base_keys.json   the 400 real token ids of the reference fixture
                     tests/integration/testdata/kv_event_base.json (seed "42", block 16), its 25
                     vLLM sha256_cbor block hashes (used as ENGINE keys) and the 25 expected
                     request keys (cbor2 + FNV).
  scenario_small.json  a seeded event stream + prompts with the expected keys / lookups / scores
                     produced by the pure-Python oracle (oracle/kvoracle.py), used to pin the C++
                     oracle and the CUDA path on identical inputs.
"""
import json
import os
import random
import sys

import cbor2

HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(os.path.dirname(HERE))
sys.path.insert(0, ROOT)

M64 = (1 << 64) - 1


def fnv64a(b, h=0xCBF29CE484222325):
    for x in b:
        h = ((h ^ x) * 0x100000001B3) & M64
    return h


def chain(seed, tokens, bs, parent=None):
    p = fnv64a(seed.encode()) if parent is None else parent
    out = []
    for i in range(0, len(tokens) - bs + 1, bs):
        payload = cbor2.dumps([p, list(tokens[i:i + bs]), None], canonical=True)
        p = fnv64a(payload)
        out.append(p)
    return out


def hash_kats():
    rnd = random.Random(20240921)
    cases = []

    def add(name, seed, bs, tokens, parent=None):
        cases.append({"name": name, "seed": seed, "block_size": bs, "parent": parent, "tokens": list(tokens),
                      "keys": chain(seed, tokens, bs, parent)})

    add("seed-empty-1..16", "", 16, range(1, 17))
    add("seed-empty-1..32", "", 16, range(1, 33))
    add("seed-empty-35-tokens-tail-dropped", "", 16, range(1, 36))
    add("short-no-keys", "", 16, range(1, 16))
    add("parent-1", "", 16, range(1, 17), parent=1)
    add("parent-23", "", 16, range(1, 17), parent=23)
    add("parent-24", "", 16, range(1, 17), parent=24)
    add("parent-255", "", 16, range(1, 17), parent=255)
    add("parent-256", "", 16, range(1, 17), parent=256)
    add("parent-65535", "", 16, range(1, 17), parent=65535)
    add("parent-65536", "", 16, range(1, 17), parent=65536)
    add("parent-2^32-1", "", 16, range(1, 17), parent=(1 << 32) - 1)
    add("parent-2^32", "", 16, range(1, 17), parent=1 << 32)
    add("parent-2^64-1", "", 16, range(1, 17), parent=M64)
    add("parent-0", "", 16, range(1, 17), parent=0)
    add("seed-42-wide-tokens", "42", 16, [70000 + 4099 * i for i in range(16)])
    edge = [0, 23, 24, 255, 256, 65535, 65536, (1 << 32) - 1, 1, 22, 25, 254, 257, 65534, 65537, (1 << 32) - 2]
    add("token-width-edges", "", 16, edge * 3)
    add("block-size-4", "", 4, [rnd.randrange(0, 50000) for _ in range(23)])
    add("block-size-1", "s", 1, [5, 24, 256, 65536])
    add("block-size-23", "", 23, [rnd.randrange(0, 1 << 32) for _ in range(70)])
    add("block-size-24", "", 24, [rnd.randrange(0, 300) for _ in range(72)])
    add("block-size-256", "", 256, [rnd.randrange(0, 128256) for _ in range(600)])
    add("block-size-300", "", 300, [rnd.randrange(0, 128256) for _ in range(650)])
    add("seed-12345-random-4k", "12345", 16, [rnd.randrange(0, 128256) for _ in range(4096)])
    add("all-zero-tokens", "", 16, [0] * 64)
    add("all-max-tokens", "", 16, [(1 << 32) - 1] * 64)
    kat = {"fnv64a": {"": fnv64a(b""), "42": fnv64a(b"42"), "12345": fnv64a(b"12345"), "a": fnv64a(b"a"),
                      "foobar": fnv64a(b"foobar")}, "cases": cases}
    # published FNV-1a 64-bit test vectors (Fowler/Noll/Vo reference suite)
    assert kat["fnv64a"][""] == 0xCBF29CE484222325
    assert kat["fnv64a"]["a"] == 0xAF63DC4C8601EC8C
    assert kat["fnv64a"]["foobar"] == 0x85944171F73967E8
    # values quoted in SURVEY.md 8(c)
    assert kat["fnv64a"]["42"] == 571532774284038691 and kat["fnv64a"]["12345"] == 16534377278781491704
    assert cases[0]["keys"] == [14388088054628765202]
    assert cases[1]["keys"][1] == 16757933279298582072 and len(cases[2]["keys"]) == 2
    assert cases[4]["keys"] == [9771344617790079767]
    assert cases[15]["keys"] == [8986345644883239756]
    return kat


def kv_event_base():
    src = os.path.join(sys.argv[1], "tests", "integration", "testdata", "kv_event_base.json")
    d = json.load(open(src))
    keys = chain(d["hash_seed"], d["token_ids"], d["block_size"])
    assert keys[:3] == [1232996234064703281, 4081027702767042585, 6770700869230650880] and keys[-1] == 4842047765409919357
    return {"source": "reference tests/integration/testdata/kv_event_base.json (token_ids, block_hashes, hash_seed, block_size)",
            "hash_seed": d["hash_seed"], "block_size": d["block_size"], "token_ids": d["token_ids"],
            "engine_hashes": d["block_hashes"], "request_keys": keys}


def scenario_small():
    """Random event stream over a small universe so that every branch is hit: shared prefixes,
    two tiers, pod-cap eviction, BlockRemoved of live / dead / unknown keys, parent chaining incl.
    unknown parents, dropped events (length mismatch, no full block), filters."""
    from oracle import kvoracle as ko
    rnd = random.Random(77)
    BS, NP, NT = 4, 24, 3
    pods = ["pod-%d" % i for i in range(NP)]
    tiers = ["gpu", "cpu", "disk"]
    weights = {"gpu": 1.0, "cpu": 0.8}
    model = "m0"
    ix = ko.Indexer(block_size=BS, hash_seed="7", size=10 ** 6, pod_cache_size=3, weights=weights)
    pool = ko.EventsPool(ix.index, ix.tokens_processor)
    docs = [[rnd.randrange(0, 200000) for _ in range(BS * rnd.randrange(1, 12))] for _ in range(12)]
    # documents 6..11 share a prefix with 0..5
    for i in range(6, 12):
        cut = BS * rnd.randrange(1, 4)
        docs[i] = docs[i - 6][:cut] + docs[i]
    stored = {}      # (pod) -> list of engine hashes stored
    events = []      # serialisable log
    next_engine = [1000]

    def engine_for(doc, blk):
        return (doc * 1000003 + blk * 7919 + 0xABCDEF0123) & M64

    for step in range(400):
        pod = rnd.choice(pods)
        r = rnd.random()
        if r < 0.6:
            d = rnd.randrange(len(docs))
            nb = len(docs[d]) // BS
            b0 = rnd.randrange(0, nb)
            b1 = rnd.randrange(b0 + 1, nb + 1)
            toks = docs[d][b0 * BS:b1 * BS]
            hashes = [engine_for(d, b) for b in range(b0, b1)]
            parent = engine_for(d, b0 - 1) if b0 > 0 else None
            if rnd.random() < 0.05:
                parent = 0xDEAD0000 + step            # unknown parent -> chain restarts at the seed
            if rnd.random() < 0.05:
                hashes = hashes[:-1] if len(hashes) > 1 else hashes + [123]   # length mismatch -> dropped
            if rnd.random() < 0.03:
                toks = toks[:BS - 1]                  # no full block -> dropped
            medium = rnd.choice([None, "GPU", "cpu", "Disk"])
            ev = {"type": "BlockStored", "pod": pod, "hashes": hashes, "parent": parent, "tokens": toks, "medium": medium}
            pool.digest_events(pod, model, [ko.BlockStored(hashes, parent, toks, BS, None, medium)])
            stored.setdefault(pod, []).extend(hashes)
        elif r < 0.95:
            cand = stored.get(pod) or [engine_for(0, 0)]
            hashes = [rnd.choice(cand) for _ in range(rnd.randrange(1, 4))]
            if rnd.random() < 0.2:
                hashes.append(0xFEED0000 + step)      # unknown engine key: silent no-op
            medium = rnd.choice([None, "GPU", "cpu"])
            ev = {"type": "BlockRemoved", "pod": pod, "hashes": hashes, "medium": medium}
            pool.digest_events(pod, model, [ko.BlockRemoved(hashes, medium)])
        else:
            ev = {"type": "AllBlocksCleared", "pod": pod}
            pool.digest_events(pod, model, [ko.AllBlocksCleared()])
        events.append(ev)

    prompts = []
    for q in range(60):
        d = rnd.randrange(len(docs))
        mlen = rnd.randrange(0, len(docs[d]) + 1)
        toks = docs[d][:mlen] + [rnd.randrange(0, 200000) for _ in range(rnd.randrange(0, 9))]
        filt = [] if rnd.random() < 0.6 else rnd.sample(pods, rnd.randrange(1, 6))
        keys = ix.tokens_processor.tokens_to_kv_block_keys(None, toks, model)
        exp = {"tokens": toks, "filter": filt, "keys": [k.chunk_hash for k in keys]}
        if keys:
            hits = ix.index.lookup(keys, set(filt))
            exp["lookup"] = [[[e.pod, e.tier] for e in hits.get(k, [])] for k in keys]
            exp["scores"] = ix.scorer.score(keys, hits)
        else:
            exp["lookup"] = None
            exp["scores"] = None
        prompts.append(exp)
    return {"block_size": BS, "hash_seed": "7", "pod_cache_size": 3, "model": model, "pods": pods, "tiers": tiers,
            "weights": weights, "events": events, "prompts": prompts,
            "final_request_keys": len(ix.index.data), "final_engine_keys": len(ix.index.engine_to_request)}


def prefix_store_kats():
    """XXH64 vectors and chained block keys of the reference's prefix-store test text (lru_store_test.go:36-44), computed with
    the xxhash package (C library binding) -- independent of oracle/ and of the C++ host layer."""
    import xxhash
    vec = [b"", b"a", b"abc", b"The capital of France is Paris", bytes(range(256)), b"x" * 31, b"y" * 32, b"z" * 33, bytes(range(97, 123)) * 11]
    kats = [{"hex": v.hex(), "seed": sd, "xxh64": xxhash.xxh64(v, seed=sd).intdigest()} for v in vec for sd in (0, 1, 0x9E3779B97F4A7C15)]
    text = b"The capital of France is Paris"
    chains = {}
    for bs in (4, 8, 30):
        prev, keys = 0, []
        for st in range(0, len(text) - bs + 1, bs):
            prev = xxhash.xxh64(prev.to_bytes(8, "little") + text[st:st + bs], seed=0).intdigest()
            keys.append(prev)
        chains[str(bs)] = keys
    return {"xxh64": kats, "text": text.decode(), "block_keys": chains}


def main():
    for name, fn in (("hash_kats.json", hash_kats), ("kv_event_base_keys.json", kv_event_base),
                     ("scenario_small.json", scenario_small), ("prefix_store_kats.json", prefix_store_kats)):
        with open(os.path.join(HERE, name), "w") as f:
            json.dump(fn(), f, separators=(",", ":"))
        print("wrote", name, os.path.getsize(os.path.join(HERE, name)), "bytes")


if __name__ == "__main__":
    main()
