"""GPU parity tests: the CUDA engine (through the C ABI) vs the CPU oracle on the same seeded inputs, vs the
committed golden vectors, and through the reference-interface mirror (KATs of the reference's own tests).
Bar: bit-exact for hashes / counts / picks, bit-exact fp64 score bits.  Run on the B200 box: pytest -m gpu."""
import dataclasses
import json
import os
import random
import struct

import numpy as np
import pytest

pytestmark = pytest.mark.gpu

GOLD = os.path.join(os.path.dirname(__file__), "golden", "xxh64_vectors.json")


@pytest.fixture(scope="module")
def epp():
    import torch
    if not torch.cuda.is_available():
        pytest.skip("no CUDA device")
    import epp_b200
    epp_b200.build.build()
    return epp_b200


@pytest.fixture(scope="module")
def tg():
    from tools import tracegen
    tracegen.build()
    return tracegen


def _pack(prompts):
    offs = np.zeros(len(prompts) + 1, dtype=np.uint64)
    np.cumsum([len(p) for p in prompts], out=offs[1:])
    blob = b"".join(prompts)
    data = np.frombuffer(blob, dtype=np.uint8).copy() if blob else np.zeros(16, np.uint8)
    return data, offs


def _pack_aligned(prompts, align=16):
    offs = np.zeros(len(prompts) + 1, dtype=np.uint64)
    chunks, pos = [], 0
    starts = []
    for p in prompts:
        pad = (-pos) % align
        chunks.append(b"\0" * pad)
        pos += pad
        starts.append(pos)
        chunks.append(p)
        pos += len(p)
    return np.frombuffer(b"".join(chunks) + b"\0" * 16, dtype=np.uint8).copy(), starts


# ------------------------------------------------------------------------------------------------
# a1 hashing
# ------------------------------------------------------------------------------------------------
def test_model_seed(epp, orc):
    with epp.Engine(8) as eng:
        for m, s in ((b"test-model1", b""), (b"synthetic-model", b""), (b"test-model1", b"s1"), (b"", b""),
                     (b"x" * 100, b"y" * 33)):
            mid = eng.register_model(m, s)
            assert eng.model_seed(mid) == orc.xxh64(m + s)
        assert eng.model_seed(0) == 0x55B9CE9184DD8509         # SURVEY B.2


def test_hash_golden_vectors(epp):
    """Every prompt vector of tests/golden/xxh64_vectors.json (python-xxhash), each with its own engine config."""
    with open(GOLD) as f:
        gold = json.load(f)
    for v in gold["prompts"]:
        data = bytes.fromhex(v["data_hex"])
        want = [int(h, 16) for h in v["hashes"]]
        with epp.Engine(8, block_size_tokens=v["block_size_tokens"], max_prefix_blocks=v["max_blocks"]) as eng:
            mid = eng.register_model(v["model"].encode(), v["salt"].encode())
            d, offs = _pack([data])
            hs, nb = eng.hash_prompts(d, offsets=offs, model_ids=np.array([mid], np.uint32))
            assert nb[0] == len(want), v["name"]
            assert [int(x) for x in hs[0, : nb[0]]] == want, v["name"]


@pytest.mark.parametrize("bst,maxb", [pytest.param(b, m, id=str(b) if m == 12 else f"{b}-cap{m}")
                                      for m in (12, 9) for b in (1, 2, 3, 6, 7, 8, 16, 24, 32)])
def test_hash_ragged_vs_oracle(epp, orc, bst, maxb):
    """Ragged batch (empty, shorter than a block, partial tail, truncated) for block sizes hitting every XXH64 tail
    class: bs%32==0 (vector path), bs%32 in {24,28} (mixed stripe), tiny blocks (<32 bytes, no stripe); even and odd
    caps (an odd cap gives the hash rows an odd pitch)."""
    rng = random.Random(bst)
    prompts = [b"", b"a", bytes(rng.getrandbits(8) for _ in range(bst * 4 - 1)), bytes(rng.getrandbits(8) for _ in range(bst * 4))]
    for _ in range(60):
        n = rng.randint(0, bst * 4 * (maxb + 3))
        prompts.append(bytes(rng.getrandbits(8) for _ in range(n)))
    with epp.Engine(8, block_size_tokens=bst, max_prefix_blocks=maxb) as eng:
        mid = eng.register_model(b"mdl")
        # (a) tightly packed (unaligned offsets -> generic path)
        d, offs = _pack(prompts)
        hs, nb = eng.hash_prompts(d, offsets=offs)
        for i, p in enumerate(prompts):
            want = orc.hash_prompt(p, b"mdl", bst, maxb)
            assert nb[i] == len(want), (i, len(p))
            assert [int(x) for x in hs[i, : nb[i]]] == want, (i, len(p))
        # (b) 16-byte aligned prompt starts with explicit offsets (vector path when bs % 32 == 0); the padded rows make
        # offsets[r+1]-offsets[r] longer than the prompt, so the lengths go with them
        d2, starts = _pack_aligned(prompts)
        offs2 = np.array(starts + [starts[-1] + len(prompts[-1])], dtype=np.uint64)
        assert any(s % 32 == 16 for s in starts)
        lens2 = np.array([len(p) for p in prompts], dtype=np.uint64)
        hs2, nb2 = eng.hash_prompts(d2, offsets=offs2, lengths=lens2)
        for i, p in enumerate(prompts):
            want = orc.hash_prompt(p, b"mdl", bst, maxb)
            assert nb2[i] == len(want), (i, len(p))
            assert [int(x) for x in hs2[i, : nb2[i]]] == want, (i, len(p))
        # single prompts at offset 0 of a buffer of their own
        for i in (0, 1, 2, 3, 10, 33):
            di = np.zeros(((len(prompts[i]) + 31) // 16) * 16 + 16, np.uint8)
            di[: len(prompts[i])] = np.frombuffer(prompts[i], np.uint8)
            h1, n1 = eng.hash_prompts(di, offsets=np.array([0, len(prompts[i])], np.uint64))
            assert [int(x) for x in h1[0, : n1[0]]] == orc.hash_prompt(prompts[i], b"mdl", bst, maxb)
        assert mid == 0


def test_hash_ragged_aligned_starts_with_lengths(epp, orc):
    """Ragged prompts whose STARTS sit on 32-byte boundaries (epp_batch.lengths): the fused 256-bit-load kernel with
    per-request block counts, partial tail blocks, prompts shorter than a block and truncation, hashes AND decisions."""
    rng = random.Random(77)
    maxb = 20
    lens = [0, 5, 63, 64, 65, 127, 128, 64 * maxb, 64 * maxb + 9, 64 * (maxb + 3)] + [rng.randint(0, 64 * (maxb + 4)) for _ in range(90)]
    prompts = [bytes(rng.getrandbits(8) for _ in range(n)) for n in lens]
    starts, pos = [], 0
    for p in prompts:
        starts.append(pos)
        pos += (len(p) + 31) // 32 * 32
    blob = np.zeros(pos + 64, np.uint8)
    for st, p in zip(starts, prompts):
        blob[st:st + len(p)] = np.frombuffer(p, np.uint8)
    offs = np.array(starts + [pos], dtype=np.uint64)
    lengths = np.array(lens, dtype=np.uint64)
    E = 12
    with epp.Engine(E, epp.ProfileSpec(0, [epp.ScorerSpec(2, 2.0), epp.ScorerSpec(1, 2.0), epp.ScorerSpec(0, 3.0)]),
                    max_prefix_blocks=maxb) as eng:
        eng.register_model(b"mdl")
        hs, nb = eng.hash_prompts(blob, offsets=offs, lengths=lengths)
        for i, p in enumerate(prompts):
            want = orc.hash_prompt(p, b"mdl", 16, maxb)
            assert nb[i] == len(want), (i, len(p))
            assert [int(x) for x in hs[i, : nb[i]]] == want, (i, len(p))
        # decisions on a small pool whose endpoints cache prefixes of some of these prompts
        kv = np.linspace(0, 0.9, E)
        waiting = np.arange(E, dtype=np.int32) % 3
        eng.pool_set(np.arange(E), np.zeros(E, np.uint8), kv, waiting)
        ix = orc.Indexer()
        ph, pe = [], []
        for e in range(E):
            h = orc.hash_prompt(prompts[10 + e], b"mdl", 16, maxb)
            ph += h[: max(1, len(h) // 2)]
            pe += [e] * max(1, len(h) // 2)
        ix.load_pairs(ph, pe)
        eng.index_load_snapshot(ph, pe)
        dec, det = eng.schedule(blob, offsets=offs, lengths=lengths)
        pool = orc.PoolState(np.zeros(E, np.uint8), kv, waiting)
        prof = orc.make_profile(0, [(2, 2.0, 0), (1, 2.0, 0), (0, 3.0, 0)])
        for i, p in enumerate(prompts):
            h = orc.hash_prompt(p, b"mdl", 16, maxb)
            m, _ = ix.match_longest_prefix(h, E)
            d = orc.schedule(prof, None, pool, m, len(h), 16, len(p), 0)
            assert (dec["status"][i], dec["pick"][i], dec["tie_count"][i], dec["total_blocks"][i]) == (d.status, d.pick, d.tie_count, len(h)), i
            assert dec["score"][i] == d.score and dec["match_blocks"][i] == m[d.pick]


def test_hash_uniform_tokens_vs_oracle(epp, orc):
    """uint32 token arrays (4 bytes/token), T = 4096 -> 256 blocks of 64 bytes (BASELINE config 3 shape), host and
    device-pointer batches."""
    import torch
    rng = np.random.default_rng(3)
    R, T = 96, 4096
    toks = rng.integers(0, 128000, size=(R, T), dtype=np.uint32)
    with epp.Engine(8) as eng:
        eng.register_model(b"synthetic-model")
        hs, nb = eng.hash_prompts(toks, uniform_len=T * 4)
        assert (nb == 256).all()
        for r in (0, 1, 50, R - 1):
            want = orc.hash_prompt(toks[r].tobytes(), b"synthetic-model", 16, 256)
            assert [int(x) for x in hs[r]] == want
        dt = torch.from_numpy(toks.view(np.int32)).cuda()
        hd, nd = eng.hash_prompts(dt, uniform_len=T * 4)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(hd.cpu().numpy().view(np.uint64), hs)
        np.testing.assert_array_equal(nd.cpu().numpy(), nb)
        # prefix property (size-independent): changing token t only changes hashes of blocks >= t // 16
        t2 = toks.copy()
        t2[:, 1000] ^= 1
        h2, _ = eng.hash_prompts(t2, uniform_len=T * 4)
        blk = 1000 // 16
        assert (h2[:, :blk] == hs[:, :blk]).all() and (h2[:, blk:] != hs[:, blk:]).all()


def test_hash_truncation_and_short(epp, orc):
    toks = np.arange(40, dtype=np.uint32)
    with epp.Engine(8, max_prefix_blocks=2) as eng:
        eng.register_model(b"synthetic-model")
        hs, nb = eng.hash_prompts(toks, uniform_len=160)
        assert nb[0] == 2 and [int(x) for x in hs[0, :2]] == [0x8A787856B0C98B2D, 0xC57021EFCC0A8595]
    with epp.Engine(8) as eng:
        eng.register_model(b"synthetic-model")
        hs, nb = eng.hash_prompts(toks, uniform_len=160)
        assert [int(x) for x in hs[0, :3]] == [0x8A787856B0C98B2D, 0xC57021EFCC0A8595, 0xA8A7E535C242C990]
        hs, nb = eng.hash_prompts(toks[:15], uniform_len=60)         # shorter than one block -> nil
        assert nb[0] == 0
        hs, nb = eng.hash_prompts(np.zeros(16, np.uint8), offsets=np.zeros(1, np.uint64))   # empty batch
        assert hs.shape[0] == 0


# ------------------------------------------------------------------------------------------------
# a2 index (write side: HBM-resident LRU store; read side: device table)
# ------------------------------------------------------------------------------------------------
def test_index_store_vs_oracle_indexer(epp, orc):
    rng = random.Random(5)
    with epp.Engine(16, lru_capacity_per_server=5) as eng:
        ix = orc.Indexer(5)
        for step in range(1500):
            op = rng.random()
            srv = rng.randrange(8)
            if op < 0.85:
                hs = [rng.randrange(60) for _ in range(rng.randint(1, 8))]
                cap = rng.choice([0, 3, 7])
                eng.index_add(srv, hs, cap)
                ix.add(hs, srv, cap)
            elif op < 0.92:
                eng.index_remove_endpoint(srv)
                ix.remove_pod(srv)
            if step % 100 == 99:
                for h in range(60):
                    assert eng.index_get(h) == ix.get(h), (step, h)


@pytest.mark.parametrize("seed,n_srv,universe,default_cap", [(11, 6, 90, 5), (12, 40, 4000, 64), (13, 3, 40, 1)])
def test_index_store_batched_adds_vs_oracle(epp, orc, seed, n_srv, universe, default_cap):
    """indexer.Add / RemovePod applied to the device store in LARGE batches (thousands of queued calls, several calls per
    endpoint and chunk, duplicates inside and across calls, calls longer than the LRU, the all-ones hash) must leave
    exactly the inverted map the reference leaves after running the same calls one by one."""
    rng = random.Random(seed)
    ALL1 = 0xFFFFFFFFFFFFFFFF

    def hash_of(k):
        return ALL1 if k == 0 else (k * 0x9E3779B97F4A7C15) & ALL1

    patched = 0
    with epp.Engine(64, lru_capacity_per_server=default_cap) as eng:
        ix = orc.Indexer(default_cap)
        for rnd in range(6):
            for _ in range(rng.choice([1, 700, 2600])):
                srv = rng.randrange(n_srv)
                n = rng.choice([0, 1, 2, 5, 9, 17, 70]) if default_cap <= 5 else rng.randint(0, 96)
                base = rng.randrange(universe)
                hs = [hash_of((base + (j if rng.random() < 0.8 else rng.randrange(universe))) % universe) for j in range(n)]
                cap = rng.choice([0, 0, 3, 7, 33])
                eng.index_add(srv, hs, cap)
                ix.add(hs, srv, cap)
                if rng.random() < 0.002:
                    eng.index_remove_endpoint(srv)
                    ix.remove_pod(srv)
            if rnd == 3:                                               # CleanUpInactivePods (plugin.go:99-122)
                active = [p for p in range(n_srv) if p % 3 != 1]
                eng.index_retain_endpoints(active)
                for p in ix.pods():
                    if p not in active:
                        ix.remove_pod(p)
            for k in range(universe):
                assert eng.index_get(hash_of(k)) == ix.get(hash_of(k)), (rnd, k)
            assert eng.stats()["index_pairs"] == len(ix.export()[0])
            patched += int(eng.stats()["last_index_patched"])
        # some of the commits above brought the read table up to date from the change log instead of rebuilding it
        # (never when the all-ones hash is involved: that one lives in the side record of the bulk build)
        assert patched > 0 or universe == 90


def test_index_add_picked_many_batches_vs_oracle(epp, orc, tg):
    """PreRequest at batch rate: after every scheduled batch the picks (and prefill picks) are indexed ON THE DEVICE;
    the next batch's decisions must equal the oracle's, whose indexer ran the same Adds one request at a time.  LRU
    capacity is far below the working set, so every batch evicts."""
    import torch
    import helpers
    w = tg.baseline_configs()["config4"].scaled(E=48, R=640, T=1024, name="config4")
    w.non_cached_tokens = 128
    trace = tg.Trace(w)
    role, kv, waiting, running = trace.pool()
    lru = 150
    pool = orc.PoolState(role, kv, waiting, running)
    ix = orc.Indexer(lru)
    primary = orc.make_profile(w.primary_filter, list(w.primary_scorers))
    prefill = orc.make_profile(tg.FILTER_PREFILL, list(w.prefill_scorers))
    with helpers.make_engine(w, lru_capacity_per_server=lru) as eng:
        eng.register_model(tg.MODEL)
        eng.pool_set(np.arange(w.E, dtype=np.uint32), role, kv, waiting, running)
        seen_prefill = 0
        patched = 0
        for b in range(5):
            tokens, _, _ = trace.requests(b * w.R, w.R)
            odec, ototal = helpers.oracle_decisions(orc, w, pool, ix, primary, prefill, tokens)
            if b % 2 == 0:
                dt = torch.from_numpy(tokens.view(np.int32)).cuda()
                ddec, ddet = eng.schedule(dt, uniform_len=w.prompt_bytes, keep_hashes=True)
                dec = epp.decisions_from_torch(ddec)
                det = ddet.cpu().numpy().view(epp.DETAIL_DTYPE).reshape(-1)
            else:
                dec, det = eng.schedule(tokens, uniform_len=w.prompt_bytes, keep_hashes=True)
            helpers.assert_decisions_equal(dec, det, odec, ototal, where=f"batch {b}")
            patched += int(eng.stats()["last_index_patched"])          # how the read table caught up with the previous picks
            eng.index_add_picked()
            for r in range(w.R):                                       # plugin.go:164-200, one request at a time
                if odec["status"][r] != 0:
                    continue
                hs = orc.hash_prompt(tokens[r].tobytes(), tg.MODEL, w.block_size_tokens, w.max_prefix_blocks)
                ix.add(hs, int(odec["pick"][r]))
                if odec["prefill_pick"][r] >= 0:
                    ix.add(hs, int(odec["prefill_pick"][r]))
                    seen_prefill += 1
            assert (dec["match_blocks"] > 0).any() or b == 0
        assert seen_prefill > 0 and patched >= 0       # (tiny tables rebuild: the change set exceeds their free slots)
        eng.index_commit()
        assert eng.stats()["index_pairs"] == len(ix.export()[0])


def test_full_size_write_side_vs_oracle(epp, orc, tg):
    """BASELINE config 3 at FULL size through the write side: schedule 65 536 requests, index all their picks on the
    device (16.8 M indexer.Add hashes, LRU capacity 31 250 -> the hot endpoints evict millions of entries), then
    schedule the NEXT 65 536 requests: every decision must equal the oracle's, whose indexer ran the same Adds one
    request at a time.  Also: the inverted maps have the same number of pairs."""
    import torch
    import helpers
    w = tg.baseline_configs()["config3"]
    trace = tg.Trace(w)
    role, kv, waiting, running = trace.pool()
    pool = orc.PoolState(role, kv, waiting, running)
    primary = orc.make_profile(w.primary_filter, list(w.primary_scorers))
    ix = orc.Indexer()
    nthr = min(64, os.cpu_count() or 1)
    with helpers.make_engine(w) as eng:
        eng.register_model(tg.MODEL)
        eng.pool_set(np.arange(w.E, dtype=np.uint32), role, kv, waiting, running)
        fh, _ = eng.hash_prompts(trace.family_tokens(), uniform_len=w.prompt_bytes)
        hs, es = trace.index_pairs(fh)
        order = np.argsort(es, kind="stable")
        hs, es = hs[order], es[order]
        cuts = np.flatnonzero(np.diff(es)) + 1
        for seg_h, seg_e in zip(np.split(hs, cuts), np.split(es, cuts)):     # seed through indexer.Add, not a snapshot
            eng.index_add(int(seg_e[0]), seg_h)
            ix.add(seg_h, int(seg_e[0]))
        for b in range(2):
            tokens, _, _ = trace.requests(b * w.R, w.R)
            odec, ototal = helpers.oracle_decisions(orc, w, pool, ix, primary, None, tokens, n_threads=nthr)
            dt = torch.from_numpy(tokens.view(np.int32)).cuda()
            ddec, _ = eng.schedule(dt, uniform_len=w.prompt_bytes, detail=False, keep_hashes=True)
            dec = epp.decisions_from_torch(ddec)
            helpers.assert_decisions_equal(dec, None, odec, ototal, where=f"full-size batch {b}")
            if b == 0:
                eng.index_add_picked()
                hh, nb = eng.hash_prompts(dt, uniform_len=w.prompt_bytes)
                hh = hh.cpu().numpy().view(np.uint64)
                nb = nb.cpu().numpy()
                for r in range(w.R):                                          # plugin.go:164-200, sequentially
                    if odec["status"][r] == 0:
                        ix.add(hh[r, : nb[r]], int(odec["pick"][r]))
                eng.index_commit()
                assert eng.stats()["index_pairs"] == len(ix.export()[0])
                assert eng.stats()["last_index_items"] == int(nb[odec["status"] == 0].sum())


def test_index_kats(epp):
    """indexer_test.go:27-113 re-encoded against the engine."""
    with epp.Engine(8, lru_capacity_per_server=3) as eng:
        eng.index_add(7, [1], 2)
        assert eng.index_get(1) == {7}
        eng.index_add(7, [2], 2)
        eng.index_add(7, [3], 2)
        assert eng.index_get(4) == set() and eng.index_get(1) == set()
        assert eng.index_get(2) == {7} and eng.index_get(3) == {7}
    with epp.Engine(8, lru_capacity_per_server=10) as eng:
        for j in range(10):
            eng.index_add(1, [j])
            eng.index_add(2, [j])
        eng.index_add(1, [10])
        assert eng.index_get(0) == {2}
        eng.index_remove_endpoint(2)
        assert eng.index_get(0) == set()
        for j in range(1, 11):
            assert eng.index_get(j) == {1}
    with epp.Engine(8) as eng:                       # the all-ones key uses the side record
        eng.index_load_snapshot([0xFFFFFFFFFFFFFFFF, 0xFFFFFFFFFFFFFFFF, 5, 5, 5], [1, 2, 3, 3, 4])
        assert eng.index_get(0xFFFFFFFFFFFFFFFF) == {1, 2}
        assert eng.index_get(5) == {3, 4}            # duplicate pair removed
        assert eng.index_get(6) == set()


# ------------------------------------------------------------------------------------------------
# a3/a4 match, a5-a9 scores, a10-a14 decisions on scaled BASELINE configs
# ------------------------------------------------------------------------------------------------
def _scaled(tg, name):
    c = tg.baseline_configs()
    return {
        "config1": c["config1"].scaled(R=512),
        "config2": c["config2"].scaled(E=256, R=384, T=512),
        "config3": c["config3"].scaled(E=512, R=512, T=1024),
        # nonCachedTokens raised from 16 so that BOTH decider outcomes occur on 1K-token prompts
        "config4": dataclasses.replace(c["config4"].scaled(E=320, R=512, T=1024), non_cached_tokens=512),
    }[name]


@pytest.mark.parametrize("name", ["config1", "config2", "config3", "config4"])
def test_schedule_vs_oracle(epp, orc, tg, name):
    import helpers
    w = _scaled(tg, name)
    trace = tg.Trace(w)
    tokens, fam_of, shared = trace.requests()
    pool, ix, primary, prefill, (ohs, oes) = helpers.setup_oracle(orc, w, trace)
    odec, ototal = helpers.oracle_decisions(orc, w, pool, ix, primary, prefill, tokens)
    with helpers.make_engine(w) as eng:
        _, (hs, es) = helpers.setup_engine(eng, w, trace)
        np.testing.assert_array_equal(np.sort(hs), np.sort(ohs))       # same index snapshot on both sides
        dec, det = eng.schedule(tokens, uniform_len=w.prompt_bytes)
        helpers.assert_decisions_equal(dec, det, odec, ototal, where=name)
        # the workload must actually exercise the interesting paths
        assert (dec["match_blocks"] > 0).sum() > w.R // 10
        if name == "config1":
            assert (dec["tie_count"] > 1).any()       # ties are real in this workload: the tie rule is exercised
        if name == "config4":
            assert (det["prefill_ran"] == 1).any() and (det["prefill_ran"] == 0).any()
        # Produce parity (dense match rows) vs the oracle's matchLongestPrefix
        match, total = eng.prefix_match(tokens[:64], uniform_len=w.prompt_bytes)
        for r in range(64):
            oh = orc.hash_prompt(tokens[r].tobytes(), tg.MODEL, w.block_size_tokens, w.max_prefix_blocks)
            want, _ = ix.match_longest_prefix(oh, w.E)
            np.testing.assert_array_equal(match[r], want)
            assert total[r] == len(oh)
        # device-pointer batch gives the same records
        import torch
        dt = torch.from_numpy(tokens.view(np.int32)).cuda()
        ddec, _ = eng.schedule(dt, uniform_len=w.prompt_bytes)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(epp.decisions_from_torch(ddec), dec)


@pytest.mark.parametrize("name,R", [("config3", 65536), ("config4", 16384), ("config2", 8192)])
def test_full_size_baseline_configs_vs_oracle(epp, orc, tg, name, R):
    """BASELINE.json's FULL sizes (config 3: 4 096 endpoints x 4 096-token prompts x 65 536 requests): every decision
    of the batch against the multi-threaded oracle -- status, pick, tie count, fp64 score bits, prefill pick -- plus
    the size-independent properties: device-pointer == host-pointer results, and a second run is bit-identical."""
    import torch
    import helpers
    w = tg.baseline_configs()[name].scaled(R=R, name=name)
    trace = tg.Trace(w)
    tokens, fam_of, shared = trace.requests()
    pool, ix, primary, prefill, _ = helpers.setup_oracle(orc, w, trace)
    odec, ototal = helpers.oracle_decisions(orc, w, pool, ix, primary, prefill, tokens, n_threads=min(64, os.cpu_count() or 1))
    with helpers.make_engine(w) as eng:
        helpers.setup_engine(eng, w, trace)
        dt = torch.from_numpy(tokens.view(np.int32)).cuda()
        ddec, ddet = eng.schedule(dt, uniform_len=w.prompt_bytes)
        torch.cuda.synchronize()
        dec = epp.decisions_from_torch(ddec)
        det = ddet.cpu().numpy().view(epp.DETAIL_DTYPE).reshape(-1)
        helpers.assert_decisions_equal(dec, det, odec, ototal, where=name + " full size")
        ddec2, _ = eng.schedule(dt, uniform_len=w.prompt_bytes)
        torch.cuda.synchronize()
        np.testing.assert_array_equal(epp.decisions_from_torch(ddec2), dec)            # idempotent / deterministic
        hdec, _ = eng.schedule(tokens[: R // 4], uniform_len=w.prompt_bytes)            # host path, chunked + pipelined
        np.testing.assert_array_equal(hdec, dec[: R // 4])
        st = eng.stats()
        assert st["index_pairs"] > 0
        # the trace exercises what it claims: hot prefixes, cold prompts, ties, early stops
        assert 0.2 < (dec["match_blocks"] > 0).mean() < 0.9 and (dec["tie_count"] > 1).any()


def test_async_device_batches_match_synchronous_ones(epp, orc, tg):
    """EPP_BATCH_ASYNC: several device batches enqueued back to back; after epp_synchronize every output equals the
    synchronous call's, the stats describe the last batch, and the engine's stream events bracket the work."""
    import torch
    import helpers
    w = tg.baseline_configs()["config3"].scaled(E=256, R=768, name="config3")
    trace = tg.Trace(w)
    tokens, _, _ = trace.requests()
    with helpers.make_engine(w) as eng:
        helpers.setup_engine(eng, w, trace)
        parts = [torch.from_numpy(tokens[i * 256:(i + 1) * 256].view(np.int32)).cuda() for i in range(3)]
        want = [epp.decisions_from_torch(eng.schedule(p, uniform_len=w.prompt_bytes, detail=False)[0]) for p in parts]
        outs = [torch.zeros((256, 32), dtype=torch.uint8, device="cuda") for _ in parts]
        torch.cuda.synchronize()
        eng.event_record(0)
        for p, o in zip(parts, outs):
            eng.schedule(p, uniform_len=w.prompt_bytes, detail=False, out=o, asynchronous=True)
        eng.event_record(1)
        eng.synchronize()
        assert eng.event_elapsed_ms() > 0.0
        for o, wnt in zip(outs, want):
            np.testing.assert_array_equal(epp.decisions_from_torch(o), wnt)
        st = eng.stats()
        assert st["last_kernels_ms"] > 0 and st["last_probes"] > 0
        with pytest.raises(epp.EngineError):
            eng.schedule(tokens[:8], uniform_len=w.prompt_bytes, asynchronous=True)      # host buffers cannot be async


@pytest.mark.parametrize("chunks", [2, 4])
def test_async_chunk_pipelined_batches(epp, orc, tg, monkeypatch, chunks):
    """Async device batches run as EPP_DEV_CHUNKS chunks alternating between the engine's two streams (default 2; ragged
    tail chunk included) and must produce exactly the synchronous single-pass decisions."""
    import torch
    import helpers
    monkeypatch.setenv("EPP_DEV_CHUNKS", str(chunks))
    w = tg.baseline_configs()["config4"].scaled(E=192, R=20000 + 37, T=512, name="config4")
    w.non_cached_tokens = 64
    trace = tg.Trace(w)
    tokens, _, _ = trace.requests()
    with helpers.make_engine(w) as eng:
        helpers.setup_engine(eng, w, trace)
        dt = torch.from_numpy(tokens.view(np.int32)).cuda()
        want, want_det = eng.schedule(dt, uniform_len=w.prompt_bytes)
        want = epp.decisions_from_torch(want)
        out = torch.zeros((w.R, 32), dtype=torch.uint8, device="cuda")
        torch.cuda.synchronize()
        for _ in range(3):
            eng.schedule(dt, uniform_len=w.prompt_bytes, detail=False, out=out, asynchronous=True)
        eng.synchronize()
        np.testing.assert_array_equal(epp.decisions_from_torch(out), want)
        assert (want["prefill_pick"] != 0xFFFFFFFF).any()
        assert eng.stats()["last_kernel_launches"] >= 2 * chunks
        # different batches back to back (each buffer set is reused only after its match kernel has finished), then a
        # kept batch: PreRequest must index the hashes of the LAST batch
        outs = [torch.zeros((w.R, 32), dtype=torch.uint8, device="cuda") for _ in range(4)]
        dts = [torch.roll(dt, shifts=7 * i, dims=0) for i in range(4)]
        torch.cuda.synchronize()
        for i in range(4):
            eng.schedule(dts[i], uniform_len=w.prompt_bytes, detail=False, out=outs[i], asynchronous=True)
        eng.synchronize()
        for i in range(4):
            np.testing.assert_array_equal(epp.decisions_from_torch(outs[i]), np.roll(want, 7 * i))
        # ragged offsets through the same path
        offs = torch.arange(w.R + 1, dtype=torch.int64, device="cuda") * w.prompt_bytes
        out.zero_()
        eng.schedule(dt, offsets=offs, detail=False, out=out, asynchronous=True)
        eng.synchronize()
        np.testing.assert_array_equal(epp.decisions_from_torch(out), want)


def test_global_stop_rule_and_holes(epp, orc):
    """Non-prefix-closed index states: the walk stops at the first block NOBODY holds; endpoints missing earlier
    blocks still count later ones; endpoints outside the slot range keep the walk alive (App. C.5)."""
    with epp.Engine(4, epp.ProfileSpec(0, [epp.ScorerSpec(0, 1.0)]), block_size_tokens=1, max_prefix_blocks=8) as eng:
        eng.register_model(b"m")
        eng.pool_set([0, 1, 2, 3], [1, 1, 1, 1], [0, 0, 0, 0], [0, 0, 0, 0])
        prompt = b"aaaabbbbccccddddeeee"
        h = orc.hash_prompt(prompt, b"m", 1, 8)
        # ep0: blocks 0,1,2 ; ep1: blocks 1,2,4 ; ep 9 (outside the pool): block 3
        eng.index_load_snapshot([h[0], h[1], h[2], h[1], h[2], h[4]], [0, 0, 0, 1, 1, 1])
        d, offs = _pack([prompt])
        m, t = eng.prefix_match(d, offsets=offs)
        assert list(m[0]) == [3, 2, 0, 0] and t[0] == 5
        eng.index_load_snapshot([h[0], h[1], h[2], h[1], h[2], h[4], h[3]], [0, 0, 0, 1, 1, 1, 9])
        m, t = eng.prefix_match(d, offsets=offs)
        assert list(m[0]) == [3, 3, 0, 0]
        dec, _ = eng.schedule(d, offsets=offs)
        assert dec["pick"][0] == 0 and dec["tie_count"][0] == 2 and dec["score"][0] == 3 / 5


def test_many_matched_endpoints_dense_fallback(epp, orc):
    """More than 128 distinct matched endpoints per request -> the warp's dense-scan path; must agree with the oracle."""
    import helpers
    E = 600
    rng = np.random.default_rng(9)
    with epp.Engine(E, epp.ProfileSpec(1, [epp.ScorerSpec(2, 2.0), epp.ScorerSpec(1, 2.0), epp.ScorerSpec(0, 3.0)]),
                    block_size_tokens=2, max_prefix_blocks=32) as eng:
        eng.register_model(b"m")
        kv = rng.integers(0, 1001, E) / 1000.0
        waiting = rng.integers(0, 5, E).astype(np.int32)
        eng.pool_set(np.arange(E), np.ones(E, np.uint8), kv, waiting)
        prompts = [bytes(rng.integers(0, 256, 8 * 20, dtype=np.uint8)) for _ in range(8)]
        ix = orc.Indexer()
        pairs_h, pairs_e = [], []
        for p in prompts[:4]:
            h = orc.hash_prompt(p, b"m", 2, 32)
            for e in range(0, E, 2):                       # 300 endpoints hold a random-depth prefix
                depth = int(rng.integers(1, len(h) + 1))
                pairs_h += h[:depth]
                pairs_e += [e] * depth
        ix.load_pairs(pairs_h, pairs_e)
        eng.index_load_snapshot(pairs_h, pairs_e)
        d, offs = _pack(prompts)
        dec, det = eng.schedule(d, offsets=offs)
        pool = orc.PoolState(np.ones(E, np.uint8), kv, waiting)
        prof = orc.make_profile(1, [(2, 2.0, 0), (1, 2.0, 0), (0, 3.0, 0)])
        odec, ototal = orc.cycle_batch(b"m", 2, 32, 0, False, ix, prof, None, pool, d, offs, 1)
        helpers.assert_decisions_equal(dec, det, odec, ototal, where="dense-fallback")
        m, t = eng.prefix_match(d, offsets=offs)
        for r in range(8):
            want, _ = ix.match_longest_prefix(orc.hash_prompt(prompts[r], b"m", 2, 32), E)
            np.testing.assert_array_equal(m[r], want)


def _tied_pool(rng, E, n_levels):
    """A pool where many endpoints share a load level, so that arg-max sets are large."""
    kv = rng.integers(0, n_levels, E) / float(n_levels)
    waiting = rng.integers(0, 2, E).astype(np.int32)
    return kv, waiting


@pytest.mark.parametrize("tie_seed", [0x5EED, 1])
def test_random_tie_rule_vs_oracle(epp, orc, tie_seed):
    """epp_config.tie_seed != 0: the pick is the member of rank orc_tie_rank(seed, 4 * ordinal + profile, |set|) of the
    arg-max set in ascending slot order (include/epp_engine.h, "Tie rule") -- through the sparse kernel (matched and
    unmatched members mixed), the dense-counter kernel (> 32 matched endpoints) and the injected-match entry point;
    the ordinal keeps counting across batches.  The reference draws a uniformly random member
    (picker/maxscore/picker.go:91-102): the picks of a batch of equal requests must spread over the set."""
    import helpers
    E, bst, B = 96, 2, 16
    rng = np.random.default_rng(41)
    primary_spec = [epp.ScorerSpec(2, 1.0), epp.ScorerSpec(1, 1.0), epp.ScorerSpec(0, 2.0)]
    with epp.Engine(E, epp.ProfileSpec(1, primary_spec), epp.ProfileSpec(2, [epp.ScorerSpec(2, 1.0), epp.ScorerSpec(0, 1.0)]),
                    block_size_tokens=bst, max_prefix_blocks=B, non_cached_tokens=4, tie_seed=tie_seed) as eng:
        eng.register_model(b"m")
        kv, waiting = _tied_pool(rng, E, 2)
        role = np.where(np.arange(E) % 3 == 0, 2, 1).astype(np.uint8)        # a third prefill, the rest decode
        eng.pool_set(np.arange(E), role, kv, waiting)
        fam = [bytes(rng.integers(0, 256, 8 * B, dtype=np.uint8)) for _ in range(6)]
        pairs_h, pairs_e = [], []
        for g, p in enumerate(fam):
            h = orc.hash_prompt(p, b"m", bst, B)
            holders = rng.choice(E, size=[2, 5, 9, 20, 40, 70][g], replace=False)   # the last two overflow the 32-entry map
            for e in holders:
                depth = int(rng.choice([len(h) // 2, len(h)]))          # few distinct depths: equal scores among holders
                pairs_h += h[:depth]
                pairs_e += [int(e)] * depth
        ix = orc.Indexer()
        ix.load_pairs(pairs_h, pairs_e)
        eng.index_load_snapshot(pairs_h, pairs_e)
        pool = orc.PoolState(role, kv, waiting)
        prim = orc.make_profile(1, [(2, 1.0, 0), (1, 1.0, 0), (0, 2.0, 0)])
        pref = orc.make_profile(2, [(2, 1.0, 0), (0, 1.0, 0)])
        spread = set()
        for batch in range(3):
            prompts = []
            for _ in range(400):
                g = int(rng.integers(0, len(fam) + 2))
                if g >= len(fam):
                    prompts.append(bytes(rng.integers(0, 256, 8 * B, dtype=np.uint8)))      # cold: the whole top group ties
                else:
                    keep = int(rng.integers(1, B + 1)) * 8
                    prompts.append(fam[g][:keep] + bytes(rng.integers(0, 256, 8 * B - keep, dtype=np.uint8)))
            d, offs = _pack(prompts)
            base = eng.stats()["n_decisions"]
            assert base == 400 * batch
            dec, det = eng.schedule(d, offsets=offs)
            odec, ototal = orc.cycle_batch(b"m", bst, B, 4, False, ix, prim, pref, pool, d, offs, 2, tie_seed=tie_seed, tie_base=base)
            helpers.assert_decisions_equal(dec, det, odec, ototal, where=f"tie rule, batch {batch}")
            assert (dec["tie_count"] > 1).sum() > 100 and (det["prefill_tie_count"] > 1).any()
            spread |= set(int(x) for x in dec["pick"][dec["tie_count"] > 6])
        assert len(spread) > 6                                  # not one hot endpoint
        # injected match rows (dense pick kernel): same rule, ordinals keep counting
        match = rng.integers(0, 3, size=(64, E)).astype(np.int32) * 4
        total = np.full(64, B, np.int32)
        base = eng.stats()["n_decisions"]
        dec2, det2 = eng.schedule_with_match(match, total, input_len_bytes=np.full(64, 8 * B, np.int64))
        scratch = np.zeros(E)
        for r in range(64):
            want = orc.schedule(prim, pref, pool, match[r], B, bst, 8 * B, 4)
            scores, mx, lowest, amax = orc.profile_run(prim, pool, match[r], B)
            k = orc.tie_rank(tie_seed, 4 * (base + r), len(amax))
            assert dec2["pick"][r] == amax[k] and dec2["tie_count"][r] == len(amax) and dec2["score"][r] == mx
        assert eng.stats()["n_decisions"] == base + 64


def test_encode_stage_vs_oracle(epp, orc):
    """The optional encode stage of the disagg handler (disagg_profile_handler.go:284-295): decode pick, then -- for
    requests with multimodal content (always-disagg-multimodal-decider) -- the encode profile (encode-filter + scorers),
    then the P/D decider and the prefill profile.  EPD style (no prefill stage) = nonCachedTokens 0."""
    import helpers
    E, bst, B = 80, 2, 16
    rng = np.random.default_rng(43)
    enc_spec = epp.ProfileSpec(3, [epp.ScorerSpec(2, 1.0), epp.ScorerSpec(1, 2.0)])
    for nct in (4, 0):
        with epp.Engine(E, epp.ProfileSpec(1, [epp.ScorerSpec(2, 1.0), epp.ScorerSpec(0, 2.0)]),
                        epp.ProfileSpec(2, [epp.ScorerSpec(2, 1.0), epp.ScorerSpec(0, 1.0)]), block_size_tokens=bst,
                        max_prefix_blocks=B, non_cached_tokens=nct, encode=enc_spec) as eng:
            eng.register_model(b"m")
            kv = rng.integers(0, 11, E) / 10.0
            waiting = rng.integers(0, 4, E).astype(np.int32)
            role = rng.choice([1, 2, 3, 5, 6, 7, 0, 8], size=E).astype(np.uint8)     # every role of roles.go:25-44
            eng.pool_set(np.arange(E), role, kv, waiting)
            fam = [bytes(rng.integers(0, 256, 8 * B, dtype=np.uint8)) for _ in range(4)]
            pairs_h, pairs_e = [], []
            for p in fam:
                h = orc.hash_prompt(p, b"m", bst, B)
                for e in rng.choice(E, size=6, replace=False):
                    depth = int(rng.integers(1, len(h) + 1))
                    pairs_h += h[:depth]
                    pairs_e += [int(e)] * depth
            ix = orc.Indexer()
            ix.load_pairs(pairs_h, pairs_e)
            eng.index_load_snapshot(pairs_h, pairs_e)
            prompts = []
            for _ in range(300):
                g = int(rng.integers(0, 5))
                keep = int(rng.integers(1, B + 1)) * 8
                prompts.append((fam[g][:keep] if g < 4 else b"") + bytes(rng.integers(0, 256, 8 * B - (keep if g < 4 else 0), dtype=np.uint8)))
            d, offs = _pack(prompts)
            mm = (rng.random(300) < 0.4).astype(np.uint8)
            dec, det = eng.schedule(d, offsets=offs, multimodal=mm)
            pool = orc.PoolState(role, kv, waiting)
            odec, ototal = orc.cycle_batch(b"m", bst, B, nct, False, ix, orc.make_profile(1, [(2, 1.0, 0), (0, 2.0, 0)]),
                                           orc.make_profile(2, [(2, 1.0, 0), (0, 1.0, 0)]), pool, d, offs, 2,
                                           encode=orc.make_profile(3, [(2, 1.0, 0), (1, 2.0, 0)]), multimodal=mm)
            helpers.assert_decisions_equal(dec, det, odec, ototal, where=f"encode stage nct={nct}")
            ok = dec["status"] == 0
            np.testing.assert_array_equal(det["encode_ran"][ok], mm[ok].astype(np.uint32))
            assert (det["encode_pick"][ok & (mm == 1)] != 0xFFFFFFFF).all()
            if nct == 0:
                assert (det["prefill_ran"] == 0).all()             # EPD: encode + decode only
            else:
                assert (det["prefill_ran"] == 1).any()
            # the same batch through device pointers
            import torch
            dd, do = torch.from_numpy(d).cuda(), torch.from_numpy(offs.view(np.int64)).cuda()
            ddec, ddet = eng.schedule(dd, offsets=do, multimodal=torch.from_numpy(mm).cuda())
            torch.cuda.synchronize()
            np.testing.assert_array_equal(epp.decisions_from_torch(ddec), dec)
            np.testing.assert_array_equal(ddet.cpu().numpy().view(epp.DETAIL_DTYPE).reshape(-1), det)
            with pytest.raises(epp.EngineError):
                eng.schedule(d, offsets=offs, multimodal=mm, detail=False)      # the encode pick needs the detail record


@pytest.mark.parametrize("tie_seed", [0, 99])
def test_small_batch_zero_copy_path_vs_oracle(epp, orc, tie_seed, monkeypatch):
    """Host batches of 1 .. 600 requests whose prompts live in pinned memory take the single-launch path of
    csrc/cycle_small.cu (one CTA per request, prompts read over PCIe, decisions written to pinned memory, no copy
    engine): ragged prompts incl. empty / shorter than a block / partial trailing block / longer than the cap, P/D and
    encode stages, > 32 holders (dense-counter pass), both tie rules -- all equal to the oracle and to the ordinary
    path (EPP_SMALL_BATCH=0)."""
    import helpers
    E, bst, B = 96, 8, 24                          # 32-byte blocks
    rng = np.random.default_rng(71)
    bb = 4 * bst
    kv = rng.integers(0, 3, E) / 3.0
    waiting = rng.integers(0, 3, E).astype(np.int32)
    role = rng.choice([1, 2, 3, 5, 7, 0], size=E).astype(np.uint8)
    prim, pref, enc = [(2, 1.0, 0), (1, 1.0, 0), (0, 2.0, 0)], [(2, 1.0, 0), (0, 1.0, 0)], [(1, 1.0, 0)]
    spec = lambda f, sc: epp.ProfileSpec(f, [epp.ScorerSpec(k, w, p) for k, w, p in sc])
    fam = [bytes(rng.integers(0, 256, bb * B, dtype=np.uint8)) for _ in range(5)]
    pairs_h, pairs_e = [], []
    for g, p in enumerate(fam):
        h = orc.hash_prompt(p, b"m", bst, B)
        for e in rng.choice(E, size=[2, 6, 12, 30, 70][g], replace=False):     # the last family overflows the sparse map
            depth = int(rng.choice([len(h) // 2, len(h)]))
            pairs_h += h[:depth]
            pairs_e += [int(e)] * depth
    ix = orc.Indexer()
    ix.load_pairs(pairs_h, pairs_e)
    pool = orc.PoolState(role, kv, waiting)

    def make_batch(n):
        prompts = []
        for i in range(n):
            g = int(rng.integers(0, len(fam) + 2))
            kind = int(rng.integers(0, 8))
            if kind == 0:
                prompts.append(b"" if i % 2 else bytes(rng.integers(0, 256, bb - 1, dtype=np.uint8)))   # no hash at all
            elif g >= len(fam):
                prompts.append(bytes(rng.integers(0, 256, int(rng.integers(bb, bb * B + 40)), dtype=np.uint8)))
            else:
                keep = int(rng.integers(1, B + 1)) * bb
                tail = int(rng.integers(0, 2 * bb))                # partial trailing block / beyond the cap
                prompts.append(fam[g][:keep] + bytes(rng.integers(0, 256, tail, dtype=np.uint8)))
        starts, pos = [], 0
        for p in prompts:                                          # rows start on 32-byte boundaries, like the batcher's
            starts.append(pos)
            pos += (len(p) + 31) & ~31
        buf = epp.PinnedBuffer(pos + 64)
        offs = np.array(starts + [pos], dtype=np.uint64)
        lens = np.array([len(p) for p in prompts], dtype=np.uint64)
        for p, st in zip(prompts, starts):
            buf.array[st: st + len(p)] = np.frombuffer(p, dtype=np.uint8)
        d, o = _pack(prompts)
        return buf, offs, lens, d, o

    results = {}
    for small, pipe in (("1024", "16"), ("1024", "0"), ("0", "16")):
        monkeypatch.setenv("EPP_SMALL_BATCH", small)
        monkeypatch.setenv("EPP_SMALL_PIPELINE", pipe)     # kernel started before the copies land (1 / 2 / 4 copies) or behind one copy
        rng = np.random.default_rng(72)
        with epp.Engine(E, spec(1, prim), spec(2, pref), block_size_tokens=bst, max_prefix_blocks=B, non_cached_tokens=8,
                        encode=spec(3, enc), tie_seed=tie_seed) as eng:
            eng.register_model(b"m")
            eng.pool_set(np.arange(E), role, kv, waiting)
            eng.index_load_snapshot(pairs_h, pairs_e)
            got = []
            for n in (1, 2, 20, 33, 130, 600, 1):
                buf, offs, lens, d, o = make_batch(n)
                mm = (rng.random(n) < 0.5).astype(np.uint8)
                base = eng.stats()["n_decisions"]
                dec, det = eng.schedule(buf.array, offsets=offs, lengths=lens, multimodal=mm, n_requests=n)
                st = eng.stats()
                if small != "0":
                    assert st["last_kernel_launches"] in (1, 2), st["last_kernel_launches"]   # 2: + the dense-counter pass
                    assert st["last_kernels_ms"] > 0
                else:
                    assert st["last_kernel_launches"] >= 3
                odec, ototal = orc.cycle_batch(b"m", bst, B, 8, False, ix, orc.make_profile(1, prim), orc.make_profile(2, pref),
                                               pool, d, o, 2, tie_seed=tie_seed, tie_base=base,
                                               encode=orc.make_profile(3, enc), multimodal=mm)
                helpers.assert_decisions_equal(dec, det, odec, ototal, where=f"small={small} pipeline={pipe} n={n}")
                got.append((dec.copy(), det.copy()))
                buf.close()
            results[small, pipe] = got
    for other in (("1024", "0"), ("0", "16")):
        for (a, ad), (b, bd) in zip(results["1024", "16"], results[other]):
            np.testing.assert_array_equal(a, b)
            np.testing.assert_array_equal(ad, bd)


def test_small_batch_prompt_buffer_may_be_rewritten_when_the_call_returns(epp, orc):
    """A cold request is decided by the global-stop rule long before its hash chain has reached the end of the prompt,
    and epp_schedule returns as soon as every request is decided.  From then on the caller may rewrite its prompt
    buffer, and the next batch's copy may refill the engine's staging buffer -- the hashes PreRequest indexes afterwards
    (incl. the one of the trailing PARTIAL block, hashing.go:90-96, which the chain reaches last) must still be those
    of the prompts that were scheduled.  1 request = the kernel reads the caller's pinned buffer; 24 = DMA-copied."""
    E, bst, B = 8, 8, 2048                         # 64 KiB prompts: the chain runs for > 100 us
    bb = 4 * bst
    rng = np.random.default_rng(99)
    role = np.full(E, 3, dtype=np.uint8)
    spec = epp.ProfileSpec(1, [epp.ScorerSpec(2, 1.0, 0)])
    for n in (1, 24):
        with epp.Engine(E, spec, None, block_size_tokens=bst, max_prefix_blocks=B, lru_capacity_per_server=100000) as eng:
            eng.register_model(b"m")
            eng.pool_set(np.arange(E), role, np.zeros(E), np.zeros(E, dtype=np.int32))
            row = bb * B
            buf = epp.PinnedBuffer(2 * n * row)
            batches = []
            for k in range(2):
                prompts = [bytes(rng.integers(0, 256, row - int(rng.integers(1, bb)), dtype=np.uint8)) for _ in range(n)]
                batches.append(prompts)
            offs = np.arange(n + 1, dtype=np.uint64) * np.uint64(row)

            def fill(prompts):
                for i, p in enumerate(prompts):
                    buf.array[i * row: i * row + len(p)] = np.frombuffer(p, dtype=np.uint8)
                return np.array([len(p) for p in prompts], dtype=np.uint64)

            lens = fill(batches[0])
            dec0, _ = eng.schedule(buf.array, offsets=offs, lengths=lens, n_requests=n, keep_hashes=True)
            buf.array[: n * row] = 0xA5             # the caller's buffer is the caller's again
            eng.index_add_picked()                  # PreRequest of batch 0 (stream-ordered behind its kernel)
            lens = fill(batches[1])
            dec1, _ = eng.schedule(buf.array, offsets=offs, lengths=lens, n_requests=n, keep_hashes=True)   # refills the staging buffer
            eng.index_commit()
            assert (dec0["status"] == 0).all() and (dec1["status"] == 0).all()
            assert (dec0["match_blocks"] == 0).all()
            for i, p in enumerate(batches[0]):
                hs = orc.hash_prompt(p, b"m", bst, B)
                assert len(hs) == B                # B - 1 full blocks + the partial one
                for j in (0, B // 2, B - 2, B - 1):
                    assert eng.index_get(int(hs[j])) == {int(dec0["pick"][i])}, (n, i, j)
            buf.close()


def test_index_commit_interval_bounds_the_staleness(epp, orc):
    """epp_config.index_commit_interval_us: with a long interval a scheduling call keeps reading the table of the last
    commit (the reference applies PreRequest in a goroutine of its own, approximateprefix/plugin.go:189-194), an
    explicit epp_index_commit makes the picks visible at once; with interval 0 the next call sees them."""
    E, bst, B = 16, 8, 8
    rng = np.random.default_rng(5)
    prompts = [bytes(rng.integers(0, 256, 4 * bst * B, dtype=np.uint8)) for _ in range(40)]
    d, offs = _pack(prompts)
    for interval, stale in ((10_000_000, True), (0, False)):
        with epp.Engine(E, epp.ProfileSpec(0, [epp.ScorerSpec(0, 1.0)]), block_size_tokens=bst, max_prefix_blocks=B,
                        index_commit_interval_us=interval) as eng:
            eng.register_model(b"m")
            eng.pool_set(np.arange(E), np.zeros(E, np.uint8), np.zeros(E), np.zeros(E, np.int32))
            dec0, _ = eng.schedule(d, offsets=offs, keep_hashes=True)          # first call: commits (nothing to commit)
            assert (dec0["match_blocks"] == 0).all()
            eng.index_add_picked()
            dec1, _ = eng.schedule(d, offsets=offs)
            if stale:
                np.testing.assert_array_equal(dec1, dec0)                       # the picks are not visible yet
                eng.index_commit()
                dec1, _ = eng.schedule(d, offsets=offs)
            assert (dec1["match_blocks"] == B).all() and (dec1["pick"] == dec0["pick"]).all()


def test_large_pool_global_counters(epp, orc, tg):
    """E too large for per-warp shared-memory counters -> zeroed global scratch path (config-5-sized pool on 1 GPU)."""
    import helpers
    w = tg.baseline_configs()["config5"].scaled(R=256, T=512, name="config5-smallR")
    trace = tg.Trace(w)
    tokens, _, _ = trace.requests()
    pool, ix, primary, prefill, _ = helpers.setup_oracle(orc, w, trace)
    odec, ototal = helpers.oracle_decisions(orc, w, pool, ix, primary, prefill, tokens)
    with helpers.make_engine(w) as eng:
        helpers.setup_engine(eng, w, trace)
        for _ in range(2):                                  # twice: counters must come back to zero
            dec, det = eng.schedule(tokens, uniform_len=w.prompt_bytes)
            helpers.assert_decisions_equal(dec, det, odec, ototal, where="config5")


def test_score_columns_vs_oracle(epp, orc):
    """Scorer.Score parity (dense [R][E] rows): every scorer kind, clamp, filters, ordered weighted sum."""
    rng = np.random.default_rng(21)
    E, R = 97, 9
    roles = rng.choice([0, 1, 2, 3, 4, 5, 8], E).astype(np.uint8)
    kv = np.where(rng.random(E) < 0.2, rng.choice([0.0, 1.0, 1.5, -0.25], E), rng.random(E))
    waiting = np.where(rng.random(E) < 0.6, 0, rng.integers(1, 300, E)).astype(np.int32)
    running = rng.integers(0, 50, E).astype(np.int32)
    ext = rng.random((4, E)) * 1.4 - 0.2
    ext[2] = np.where(rng.random(E) < 0.3, 0, rng.integers(0, 9000, E))        # InFlightLoad.Tokens
    ext[3] = np.where(rng.random(E) < 0.3, 0, rng.integers(0, 40, E))          # InFlightLoad.Requests
    scorers = [(0, 3.0, 0), (1, 2.0, 0), (2, 2.0, 0), (3, 1.0, 10), (4, 0.37, 1), (5, 1.5, 0), (6, 1.25, 5000.0, 2),
               (7, 0.8, 0.5, 3, 2.0)]
    total = rng.choice([0, 1, 7, 256], R).astype(np.int32)
    match = (rng.random((R, E)) * (total[:, None] + 1)).astype(np.int32)
    match = np.minimum(match, total[:, None])
    for filt in (0, 1, 2):
        with epp.Engine(E, epp.ProfileSpec(filt, [epp.ScorerSpec(*s) for s in scorers]), n_ext_cols=4) as eng:
            eng.pool_set(np.arange(E), roles, kv, waiting, running, ext)
            pool = orc.PoolState(roles, kv, waiting, running, ext)
            prof = orc.make_profile(filt, scorers)
            cand = np.array([orc.lib().orc_role_filter_keeps(filt, int(r)) for r in roles], np.uint8)
            got = eng.score(match, total, 0, -1)
            for r in range(R):
                want, _, _, _ = orc.profile_run(prof, pool, match[r], int(total[r]))
                if cand.any():
                    np.testing.assert_array_equal(got[r].view(np.uint64), want.view(np.uint64))
            for si, s in enumerate(scorers):
                col = eng.score(match, total, 0, si)
                for r in range(R):
                    want = orc.score_column(s, pool, cand, match[r], int(total[r]))
                    np.testing.assert_array_equal(col[r].view(np.uint64), want.view(np.uint64))
            dec, det = eng.schedule_with_match(match, total)
            for r in range(R):
                d = orc.schedule(prof, None, pool, match[r], int(total[r]), 16, 0, 0)
                assert dec["status"][r] == d.status
                if d.status == 0:
                    assert dec["pick"][r] == d.pick and dec["tie_count"][r] == d.tie_count
                    assert dec["score"][r : r + 1].view(np.uint64)[0] == np.float64(d.score).view(np.uint64)


def test_token_load_and_active_request_kats(epp):
    """token_load_test.go:32-61 and active_request_test.go:36-92, 172-216 re-encoded against the engine."""
    P = epp.plugins

    def scores(scorer, column_values):
        n = len(column_values)
        prof = epp.ProfileSpec(0, [epp.ScorerSpec(scorer.kind, 1.0, scorer.param, scorer.column, scorer.param2)])
        with epp.Engine(n, prof, n_ext_cols=1) as eng:
            eng.pool_set(np.arange(n), np.zeros(n, np.uint8), np.zeros(n), np.zeros(n, np.int32), np.zeros(n, np.int32),
                         np.asarray(column_values, dtype=np.float64).reshape(1, n))
            return list(eng.score(np.zeros((1, n), np.int32), np.zeros(1, np.int32), 0, 0)[0])

    assert scores(P.TokenLoadScorer(0, 1000), [0, 500, 1000]) == [1.0, 0.5, 0.0]
    assert scores(P.TokenLoadScorer(0, 1000), [-5, 2500, 250]) == [1.0, 0.0, 0.75]
    assert scores(P.TokenLoadScorer(0, 0), [4194304 // 2]) == [0.5]                  # <= 0 -> default threshold
    assert scores(P.NewActiveRequest(0), [0, 0, 0]) == [1.0, 1.0, 1.0]               # no load attribute set
    assert scores(P.NewActiveRequest(0), [3, 0, 6]) == [0.5, 1.0, 0.0]
    assert scores(P.NewActiveRequest(0), [4, 0, 1]) == [0.0, 1.0, 0.75]
    assert scores(P.NewActiveRequest(0, 0, 0.0), [0, 0]) == [1.0, 1.0]               # binary mode
    assert scores(P.NewActiveRequest(0, 0, 0.0), [1, 0]) == [0.0, 1.0]
    assert scores(P.NewActiveRequest(0, 1, 0.5), [1, 2, 0]) == [1.0, 0.0, 1.0]       # hybrid mode
    assert scores(P.NewActiveRequest(0, -3, 7.0), [2, 4]) == [0.5, 0.0]              # invalid params -> defaults


def test_lora_affinity_kats_and_parity(epp, orc, tg):
    """lora-affinity-scorer: the reference's table (lora_affinity_test.go:30-141) through the engine, then the whole
    cycle (prefix matches from the index + queue + lora-affinity, three adapters, sparse kernel AND its dense-counter
    fallback) against the oracle evaluated per adapter."""
    import torch
    import helpers
    P = epp.plugins
    LA = P.LoraAffinityScorer()
    prof = epp.ProfileSpec(0, [epp.ScorerSpec(LA.kind, 1.0)])
    with epp.Engine(5, prof) as eng:
        m1 = eng.register_model(b"active-model-1")
        m2 = eng.register_model(b"active-model-2")
        eng.pool_set(np.arange(5), np.zeros(5, np.uint8), np.zeros(5), np.zeros(5, np.int32), np.zeros(5, np.int32))
        # pod1..pod5 of "Multiple endpoints with mixed active and waiting models"
        eng.pool_set_lora(np.arange(5), [5, 5, 2, 2, 2], [1, 2, 1, 2, 2],
                          [(0, m1, 1), (1, m2, 1), (1, m1, 2), (2, m2, 1), (3, m1, 2)])
        z = np.zeros((1, 5), np.int32)
        assert list(eng.score(z, [0], 0, 0, model_ids=[m1])[0]) == [1.0, 0.8, 0.8, 0.6, 0.0]
        assert list(eng.score(z, [0], 0, 0, model_ids=[m2])[0]) == [0.8, 1.0, 1.0, 0.0, 0.0]
        dec, _ = eng.schedule_with_match(z, [0], model_ids=[m1])
        assert dec["pick"][0] == 0 and dec["score"][0] == 1.0 and dec["tie_count"][0] == 1

    # ---- whole cycle, several adapters
    w = tg.baseline_configs()["config3"].scaled(E=96, R=1536, T=512, name="config3")
    trace = tg.Trace(w)
    role, kv, waiting, running = trace.pool()
    tokens, _, _ = trace.requests()
    rng = np.random.default_rng(5)
    A = 3
    names = [tg.MODEL] + [tg.MODEL + b"-lora%d" % a for a in range(1, A)]
    mx = rng.integers(0, 5, w.E).astype(np.int32)
    state = np.zeros((A, w.E), np.uint8)
    for a in range(A):
        k = [6, 40, 70][a]                                     # adapter 2 is resident on more endpoints than the lane map holds
        idx = rng.choice(w.E, k, replace=False)
        state[a, idx] = rng.choice([1, 2], k)
    loaded = (state != 0).sum(axis=0).astype(np.int32) + rng.integers(0, 2, w.E).astype(np.int32)
    scorers = [(0, 2.0, 0.0), (2, 1.0, 0.0), (8, 1.5, 0.0)]    # prefix, queue, lora-affinity
    model_of = rng.integers(0, A, w.R).astype(np.uint32)
    with epp.Engine(w.E, epp.ProfileSpec(0, [epp.ScorerSpec(*s) for s in scorers]), block_size_tokens=w.block_size_tokens,
                    max_prefix_blocks=w.max_prefix_blocks) as eng:
        mids = [eng.register_model(n) for n in names]
        eng.pool_set(np.arange(w.E, dtype=np.uint32), role, kv, waiting, running)
        members = [(e, mids[a], int(state[a, e])) for a in range(A) for e in range(w.E) if state[a, e]]
        eng.pool_set_lora(np.arange(w.E), mx, loaded, members)
        # index: every adapter has its own hash chain (the seed is XXH64(model)), families cached per adapter 0 only
        fh, _ = eng.hash_prompts(trace.family_tokens(), uniform_len=w.prompt_bytes)
        hs, es = trace.index_pairs(fh)
        eng.index_load_snapshot(hs, es)
        ix = orc.Indexer()
        ix.load_pairs(hs, es)
        dt = torch.from_numpy(tokens.view(np.int32)).cuda()
        ddec, _ = eng.schedule(dt, uniform_len=w.prompt_bytes, model_ids=torch.from_numpy(np.array(mids, np.uint32)[model_of].view(np.int32)).cuda())
        dec = epp.decisions_from_torch(ddec)
        hdec, _ = eng.schedule(tokens, uniform_len=w.prompt_bytes, model_ids=np.array(mids, np.uint32)[model_of])
        np.testing.assert_array_equal(hdec, dec)
        prof_o = orc.make_profile(0, scorers)
        st = eng.stats()
        for a in range(A):
            pool = orc.PoolState(role, kv, waiting, running).set_lora(state[a], mx, loaded)
            sel = np.flatnonzero(model_of == a)
            offs = np.arange(len(sel) + 1, dtype=np.uint64) * np.uint64(w.prompt_bytes)
            odec, ototal = orc.cycle_batch(names[a], w.block_size_tokens, w.max_prefix_blocks, 0, False, ix, prof_o, None,
                                           pool, np.ascontiguousarray(tokens[sel]), offs, 4)
            helpers.assert_decisions_equal(dec[sel], None, odec, ototal, where=f"adapter {a}")
        assert (dec["match_blocks"] > 0).any()


# ------------------------------------------------------------------------------------------------
# the reference's own scheduler tests through the interface mirror
# ------------------------------------------------------------------------------------------------
def test_reference_TestSchedule(epp):
    """pkg/epp/scheduling/scheduler_test.go:40-157 (default 4-scorer profile -> pod2, score 2.8)."""
    P = epp.plugins
    prof = P.NewSchedulerProfile().WithScorers(
        P.NewWeightedScorer(P.KVCacheUtilizationScorer(), 1), P.NewWeightedScorer(P.QueueScorer(), 1),
        P.NewWeightedScorer(P.PrefixCacheScorer(), 1), P.NewWeightedScorer(P.ExternalScorer(0), 1),
    ).WithPicker(P.NewMaxScorePicker(1))
    sched = P.Scheduler(P.SingleProfileHandler(), {"default": prof}, ext_columns=1)
    with pytest.raises(P.SchedulingError):
        sched.Schedule(P.InferenceRequest(TargetModel="any-model"), [])
    pods = [P.NewEndpoint(P.EndpointMetadata("pod1"), P.Metrics(0, 0.2)),
            P.NewEndpoint(P.EndpointMetadata("pod2"), P.Metrics(0, 0.2)),
            P.NewEndpoint(P.EndpointMetadata("pod3"), P.Metrics(10, 0.8))]
    lora = [[0.0, 1.0, 0.8]]        # lora_affinity.go:76-100 tiers for TargetModel "critical"
    res = sched.Schedule(P.InferenceRequest(TargetModel="critical"), pods, ext=lora)
    tgt = res.ProfileResults["default"]
    assert tgt.TargetEndpoints[0].GetMetadata().Name == "pod2" and tgt.Score == 2.8
    assert res.PrimaryProfileName == "default"


def test_reference_TestPDSchedule(epp):
    """profilehandler/disagg/scheduler_test.go:34-297."""
    P = epp.plugins
    ep1 = P.NewEndpoint(P.EndpointMetadata("endpoint1", {P.RoleLabel: P.RolePrefill}, "1.2.3.4"), P.Metrics(0))
    ep2 = P.NewEndpoint(P.EndpointMetadata("endpoint2", {P.RoleLabel: P.RoleDecode}, "5.6.7.8"), P.Metrics(0))
    norole = P.NewEndpoint(P.EndpointMetadata("noRoleEndpoint1", {}, "1.1.1.1"), P.Metrics(2))

    def mk():
        prefill = P.NewSchedulerProfile().WithFilters(P.NewPrefillRole()).WithPicker(P.NewMaxScorePicker(1))
        prefill.AddPlugins(P.NewWeightedScorer(P.PrefixCacheScorer(), 50))
        decode = P.NewSchedulerProfile().WithFilters(P.NewDecodeRole()).WithScorers(
            P.NewWeightedScorer(P.NewLoadAware(128), 1)).WithPicker(P.NewMaxScorePicker(1))
        decode.AddPlugins(P.NewWeightedScorer(P.PrefixCacheScorer(), 0))
        handler = P.DisaggProfileHandler("decode", "prefill", P.PrefixBasedPDDecider(2))
        return P.Scheduler(handler, {"prefill": prefill, "decode": decode})

    def run(prompt, pods, cached):
        tokens = len(prompt) // 4
        for p in pods:
            p.Put(P.PrefixCacheMatchInfoKey, P.NewPrefixCacheMatchInfo(tokens if cached else 0, tokens, 1))
        return mk().Schedule(P.InferenceRequest(TargetModel="critical", Prompt=prompt), pods)

    def names(res):
        return {k: v.TargetEndpoints[0].GetMetadata().Name for k, v in res.ProfileResults.items()}

    with pytest.raises(P.SchedulingError):
        mk().Schedule(P.InferenceRequest(Prompt=b"12345678901"), [])
    assert names(run(b"12345678901", [ep2], False)) == {"decode": "endpoint2"}
    with pytest.raises(P.SchedulingError):
        run(b"12345678901", [ep1], False)
    assert names(run(b"12345678906", [ep1, ep2], False)) == {"decode": "endpoint2", "prefill": "endpoint1"}
    assert names(run(b"12345678906", [ep1, ep2], True)) == {"decode": "endpoint2"}
    assert names(run(b"12345", [ep1, ep2], False)) == {"decode": "endpoint2"}
    assert names(run(b"12345", [ep1, ep2], True)) == {"decode": "endpoint2"}
    assert names(run(b"12345678901", [ep1, norole], False)) == {"decode": "noRoleEndpoint1", "prefill": "endpoint1"}
    long = b"1234567890123456789012345678901234567890"
    r = run(long, [ep1, ep2, norole], False)
    assert names(r) == {"decode": "endpoint2", "prefill": "endpoint1"} and r.ProfileResults["decode"].Score == 0.5
    assert names(run(long, [ep1, ep2, norole], True)) == {"decode": "endpoint2"}


def test_reference_prefix_plugin_flow(epp):
    """approximateprefix/plugin_test.go:37-82 and :174-226 through Produce / PreRequest on the engine."""
    P = epp.plugins
    with epp.Engine(3, epp.ProfileSpec(0, [epp.ScorerSpec(0, 1.0)]), block_size_tokens=1) as eng:
        eng.pool_set([0, 1, 2], [0, 0, 0], [0, 0, 0], [0, 0, 0])
        prod = P.ApproxPrefixCacheProducer(eng, b"test-model1")
        pods = [P.NewEndpoint(P.EndpointMetadata(f"pod{i+1}")) for i in range(3)]
        m, t = prod.Produce([b"aaaabbbb"], pods)                     # empty index
        assert list(m[0]) == [0, 0, 0] and t[0] == 2
        info, ok = pods[0].Get(P.PrefixCacheMatchInfoKey)
        assert ok and (info.MatchBlocks(), info.TotalBlocks()) == (0, 2)
        m, t = prod.Produce([b"aaaaaa"], pods)
        assert t[0] == 2                                             # 1 full + 1 partial block
        prod.PreRequest(0, [0, 2])                                   # pod1 primary, pod3 prefill
        m, t = prod.Produce([b"aaaabbbb"], pods)
        assert list(m[0]) == [1, 0, 1] and t[0] == 2
        # keep_hashes + epp_index_add_picked == PreRequest for the picked endpoint
        d, offs = _pack([b"ccccdddd"])
        dec, _ = eng.schedule(d, offsets=offs, keep_hashes=True)
        eng.index_add_picked()
        m, t = eng.prefix_match(d, offsets=offs)
        assert m[0, int(dec["pick"][0])] == 2


def test_errors(epp):
    with pytest.raises(epp.EngineError):
        epp.Engine(0)
    with pytest.raises(epp.EngineError):
        epp.Engine(8, epp.ProfileSpec(0, [epp.ScorerSpec(99, 1.0)]))
    with epp.Engine(8) as eng:
        toks = np.zeros(64, np.uint32)
        with pytest.raises(epp.EngineError):                        # no model registered
            eng.hash_prompts(toks, uniform_len=256)
        eng.register_model(b"m")
        with pytest.raises(epp.EngineError):                        # schedule before pool_set
            eng.schedule(toks, uniform_len=256)
        with pytest.raises(epp.EngineError):
            eng.pool_set([9], [0], [0.0], [0])                      # slot id out of range
        with pytest.raises(epp.EngineError):
            eng.pool_set([1], [0], [float("nan")], [0])
        eng.pool_set([], [], [], [])                                # empty pool -> every decision is an error
        dec, _ = eng.schedule(toks, uniform_len=256)
        assert dec["status"][0] == -1 and dec["pick"][0] == 0xFFFFFFFF
