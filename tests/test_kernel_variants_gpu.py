"""One oracle parity case per templated kernel instantiation of libepp_engine.so.

The engine picks a template instantiation from properties of the input (layout alignment, block size, prompt length
against the small-batch staging buffer, profile count, tie rule) or from an A/B switch (EPP_HASH_STAGED,
EPP_MATCH_CTAS).  Every case below runs under a kernel recorder (torch.profiler, CUDA activity) and asserts that its
target instantiation actually ran -- and, where it matters, that the fallback did not -- then compares hashes and
decisions bit for bit with the CPU oracle.  Expected values never come from the engine's own hash kernel.

VARIANTS maps every templated __global__ of the library to the test that covers it; the CPU test
test_variant_table_matches_library keeps that table equal to what `cuobjdump -symbols` lists, so a new instantiation
fails the suite until it has a parity case.  GPU cases are marked one by one (the guard runs without a device).

EPP_KERNEL_RECORDER=off turns the recorder's assertions off and nothing else (every check it skips raises a warning):
compute-sanitizer holds the CUPTI subscription torch.profiler needs (profiles/r3_sanitizer_memcheck_variants.log), so a
memcheck run of this file sets it and still runs every parity check."""
import ast
import contextlib
import json
import os
import re
import shutil
import subprocess
import sys
import tempfile
import warnings

import numpy as np
import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
HERE = os.path.dirname(os.path.abspath(__file__))

VARIANTS = {
    "k_hash_fused<true>": "test_hash_fused_32_byte_layouts_vs_oracle",
    "k_hash_fused<false>": "test_hash_fused_16_byte_layouts_vs_oracle",
    "k_hash_staged<16,4,4>": "test_hash_staged_shapes_vs_oracle",
    "k_hash_staged<16,3,4>": "test_hash_staged_shapes_vs_oracle",
    "k_hash_staged<32,4,4>": "test_hash_staged_shapes_vs_oracle",
    "k_cycle_small<true,true>": "test_small_batch_variants_vs_oracle",
    "k_cycle_small<false,true>": "test_small_batch_variants_vs_oracle",
    "k_cycle_small<true,false>": "test_small_batch_variants_vs_oracle",
    "k_cycle_small<false,false>": "test_small_batch_variants_vs_oracle",
    "k_match_pick_sparse<8,false,false,1>": "test_match_pick_sparse_stages_and_tie_rules_vs_oracle",
    "k_match_pick_sparse<6,false,false,2>": "test_match_pick_sparse_stages_and_tie_rules_vs_oracle",
    "k_match_pick_sparse<6,false,true,2>": "test_match_pick_sparse_stages_and_tie_rules_vs_oracle",
    "k_match_pick_sparse<6,false,false,3>": "test_match_pick_sparse_stages_and_tie_rules_vs_oracle",
    "k_match_pick_sparse<6,false,true,3>": "test_match_pick_sparse_stages_and_tie_rules_vs_oracle",
    "k_match_pick_sparse<6,false,true,1>": "test_single_profile_random_ties_vs_oracle",
    "k_match_pick_sparse<6,false,false,1>": "test_match_ctas_6_vs_oracle",
    "k_match_pick_sparse<6,true,false,1>": "tests/test_sharded.py::test_sharded_two_shards_one_gpu",
}

TIE_SEED = 0x7153ED          # bench.py's index-write leg ("random_ties")


# ------------------------------------------------------------------------------------------------
# kernel names and the recorder
# ------------------------------------------------------------------------------------------------
def kernel_key(name: str) -> str:
    """'void epp::(anonymous namespace)::k_cycle_small<false, true>(epp::HashParams, ...)' -> 'k_cycle_small<false,true>'
    (non-templated kernels: the bare name)."""
    name = name.replace("(anonymous namespace)::", "")
    if "(" not in name:
        name += "("
    m = re.search(r"([A-Za-z_]\w*)\s*(<[^()]*>)?\s*\(", name)
    if not m:
        return name
    return m.group(1) + (re.sub(r"\s+", "", m.group(2)) if m.group(2) else "")


class KernelLog:
    def __init__(self, off=False):
        self.off = off               # EPP_KERNEL_RECORDER=off: nothing recorded, nothing asserted
        self.names = set()
        self.grids = {}              # kernel key -> list of grid dimensions, in launch order
        self.copies = []             # (memcpy name, bytes), e.g. ("Memcpy HtoD (Pinned -> Device)", 4096)

    def add(self, name, grid):
        k = kernel_key(name)
        self.names.add(k)
        self.grids.setdefault(k, []).append(grid)

    @staticmethod
    def union(logs):
        u = KernelLog(off=any(g.off for g in logs))
        for g in logs:
            u.names |= g.names
            u.copies += g.copies
            for k, v in g.grids.items():
                u.grids.setdefault(k, []).extend(v)
        return u

    def __repr__(self):
        return "kernels seen: " + ", ".join(sorted(self.names))


@contextlib.contextmanager
def record_kernels():
    """Runs the body under torch.profiler (CUDA activity) and fills the yielded KernelLog with every kernel launched,
    whatever library launched it.  A trace without a single kernel is an error, never a pass."""
    import torch
    from torch.profiler import ProfilerActivity, profile
    if os.environ.get("EPP_KERNEL_RECORDER") == "off":
        yield KernelLog(off=True)
        return
    log = KernelLog()
    torch.cuda.synchronize()
    with profile(activities=[ProfilerActivity.CPU, ProfilerActivity.CUDA]) as prof:
        yield log
        torch.cuda.synchronize()
    with tempfile.TemporaryDirectory() as d:
        path = os.path.join(d, "trace.json")
        prof.export_chrome_trace(path)
        with open(path) as f:
            events = json.load(f).get("traceEvents", [])
    kernels = [e for e in events if e.get("cat") == "kernel"]
    if not kernels:
        raise AssertionError("torch.profiler recorded no CUDA kernel at all: the kernel recorder is blind, so this case "
                             "cannot tell which instantiation ran")
    for e in kernels:
        log.add(e.get("name", ""), (e.get("args") or {}).get("grid"))
    log.copies = [(e.get("name", ""), (e.get("args") or {}).get("bytes")) for e in events if e.get("cat") == "gpu_memcpy"]


def _expect(log, ran=(), not_ran=()):
    if log.off:
        warnings.warn(f"EPP_KERNEL_RECORDER=off: NOT checked that {list(ran)} ran and {list(not_ran)} did not")
        return
    print(f"expected {list(ran)}, {log!r}")
    for k in ran:
        assert k in log.names, f"{k} did not run; {log!r}"
    for k in not_ran:
        assert k not in log.names, f"{k} ran; {log!r}"


# ------------------------------------------------------------------------------------------------
# fixtures and input builders
# ------------------------------------------------------------------------------------------------
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


@pytest.fixture(scope="module")
def engine_library():
    """Build only: the cross-compiled library, no device needed."""
    import epp_b200
    return epp_b200.build.build()


MODELS = [b"mdl", b"other-model", b"third"]


def _pack(prompts):
    """Tightly packed bytes + offsets: the oracle's view of a batch."""
    offs = np.zeros(len(prompts) + 1, dtype=np.uint64)
    np.cumsum([len(p) for p in prompts], out=offs[1:])
    blob = b"".join(prompts)
    data = np.frombuffer(blob, dtype=np.uint8).copy() if blob else np.zeros(16, np.uint8)
    return data, offs


def _starts(lengths, align):
    """Row starts: align 32 = every start on a 32-byte boundary; align 16 = every start at 16 mod 32 (16-byte but not
    32-byte aligned, so the batch layout is exactly 16-byte aligned)."""
    starts, pos = [], 0
    for n in lengths:
        pos = (pos + 31) & ~31
        if align == 16:
            pos += 16
        starts.append(pos)
        pos += n
    return starts, pos


def _layout(prompts, align, out=None):
    """Ragged rows at the starts of _starts(); offsets[r + 1] - offsets[r] is longer than a prompt, so the lengths go
    with it.  out: a pinned array to write into."""
    starts, end = _starts([len(p) for p in prompts], align)
    blob = np.zeros(end + 64, np.uint8) if out is None else out
    for st, p in zip(starts, prompts):
        blob[st: st + len(p)] = np.frombuffer(p, np.uint8)
    offs = np.array(starts + [end], dtype=np.uint64)
    lens = np.array([len(p) for p in prompts], dtype=np.uint64)
    return blob, offs, lens


def _ragged_prompts(rng, bb, maxb, R):
    """Empty, shorter than a block, whole 8-block windows, one block either side of a window edge, partial tails, the
    cap exactly and past it; the rest random."""
    fixed = [0, 1, bb - 1, bb, bb + 5, 8 * bb, 16 * bb, 7 * bb, 9 * bb, 15 * bb, 17 * bb, 8 * bb + 5, 8 * bb - 3,
             maxb * bb, maxb * bb - 1, maxb * bb + 7, (maxb + 3) * bb, (maxb - 1) * bb + bb // 2]
    lens = [n for n in fixed if n >= 0][:R]
    while len(lens) < R:
        lens.append(int(rng.integers(0, bb * (maxb + 4))))
    return [bytes(rng.integers(0, 256, n, dtype=np.uint8)) for n in lens]


def _assert_hashes(orc, hs, nb, prompts, models, bst, maxb, where):
    hs = np.asarray(hs).view(np.uint64)
    nb = np.asarray(nb)
    for i, p in enumerate(prompts):
        want = orc.hash_prompt(p, models[i], bst, maxb)
        assert nb[i] == len(want), (where, i, len(p))
        assert [int(x) for x in hs[i, : nb[i]]] == want, (where, i, len(p))


def _hash_layout_cases(epp, orc, eng, bst, maxb, align, seed, kernel, R=77):
    """Hashes of one engine across the layouts of one alignment class, each against the oracle: host ragged rows with
    lengths and mixed models; the same as device pointers (offsets alignment probed on the device); host and device
    uniform rows whose length is past the cap, and shorter ones with a partial tail."""
    import torch
    bb = 4 * bst
    rng = np.random.default_rng(seed)
    mids = [eng.register_model(m) for m in MODELS]
    assert mids == [0, 1, 2]
    prompts = _ragged_prompts(rng, bb, maxb, R)
    model_of = rng.integers(0, len(MODELS), R).astype(np.uint32)
    models = [MODELS[m] for m in model_of]
    blob, offs, lens = _layout(prompts, align)
    hs, nb = eng.hash_prompts(blob, offsets=offs, lengths=lens, model_ids=model_of)
    _assert_hashes(orc, hs, nb, prompts, models, bst, maxb, f"{kernel}: host ragged, align {align}")
    dh, dn = eng.hash_prompts(torch.from_numpy(blob).cuda(), offsets=torch.from_numpy(offs.view(np.int64)).cuda(),
                              lengths=torch.from_numpy(lens.view(np.int64)).cuda(),
                              model_ids=torch.from_numpy(model_of.view(np.int32)).cuda())
    torch.cuda.synchronize()
    _assert_hashes(orc, dh.cpu().numpy(), dn.cpu().numpy(), prompts, models, bst, maxb, f"{kernel}: device ragged, align {align}")
    extra = 16 if align == 16 else 32
    for L in (maxb * bb + extra, 3 * bb + extra):            # past the cap / a partial trailing block
        assert L % 32 == (16 if align == 16 else 0)
        Ru = 45
        rows = rng.integers(0, 256, (Ru, L), dtype=np.uint8)
        mu = rng.integers(0, len(MODELS), Ru).astype(np.uint32)
        want_p = [rows[r].tobytes() for r in range(Ru)]
        want_m = [MODELS[m] for m in mu]
        hs, nb = eng.hash_prompts(rows, uniform_len=L, model_ids=mu)
        _assert_hashes(orc, hs, nb, want_p, want_m, bst, maxb, f"{kernel}: host uniform {L}")
        dh, dn = eng.hash_prompts(torch.from_numpy(rows).cuda(), uniform_len=L,
                                  model_ids=torch.from_numpy(mu.view(np.int32)).cuda())
        torch.cuda.synchronize()
        _assert_hashes(orc, dh.cpu().numpy(), dn.cpu().numpy(), want_p, want_m, bst, maxb, f"{kernel}: device uniform {L}")


def _holders_index(orc, rng, fam, model, bst, B, E, counts):
    """Index pairs: family g cached by counts[g] endpoints at few distinct depths (equal scores among holders); counts
    above 32 overflow the sparse kernel's per-request map (dense-counter pass)."""
    ph, pe = [], []
    for g, p in enumerate(fam):
        h = orc.hash_prompt(p, model, bst, B)
        for e in rng.choice(E, size=counts[g], replace=False):
            depth = int(rng.choice([max(1, len(h) // 2), len(h)]))
            ph += h[:depth]
            pe += [int(e)] * depth
    return np.array(ph, np.uint64), np.array(pe, np.uint32)


def _spec(epp, f, scorers):
    return epp.ProfileSpec(f, [epp.ScorerSpec(k, w, p) for k, w, p in scorers])


PRIM = [(2, 1.0, 0), (1, 1.0, 0), (0, 2.0, 0)]
PREF = [(2, 1.0, 0), (0, 1.0, 0)]
ENC = [(1, 1.0, 0)]


# ------------------------------------------------------------------------------------------------
# hashing: k_hash_fused<true / false>, k_hash_staged<...>
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("maxb", [9, 12])
@pytest.mark.parametrize("bst", [8, 16, 24, 32])
def test_hash_fused_16_byte_layouts_vs_oracle(epp, orc, bst, maxb):
    """k_hash_fused<false> (128-bit loads): 1-4 XXH64 stripes per block, odd and even caps (odd: the chain warp's
    scalar-store branch), ragged rows at 16 mod 32 with lengths, device offsets at 16 mod 32 (k_offsets_aligned),
    uniform rows of length 16 mod 32, mixed models."""
    with epp.Engine(8, block_size_tokens=bst, max_prefix_blocks=maxb) as eng:
        with record_kernels() as k:
            _hash_layout_cases(epp, orc, eng, bst, maxb, 16, seed=bst * 100 + maxb, kernel="k_hash_fused<false>")
    _expect(k, ran=["k_hash_fused<false>", "k_offsets_aligned"], not_ran=["k_hash_fused<true>", "k_hash_generic"])


@pytest.mark.gpu
@pytest.mark.parametrize("bst,maxb", [(16, 255), (8, 9), (32, 12), (24, 9)])
def test_hash_fused_32_byte_layouts_vs_oracle(epp, orc, bst, maxb):
    """k_hash_fused<true> (256-bit loads) on the same generators: 32-byte row starts and uniform rows, odd caps."""
    with epp.Engine(8, block_size_tokens=bst, max_prefix_blocks=maxb) as eng:
        with record_kernels() as k:
            _hash_layout_cases(epp, orc, eng, bst, maxb, 32, seed=bst * 100 + maxb + 1, kernel="k_hash_fused<true>")
    _expect(k, ran=["k_hash_fused<true>"], not_ran=["k_hash_fused<false>", "k_hash_generic"])


@pytest.mark.gpu
def test_hash_fused_16_byte_grid_stride_vs_oracle(epp, orc):
    """k_hash_fused<false> with more 32-request tiles than resident CTAs (grid capped at SMs x occupancy, so CTAs loop
    over tiles): 40 000 short ragged prompts at 16 mod 32, odd cap -- hashes against the oracle, then the decisions of
    the same batch against cycle_batch."""
    import helpers
    bst, B, E = 8, 9, 64
    bb = 4 * bst
    R = 40_000
    rng = np.random.default_rng(404)
    fam = [bytes(rng.integers(0, 256, bb * B, dtype=np.uint8)) for _ in range(4)]
    prompts = []
    for _ in range(R):
        g = int(rng.integers(0, len(fam) + 1))
        if g < len(fam):
            keep = int(rng.integers(0, B + 1)) * bb
            prompts.append(fam[g][:keep] + bytes(rng.integers(0, 256, int(rng.integers(0, 2 * bb)), dtype=np.uint8)))
        else:
            prompts.append(bytes(rng.integers(0, 256, int(rng.integers(0, bb * (B + 2))), dtype=np.uint8)))
    blob, offs, lens = _layout(prompts, 16)
    kv = rng.integers(0, 3, E) / 3.0
    waiting = rng.integers(0, 3, E).astype(np.int32)
    ph, pe = _holders_index(orc, rng, fam, b"mdl", bst, B, E, [3, 9, 20, 40])
    with epp.Engine(E, _spec(epp, 0, PRIM), block_size_tokens=bst, max_prefix_blocks=B) as eng:
        eng.register_model(b"mdl")
        eng.pool_set(np.arange(E), np.zeros(E, np.uint8), kv, waiting)
        eng.index_load_snapshot(ph, pe)
        with record_kernels() as k:
            hs, nb = eng.hash_prompts(blob, offsets=offs, lengths=lens)
            dec, det = eng.schedule(blob, offsets=offs, lengths=lens)
    _expect(k, ran=["k_hash_fused<false>"], not_ran=["k_hash_generic", "k_hash_fused<true>"])
    if not k.off:
        n_tiles = (R + 31) // 32
        grids = [g for g in k.grids["k_hash_fused<false>"] if g]
        assert grids, "the trace carries no grid size for k_hash_fused<false>"
        assert all(g[0] < n_tiles for g in grids), (grids, n_tiles)         # every CTA walks more than one tile
    ix = orc.Indexer()
    ix.load_pairs(ph, pe)
    d, o = _pack(prompts)
    _assert_hashes(orc, hs, nb, prompts, [b"mdl"] * R, bst, B, "k_hash_fused<false>: grid-stride")
    pool = orc.PoolState(np.zeros(E, np.uint8), kv, waiting)
    odec, ototal = orc.cycle_batch(b"mdl", bst, B, 0, False, ix, orc.make_profile(0, PRIM), None, pool, d, o, 8)
    helpers.assert_decisions_equal(dec, det, odec, ototal, where="k_hash_fused<false>: grid-stride batch")
    assert (dec["match_blocks"] > 0).sum() > R // 10


@pytest.mark.gpu
@pytest.mark.parametrize("maxb", [9, 12, 255])
@pytest.mark.parametrize("shape,kernel", [("1", "k_hash_staged<16,4,4>"), ("1634", "k_hash_staged<16,3,4>"),
                                          ("3244", "k_hash_staged<32,4,4>")])
def test_hash_staged_shapes_vs_oracle(epp, orc, monkeypatch, shape, kernel, maxb):
    """EPP_HASH_STAGED (64-byte blocks only): every task shape, 16- and 32-byte layouts, odd and even caps, batch sizes
    that are not a multiple of the task size, mixed models."""
    monkeypatch.setenv("EPP_HASH_STAGED", shape)           # read at engine creation
    with epp.Engine(8, block_size_tokens=16, max_prefix_blocks=maxb) as eng:
        with record_kernels() as k:
            _hash_layout_cases(epp, orc, eng, 16, maxb, 16, seed=maxb * 7 + len(shape), kernel=kernel, R=77)
        _expect(k, ran=[kernel], not_ran=["k_hash_fused<false>", "k_hash_fused<true>", "k_hash_generic"])
    with epp.Engine(8, block_size_tokens=16, max_prefix_blocks=maxb) as eng:
        with record_kernels() as k:
            _hash_layout_cases(epp, orc, eng, 16, maxb, 32, seed=maxb * 7 + len(shape) + 1, kernel=kernel, R=53)
        _expect(k, ran=[kernel], not_ran=["k_hash_fused<false>", "k_hash_fused<true>", "k_hash_generic"])


# ------------------------------------------------------------------------------------------------
# small host batches: k_cycle_small<kAlign32, kStage>
# ------------------------------------------------------------------------------------------------
def _expect_prompt_copy(log, offs, zero_copy):
    """Zero-copy batches leave the prompts in pinned host memory (no host-to-device copy but the 4-byte epoch word);
    the others bring them into HBM with one copy of the whole row span."""
    if log.off:
        warnings.warn("EPP_KERNEL_RECORDER=off: NOT checked whether the prompts were read in place or copied")
        return
    htod = [b for name, b in log.copies if "HtoD" in name]
    span = int(offs[-1] - offs[0])
    if zero_copy:
        assert not [b for b in htod if b is None or b > 4], f"zero-copy batch copied its prompts: {log.copies}"
    else:
        assert span in htod, f"no {span}-byte prompt copy: {log.copies}"


@pytest.mark.gpu
@pytest.mark.parametrize("shape", ["staged", "unstaged"])
@pytest.mark.parametrize("row_align", [16, 32])
def test_small_batch_variants_vs_oracle(epp, orc, monkeypatch, row_align, shape):
    """The single-launch small-batch kernel in all four builds: pinned rows on 16- or 32-byte boundaries; prompts
    staged into shared memory (32-byte blocks, odd cap 25) or, past the 160 KiB staging buffer, read by the digest
    threads themselves (64-byte blocks, odd cap 2 601: prompts from empty to past the cap, more than 32 full blocks, the
    trailing partial block parked behind the stripe states).  Zero-copy (1, 3 requests) and DMA-copied (40, 300)
    batches; P/D + encode stages; both tie rules.  Every decision equals the oracle's and the ordinary path's
    (EPP_SMALL_BATCH=0)."""
    import helpers
    a32 = "true" if row_align == 32 else "false"
    stage = "true" if shape == "staged" else "false"
    target = f"k_cycle_small<{a32},{stage}>"
    E = 96
    bst, B = (8, 25) if shape == "staged" else (16, 2601)
    bb = 4 * bst
    rng = np.random.default_rng(71 + row_align + len(shape))
    kv = rng.integers(0, 3, E) / 3.0
    waiting = rng.integers(0, 3, E).astype(np.int32)
    role = rng.choice([1, 2, 3, 5, 7, 0], size=E).astype(np.uint8)
    # three families as long as the cap, two that end in a partial block of 17 and 29 bytes in both shapes (not a
    # multiple of 16: the tail copy's byte loop runs); requests that repeat one of those whole match their cached
    # trailing block only if its hash is right
    fam = [bytes(rng.integers(0, 256, n, dtype=np.uint8)) for n in (bb * B, bb * B, bb * B, bb * (B // 3) + 17, bb * (B - 2) + 29)]
    ph, pe = _holders_index(orc, rng, fam, b"m", bst, B, E, [2, 6, 12, 30, 70])
    ix = orc.Indexer()
    ix.load_pairs(ph, pe)
    pool = orc.PoolState(role, kv, waiting)

    def make_batch(n):
        prompts = []
        for i in range(n):
            g = int(rng.integers(0, len(fam) + 2))
            kind = int(rng.integers(0, 8))
            if kind == 0 or (n == 3 and i == 0):
                prompts.append(b"" if i % 2 == 0 else bytes(rng.integers(0, 256, bb - 1, dtype=np.uint8)))
            elif kind == 1 or n == 1:
                prompts.append(fam[3 + i % 2])                # a cached prompt with a partial trailing block, whole
            elif g >= len(fam):
                prompts.append(bytes(rng.integers(0, 256, int(rng.integers(bb, bb * B + 3 * bb)), dtype=np.uint8)))
            else:
                keep = int(rng.integers(1, B + 1)) * bb
                tail = int(rng.integers(0, 2 * bb))          # partial trailing block / past the cap
                prompts.append(fam[g][:keep] + bytes(rng.integers(0, 256, tail, dtype=np.uint8)))
        if n == 3:                                           # a whole-prompt request past the cap, with a tail
            prompts[1] = fam[2] + bytes(rng.integers(0, 256, bb + 9, dtype=np.uint8))
            prompts[2] = fam[4]
        starts, end = _starts([len(p) for p in prompts], row_align)
        buf = epp.PinnedBuffer(end + 64)
        _, offs, lens = _layout(prompts, row_align, out=buf.array)
        d, o = _pack(prompts)
        mm = (rng.random(n) < 0.5).astype(np.uint8)
        return buf, offs, lens, d, o, mm

    sizes = (1, 3, 40, 300)
    batches = [make_batch(n) for n in sizes]
    if shape == "unstaged":
        assert max(int(b[2].max()) for b in batches) > bb * B and any(int(b[2].max()) > 32 * bb for b in batches)
    try:
        for tie_seed in (0, TIE_SEED):
            got = {}
            for small in ("1024", "0"):
                monkeypatch.setenv("EPP_SMALL_BATCH", small)
                with epp.Engine(E, _spec(epp, 1, PRIM), _spec(epp, 2, PREF), block_size_tokens=bst, max_prefix_blocks=B,
                                non_cached_tokens=8, encode=_spec(epp, 3, ENC), tie_seed=tie_seed) as eng:
                    eng.register_model(b"m")
                    eng.pool_set(np.arange(E), role, kv, waiting)
                    eng.index_load_snapshot(ph, pe)
                    out, logs = [], []
                    for n, (buf, offs, lens, d, o, mm) in zip(sizes, batches):
                        base = eng.stats()["n_decisions"]
                        with record_kernels() as kb:
                            dec, det = eng.schedule(buf.array, offsets=offs, lengths=lens, multimodal=mm, n_requests=n)
                        if small != "0":
                            assert eng.stats()["last_kernel_launches"] in (1, 2)     # 2: + the dense-counter pass
                            _expect_prompt_copy(kb, offs, zero_copy=n <= 8)          # EPP_SMALL_ZEROCOPY default: 8
                        logs.append(kb)
                        out.append((dec.copy(), det.copy(), base))
                    k = KernelLog.union(logs)
                    if small != "0":
                        _expect(k, ran=[target], not_ran=["k_hash_generic"])
                    else:
                        _expect(k, ran=[f"k_hash_fused<{a32}>"], not_ran=[target])
                    got[small] = out
            for n, (buf, offs, lens, d, o, mm), (dec, det, base) in zip(sizes, batches, got["1024"]):
                odec, ototal = orc.cycle_batch(b"m", bst, B, 8, False, ix, orc.make_profile(1, PRIM), orc.make_profile(2, PREF),
                                               pool, d, o, 8, tie_seed=tie_seed, tie_base=base,
                                               encode=orc.make_profile(3, ENC), multimodal=mm)
                helpers.assert_decisions_equal(dec, det, odec, ototal, where=f"{target} tie_seed={tie_seed} n={n}")
            for (a, ad, _), (b, bd, _) in zip(got["1024"], got["0"]):
                np.testing.assert_array_equal(a, b)
                np.testing.assert_array_equal(ad, bd)
        assert (got["1024"][-1][0]["match_blocks"] > 0).any()
        whole = [np.isin(lens, [len(fam[3]), len(fam[4])]) & (dec["match_blocks"] == dec["total_blocks"])   # cached prompts
                 for (dec, _, _), (_, _, lens, _, _, _) in zip(got["1024"], batches)]                        # matched to the end
        assert sum(int(x.sum()) for x in whole) > 3
    finally:
        for b in batches:
            b[0].close()


# ------------------------------------------------------------------------------------------------
# match / score / pick: k_match_pick_sparse<MINCTA, kSharded, kTie, kStages>
# ------------------------------------------------------------------------------------------------
@pytest.mark.gpu
@pytest.mark.parametrize("tie_seed", [0, 0x5EED])
@pytest.mark.parametrize("stages", [1, 2, 3])
def test_match_pick_sparse_stages_and_tie_rules_vs_oracle(epp, orc, stages, tie_seed):
    """The throughput match kernel for 1 / 2 / 3 handler stages (primary; + prefill; + encode) x both tie rules, on a
    device batch with a tied pool and families held by more than 32 endpoints (the dense overflow pass behind it)."""
    import torch
    import helpers
    E, bst, B, R = 96, 8, 16, 700
    bb = 4 * bst
    rng = np.random.default_rng(stages * 10 + (tie_seed & 7))
    kv = rng.integers(0, 2, E) / 2.0
    waiting = rng.integers(0, 2, E).astype(np.int32)
    role = rng.choice([1, 2, 3, 5, 7, 0], size=E).astype(np.uint8) if stages > 1 else np.zeros(E, np.uint8)
    fam = [bytes(rng.integers(0, 256, bb * B, dtype=np.uint8)) for _ in range(5)]
    ph, pe = _holders_index(orc, rng, fam, b"m", bst, B, E, [2, 6, 12, 40, 70])
    ix = orc.Indexer()
    ix.load_pairs(ph, pe)
    prompts = []
    for _ in range(R):
        g = int(rng.integers(0, len(fam) + 2))
        if g >= len(fam):
            prompts.append(bytes(rng.integers(0, 256, int(rng.integers(0, bb * (B + 2))), dtype=np.uint8)))
        else:
            keep = int(rng.integers(1, B + 1)) * bb
            prompts.append(fam[g][:keep] + bytes(rng.integers(0, 256, int(rng.integers(0, bb)), dtype=np.uint8)))
    blob, offs, lens = _layout(prompts, 32)
    mm = (rng.random(R) < 0.5).astype(np.uint8)
    prim_f = 1 if stages > 1 else 0
    kw = dict(block_size_tokens=bst, max_prefix_blocks=B, tie_seed=tie_seed)
    if stages >= 2:
        kw["non_cached_tokens"] = 8
    if stages == 3:
        kw["encode"] = _spec(epp, 3, ENC)
    with epp.Engine(E, _spec(epp, prim_f, PRIM), _spec(epp, 2, PREF) if stages >= 2 else None, **kw) as eng:
        eng.register_model(b"m")
        eng.pool_set(np.arange(E), role, kv, waiting)
        eng.index_load_snapshot(ph, pe)
        base = eng.stats()["n_decisions"]
        with record_kernels() as k:
            ddec, ddet = eng.schedule(torch.from_numpy(blob).cuda(), offsets=torch.from_numpy(offs.view(np.int64)).cuda(),
                                      lengths=torch.from_numpy(lens.view(np.int64)).cuda(),
                                      multimodal=torch.from_numpy(mm).cuda() if stages == 3 else None)
            torch.cuda.synchronize()
    tie = "true" if tie_seed else "false"
    mincta = 8 if (stages == 1 and not tie_seed) else 6
    _expect(k, ran=[f"k_match_pick_sparse<{mincta},false,{tie},{stages}>"])
    dec = epp.decisions_from_torch(ddec)
    det = ddet.cpu().numpy().view(epp.DETAIL_DTYPE).reshape(-1)
    d, o = _pack(prompts)
    pool = orc.PoolState(role, kv, waiting)
    odec, ototal = orc.cycle_batch(b"m", bst, B, kw.get("non_cached_tokens", 0), False, ix, orc.make_profile(prim_f, PRIM),
                                   orc.make_profile(2, PREF) if stages >= 2 else None, pool, d, o, 8, tie_seed=tie_seed,
                                   tie_base=base, encode=orc.make_profile(3, ENC) if stages == 3 else None,
                                   multimodal=mm if stages == 3 else None)
    helpers.assert_decisions_equal(dec, det, odec, ototal, where=f"k_match_pick_sparse<{mincta},false,{tie},{stages}>: tie_seed={tie_seed}")
    assert (dec["tie_count"] > 1).sum() > R // 10
    if stages >= 2:
        assert (det["prefill_ran"] == 1).any()


def _config3_scaled(tg, R=1536):
    return tg.baseline_configs()["config3"].scaled(E=512, R=R, T=1024, name="config3")


def _tied_config3(orc, tg, w, trace, rng):
    """Scaled config 3 with a pool of few load levels (large arg-max sets) and the trace's index plus three families
    held by 40 / 70 / 100 more endpoints (past the sparse map: the dense pass runs under the same tie rule)."""
    import helpers
    role, _, _, running = trace.pool()
    kv = rng.integers(0, 2, w.E) / 2.0
    waiting = rng.integers(0, 2, w.E).astype(np.int32)
    _, _, primary, _, (hs, es) = helpers.setup_oracle(orc, w, trace)
    fam = trace.family_tokens()
    eh, ee = _holders_index(orc, rng, [fam[g].tobytes() for g in range(3)], tg.MODEL, w.block_size_tokens,
                            w.max_prefix_blocks, w.E, [40, 70, 100])
    hs, es = np.concatenate([hs, eh]), np.concatenate([es, ee])
    ix = orc.Indexer()
    ix.load_pairs(hs, es)
    return (role, kv, waiting, running), orc.PoolState(role, kv, waiting, running), ix, primary, (hs, es)


@pytest.mark.gpu
def test_single_profile_random_ties_vs_oracle(epp, orc, tg):
    """One profile with tie_seed != 0 (what a deployment runs: bench.py's seed): a host batch then a device batch of
    scaled config 3 on a tied pool -- the tie ordinal keeps counting across calls -- bit-exact against the oracle; the
    ties are real and the picks spread over the arg-max sets instead of landing on the lowest slot."""
    import torch
    import helpers
    w = _config3_scaled(tg)
    trace = tg.Trace(w)
    rng = np.random.default_rng(3)
    (role, kv, waiting, running), pool, ix, primary, (hs, es) = _tied_config3(orc, tg, w, trace, rng)
    with helpers.make_engine(w, tie_seed=TIE_SEED) as eng:
        eng.register_model(tg.MODEL)
        eng.pool_set(np.arange(w.E, dtype=np.uint32), role, kv, waiting, running)
        eng.index_load_snapshot(hs, es)
        for b in range(2):
            tokens, _, _ = trace.requests(b * w.R, w.R)
            base = eng.stats()["n_decisions"]
            assert base == b * w.R
            with record_kernels() as k:
                if b == 0:
                    dec, det = eng.schedule(tokens, uniform_len=w.prompt_bytes)          # > 1024: the ordinary host path
                else:
                    ddec, ddet = eng.schedule(torch.from_numpy(tokens.view(np.int32)).cuda(), uniform_len=w.prompt_bytes)
                    torch.cuda.synchronize()
                    dec = epp.decisions_from_torch(ddec)
                    det = ddet.cpu().numpy().view(epp.DETAIL_DTYPE).reshape(-1)
            _expect(k, ran=["k_match_pick_sparse<6,false,true,1>"],
                    not_ran=["k_match_pick_sparse<8,false,false,1>", "k_match_pick_sparse<6,false,false,1>"])
            odec, ototal = helpers.oracle_decisions(orc, w, pool, ix, primary, None, tokens, n_threads=8,
                                                    tie_seed=TIE_SEED, tie_base=base)
            helpers.assert_decisions_equal(dec, det, odec, ototal, where=f"k_match_pick_sparse<6,false,true,1>: single-profile random ties, batch {b}")
            low, _ = helpers.oracle_decisions(orc, w, pool, ix, primary, None, tokens, n_threads=8)
            tied = dec["tie_count"] > 1
            assert tied.sum() > w.R // 4, tied.sum()
            assert (dec["pick"][tied] != low["pick"][tied]).mean() > 0.5, \
                "k_match_pick_sparse<6,false,true,1>: tied picks land on the lowest slot"          # not the rule of tie_seed 0
            assert len(set(dec["pick"][dec["tie_count"] > 4].tolist())) > 20    # not one hot endpoint
            assert (dec["match_blocks"] > 0).sum() > w.R // 10


@pytest.mark.gpu
def test_single_profile_random_ties_full_size_config3_vs_oracle(epp, orc, tg):
    """BASELINE config 3 at full size (4 096 endpoints, 65 536 requests of 4 096 tokens) with bench.py's tie seed: every
    decision of the device batch against the multi-threaded oracle."""
    import torch
    import helpers
    w = tg.baseline_configs()["config3"].scaled(R=65536, name="config3")
    trace = tg.Trace(w)
    tokens, _, _ = trace.requests()
    pool, ix, primary, _, (hs, es) = helpers.setup_oracle(orc, w, trace)
    odec, ototal = helpers.oracle_decisions(orc, w, pool, ix, primary, None, tokens, n_threads=min(64, os.cpu_count() or 1),
                                            tie_seed=TIE_SEED, tie_base=0)
    role, kv, waiting, running = trace.pool()
    with helpers.make_engine(w, tie_seed=TIE_SEED) as eng:
        eng.register_model(tg.MODEL)
        eng.pool_set(np.arange(w.E, dtype=np.uint32), role, kv, waiting, running)
        eng.index_load_snapshot(hs, es)
        dt = torch.from_numpy(tokens.view(np.int32)).cuda()
        with record_kernels() as k:
            ddec, ddet = eng.schedule(dt, uniform_len=w.prompt_bytes)
            torch.cuda.synchronize()
    _expect(k, ran=["k_match_pick_sparse<6,false,true,1>"])
    dec = epp.decisions_from_torch(ddec)
    det = ddet.cpu().numpy().view(epp.DETAIL_DTYPE).reshape(-1)
    helpers.assert_decisions_equal(dec, det, odec, ototal, where="k_match_pick_sparse<6,false,true,1>: config3 full size, random ties")
    assert (dec["tie_count"] > 1).any()


_CTAS_CHILD = r"""
import json, sys
root, tests, out = sys.argv[1:4]
sys.path[:0] = [root, tests]
import numpy as np
import torch
import epp_b200 as epp
import helpers
import test_kernel_variants_gpu as T
from tools import tracegen as tg
w = T._config3_scaled(tg, R=2048)
trace = tg.Trace(w)
tokens, _, _ = trace.requests()
role, kv, waiting, running = trace.pool()
with helpers.make_engine(w) as eng:
    eng.register_model(tg.MODEL)
    eng.pool_set(np.arange(w.E, dtype=np.uint32), role, kv, waiting, running)
    eng.index_load_snapshot(np.load(out + "/index_h.npy"), np.load(out + "/index_e.npy"))
    with T.record_kernels() as k:
        ddec, ddet = eng.schedule(torch.from_numpy(tokens.view(np.int32)).cuda(), uniform_len=w.prompt_bytes)
        torch.cuda.synchronize()
    np.save(out + "/dec.npy", epp.decisions_from_torch(ddec))
    np.save(out + "/det.npy", ddet.cpu().numpy().view(epp.DETAIL_DTYPE).reshape(-1))
with open(out + "/kernels.json", "w") as f:
    json.dump(None if k.off else sorted(k.names), f)
"""


@pytest.mark.gpu
def test_match_ctas_6_vs_oracle(epp, orc, tg, tmp_path):
    """EPP_MATCH_CTAS=6 (the 40-register build of the one-profile kernel).  The switch is read once per process, so a
    child process schedules a scaled config-3 device batch with it; its decisions must equal the oracle's."""
    import helpers
    w = _config3_scaled(tg, R=2048)
    trace = tg.Trace(w)
    tokens, _, _ = trace.requests()
    pool, ix, primary, _, (hs, es) = helpers.setup_oracle(orc, w, trace)
    np.save(tmp_path / "index_h.npy", hs)
    np.save(tmp_path / "index_e.npy", es)
    env = dict(os.environ, EPP_MATCH_CTAS="6")
    r = subprocess.run([sys.executable, "-c", _CTAS_CHILD, ROOT, HERE, str(tmp_path)], env=env, cwd=ROOT,
                       capture_output=True, text=True, timeout=900)
    assert r.returncode == 0, r.stdout[-4000:] + r.stderr[-4000:]
    with open(tmp_path / "kernels.json") as f:
        seen = json.load(f)
    if seen is not None:
        log = KernelLog()
        log.names = set(seen)
        _expect(log, ran=["k_match_pick_sparse<6,false,false,1>"], not_ran=["k_match_pick_sparse<8,false,false,1>"])
    dec = np.load(tmp_path / "dec.npy")
    det = np.load(tmp_path / "det.npy")
    odec, ototal = helpers.oracle_decisions(orc, w, pool, ix, primary, None, tokens, n_threads=8)
    helpers.assert_decisions_equal(dec, det, odec, ototal, where="k_match_pick_sparse<6,false,false,1>: EPP_MATCH_CTAS=6")
    assert (dec["match_blocks"] > 0).sum() > w.R // 10


# ------------------------------------------------------------------------------------------------
# CPU guard: the table above lists exactly the library's templated kernels
# ------------------------------------------------------------------------------------------------
def _cuda_tool(*names):
    home = os.environ.get("CUDA_HOME") or os.environ.get("CUDA_PATH") or "/usr/local/cuda"
    for n in names:
        for c in (shutil.which(n), os.path.join(home, "bin", n)):
            if c and os.path.exists(c):
                return c
    pytest.fail(f"none of {names} found (CUDA toolkit / binutils)")


def library_template_kernels(so_path):
    """Templated __global__ instantiations of a library: cuobjdump -symbols (STO_ENTRY), demangled, as kernel_key()."""
    out = subprocess.run([_cuda_tool("cuobjdump"), "-symbols", so_path], capture_output=True, text=True, check=True).stdout
    mangled = [line.split()[-1] for line in out.splitlines() if "STO_ENTRY" in line]
    assert mangled, "cuobjdump lists no kernel entry in " + so_path
    dem = subprocess.run([_cuda_tool("c++filt", "cu++filt")], input="\n".join(mangled) + "\n", capture_output=True,
                         text=True, check=True).stdout.split("\n")
    keys = {kernel_key(d) for d in dem if d.strip()}
    return {k for k in keys if "<" in k}


def _test_exists(ref):
    if "::" in ref:
        path, name = ref.split("::", 1)
        with open(os.path.join(ROOT, path)) as f:
            tree = ast.parse(f.read())
        return any(isinstance(n, ast.FunctionDef) and n.name == name for n in tree.body)
    return ref.startswith("test_") and callable(globals().get(ref))


def test_variant_table_matches_library(engine_library):
    """Every templated kernel of libepp_engine.so has a parity case in VARIANTS, and every entry names a kernel the
    library still has and a test that exists."""
    have = library_template_kernels(engine_library)
    missing = sorted(have - set(VARIANTS))
    stale = sorted(set(VARIANTS) - have)
    assert not missing and not stale, f"kernels without a parity case: {missing}; table entries the library lacks: {stale}"
    bad = sorted(f"{k} -> {v}" for k, v in VARIANTS.items() if not _test_exists(v))
    assert not bad, f"VARIANTS names tests that do not exist: {bad}"


def test_kernel_key_forms():
    assert kernel_key("void epp::(anonymous namespace)::k_cycle_small<false, true>(epp::HashParams, epp::PickParams, "
                      "epp::SmallOut, unsigned int)") == "k_cycle_small<false,true>"
    assert kernel_key("void epp::k_match_pick_sparse<6, false, true, 1>(epp::PickParams)") == "k_match_pick_sparse<6,false,true,1>"
    assert kernel_key("epp::k_hash_generic(epp::HashParams)") == "k_hash_generic"
    assert kernel_key("k_offsets_aligned") == "k_offsets_aligned"
