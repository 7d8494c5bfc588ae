"""The quantizing encode split into launches (-m gpu), against the C oracle byte for byte.

An aligned 4-level quantizing pass of a job with at least split_min_tiles() tiles (hgi_tile_fast.cu) runs as
launch_fast_split: PART 1 (interior tiles, with the L2 prefetch), PART 2 or PART 4 (the right tile columns; PART 4 when
the width is a multiple of 128) and PART 3 (the bottom tile rows), the edge launches forked onto the scratch set's side
stream on a real stream.  HGI_B200_SPLIT_MIN=1 sends every such pass of these small planes through it.  Each knob
setting runs in a process of its own (tests/launch_shapes_worker.py: the knobs are read once per process); this
process holds the oracle and compares every output and every call's kernel count (tile_model.expected_launches).

Entry points of every case:
  (a) host API encode_batch (with and without histograms), decode_batch, encode with the reconstruction;
  (b) device API on a torch.cuda.Stream, three calls with the same buffers (plain, captured, replayed), with
      recon_out + hist_out and without;  (c) the same once on torch's default stream (no fork, no graph);
  (d) padded rows (hgi_*_dev_pitched): pitch align16(w) + 0 / 16, garbage in the input padding;
  (e) the caller's own torch.cuda.graph capture of encode_device + decode_device on a stream, after one warm-up call
      on that stream, replayed on three inputs.

Every instantiation of hgi_tile_fast_part_kernel (PART 1/2/3/4 x EXTRA x interpolator; the split is ALIGNED only)
runs under HGI_B200_SPLIT_MIN=1.  EXTRA = false: entry points (b-), (c-), (d-) and the grid-only host calls of a
case with L <= 7; EXTRA = true: (a) encode, (b+), (c+), (d+), (e), and the coarse pass of every L >= 8 case.
  PART 1 + 2 + 3:  160x146 (Crossed Medium L5 / LeftTop High L7 ...), 272x81 and 400x82 (two right columns);
  PART 1 + 4 + 3:  256x145 and 256x144 (both interpolators), 640x520 (the multi-chunk case);
  PART 3 alone:    128x64, 144x96, 160x80 (an interior column, no interior row), 96x160 (the reverse), and the coarse
                   pass of the L >= 8 cases on planes up to 2048 wide;
  coarse pass with PART 1 + 2 + 3 (EXTRA, vec_ok 2: the 145-wide decimated plane): 2320x1296 L8.
Padded rows whose width is not a multiple of 16 (vec_ok 2, the `ragged` loads of PARTs 2 and 3) are the (d) entry
points of 161x145, 273x96 and 250x146, both interpolators; PART 4 cannot meet them (its width is a multiple of 128).
Lossless and NoOp cases are the controls: they must not split.
"""
import json
import os
import subprocess
import sys

import numpy as np
import pytest

import rustyhgi_b200 as hgi
import tile_model as tm
from conftest import photo_like
from oracle import c as oc

pytestmark = pytest.mark.gpu
HERE = os.path.dirname(os.path.abspath(__file__))
ROOT = os.path.dirname(HERE)
WORKER = os.path.join(HERE, "launch_shapes_worker.py")

# (w, h): around the split geometry (interior columns (w - 17) // 128, interior rows (h - 17) // 64)
GEOMS = [(128, 64), (144, 96), (160, 80), (96, 160), (256, 145), (256, 144), (160, 146), (272, 81), (400, 82),
         (161, 145), (273, 96), (250, 146)]
PARAMS = [("Crossed", "Linear", 2), ("LeftTop", "Linear", 3), ("Crossed", "Linear", 1), ("LeftTop", "Linear", 2)]
LEVELS = [4, 5, 7, 8, 9]
CONTENTS = ["noise", "photo", "saturated"]

KNOBS = [
    ("defaults", {}),
    ("split_min_1", {"HGI_B200_SPLIT_MIN": "1"}),
    ("prefetch_0", {"HGI_B200_SPLIT_MIN": "1", "HGI_B200_PREFETCH": "0"}),
    ("prefetch_0.5", {"HGI_B200_SPLIT_MIN": "1", "HGI_B200_PREFETCH": "0.5"}),
    ("prefetch_2", {"HGI_B200_SPLIT_MIN": "1", "HGI_B200_PREFETCH": "2"}),
    ("graphs_0", {"HGI_B200_GRAPHS": "0"}),
    ("poison_00", {"HGI_B200_SPLIT_MIN": "1", "HGI_B200_POISON_SCRATCH": "0x00"}),
    ("poison_ff", {"HGI_B200_SPLIT_MIN": "1", "HGI_B200_POISON_SCRATCH": "0xFF"}),
    ("poison_a5", {"HGI_B200_SPLIT_MIN": "1", "HGI_B200_POISON_SCRATCH": "0xA5"}),
    ("slots_1", {"HGI_B200_SLOTS": "1", "HGI_B200_CHUNK_MB": "1", "HGI_B200_SPLIT_MIN": "1"}),
    ("slots_2", {"HGI_B200_SLOTS": "2", "HGI_B200_CHUNK_MB": "1", "HGI_B200_SPLIT_MIN": "1"}),
]
KNOB_VARS = ("HGI_B200_SPLIT_MIN", "HGI_B200_PREFETCH", "HGI_B200_GRAPHS", "HGI_B200_POISON_SCRATCH", "HGI_B200_SLOTS",
             "HGI_B200_CHUNK_MB")


def make_cases():
    cases = []
    for gi, (w, h) in enumerate(GEOMS):
        for pj, (interp, quant, q) in enumerate(PARAMS):
            cases.append(dict(w=w, h=h, n=1 + (gi + pj) % 2, levels=LEVELS[(gi + pj) % 5], interp=interp, quant=quant,
                              q=q, content=CONTENTS[(gi + 2 * pj) % 3]))
    for (w, h), (interp, quant, levels) in zip([(256, 145), (160, 146), (161, 145), (272, 81)],
                                               [("Crossed", "Linear", 4), ("LeftTop", "NoOp", 5), ("Crossed", "NoOp", 8),
                                                ("LeftTop", "Linear", 9)]):
        cases.append(dict(w=w, h=h, n=2, levels=levels, interp=interp, quant=quant, q=0, content="noise"))   # controls
    cases.append(dict(w=2320, h=1296, n=1, levels=8, interp="Crossed", quant="Linear", q=2, content="photo"))
    cases.append(dict(w=640, h=520, n=14, levels=6, interp="Crossed", quant="Linear", q=2, content="photo"))   # 3 per MB
    return cases


def planes(kind, n, h, w, seed):
    rng = np.random.default_rng(seed)
    if kind == "noise":
        return rng.integers(0, 256, (n, h, w)).astype(np.uint8)
    if kind == "photo":
        return np.stack([photo_like(w, h, seed + k) for k in range(n)])
    blk = 1 + seed % 7                                   # saturated blocks: every pixel 0 or 255
    m = rng.integers(0, 2, (n, -(-h // blk), -(-w // blk))).astype(np.uint8) * 255
    return np.repeat(np.repeat(m, blk, 1), blk, 2)[:, :h, :w].copy()


def oracle(imgs, levels, interp, quant, q):
    oi = oc.INTERP_CROSSED if interp == "Crossed" else oc.INTERP_LEFTTOP
    qk = oc.QUANT_LINEAR if quant == "Linear" else oc.QUANT_NOOP
    out = [oc.encode(im, levels, interp=oi, qkind=qk, qlevel=q, want_recon=True) for im in imgs]
    g = np.stack([a for a, _ in out])
    r = np.stack([b for _, b in out])
    hist = np.stack([np.bincount(x.reshape(-1), minlength=256).astype(np.uint32) for x in g])
    return g, r, hist


def run_worker(mode, inp, outp, env_over, timeout=600):
    env = {k: v for k, v in os.environ.items() if k not in KNOB_VARS}
    env.update(env_over)
    r = subprocess.run([sys.executable, WORKER, mode, str(inp), str(outp)], env=env, capture_output=True, text=True,
                       timeout=timeout)
    assert r.returncode == 0 and "worker ok" in r.stdout, r.stdout[-2000:] + r.stderr[-3000:]
    return np.load(outp)


def first_difference(got, want):
    if got.shape != want.shape:
        return f"shape {got.shape} != {want.shape}"
    idx = tuple(int(v) for v in np.argwhere(got != want)[0])
    return f"first differing byte at {idx}: got {got[idx]}, want {want[idx]} ({int((got != want).sum())} differ)"


def compare(res, want, describe, expected_launches, expected_graphs):
    """Every output against the oracle and every call's kernel / graph launches against the plain statement; the
    message names the first failing case, entry point and byte."""
    errors, blobs = [], {}
    for o in json.loads(str(res["outputs"])):
        if o["sha"] not in blobs:
            blobs[o["sha"]] = res[f"blob/{o['sha']}"]
        got = blobs[o["sha"]]
        g, r, hist = want(o["case"], o["variant"])
        exp = {"grid": g, "recon": r, "dec": r, "hist": hist}[o["what"]]
        if o["first"]:
            exp = exp[:o["first"]]
        if got.shape != exp.shape or not np.array_equal(got, exp):
            errors.append(f"{describe(o['case'])} entry {o['entry']} {o['what']} (input {o['variant']}): "
                          f"{first_difference(got, exp)}")
    for c in json.loads(str(res["calls"])):
        el, eg = expected_launches(c), expected_graphs(c)
        if c["launches"] != el or c["graphs"] != eg:
            errors.append(f"{describe(c['case'])} entry {c['entry']} call {c['call']} ({c['mode']}): "
                          f"{c['launches']} kernel / {c['graphs']} graph launches, expected {el} / {eg}")
    assert not errors, f"{len(errors)} mismatches; first: {errors[0]}" + "".join("\n  " + e for e in errors[1:8])


@pytest.fixture(scope="module")
def matrix(tmp_path_factory):
    """The case list, its inputs (three variants per case) and the oracle's outputs, written once."""
    d = tmp_path_factory.mktemp("launch_shapes")
    cases = make_cases()
    inputs, want = {}, {}
    for i, c in enumerate(cases):
        for v in range(3):
            kind = c["content"] if v == 0 else CONTENTS[(CONTENTS.index(c["content"]) + v) % 3]
            imgs = planes(kind, c["n"], c["h"], c["w"], 31 * i + v)
            inputs[f"in/{i}/{v}"] = imgs
            want[(i, v)] = oracle(imgs, c["levels"], c["interp"], c["quant"], c["q"])
    np.savez(d / "in.npz", cases=np.array(json.dumps(cases)), **inputs)
    np.savez(d / "oracle.npz", **{f"{k}/{i}/{v}": a for (i, v), arrs in want.items() for k, a in zip("grh", arrs)})
    return d, cases, want


def _qerr(c):
    return 10 * c["q"] if c["quant"] == "Linear" else 0


@pytest.mark.parametrize("name,env", KNOBS, ids=[k for k, _ in KNOBS])
def test_split_launches_equal_the_oracle_under_every_knob(matrix, name, env):
    """Every case x entry point under one knob setting: grid, reconstruction, histogram and decoded bytes equal the
    oracle, and every call launched the kernels the dispatch statement says (so a split that did not happen fails)."""
    d, cases, want = matrix
    res = run_worker("matrix", d / "in.npz", d / f"out_{name}.npz", env)
    split_min = int(env.get("HGI_B200_SPLIT_MIN", tm.SPLIT_MIN_TILES))
    chunk_bytes = int(env.get("HGI_B200_CHUNK_MB", 64)) << 20
    graphs_on = env.get("HGI_B200_GRAPHS", "1")[:1] != "0"

    def dev(c, mode, hist, n, pitch):
        return tm.expected_launches(mode, _qerr(c) if mode == "enc" else 0, c["w"], c["h"], pitch % 16 == 0,
                                    c["levels"], n, split_min, hist)

    def expected_launches(call):
        c = cases[call["case"]]
        n, pitch = call["n"], call["pitch"]
        if call["mode"] == "replay":
            return 0
        if call["mode"] == "enc+dec":
            return dev(c, "enc", True, n, pitch) + dev(c, "dec", False, n, pitch)
        if call.get("host"):          # run_host_chunks: chunks of chunk_bytes // plane images
            per = max(1, min(n, chunk_bytes // (c["w"] * c["h"])))
            return sum(dev(c, call["mode"], call["hist"], min(per, n - f), pitch) for f in range(0, n, per))
        return dev(c, call["mode"], call["hist"], n, pitch)

    def expected_graphs(call):        # run_dev_cached: chains of L > 4 on a real stream replay from the second call
        c = cases[call["case"]]
        L = tm.effective_levels(c["levels"], c["w"], c["h"])
        return int(graphs_on and call["entry"][0] == "b" and call["call"] >= 1 and L > 4)

    def describe(i):
        c = cases[i]
        return (f"[{name}] case {i} {c['w']}x{c['h']} n={c['n']} L{c['levels']} {c['interp']} {c['quant']}({c['q']}) "
                f"{c['content']}")

    compare(res, lambda i, v: want[(i, v)], describe, expected_launches, expected_graphs)


def test_graph_cache_keys_separate_calls_that_differ_in_one_field(tmp_path):
    """On one stream with one src / grid pair, calls A, B, A, B, ... (five each) that differ in exactly one ChainKey
    field: each must get its own captured chain (8 graph launches per sequence) and its own bytes; the two level
    counts that clamp to the same effective L share one (9).  Every output buffer is reset before every call, so a
    replay of the other call's graph -- into the other recon / hist buffer, all of them live -- shows."""
    w, h = 256, 146                   # effective L = 8; HGI_B200_SPLIT_MIN=1: both passes split (side-stream fork in the graph)
    src = np.stack([photo_like(w, h, 77), np.random.default_rng(78).integers(0, 256, (h, w)).astype(np.uint8)])
    seqs = []
    for L in (6, 8):
        base = dict(levels=L, interp="Crossed", quant="Linear", q=2, recon=0, hist=0)
        for field, change in (("interpolator", {"interp": "LeftTop"}), ("quant_level", {"q": 3}),
                              ("Lossless against Medium", {"q": 0}), ("recon_out", {"recon": 1}), ("hist", {"hist": 1})):
            seqs.append(dict(name=f"L{L} {field}", calls=[base, dict(base, **change)] * 5))
    base = dict(levels=8, interp="Crossed", quant="Linear", q=2, recon=0, hist=0)
    seqs.append(dict(name="levels 8 / 9 (same effective L)", calls=[base, dict(base, levels=9)] * 5))
    seqs.append(dict(name="levels 6 / 8", calls=[dict(base, levels=6), base] * 5))
    np.savez(tmp_path / "in.npz", seqs=np.array(json.dumps(seqs)), src=src)
    res = run_worker("keys", tmp_path / "in.npz", tmp_path / "out.npz", {"HGI_B200_SPLIT_MIN": "1"})

    want = {}

    def key(p):
        return (p["interp"], p["q"], p["recon"], p["hist"], tm.effective_levels(p["levels"], w, h))

    def oracle_of(i, k):
        p = seqs[i]["calls"][k]
        t = (p["interp"], p["q"], tm.effective_levels(p["levels"], w, h))
        if t not in want:
            want[t] = oracle(src, p["levels"], p["interp"], "Linear", p["q"])
        return want[t]

    def expected_launches(call):
        p = seqs[call["case"]]["calls"][call["call"]]
        return tm.expected_launches("enc", 10 * p["q"], w, h, True, p["levels"], 2, 1, True)

    def expected_graphs(call):        # first sighting plain, second captured + launched, then replayed
        calls = seqs[call["case"]]["calls"]
        return int(any(key(calls[j]) == key(calls[call["call"]]) for j in range(call["call"])))

    compare(res, oracle_of, lambda i: seqs[i]["name"], expected_launches, expected_graphs)
    per_seq = {}
    for c in json.loads(str(res["calls"])):
        per_seq[c["case"]] = per_seq.get(c["case"], 0) + c["graphs"]
    assert [per_seq[i] for i in range(len(seqs))] == [8] * (len(seqs) - 2) + [9, 8]


def test_batches_beyond_grid_z_on_the_split_path():
    """66 000 planes of 160x96 (one interior tile each, so PART 1 and its prefetch run) at L4 and L5, Medium, with
    recon_out and hist_out, on a real stream: the job is cut into launches of 65 535 images; the first chunk splits and
    prefetches 370 images ahead (ceil(1480 / 4 tiles)), the remaining 465 images are below split_min_tiles().  The
    batch repeats 7 base planes, so every plane is checked on the GPU against its base plane, and the base planes and
    the planes at the chunk and prefetch edges against the oracle."""
    import torch
    w, h, n = 160, 96, 66000
    bases = np.stack([photo_like(w, h, 500 + k) for k in range(6)] +
                     [np.random.default_rng(506).integers(0, 256, (h, w)).astype(np.uint8)])
    nb = len(bases)
    ctx = hgi.Context(0)
    src = torch.from_numpy(bases).cuda().repeat(-(-n // nb), 1, 1)[:n]
    grid, recon = torch.empty_like(src), torch.empty_like(src)
    hist = torch.empty((n, 256), dtype=torch.int32, device="cuda")
    s = torch.cuda.Stream()
    pf = -(-1480 // 4)
    check = sorted(set(list(range(nb)) + [65535 - 1480 - 1, 65535 - 1480, 65535 - 1480 + 1, 65535 - pf - 1, 65535 - pf,
                                          65535 - pf + 1, 65534, 65535, 65536, n - 1]))
    m = n // nb * nb
    for levels in (4, 5):
        want_g, want_r, want_h = oracle(bases, levels, "Crossed", "Linear", 2)
        for t in (grid, recon):
            t.fill_(0x5A)
        hist.fill_(-1)
        torch.cuda.synchronize()
        k0 = ctx.kernel_launches
        hgi.Encoder(hgi.Crossed, hgi.Linear(hgi.QuantizationLevel.Medium), levels, ctx=ctx).encode_device(
            src, grids_out=grid, recon_out=recon, hist_out=hist, stream=s.cuda_stream)
        s.synchronize()
        assert ctx.kernel_launches - k0 == tm.expected_launches("enc", 20, w, h, True, levels, n, hist=True), levels
        for t in (grid, recon, hist):
            head = t[:nb]
            assert torch.equal(t[:m].view(m // nb, *head.shape), head.unsqueeze(0).expand(m // nb, *head.shape)), levels
            assert torch.equal(t[m:], head[:n - m]), levels
        for p in check:
            b = p % nb
            assert (grid[p].cpu().numpy() == want_g[b]).all(), (levels, p)
            assert (recon[p].cpu().numpy() == want_r[b]).all(), (levels, p)
            assert (hist[p].cpu().numpy().view(np.uint32) == want_h[b]).all(), (levels, p)
    del src, grid, recon, hist
    torch.cuda.synchronize()
    ctx.close()


def test_fuzz_through_the_split():
    """tools/fuzz_parity.py (120 random cases) with HGI_B200_SPLIT_MIN=1: random sizes, pitches, levels, quantizers
    and interpolators through the split parts."""
    env = {k: v for k, v in os.environ.items() if k not in KNOB_VARS}
    env["HGI_B200_SPLIT_MIN"] = "1"
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tools", "fuzz_parity.py"), "--cases", "120", "--seed", "303"],
                       env=env, capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "fuzz ok: 120 cases" in r.stdout, r.stdout[-1500:] + r.stderr[-1500:]
