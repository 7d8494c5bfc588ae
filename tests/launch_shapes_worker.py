"""Worker of tests/test_gpu_launch_shapes.py: runs the cases of an input .npz through the library in a process of its
own (the HGI_B200_* knobs are read once per process) and writes what came back to an output .npz.

    python tests/launch_shapes_worker.py matrix|keys IN.npz OUT.npz

It compares nothing: the parent holds the oracle.  Outputs are stored once per distinct content (`blob/<sha1>`) and
listed in `outputs` (JSON: case, entry point, what, input variant, sha1); every library call is listed in `calls`
(JSON: case, entry point, call, kernel launches, graph launches, and what the launch count depends on)."""
import hashlib
import json
import os
import sys

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))

import numpy as np  # noqa: E402
import torch  # noqa: E402

import rustyhgi_b200 as hgi  # noqa: E402

SENTINEL = 0x5A


def _interp(name):
    return hgi.Crossed if name == "Crossed" else hgi.LeftTop


def _quant(c):
    q = hgi.QuantizationLevel(c["q"])
    return hgi.Linear(q) if c["quant"] == "Linear" else hgi.NoOp(q)


class Recorder:
    def __init__(self):
        self.blobs, self.outputs, self.calls = {}, [], []

    def out(self, case, entry, what, variant, t, first=None):
        a = t.cpu().numpy() if isinstance(t, torch.Tensor) else np.asarray(t)
        if what == "hist":
            a = a.view(np.uint32)
        a = np.ascontiguousarray(a)
        sha = hashlib.sha1(a.tobytes() + repr(a.shape).encode()).hexdigest()
        self.blobs.setdefault(sha, a)
        self.outputs.append(dict(case=case, entry=entry, what=what, variant=variant, sha=sha, first=first))

    def call(self, ctx, case, entry, call, fn, **desc):
        k0, g0 = ctx.kernel_launches, ctx.graph_launches
        r = fn()
        self.calls.append(dict(case=case, entry=entry, call=call, launches=ctx.kernel_launches - k0,
                               graphs=ctx.graph_launches - g0, **desc))
        return r

    def save(self, path):
        arrays = {f"blob/{k}": v for k, v in self.blobs.items()}
        np.savez(path, outputs=np.array(json.dumps(self.outputs)), calls=np.array(json.dumps(self.calls)), **arrays)


def run_case(rec, i, c, inputs):
    """Entry points (a)..(e) of the test's docstring on case `c`; inputs[v] is input variant v (n, h, w)."""
    n, h, w, levels = c["n"], c["h"], c["w"], c["levels"]
    ctx = hgi.Context(0)        # a context of its own: no launch chain of another case is cached
    enc = hgi.Encoder(_interp(c["interp"]), _quant(c), levels, ctx=ctx)
    dec = hgi.Decoder(_interp(c["interp"]), ctx=ctx)
    img = inputs[0]
    desc = dict(n=n, pitch=w)

    # (a) host API: slot streams (they fork the split launches)
    g, hist = rec.call(ctx, i, "a", 0, lambda: enc.encode_batch(img, want_hist=True), mode="enc", hist=True, host=True, **desc)
    rec.out(i, "a", "grid", 0, g)
    rec.out(i, "a", "hist", 0, hist)
    g = rec.call(ctx, i, "a", 1, lambda: enc.encode_batch(img), mode="enc", hist=False, host=True, **desc)
    rec.out(i, "a", "grid", 0, g)
    back = rec.call(ctx, i, "a", 2, lambda: dec.decode_batch(levels, g), mode="dec", hist=False, host=True, **desc)
    rec.out(i, "a", "dec", 0, back)
    g1, r1 = rec.call(ctx, i, "a", 3, lambda: enc.encode(img[0], want_recon=True), mode="enc", hist=False, host=True,
                      n=1, pitch=w)
    rec.out(i, "a", "grid", 0, g1.as_plane()[None], first=1)
    rec.out(i, "a", "recon", 0, r1[None], first=1)

    src = torch.from_numpy(img).cuda()
    s = torch.cuda.Stream()
    keep = []                   # every buffer a cached chain may point into stays alive until the case ends

    def buffers():
        b = [torch.full_like(src, SENTINEL), torch.full_like(src, SENTINEL), torch.full_like(src, SENTINEL),
             torch.full((n, 256), -1, dtype=torch.int32, device="cuda")]
        keep.append(b)
        return b

    # (b) device API on a real stream, three calls with the same buffers: plain, captured, replayed
    # (c) device API on torch's default stream (cudaStreamLegacy: no fork, no graph)
    for entry, stream, calls in (("b", s, 3), ("c", None, 1)):
        for extra in (True, False):
            ent = entry + ("+" if extra else "-")
            grid, recon, out, hist = buffers()
            torch.cuda.synchronize()
            for k in range(calls):
                with torch.cuda.stream(stream if stream is not None else torch.cuda.current_stream()):
                    grid.fill_(SENTINEL)
                    recon.fill_(SENTINEL)
                    out.fill_(SENTINEL)
                    hist.fill_(-1)
                sh = stream.cuda_stream if stream is not None else None
                rec.call(ctx, i, ent, k, lambda: enc.encode_device(src, grids_out=grid, recon_out=recon if extra else None,
                                                                  hist_out=hist if extra else None, stream=sh),
                         mode="enc", hist=extra, **desc)
                rec.call(ctx, i, ent, k, lambda: dec.decode_device(levels, grid, images_out=out, stream=sh),
                         mode="dec", hist=False, **desc)
                torch.cuda.synchronize()
                rec.out(i, ent, "grid", 0, grid)
                rec.out(i, ent, "dec", 0, out)
                if extra:
                    rec.out(i, ent, "recon", 0, recon)
                    rec.out(i, ent, "hist", 0, hist)

    # (d) padded rows (hgi_*_dev_pitched): garbage in the input padding; output padding bytes are unspecified
    rng = np.random.default_rng(1000 + i)
    for pad in (0, 16):
        pitch = (w + 15) // 16 * 16 + pad
        for extra in (True, False):
            ent = f"d{pad}" + ("+" if extra else "-")
            buf = torch.from_numpy(rng.integers(0, 256, (n, h, pitch)).astype(np.uint8)).cuda()
            buf[:, :, :w] = src
            gb, rb, ob = (torch.full((n, h, pitch), SENTINEL, dtype=torch.uint8, device="cuda") for _ in range(3))
            hist = torch.full((n, 256), -1, dtype=torch.int32, device="cuda")
            keep.append((buf, gb, rb, ob, hist))
            torch.cuda.synchronize()
            rec.call(ctx, i, ent, 0, lambda: enc.encode_device(buf[:, :, :w], grids_out=gb[:, :, :w],
                                                              recon_out=rb[:, :, :w] if extra else None,
                                                              hist_out=hist if extra else None, stream=s.cuda_stream),
                     mode="enc", hist=extra, n=n, pitch=pitch)
            rec.call(ctx, i, ent, 0, lambda: dec.decode_device(levels, gb[:, :, :w], images_out=ob[:, :, :w], stream=s.cuda_stream),
                     mode="dec", hist=False, n=n, pitch=pitch)
            torch.cuda.synchronize()
            rec.out(i, ent, "grid", 0, gb[:, :, :w])
            rec.out(i, ent, "dec", 0, ob[:, :, :w])
            if extra:
                rec.out(i, ent, "recon", 0, rb[:, :, :w])
                rec.out(i, ent, "hist", 0, hist)

    # (e) the caller's own capture around encode_device + decode_device, after one warm-up call on the same stream;
    # replayed on three different inputs
    s2 = torch.cuda.Stream()
    st_src = torch.from_numpy(inputs[1]).cuda()
    grid, recon, out, hist = buffers()
    keep.append(st_src)
    torch.cuda.synchronize()

    def both():
        enc.encode_device(st_src, grids_out=grid, recon_out=recon, hist_out=hist)
        dec.decode_device(levels, grid, images_out=out)

    with torch.cuda.stream(s2):
        rec.call(ctx, i, "e", 0, both, mode="enc+dec", hist=True, **desc)
    s2.synchronize()
    rec.out(i, "e", "grid", 1, grid)
    rec.out(i, "e", "dec", 1, out)
    g = torch.cuda.CUDAGraph()
    with torch.cuda.graph(g, stream=s2):
        rec.call(ctx, i, "e", 1, both, mode="enc+dec", hist=True, **desc)
    for v in (0, 2, 1):
        st_src.copy_(torch.from_numpy(inputs[v]).cuda())
        for t in (grid, recon, out):
            t.fill_(SENTINEL)
        hist.fill_(-1)
        torch.cuda.synchronize()
        rec.call(ctx, i, "e", 2 + v, g.replay, mode="replay", hist=False, **desc)
        torch.cuda.synchronize()
        rec.out(i, "e", "grid", v, grid)
        rec.out(i, "e", "recon", v, recon)
        rec.out(i, "e", "dec", v, out)
        rec.out(i, "e", "hist", v, hist)
    torch.cuda.synchronize()
    del g
    ctx.close()


def run_keys(rec, seqs, src_np):
    """Graph-cache keys: on one stream and one src / grid pair, alternate calls A, B, A, B, ... that differ in one
    ChainKey field.  Before every call all output buffers are reset, so a replay of the other call's graph shows."""
    n, h, w = src_np.shape
    src = torch.from_numpy(src_np).cuda()
    grid = torch.empty_like(src)
    recons = [torch.empty_like(src), torch.empty_like(src)]
    hists = [torch.empty((n, 256), dtype=torch.int32, device="cuda") for _ in range(2)]
    for si, seq in enumerate(seqs):
        ctx = hgi.Context(0)
        s = torch.cuda.Stream()
        for k, p in enumerate(seq["calls"]):
            enc = hgi.Encoder(_interp(p["interp"]), _quant(p), p["levels"], ctx=ctx)
            with torch.cuda.stream(s):
                for t in [grid] + recons:
                    t.fill_(SENTINEL)
                for t in hists:
                    t.fill_(-1)
            r, hh = recons[p["recon"]], hists[p["hist"]]
            rec.call(ctx, si, "keys", k, lambda: enc.encode_device(src, grids_out=grid, recon_out=r, hist_out=hh,
                                                                  stream=s.cuda_stream), mode="enc", hist=True, n=n, pitch=w)
            s.synchronize()
            rec.out(si, "keys", "grid", k, grid)
            rec.out(si, "keys", "recon", k, r)
            rec.out(si, "keys", "hist", k, hh)
        torch.cuda.synchronize()
        ctx.close()


def main():
    mode, inp, outp = sys.argv[1:4]
    d = np.load(inp)
    rec = Recorder()
    if mode == "matrix":
        cases = json.loads(str(d["cases"]))
        for i, c in enumerate(cases):
            run_case(rec, i, c, [d[f"in/{i}/{v}"] for v in range(3)])
    else:
        run_keys(rec, json.loads(str(d["seqs"])), d["src"])
    torch.cuda.synchronize()
    rec.save(outp)
    print(f"worker ok: {len(rec.calls)} calls, {len(rec.outputs)} outputs")


if __name__ == "__main__":
    main()
