"""Token-range reads of an LACB file (sharding.decompress_sharded(start, stop)) with a reversible stand-in coder:
which batches are decoded, what each slot is given, and the 2-rank deal (gloo, CPU)."""
import os
import socket

import numpy as np
import pytest
import torch.distributed as dist
import torch.multiprocessing as mp

from lac_b200 import container, sharding


def _encode(tokens, ntok):
    streams = [np.asarray(row[:n], dtype="<i4").tobytes() for row, n in zip(tokens, ntok)]
    return streams, [8 * len(s) for s in streams]


class Decoder:
    """decode_batch stand-in that decodes any prefix of a stream (as the GPU decoder does) and records its calls."""

    def __init__(self, chunk_tokens):
        self.T, self.calls = chunk_tokens, []

    def __call__(self, streams, ntok):
        self.calls.append((list(streams), ntok.copy()))
        out = np.zeros((len(streams), self.T), dtype=np.int32)
        for i, (s, n) in enumerate(zip(streams, ntok)):
            assert len(s) >= 4 * n
            out[i, :n] = np.frombuffer(s, dtype="<i4")[:n]
        return out


def _file(n_tokens, chunk, B, header_B=None):
    toks = np.random.default_rng(n_tokens).integers(0, 1000, n_tokens).astype(np.int32)
    blob = sharding.compress_sharded(toks, chunk, B, _encode, 48, 1000, "cpu", tag=5)
    if header_B is not None:   # rewrite the header's batch_streams (0: one batch of all chunks)
        c = container.unpack(blob)
        blob = container.pack(c.streams(), c.ntok, c.nbits, 48, 1000, chunk, batch_streams=header_B, tag=5)
    return toks, blob


def _expected_calls(blob, start, stop):
    """The decode_batch calls a range read must make, from the index alone."""
    c = container.unpack(blob)
    B = c.batch_streams or max(c.n_chunks, 1)
    streams = c.streams()
    first = np.concatenate([[0], np.cumsum(c.ntok.astype(np.int64))])
    calls = []
    for k in range(-(-c.n_chunks // B)):
        bs, bn = [b""] * B, np.zeros(B, dtype=np.int32)
        for j in range(B):
            i = k * B + j
            if i < c.n_chunks and max(first[i], start) < min(first[i + 1], stop):   # overlaps [start, stop)
                bs[j], bn[j] = streams[i], min(int(c.ntok[i]), stop - int(first[i]))
        if bn.any():
            calls.append((bs, bn))
    return calls


def _same_calls(got, want):
    assert len(got) == len(want)
    for (gs, gn), (ws, wn) in zip(got, want):
        assert gs == ws and gn.dtype == np.int32 and np.array_equal(gn, wn)


FILES = [(37, 8, 3, None), (1000, 16, 4, None), (37, 8, 3, 0), (20, 4, 8, None)]


@pytest.mark.parametrize("n_tokens,chunk,B,header_B", FILES)
def test_every_range_reads_its_tokens_and_decodes_only_what_it_needs(n_tokens, chunk, B, header_B):
    toks, blob = _file(n_tokens, chunk, B, header_B)
    step = 1 if n_tokens < 100 else 37           # 1000 tokens: every start, stops at a stride plus the edges
    for start in range(n_tokens + 1):
        stops = set(range(start, n_tokens + 1, step)) | {start, start + 1, n_tokens}
        for stop in sorted(s for s in stops if s <= n_tokens):
            dec = Decoder(chunk)
            got = sharding.decompress_sharded(blob, dec, "cpu", start=start, stop=stop)
            assert got.dtype == np.int32 and np.array_equal(got, toks[start:stop]), (start, stop)
            _same_calls(dec.calls, _expected_calls(blob, start, stop))


@pytest.mark.parametrize("n_tokens,chunk,B,header_B", FILES)
def test_whole_file_is_one_call_per_batch_with_full_counts(n_tokens, chunk, B, header_B):
    toks, blob = _file(n_tokens, chunk, B, header_B)
    c = container.unpack(blob)
    Bh = c.batch_streams or c.n_chunks
    d0, d1, d2 = Decoder(chunk), Decoder(chunk), Decoder(chunk)
    assert np.array_equal(sharding.decompress_sharded(blob, d0, "cpu"), toks)
    assert np.array_equal(sharding.decompress_sharded(blob, d1, "cpu", start=0, stop=n_tokens), toks)
    assert np.array_equal(sharding.decompress_sharded(blob, d2, "cpu", start=0, stop=None), toks)
    streams = c.streams()
    want = []
    for c0 in range(0, c.n_chunks, Bh):
        c1 = min(c.n_chunks, c0 + Bh)
        bn = np.zeros(Bh, dtype=np.int32)
        bn[: c1 - c0] = c.ntok[c0:c1]
        want.append((streams[c0:c1] + [b""] * (Bh - (c1 - c0)), bn))
    for d in (d0, d1, d2):
        _same_calls(d.calls, want)


def test_empty_ranges_and_empty_file_decode_nothing():
    toks, blob = _file(37, 8, 3)
    for start in (0, 8, 20, 37):
        dec = Decoder(8)
        got = sharding.decompress_sharded(blob, dec, "cpu", start=start, stop=start)
        assert got.dtype == np.int32 and got.shape == (0,) and dec.calls == []
    _, empty = _file(0, 8, 3)
    dec = Decoder(8)
    got = sharding.decompress_sharded(empty, dec, "cpu")
    assert got.dtype == np.int32 and got.shape == (0,) and dec.calls == []


@pytest.mark.parametrize("start,stop", [(-1, 5), (0, -1), (5, 4), (0, 38), (38, 38), (1.0, 5), (0, 5.0),
                                        ("0", 5), (None, 5), (True, 5), (0, np.float64(3))])
def test_bad_ranges_raise(start, stop):
    _, blob = _file(37, 8, 3)
    dec = Decoder(8)
    with pytest.raises(ValueError):
        sharding.decompress_sharded(blob, dec, "cpu", start=start, stop=stop)
    assert dec.calls == []


def test_numpy_integers_are_accepted():
    toks, blob = _file(37, 8, 3)
    got = sharding.decompress_sharded(blob, Decoder(8), "cpu", start=np.int64(9), stop=np.uint32(30))
    assert np.array_equal(got, toks[9:30])


# ------------------------------------------------------------------ two ranks
RANGES = [(0, None), (0, 1), (9, 30), (16, 17), (23, 25), (60, 1000), (500, 900), (300, 300), (999, 1000)]


def _range_worker(rank, world, port, q):
    _, blob = _file(1000, 16, 4)                 # written by one process: every rank builds the same file
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    out = []
    for start, stop in RANGES:
        dec = Decoder(16)
        got = sharding.decompress_sharded(blob, dec, "cpu", start=start, stop=stop)
        out.append((got, dec.calls))
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_read_the_same_range_and_split_the_batches():
    toks, blob = _file(1000, 16, 4)
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_range_worker, args=(r, 2, port, q)) for r in range(2)]
    for p in procs:
        p.start()
    res = dict(q.get(timeout=120) for _ in procs)
    for p in procs:
        p.join(timeout=120)
        assert p.exitcode == 0
    for n, (start, stop) in enumerate(RANGES):
        stop = len(toks) if stop is None else stop
        got0, calls0 = res[0][n]
        got1, calls1 = res[1][n]
        assert got1 is None
        assert np.array_equal(got0, toks[start:stop])
        assert np.array_equal(got0, sharding.decompress_sharded(blob, Decoder(16), "cpu", start=start, stop=stop))
        # every needed batch exactly once over the two ranks, rank 0 the earlier ones, balanced
        want = _expected_calls(blob, start, stop)
        _same_calls(calls0 + calls1, want)
        assert len(calls0) - len(calls1) in (0, 1)
