"""Packed token-range reads of batch-invariant files (sharding.decompress_packed) with a reversible stand-in coder:
every needed chunk decoded exactly once for its needed prefix, batch sizes, the deal over ranks, and a 2-rank gloo
run (CPU)."""
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
    """decode_batch stand-in of a decoder with S streams: decodes any prefix of up to S streams, records its calls.
    packed=False for the batched read of decompress_sharded, whose padding slots ask for 0 tokens."""

    def __init__(self, chunk_tokens, S, packed=True):
        self.T, self.S, self.packed, self.calls = chunk_tokens, S, packed, []

    def __call__(self, streams, ntok):
        assert 1 <= len(streams) <= self.S and ntok.shape == (len(streams),) and ntok.dtype == np.int32
        self.calls.append((list(streams), ntok.copy()))
        out = np.zeros((len(streams), self.T), dtype=np.int32)
        for i, (s, n) in enumerate(zip(streams, ntok)):
            assert (n >= 1 or not self.packed) and len(s) >= 4 * n
            out[i, :n] = np.frombuffer(s, dtype="<i4")[:n]
        return out


def _file(n_tokens, chunk, B):
    toks = np.random.default_rng(n_tokens + chunk).integers(0, 1000, n_tokens).astype(np.int32)
    return toks, sharding.compress_sharded(toks, chunk, B, _encode, 48, 1000, "cpu", tag=5)


def _needed(blob, start, stop):
    """{chunk: tokens to decode} for a range, from the index alone."""
    c = container.unpack(blob)
    first = np.concatenate([[0], np.cumsum(c.ntok.astype(np.int64))])
    return {i: min(int(c.ntok[i]), stop - int(first[i])) for i in range(c.n_chunks)
            if max(first[i], start) < min(first[i + 1], stop)}


def _check_calls(blob, calls, start, stop, S):
    """Every needed chunk exactly once, for its needed prefix; no batch above S; longest prefixes first."""
    c = container.unpack(blob)
    streams = c.streams()
    want = _needed(blob, start, stop)
    seen = {}
    for bs, bn in calls:
        assert 1 <= len(bs) <= S
        for s, n in zip(bs, bn):
            i = [j for j in want if streams[j] == s and j not in seen and want[j] == n]
            assert i, "a decoded stream is not a needed chunk (or was decoded twice)"
            seen[i[0]] = int(n)
    assert seen == want


# (tokens, chunk length, decoder S, file batch_streams)
FILES = [(37, 8, 1, 3), (37, 8, 3, 3), (37, 8, 16, 3), (1000, 16, 4, 4), (1000, 16, 7, 64), (20, 4, 8, 8),
         (203, 10, 5, 2)]


@pytest.mark.parametrize("n_tokens,chunk,S,fileB", FILES)
def test_every_range_decodes_each_needed_chunk_once(n_tokens, chunk, S, fileB):
    toks, blob = _file(n_tokens, chunk, fileB)
    step = 1 if n_tokens < 100 else 23
    for start in range(0, n_tokens + 1, 1 if n_tokens < 100 else 7):
        stops = set(range(start, n_tokens + 1, step)) | {start, start + 1, n_tokens}
        for stop in sorted(s for s in stops if s <= n_tokens):
            dec = Decoder(chunk, S)
            got = sharding.decompress_packed(blob, dec, S, "cpu", start=start, stop=stop)
            assert got.dtype == np.int32 and np.array_equal(got, toks[start:stop]), (start, stop)
            _check_calls(blob, dec.calls, start, stop, S)
            # one rank: ceil(needed / S) batches, the longest prefixes first
            assert len(dec.calls) == -(-len(_needed(blob, start, stop)) // S)
            lens = [int(n) for _, bn in dec.calls for n in bn]
            assert lens == sorted(lens, reverse=True)


def test_whole_file_and_default_range_match():
    toks, blob = _file(1000, 16, 4)
    for S in (1, 4, 5, 64, 100):
        a, b = Decoder(16, S), Decoder(16, S)
        assert np.array_equal(sharding.decompress_packed(blob, a, S, "cpu"), toks)
        assert np.array_equal(sharding.decompress_packed(blob, b, S, "cpu", start=0, stop=len(toks)), toks)
        assert [n.tolist() for _, n in a.calls] == [n.tolist() for _, n in b.calls]
        _check_calls(blob, a.calls, 0, len(toks), S)


def test_empty_ranges_bad_ranges_and_empty_file():
    toks, blob = _file(37, 8, 3)
    for start in (0, 8, 37):
        dec = Decoder(8, 4)
        got = sharding.decompress_packed(blob, dec, 4, "cpu", start=start, stop=start)
        assert got.dtype == np.int32 and got.shape == (0,) and dec.calls == []
    for start, stop in ((-1, 5), (5, 4), (0, 38), (1.0, 5)):
        dec = Decoder(8, 4)
        with pytest.raises(ValueError):
            sharding.decompress_packed(blob, dec, 4, "cpu", start=start, stop=stop)
        assert dec.calls == []
    _, empty = _file(0, 8, 3)
    dec = Decoder(8, 4)
    assert sharding.decompress_packed(empty, dec, 4, "cpu").shape == (0,) and dec.calls == []


@pytest.mark.parametrize("n_needed,S,world", [(1, 4, 1), (5, 4, 4), (7, 8, 2), (9, 4, 8), (3, 4, 8), (40, 4, 8),
                                              (256, 256, 8), (600, 256, 2), (17, 1, 3)])
def test_batches_are_bounded_and_every_rank_gets_work(n_needed, S, world):
    want = np.zeros(n_needed + 3, dtype=np.int64)
    want[1:n_needed + 1] = np.random.default_rng(n_needed).integers(1, 50, n_needed)
    batches = sharding.pack_batches(want, S, world)
    ids = np.concatenate(batches)
    assert sorted(ids.tolist()) == list(range(1, n_needed + 1))
    lens = [int(want[i]) for i in ids]
    assert lens == sorted(lens, reverse=True)
    assert all(1 <= len(b) <= S for b in batches)
    if n_needed > world * S:                       # more than one round: full batches of S from the front
        assert len(batches) == -(-n_needed // S) and all(len(b) == S for b in batches[:-1])
    else:                                          # one round: balanced, and every rank has work
        assert len(batches) == min(world, n_needed)
        assert all(len(b) <= -(-n_needed // world) for b in batches)
        assert {k % world for k in range(len(batches))} == set(range(min(world, n_needed)))


def _steps(calls):
    """Model steps a run of decode_batch calls costs: each batch runs for its longest prefix."""
    return sum(int(bn.max()) for _, bn in calls)


@pytest.mark.parametrize("n_tokens,chunk,B", [(1000, 16, 4), (203, 10, 5), (37, 8, 3), (300, 7, 8)])
def test_one_rank_never_runs_more_steps_than_the_batched_read(n_tokens, chunk, B):
    """A decoder of the file's own S: the packed read costs at most the steps of decompress_sharded's read."""
    toks, blob = _file(n_tokens, chunk, B)
    for start in range(0, n_tokens, 3):
        for stop in range(start + 1, n_tokens + 1, 5):
            old, new = Decoder(chunk, B, packed=False), Decoder(chunk, B)
            sharding.decompress_sharded(blob, old, "cpu", start=start, stop=stop)
            assert np.array_equal(sharding.decompress_packed(blob, new, B, "cpu", start=start, stop=stop),
                                  toks[start:stop])
            assert _steps(new.calls) <= _steps(old.calls), (start, stop)


def test_s_chunks_and_a_partial_one_cost_what_the_batched_read_costs():
    """S full chunks plus the first 5 tokens of the next: one batch of S for the full chunks, and the partial chunk
    alone in a batch of 1 (decoded at n = 1) -- not two half batches that both run the full chunk length."""
    S, chunk = 8, 16
    toks, blob = _file(3 * S * chunk, chunk, S)
    for first in (0, 1, S - 1):
        start, stop = first * chunk, (first + S) * chunk + 5
        old, new = Decoder(chunk, S, packed=False), Decoder(chunk, S)
        sharding.decompress_sharded(blob, old, "cpu", start=start, stop=stop)
        got = sharding.decompress_packed(blob, new, S, "cpu", start=start, stop=stop)
        assert np.array_equal(got, toks[start:stop])
        assert [len(bs) for bs, _ in new.calls] == [S, 1] and new.calls[1][1].tolist() == [5]
        assert _steps(new.calls) == chunk + 5 <= _steps(old.calls)


# ------------------------------------------------------------------ two ranks
RANGES = [(0, None), (0, 1), (9, 30), (16, 17), (23, 25), (60, 1000), (500, 900), (300, 300), (999, 1000)]
S2 = 3


def _worker(rank, world, port, q):
    _, blob = _file(1000, 16, 4)
    os.environ["MASTER_ADDR"] = "127.0.0.1"
    os.environ["MASTER_PORT"] = str(port)
    dist.init_process_group("gloo", rank=rank, world_size=world)
    out = []
    for start, stop in RANGES:
        dec = Decoder(16, S2)
        got = sharding.decompress_packed(blob, dec, S2, "cpu", start=start, stop=stop)
        out.append((got, dec.calls))
    q.put((rank, out))
    dist.barrier()
    dist.destroy_process_group()


def test_two_ranks_return_what_one_rank_returns():
    toks, blob = _file(1000, 16, 4)
    s = socket.socket()
    s.bind(("127.0.0.1", 0))
    port = s.getsockname()[1]
    s.close()
    ctx = mp.get_context("spawn")
    q = ctx.Queue()
    procs = [ctx.Process(target=_worker, args=(r, 2, port, q)) for r in range(2)]
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
        one = sharding.decompress_packed(blob, Decoder(16, S2), S2, "cpu", start=start, stop=stop)
        assert np.array_equal(got0, toks[start:stop]) and np.array_equal(got0, one)
        _check_calls(blob, calls0 + calls1, start, stop, S2)
        if len(_needed(blob, start, stop)) >= 2:
            assert calls0 and calls1                  # both ranks decode
