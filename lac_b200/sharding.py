"""Multi-GPU layout: independent chunks shard across ranks with no collective inside the coding
loop; the only exchange is the gather of per-chunk token / bit counts and, for writing one file,
of the compressed bytes (a few bits per token).  Works on NCCL (GPU tensors) and gloo (CPU tensors).

Chunks are coded in model batches of exactly `batch_streams` streams (the last batch padded with empty
streams): the predictor then sees the same batch shape whether a file is written by 1 GPU and read by 8 or the
other way round, which is what makes the logits -- and with them the decode -- bit-reproducible.  Batches, not
chunks, are what is dealt to the ranks: rank r owns a contiguous range of batches.

That batch shape binds torch-mode files only.  A batch-invariant predictor gives a stream the same logits in a
batch of any size, so such a file is decoded chunk by chunk (decompress_packed): the needed chunks are packed into
batches of the decoder's size and dealt over all ranks, whatever batch_streams the header records.
"""
from __future__ import annotations

import numbers
from typing import Callable, List, Optional, Sequence, Tuple

import numpy as np
import torch
import torch.distributed as dist

from . import container


def chunk_range(n_chunks: int, rank: int, world: int) -> Tuple[int, int]:
    """Contiguous, balanced [begin, end) of the items rank owns (first n % world ranks get one more)."""
    base, extra = divmod(n_chunks, world)
    begin = rank * base + min(rank, extra)
    return begin, begin + base + (1 if rank < extra else 0)


def batch_spans(n_chunks: int, batch_streams: int, world: int) -> List[Tuple[int, int]]:
    """Per rank the [begin, end) CHUNK range it owns: whole batches, dealt contiguously."""
    n_batches = -(-n_chunks // batch_streams) if n_chunks else 0
    spans = []
    for r in range(world):
        b, e = chunk_range(n_batches, r, world)
        spans.append((min(n_chunks, b * batch_streams), min(n_chunks, e * batch_streams)))
    return spans


def _world(group=None) -> Tuple[int, int]:
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(group), dist.get_world_size(group)
    return 0, 1


def gather_index(ntok: torch.Tensor, nbits: torch.Tensor, n_chunks: int, group=None,
                 spans: Optional[Sequence[Tuple[int, int]]] = None) -> Tuple[torch.Tensor, torch.Tensor]:
    """All ranks get the global (ntok, nbits) int64 [n_chunks] from their local shards (rank order = chunk order).
    spans: the chunk range of every rank (default: chunk_range)."""
    rank, world = _world(group)
    if spans is None:
        spans = [chunk_range(n_chunks, r, world) for r in range(world)]
    if world == 1:
        return ntok.to(torch.int64), nbits.to(torch.int64)
    width = max(max(e - b for b, e in spans), 1)
    local = torch.zeros((2, width), dtype=torch.int64, device=ntok.device)
    local[0, : ntok.numel()] = ntok.to(torch.int64)
    local[1, : nbits.numel()] = nbits.to(torch.int64)
    everyone = torch.zeros((world, 2, width), dtype=torch.int64, device=ntok.device)
    dist.all_gather_into_tensor(everyone.view(-1), local.view(-1), group=group)
    g_ntok = [everyone[r, 0, : e - b] for r, (b, e) in enumerate(spans)]
    g_nbits = [everyone[r, 1, : e - b] for r, (b, e) in enumerate(spans)]
    return torch.cat(g_ntok), torch.cat(g_nbits)


def gather_payload(local_bytes: torch.Tensor, g_nbits: torch.Tensor, n_chunks: int, dst: int = 0, group=None,
                   spans: Optional[Sequence[Tuple[int, int]]] = None) -> Optional[bytes]:
    """Concatenate every rank's (already concatenated) chunk bytes on rank dst; None elsewhere."""
    rank, world = _world(group)
    if spans is None:
        spans = [chunk_range(n_chunks, r, world) for r in range(world)]
    if world == 1:
        return local_bytes.cpu().numpy().tobytes()
    sizes = [int(((g_nbits[b:e] + 7) // 8).sum().item()) for b, e in spans]
    width = max(max(sizes), 1)
    padded = torch.zeros(width, dtype=torch.uint8, device=local_bytes.device)
    padded[: local_bytes.numel()] = local_bytes
    everyone = torch.zeros((world, width), dtype=torch.uint8, device=local_bytes.device)
    dist.all_gather_into_tensor(everyone.view(-1), padded, group=group)
    if rank != dst:
        return None
    host = everyone.cpu().numpy()
    return b"".join(host[r, : sizes[r]].tobytes() for r in range(world))


def gather_tokens(local: torch.Tensor, n_chunks: int, chunk_tokens: int, spans: Sequence[Tuple[int, int]],
                  dst: int = 0, group=None) -> Optional[torch.Tensor]:
    """Decoded tokens int32 [local chunks, chunk_tokens] of every rank -> [n_chunks, chunk_tokens] on rank dst."""
    rank, world = _world(group)
    if world == 1:
        return local
    width = max(max(e - b for b, e in spans), 1)
    padded = torch.zeros((width, chunk_tokens), dtype=torch.int32, device=local.device)
    padded[: local.shape[0]] = local
    everyone = torch.zeros((world, width, chunk_tokens), dtype=torch.int32, device=local.device)
    dist.all_gather_into_tensor(everyone.view(-1), padded.view(-1), group=group)
    if rank != dst:
        return None
    return torch.cat([everyone[r, : e - b] for r, (b, e) in enumerate(spans)])


def concat_streams(streams: Sequence[bytes], device) -> torch.Tensor:
    buf = np.frombuffer(b"".join(streams), dtype=np.uint8).copy() if streams else np.zeros(0, dtype=np.uint8)
    return torch.from_numpy(buf).to(device)


# ------------------------------------------------------------------ the sharded job (host logic only)
# encode_batch(tokens int32 [B, chunk_tokens], ntok int32 [B]) -> (streams: list of B bytes, nbits: list of B ints)
# decode_batch(streams: list of B bytes, ntok int32 [B])       -> tokens int32 [B, chunk_tokens] (numpy)
EncodeBatch = Callable[[np.ndarray, np.ndarray], Tuple[List[bytes], Sequence[int]]]
DecodeBatch = Callable[[List[bytes], np.ndarray], np.ndarray]


def split_chunks(tokens, chunk_tokens: int) -> Tuple[np.ndarray, np.ndarray]:
    toks = np.ascontiguousarray(tokens, dtype=np.int32)
    n_chunks = (len(toks) + chunk_tokens - 1) // chunk_tokens
    padded = np.zeros(n_chunks * chunk_tokens, dtype=np.int32)
    padded[: len(toks)] = toks
    ntok = np.full(n_chunks, chunk_tokens, dtype=np.int32)
    if n_chunks:
        ntok[-1] = len(toks) - (n_chunks - 1) * chunk_tokens
    return padded.reshape(n_chunks, chunk_tokens), ntok


def compress_sharded(tokens, chunk_tokens: int, batch_streams: int, encode_batch: EncodeBatch, prec: int, vocab: int,
                     device, tag: int = 0, group=None, quantiser: int = container.QUANT_LQ32) -> Optional[bytes]:
    """Every rank passes the SAME token array; rank r codes its batches; rank 0 returns the LACB file (None
    elsewhere).  One gather of the index and one of the payload, nothing inside the coding loop."""
    rank, world = _world(group)
    chunks, ntok = split_chunks(tokens, chunk_tokens)
    n_chunks = len(ntok)
    spans = batch_spans(n_chunks, batch_streams, world)
    b, e = spans[rank]
    streams: List[bytes] = []
    nbits: List[int] = []
    for c0 in range(b, e, batch_streams):
        c1 = min(e, c0 + batch_streams)
        bt = np.zeros((batch_streams, chunk_tokens), dtype=np.int32)   # padded to the full batch shape
        bn = np.zeros(batch_streams, dtype=np.int32)
        bt[: c1 - c0] = chunks[c0:c1]
        bn[: c1 - c0] = ntok[c0:c1]
        s, nb = encode_batch(bt, bn)
        streams += list(s[: c1 - c0])
        nbits += [int(x) for x in nb[: c1 - c0]]
    l_ntok = torch.from_numpy(ntok[b:e].astype(np.int64)).to(device)
    l_nbits = torch.tensor(nbits, dtype=torch.int64, device=device)
    g_ntok, g_nbits = gather_index(l_ntok, l_nbits, n_chunks, group, spans)
    payload = gather_payload(concat_streams(streams, device), g_nbits, n_chunks, 0, group, spans)
    if rank != 0:
        return None
    return container.pack_payload(payload, g_ntok.cpu().numpy(), g_nbits.cpu().numpy(), prec, vocab, chunk_tokens,
                                  quantiser, batch_streams, tag)


def _check_range(start, stop, total: int) -> Tuple[int, int]:
    for name, v in (("start", start), ("stop", stop)):
        if isinstance(v, bool) or not isinstance(v, numbers.Integral):
            raise ValueError(f"{name} must be an integer, got {v!r}")
    if not 0 <= start <= stop <= total:
        raise ValueError(f"token range [{start}, {stop}) is not inside the file's [0, {total}]")
    return int(start), int(stop)


def _plan(c: container.Container, start, stop) -> Tuple[np.ndarray, int, int]:
    """(first token of every chunk and the total, start, stop) after the bounds check."""
    first = np.zeros(c.n_chunks + 1, dtype=np.int64)
    np.cumsum(c.ntok, out=first[1:])
    start, stop = _check_range(start, first[-1] if stop is None else stop, int(first[-1]))
    return first, start, stop


def _want(c: container.Container, first: np.ndarray, start: int, stop: int) -> np.ndarray:
    """Tokens to decode per chunk: the prefix up to stop of every chunk that overlaps [start, stop), else 0."""
    want = np.minimum(c.ntok.astype(np.int64), np.maximum(stop - first[:-1], 0))
    want[first[1:] <= start] = 0
    return want


def decompress_sharded(blob: bytes, decode_batch: DecodeBatch, device, group=None, start: int = 0,
                       stop: Optional[int] = None) -> Optional[np.ndarray]:
    """Every rank passes the SAME file and range; rank 0 returns tokens[start:stop] (None elsewhere).  The default
    range is the whole file.

    Only the batches holding a chunk that overlaps [start, stop) are decoded, dealt contiguously over the ranks.  A
    needed chunk is decoded from its first token on, min(its length, stop - its first token) tokens of its stream;
    every other slot of the batch is an empty stream with 0 tokens.  The batch keeps its full shape, and the model
    keeps rows independent at a fixed shape, so a needed row sees the logits it saw when the file was written
    (tests/test_gpu_token_range.py).  A batch costs as many model steps as its longest needed prefix.  A chunk
    with no tokens overlaps no range and is never decoded."""
    rank, world = _world(group)
    c = container.unpack(blob)
    first, start, stop = _plan(c, start, stop)
    if start == stop:
        return np.zeros(0, dtype=np.int32) if rank == 0 else None
    want = _want(c, first, start, stop)
    needed = np.flatnonzero(want)
    B = c.batch_streams or max(c.n_chunks, 1)
    batches = np.unique(needed // B)
    # rank r decodes batches[b:e], (b, e) = chunk_range(len(batches), r, world), and holds the decoded rows of
    # needed[rows[b]:rows[e]]
    rows = np.append(np.searchsorted(needed // B, batches), len(needed))
    deal = [chunk_range(len(batches), r, world) for r in range(world)]
    spans = [(int(rows[b]), int(rows[e])) for b, e in deal]
    b, e = deal[rank]
    off = c.offsets()
    local = np.zeros((spans[rank][1] - spans[rank][0], c.chunk_tokens), dtype=np.int32)
    at = 0
    for k in batches[b:e]:
        c0, c1 = int(k) * B, min(c.n_chunks, (int(k) + 1) * B)
        bs = [c.payload[off[i]:off[i + 1]] if want[i] else b"" for i in range(c0, c1)] + [b""] * (B - (c1 - c0))
        bn = np.zeros(B, dtype=np.int32)
        bn[: c1 - c0] = want[c0:c1]
        got = decode_batch(bs, bn)[: c1 - c0][want[c0:c1] > 0]
        local[at:at + len(got)] = got
        at += len(got)
    got = gather_tokens(torch.from_numpy(local).to(device), len(needed), c.chunk_tokens, spans, 0, group)
    if rank != 0:
        return None
    got = got.cpu().numpy()
    flat = np.concatenate([got[j, : want[i]] for j, i in enumerate(needed)])
    return flat[start - first[needed[0]]:]


def pack_batches(want: np.ndarray, batch_streams: int, world: int) -> List[np.ndarray]:
    """The decode batches of a batch-invariant read: the chunks with want > 0, ordered by want descending (ties in
    chunk order) so that short prefixes do not wait in a batch with long ones.
      * More needed chunks than world x batch_streams: cut from the front into batches of batch_streams, so the
        shortest prefixes share the last batch (which the decoder runs at a smaller active size).  With one rank
        this is the least total of steps (the sum of every batch's longest prefix) any batching of <= S chunks
        reaches.
      * Otherwise: min(world, needed) balanced batches, none larger than ceil(needed / world) <= batch_streams,
        so every rank gets work while there are chunks for it."""
    needed = np.flatnonzero(want)
    order = needed[np.argsort(-want[needed], kind="stable")]
    if len(order) > world * batch_streams:
        return [order[b:b + batch_streams] for b in range(0, len(order), batch_streams)]
    n_batches = min(world, len(order))
    return [order[b:e] for b, e in (chunk_range(len(order), k, n_batches) for k in range(n_batches))]


def decompress_packed(blob: bytes, decode_batch: DecodeBatch, batch_streams: int, device, group=None,
                      start: int = 0, stop: Optional[int] = None) -> Optional[np.ndarray]:
    """decompress_sharded for a file of a batch-invariant predictor, whose rows do not depend on the batch they
    share: every rank passes the SAME file and range and its decoder's stream count; rank 0 returns
    tokens[start:stop] (None elsewhere).

    Each chunk that overlaps the range is decoded exactly once from its first token, for min(its length, stop -
    its first token) tokens.  pack_batches groups them into batches of at most batch_streams chunks, and batch k
    goes to rank k % world (longest batches first, so round robin also balances the steps).  decode_batch gets
    exactly the batch's streams; a batch costs as many model steps as its longest needed prefix.  The file's own
    batch_streams plays no part."""
    rank, world = _world(group)
    c = container.unpack(blob)
    first, start, stop = _plan(c, start, stop)
    if start == stop:
        return np.zeros(0, dtype=np.int32) if rank == 0 else None
    want = _want(c, first, start, stop)
    batches = pack_batches(want, int(batch_streams), world)
    mine = batches[rank::world]
    owned = [np.concatenate(batches[r::world]) if batches[r::world] else np.zeros(0, np.int64) for r in range(world)]
    spans, at = [], 0
    for o in owned:
        spans.append((at, at + len(o)))
        at += len(o)
    off = c.offsets()
    local = np.zeros((len(owned[rank]), c.chunk_tokens), dtype=np.int32)
    at = 0
    for ids in mine:
        got = decode_batch([c.payload[off[i]:off[i + 1]] for i in ids], want[ids].astype(np.int32))
        local[at:at + len(ids)] = got[: len(ids)]
        at += len(ids)
    got = gather_tokens(torch.from_numpy(local).to(device), spans[-1][1], c.chunk_tokens, spans, 0, group)
    if rank != 0:
        return None
    got = got.cpu().numpy()
    row = np.empty(c.n_chunks, dtype=np.int64)        # chunk -> its row in the gathered rank-order rows
    row[np.concatenate(owned)] = np.arange(spans[-1][1])
    needed = np.flatnonzero(want)
    flat = np.concatenate([got[row[i], : want[i]] for i in needed])
    return flat[start - first[needed[0]]:]
