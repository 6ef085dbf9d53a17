"""Chunk / stream container ("LACB" v2): the framing the reference lacks.

The reference has no file format: A_from_bin keeps emitting symbols while its bit window allows
(arith_code.py:322-326) and ACSampler's demo loops until the bits run out
(arithmetic_coding.py:288-300), so token counts must travel next to the bitstreams.  Text is cut
into independent chunks (streams); each chunk is one coder stream with its own flush.

Layout (little endian):
    0   4  magic  b"LACB"
    4   2  version (2)
    6   1  precision of the coder (AC(..., prec))
    7   1  quantiser id (2 = LQ32 block-form tables on a fixed total 2^32, 0 = caller-supplied tables)
    8   4  vocabulary size
    12  4  nominal tokens per chunk
    16  8  number of chunks N
    24  8  total tokens
    32  4  streams per model batch (chunks are coded in batches of exactly this many streams, the last batch padded
           with empty streams, so the predictor sees the same batch shape when decoding -- on any number of GPUs).
           It binds torch-mode files only: a batch-invariant predictor's file (model tag of a `:bi` configuration)
           decodes at any batch size, and there the field is informational
    36  4  model tag (CRC-32 of the predictor's configuration string; 0 = unspecified)
    40  N x (uint32 tokens in chunk, uint32 bits in chunk)      -- the index
    ..  chunk payloads, each byte aligned ((bits + 7) // 8 bytes), in chunk order
"""
from __future__ import annotations

import struct
import zlib
from dataclasses import dataclass
from typing import List, Sequence

import numpy as np

MAGIC = b"LACB"
VERSION = 2
HEADER = struct.Struct("<4sHBBIIQQII")
QUANT_TABLES = 0
QUANT_LQ32 = 2  # (1 was the round-1 row-reference form of LQ32, no longer produced or read)


def model_tag(config: str) -> int:
    return zlib.crc32(config.encode("utf-8")) & 0xFFFFFFFF


@dataclass
class Container:
    prec: int
    quantiser: int
    vocab: int
    chunk_tokens: int
    ntok: np.ndarray      # uint32 [N]
    nbits: np.ndarray     # uint32 [N]
    payload: bytes        # concatenated chunk bytes
    batch_streams: int = 0
    tag: int = 0

    @property
    def n_chunks(self) -> int:
        return len(self.ntok)

    def offsets(self) -> np.ndarray:
        """Byte offsets of the chunks inside payload, int64 [N + 1]."""
        off = np.zeros(self.n_chunks + 1, dtype=np.int64)
        np.cumsum((self.nbits.astype(np.int64) + 7) // 8, out=off[1:])
        return off

    def streams(self) -> List[bytes]:
        off = self.offsets()
        return [self.payload[off[i]:off[i + 1]] for i in range(self.n_chunks)]


def pack(streams: Sequence[bytes], ntok: Sequence[int], nbits: Sequence[int], prec: int, vocab: int,
         chunk_tokens: int, quantiser: int = QUANT_LQ32, batch_streams: int = 0, tag: int = 0) -> bytes:
    ntok = np.asarray(ntok, dtype=np.uint32)
    nbits = np.asarray(nbits, dtype=np.uint32)
    if not (len(streams) == len(ntok) == len(nbits)):
        raise ValueError("streams, ntok and nbits must have the same length")
    for i, s in enumerate(streams):
        if len(s) != (int(nbits[i]) + 7) // 8:
            raise ValueError(f"chunk {i}: {len(s)} bytes for {int(nbits[i])} bits")
    head = HEADER.pack(MAGIC, VERSION, prec, quantiser, vocab, chunk_tokens, len(streams),
                       int(ntok.sum(dtype=np.uint64)), batch_streams, tag)
    index = np.stack([ntok, nbits], axis=1).astype("<u4").tobytes()
    return head + index + b"".join(streams)


def pack_payload(payload: bytes, ntok, nbits, prec: int, vocab: int, chunk_tokens: int,
                 quantiser: int = QUANT_LQ32, batch_streams: int = 0, tag: int = 0) -> bytes:
    """Same file from an already concatenated payload (what the multi-rank gather delivers)."""
    ntok = np.asarray(ntok, dtype=np.uint32)
    nbits = np.asarray(nbits, dtype=np.uint32)
    if len(payload) != int(((nbits.astype(np.int64) + 7) // 8).sum()):
        raise ValueError("payload length does not match the index")
    head = HEADER.pack(MAGIC, VERSION, prec, quantiser, vocab, chunk_tokens, len(ntok),
                       int(ntok.sum(dtype=np.uint64)), batch_streams, tag)
    return head + np.stack([ntok, nbits], axis=1).astype("<u4").tobytes() + bytes(payload)


def unpack(blob: bytes) -> Container:
    if len(blob) < 6:
        raise ValueError("truncated container")
    magic, ver = struct.unpack_from("<4sH", blob, 0)
    if magic != MAGIC:
        raise ValueError("not a LACB container")
    if ver != VERSION:
        raise ValueError(f"LACB version {ver} is not supported (this build reads version {VERSION})")
    if len(blob) < HEADER.size:
        raise ValueError("truncated container")
    magic, ver, prec, quant, vocab, chunk_tokens, n, total, batch_streams, tag = HEADER.unpack_from(blob, 0)
    idx_end = HEADER.size + 8 * n
    if len(blob) < idx_end:
        raise ValueError("truncated index")
    index = np.frombuffer(blob, dtype="<u4", count=2 * n, offset=HEADER.size).reshape(n, 2)
    c = Container(prec, quant, vocab, chunk_tokens, index[:, 0].copy(), index[:, 1].copy(), bytes(blob[idx_end:]),
                  batch_streams, tag)
    if int(c.ntok.sum(dtype=np.uint64)) != total:
        raise ValueError("index does not add up to the total token count")
    if len(c.payload) != int(c.offsets()[-1]):
        raise ValueError("payload length does not match the index")
    return c
