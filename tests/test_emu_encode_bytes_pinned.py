"""Byte-exact pins of the emulated zstd encoder (tests/emu): SHA-1 digests of what the encoder's kernels produce for a
fixed set of inputs, at levels 1-3, with and without the frame checksum, in chunk mode and in frame mode (with history).

The digests were recorded before the literal and sequence-code histograms moved into the parse kernel and the pack
kernel began to size its sequence bitstream from the chain walk's per-block sums.  Neither change may alter a byte:
any optimisation of the entropy stages must leave these digests as they are.  Unlike the oracle-parity checks
(check_util.py), which accept any parse the entropy stage encodes faithfully, these pins catch a changed parse too.

Run this file as a script to print the current digests."""
import hashlib

import numpy as np
import pytest

import helpers as H
from emu_util import emu_encode, emu_encode_frames


def _corpus():
    return [H.golden("e.txt"), H.golden("twain.txt"), H.golden("html.txt")]


def _chunk_inputs(level):
    block = 65536 if level == 1 else 131072
    chunks = [d[i:i + block] for d in _corpus() for i in range(0, len(d), block)]
    rnd = np.random.Generator(np.random.PCG64(20261017)).integers(0, 256, 65536, dtype=np.uint8).tobytes()
    tw = H.golden("twain.txt")
    # edge chunks: empty, one byte, all zeros, incompressible, and 64 KiB + 1 (too big at level 1, a normal block above)
    return chunks + [b"", b"x", bytes(65536), rnd, tw[:65537]]


def _frame_inputs():
    e, tw, html = _corpus()
    # multi-block frames (the later blocks see the earlier ones as history), a frame of one short block, an empty frame
    return [tw, e, html + html, tw[:1000], b""]


def _sha(*parts):
    h = hashlib.sha1()
    for p in parts:
        h.update(p if isinstance(p, (bytes, bytearray)) else np.ascontiguousarray(p).tobytes())
    return h.hexdigest()


def chunk_digests(E, level, flags):
    """(output digest, parse-dump digest) of chunk mode: every frame, every output size, and the debug dump the
    device's debug entry point returns (per chunk header, sequences, literals)."""
    chunks = _chunk_inputs(level)
    frames, outs, hdr, seqs, lits = emu_encode(E, chunks, flags=flags, level=level)
    out = _sha(outs.astype(np.int64), *frames)
    dump = _sha(hdr, *(seqs[i, :min(int(hdr[i, 0]), seqs.shape[1])] for i in range(len(chunks))),
                *(lits[i, :int(hdr[i, 1])] for i in range(len(chunks)) if int(hdr[i, 2]) == 0))
    return out, dump


def frame_digest(E, level, crc):
    frames, blocks, _ = emu_encode_frames(E, _frame_inputs(), level=level, crc=crc, dump=False)
    return _sha(np.array([len(f) for f in frames], dtype=np.int64), *frames)


CHUNK_PINS = {
    (1, 3): ("d019a98c0f8f067ece8471d5988e62b6dd41d905", "02e78ed93e1bb0cf93f69e740c26fc7c4205d6b4"),
    (1, 2): ("c81b42dce00a946cb7c612045740930c0b3090b4", "02e78ed93e1bb0cf93f69e740c26fc7c4205d6b4"),
    (2, 3): ("a51a4ef87bdec8b4d641cf222df58e38e3d8c553", "91ecaba074715e89ad441002f38e1ebd3520b892"),
    (2, 2): ("49766ffa7ed4e646d4ae709030bae22b82c0dd87", "91ecaba074715e89ad441002f38e1ebd3520b892"),
    (3, 3): ("69801ce11e99cdcf63fe17ef7125c59c0df0f723", "1458a5d45595b8b32f01e67a7bdf0a2e6230bd62"),
    (3, 2): ("837728dbc7f4761f47163d1c71191b630b0d6e89", "1458a5d45595b8b32f01e67a7bdf0a2e6230bd62"),
}
FRAME_PINS = {
    (1, True): "3103fa2b79d26e20a8aefbda21d759f422e55b21",
    (1, False): "dd810df6687af8cd8868ef0291a2b0ef159c4be3",
    (2, True): "0deee32269784ad46270d5e3945329aa5ab60a92",
    (2, False): "3d34a53e5e31b71d5559f60d2d169162e4536e6d",
    (3, True): "55aaa6a3022e58d8ba2ffc6ba749a1a7082d7a84",
    (3, False): "f6d872d913bf9d39ce3ecd799bd1a5c3f5be265b",
}


@pytest.mark.parametrize("level,flags", sorted(CHUNK_PINS), ids=lambda v: str(v))
def test_chunk_mode_bytes_pinned(emu_lib, level, flags):
    assert chunk_digests(emu_lib, level, flags) == CHUNK_PINS[(level, flags)]


@pytest.mark.parametrize("level,crc", sorted(FRAME_PINS), ids=lambda v: str(v))
def test_frame_mode_bytes_pinned(emu_lib, level, crc):
    assert frame_digest(emu_lib, level, crc) == FRAME_PINS[(level, crc)]


if __name__ == "__main__":
    E = H.emu()
    for k in sorted(CHUNK_PINS):
        print("chunk", k, chunk_digests(E, *k))
    for k in sorted(FRAME_PINS):
        print("frame", k, frame_digest(E, *k))
