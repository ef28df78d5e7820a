"""Host-side mirror of the reference's zstd encoder / decoder interface for the accelerated path.

Names follow klauspost/compress/zstd: ``Encoder.EncodeAll`` (zstd/encoder.go:722),
``Encoder.MaxEncodedSize`` (:843), levels ``SpeedFastest``/``SpeedDefault``
(zstd/encoder_options.go), ``WithEncoderCRC``; ``Decoder.DecodeAll`` (zstd/decoder.go:319) with the package's
error values (zstd/zstd.go:40-96).  The work is done by libb200comp.so
(hand-written sm_100a kernels) through the C ABI in include/b2c.h; PyTorch is only the owner of
device buffers and streams.
"""
import ctypes

import numpy as np
import torch

from . import _lib
from ._lib import lib, check, B2CError

SpeedFastest = 1
SpeedDefault = 2
SpeedBetterCompression = 3
CHUNK = 1 << 16           # SpeedFastest block size, zstd/encoder_options.go:248-252
SLOT = CHUNK + 512        # per-chunk output slot (>= MaxEncodedSize(CHUNK))
BLOCK = {SpeedFastest: 1 << 16, SpeedDefault: 128 << 10, SpeedBetterCompression: 128 << 10}   # zstd/encoder_options.go:41,248-252
FLAG_CRC = 1
FLAG_FRAME = 2


class Encoder:
    """zstd.Encoder on one B200: batches of independent blocks (one-block frames: encode_device / encode_chunks /
    encode_packed) and frame mode (encode_frames / EncodeAll: one multi-block frame per input, blocks with history).
    padding: WithEncoderPadding -- EncodeAll output and a Writer's total are brought to a multiple of it with a skippable
    frame (zstd/encoder_options.go, zstd/frameenc.go:96-137)."""

    def __init__(self, level=SpeedFastest, crc=True, device=0, max_chunks=4096, padding=0):
        if not torch.cuda.is_available() or lib.b2c_device_count() == 0:
            raise B2CError("no CUDA device: compress_b200 has no CPU fallback")
        if level not in BLOCK:
            raise B2CError("levels on the GPU path: SpeedFastest, SpeedDefault, SpeedBetterCompression")
        self.level = level
        self.block = BLOCK[level]
        self.slot = self.block + 512
        self.flags = (FLAG_CRC if crc else 0) | FLAG_FRAME
        self.device = device
        self.max_chunks = max_chunks
        if padding < 0 or padding > 1 << 30:
            raise B2CError("padding must be in [0, 1 GiB]")
        self.padding = padding
        self._ctx = lib.b2c_ctx_create(device, max_chunks)
        if not self._ctx:
            raise B2CError("b2c_ctx_create failed")

    def close(self):
        if self._ctx:
            lib.b2c_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self):
        return int(lib.b2c_launch_count(self._ctx))

    @property
    def sm_count(self):
        return int(lib.b2c_sm_count(self._ctx))

    # profile slots of b2c_profile_read.  The histograms are counted inside the parse kernel, so the
    # "b2c_zstd_hist_kernel" slot is an empty interval (about 0 ms); the key stays so that readers of the profile keep working.
    KERNELS = ("b2c_zstd_xxh_kernel", "b2c_lz_parse_kernel", "b2c_zstd_hist_kernel", "b2c_zstd_tables_kernel",
               "b2c_zstd_chains_kernel", "b2c_zstd_pack_kernel")

    def profile(self, on=True):
        check(lib.b2c_profile_enable(self._ctx, 1 if on else 0), self._ctx)

    def profile_read(self):
        """-> ({kernel name: summed ms}, encode calls) since profile(True); synchronises the device."""
        ms = (ctypes.c_double * 6)()
        nc = ctypes.c_uint32(0)
        check(lib.b2c_profile_read(self._ctx, ms, ctypes.byref(nc)), self._ctx)
        return {k: float(ms[i]) for i, k in enumerate(self.KERNELS)}, int(nc.value)

    def MaxEncodedSize(self, size):
        return int(lib.b2c_zstd_bound(size, self.level))

    # ---- device-resident batch -------------------------------------------------------------
    def encode_device(self, src, sizes=None, chunk=None, dst=None, out_sizes=None, flags=None):
        """src: uint8 CUDA tensor holding nchunks chunks at stride `chunk` bytes (default: the level's block size).
        sizes: optional uint32 CUDA tensor (per-chunk sizes); default all `chunk` bytes.
        Returns (dst [nchunks, slot] uint8, out_sizes [nchunks] int64), both on the device. Async."""
        assert src.is_cuda and src.dtype == torch.uint8
        chunk = self.block if chunk is None else chunk
        SLOT = self.slot
        nchunks = src.numel() // chunk if sizes is None else sizes.numel()
        if dst is None:
            dst = torch.empty((nchunks, SLOT), dtype=torch.uint8, device=src.device)
        if out_sizes is None:
            out_sizes = torch.empty((nchunks,), dtype=torch.int64, device=src.device)
        stream = torch.cuda.current_stream(src.device).cuda_stream
        rc = lib.b2c_zstd_encode_device(
            self._ctx, self.level, self.flags if flags is None else flags, src.data_ptr(), chunk,
            None if sizes is None else sizes.data_ptr(), chunk, dst.data_ptr(), SLOT, out_sizes.data_ptr(),
            nchunks, ctypes.c_void_p(stream))
        check(rc, self._ctx)
        return dst, out_sizes

    def encode_device_debug(self, src, sizes=None, chunk=None, flags=None, seq_cap=None):
        """Like encode_device but also returns the parse (sequence triples + literals) per chunk."""
        chunk = self.block if chunk is None else chunk
        SLOT = self.slot
        seq_cap = self.block // 4 + 64 if seq_cap is None else seq_cap
        nchunks = src.numel() // chunk if sizes is None else sizes.numel()
        dev = src.device
        dst = torch.empty((nchunks, SLOT), dtype=torch.uint8, device=dev)
        out_sizes = torch.empty((nchunks,), dtype=torch.int64, device=dev)
        hdr = torch.zeros((nchunks, 4), dtype=torch.int32, device=dev)
        seqs = torch.zeros((nchunks, seq_cap, 3), dtype=torch.int32, device=dev)
        lits = torch.zeros((nchunks, self.block), dtype=torch.uint8, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib.b2c_zstd_encode_device_debug(
            self._ctx, self.level, self.flags if flags is None else flags, src.data_ptr(), chunk,
            None if sizes is None else sizes.data_ptr(), chunk, dst.data_ptr(), SLOT, out_sizes.data_ptr(), nchunks,
            hdr.data_ptr(), seqs.data_ptr(), lits.data_ptr(), seq_cap, ctypes.c_void_p(stream))
        check(rc, self._ctx)
        return dst, out_sizes, hdr, seqs, lits

    # ---- host buffers (what the cgo shim calls) -----------------------------------------------
    def encode_chunks(self, chunks):
        """chunks: list of bytes-like (each at most the level's block size).  Returns list of encoded frames (bytes)."""
        n = len(chunks)
        if n == 0:
            return []
        bufs = [np.frombuffer(c, dtype=np.uint8) if len(c) else np.zeros(0, dtype=np.uint8) for c in chunks]
        outs = [np.empty(self.MaxEncodedSize(len(c)) + 16, dtype=np.uint8) for c in chunks]
        srcs = (ctypes.c_void_p * n)(*[b.ctypes.data for b in bufs])
        ssz = (ctypes.c_size_t * n)(*[len(c) for c in chunks])
        dsts = (ctypes.c_void_p * n)(*[o.ctypes.data for o in outs])
        dcap = (ctypes.c_size_t * n)(*[o.size for o in outs])
        res = (ctypes.c_int64 * n)()
        rc = lib.b2c_zstd_encode_chunks(self._ctx, self.level, self.flags, srcs, ssz, dsts, dcap, res, n)
        check(rc, self._ctx)
        out = []
        for i in range(n):
            if res[i] < 0:
                raise B2CError(f"chunk {i}: {lib.b2c_strerror(int(res[i])).decode()}")
            out.append(outs[i][: res[i]].tobytes())
        return out

    def encode_packed(self, src, dst=None, chunk=None):
        """src: contiguous host buffer (bytes / numpy / CPU torch tensor, ideally pinned).  Returns
        (dst uint8 tensor (pinned), total, sizes int64 ndarray, offsets uint64 ndarray): dst[:total] is the
        concatenation of one frame per `chunk` bytes of src."""
        if isinstance(src, torch.Tensor):
            assert not src.is_cuda and src.dtype == torch.uint8 and src.is_contiguous()
            sptr, nbytes = src.data_ptr(), src.numel()
        else:
            arr = np.frombuffer(src, dtype=np.uint8)
            sptr, nbytes = arr.ctypes.data, arr.size
        chunk = self.block if chunk is None else chunk
        nchunks = max(1, (nbytes + chunk - 1) // chunk)
        cap = nbytes + nchunks * 32 + 64
        if dst is None:
            dst = torch.empty(cap, dtype=torch.uint8, pin_memory=True)
        sizes = np.empty(nchunks, dtype=np.int64)
        offs = np.empty(nchunks, dtype=np.uint64)
        total = ctypes.c_size_t(0)
        rc = lib.b2c_zstd_encode_packed(self._ctx, self.level, self.flags, sptr, nbytes, chunk, dst.data_ptr(),
                                        dst.numel(), sizes.ctypes.data, offs.ctypes.data, ctypes.byref(total))
        check(rc, self._ctx)
        return dst, int(total.value), sizes, offs

    # ---- frame mode: one frame per input of any size (the multi-block branch of encodeAll, zstd/encoder.go:796-830) ----
    def FrameBound(self, size):
        return int(lib.b2c_zstd_frame_bound(size, self.level))

    def encode_frames_device(self, src, offsets, sizes, dst=None):
        """src: uint8 CUDA tensor; frame f = sizes[f] bytes at src[offsets[f]:] (host sequences of ints).  Every frame's
        blocks see the bytes before them (history) and are encoded in parallel.  Returns (dst uint8 CUDA tensor,
        frame_offsets uint64 CUDA tensor, frame_sizes int64 CUDA tensor): frame f is dst[off[f] : off[f] + size[f]].  Async."""
        assert src.is_cuda and src.dtype == torch.uint8
        n = len(sizes)
        offs = np.ascontiguousarray(offsets, dtype=np.uint64)
        lens = np.ascontiguousarray(sizes, dtype=np.uint64)
        if dst is None:
            cap = sum(self.FrameBound(int(x)) for x in lens) + 64
            dst = torch.empty(cap, dtype=torch.uint8, device=src.device)
        foff = torch.empty(n, dtype=torch.uint64, device=src.device)
        fsz = torch.empty(n, dtype=torch.int64, device=src.device)
        stream = torch.cuda.current_stream(src.device).cuda_stream
        rc = lib.b2c_zstd_encode_frames_device(self._ctx, self.level, self.flags & FLAG_CRC, src.data_ptr(), offs.ctypes.data,
                                               lens.ctypes.data, n, dst.data_ptr(), dst.numel(), foff.data_ptr(),
                                               fsz.data_ptr(), ctypes.c_void_p(stream))
        check(rc, self._ctx)
        return dst, foff, fsz

    def encode_frames(self, inputs):
        """inputs: list of bytes-like of any size.  Returns one zstd frame (bytes) per input: Encoder.EncodeAll applied to
        each, all blocks of all inputs in one device batch."""
        n = len(inputs)
        if n == 0:
            return []
        bufs = [np.frombuffer(c, dtype=np.uint8) if len(c) else np.zeros(0, dtype=np.uint8) for c in inputs]
        outs = [np.empty(self.FrameBound(len(c)) + 16, dtype=np.uint8) for c in inputs]
        srcs = (ctypes.c_void_p * n)(*[b.ctypes.data for b in bufs])
        ssz = (ctypes.c_size_t * n)(*[len(c) for c in inputs])
        dsts = (ctypes.c_void_p * n)(*[o.ctypes.data for o in outs])
        dcap = (ctypes.c_size_t * n)(*[o.size for o in outs])
        res = (ctypes.c_int64 * n)()
        rc = lib.b2c_zstd_encode_frames(self._ctx, self.level, self.flags & FLAG_CRC, srcs, ssz, dsts, dcap, res, n)
        check(rc, self._ctx)
        out = []
        for i in range(n):
            if res[i] < 0:
                raise B2CError(f"input {i}: {lib.b2c_strerror(int(res[i])).decode()}")
            out.append(outs[i][: res[i]].tobytes())
        return out

    def EncodeAll(self, src, dst=None, single_frame=True):
        """EncodeAll will encode all input in src and append it to dst (zstd/encoder.go:715-729).  As in the reference the
        result is ONE frame (content size in the header, one checksum); single_frame=False gives round 1's stream of
        independent one-block frames instead (a valid zstd stream of the same content, zstd/encoder.go:719)."""
        src = bytes(src)
        if single_frame:
            out = self.encode_frames([src])[0]
        else:
            buf, total, _, _ = self.encode_packed(src)
            out = bytes(buf[:total].numpy())
        if self.padding:
            out = skippableFrame(out, calcSkippableFrame((len(dst) if dst is not None else 0) + len(out), self.padding))
        if dst is not None:
            dst += out
            return dst
        return out


class Writer:
    """The streaming face of zstd.Encoder (Write / Flush / Close, zstd/encoder.go:123-260) over frame mode: bytes written
    are gathered and leave as complete frames -- one per Flush / Close, or every `frame_bytes` of input -- each a multi-block
    frame whose blocks see their history.  Concatenated frames are one valid zstd stream (zstd/encoder.go:719)."""

    def __init__(self, w, level=SpeedFastest, crc=True, device=0, frame_bytes=None, encoder=None, padding=0):
        """frame_bytes: input bytes per frame; default four frame-mode blocks (192 KiB at SpeedFastest, 384 KiB above), the
        longest frames the staged GPU decoder takes on its fast path (DESIGN.md section 4).  encoder: an Encoder to share
        (its level and checksum setting apply); by default the writer owns one."""
        self._w = w
        self._enc = encoder if encoder is not None else Encoder(level=level, crc=crc, device=device, max_chunks=64,
                                                                padding=padding)
        self._own = encoder is None
        self._buf = bytearray()
        self._frame_bytes = frame_bytes if frame_bytes else 4 * (49152 if level == SpeedFastest else 98304)
        self._wrote = False
        self._nwritten = 0

    def Reset(self, w):
        """Discard pending state and write to w from now on, keeping the device context (zstd/encoder.go:100-121)."""
        self._w = w
        self._buf = bytearray()
        self._wrote = False
        self._nwritten = 0

    def _put(self, frame):
        self._w.write(frame)
        self._nwritten += len(frame)
        self._wrote = True

    def Write(self, p):
        self._buf += p
        while len(self._buf) >= self._frame_bytes:
            self._emit(self._frame_bytes)
        return len(p)

    def ReadFrom(self, r):
        """Encode everything r yields until EOF (frames leave as they fill); returns the byte count; does not close
        (zstd/encoder.go:203-260)."""
        n = 0
        while True:
            chunk = r.read(self._frame_bytes)
            if not chunk:
                return n
            n += len(chunk)
            self.Write(chunk)

    def _emit(self, n):
        part = bytes(self._buf[:n])
        del self._buf[:n]
        self._put(self._enc.encode_frames([part])[0])

    def Flush(self):
        if self._buf:
            self._emit(len(self._buf))

    def Close(self):
        self.Flush()
        if not self._wrote:          # an empty stream is still a frame (WithZeroFrames, zstd/encoder.go:732-751)
            self._put(self._enc.encode_frames([b""])[0])
        pad = getattr(self._enc, "padding", 0)
        if pad:                      # WithEncoderPadding: the stream's total becomes a multiple (zstd/encoder.go Close)
            self._put(skippableFrame(b"", calcSkippableFrame(self._nwritten, pad)))
        if self._own:
            self._enc.close()


# ---- decoder ------------------------------------------------------------------------------------
class ZstdError(B2CError):
    """Decode error; ``code`` is the C-ABI error code, ``str`` the reference's message class."""

    def __init__(self, code):
        self.code = int(code)
        super().__init__(lib.b2c_strerror(self.code).decode())


ErrMagicMismatch = -7
ErrWindowSizeExceeded = -8
ErrCRCMismatch = -9
ErrFrameSizeMismatch = -10
ErrCorrupt = -5
ErrDecoderSizeExceeded = -4


class Decoder:
    """zstd.Decoder for batches of independent streams on one B200 (staged kernels; a one-warp decoder for the rest)."""

    def __init__(self, device=0, max_decoded=64 << 20):
        if not torch.cuda.is_available() or lib.b2c_device_count() == 0:
            raise B2CError("no CUDA device: compress_b200 has no CPU fallback")
        self.device = device
        self.max_decoded = max_decoded       # WithDecoderMaxMemory analogue for DecodeAll without a known size
        self._ctx = lib.b2c_ctx_create(device, 0)
        if not self._ctx:
            raise B2CError("b2c_ctx_create failed")

    def close(self):
        if self._ctx:
            lib.b2c_ctx_destroy(self._ctx)
            self._ctx = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    @property
    def launches(self):
        return int(lib.b2c_launch_count(self._ctx))

    DECODE_KERNELS = ("b2c_zstd_dec_scan_kernel", "b2c_zstd_dec_lit_kernel", "b2c_zstd_dec_seq_kernel", "b2c_zstd_dec_exec_kernel",
                      "b2c_zstd_dec_xxh_kernel", "b2c_zstd_decode_kernel")

    def profile(self, on=True):
        check(lib.b2c_decode_profile_enable(self._ctx, 1 if on else 0), self._ctx)

    def profile_read(self):
        """-> {kernel name: summed ms} of the decode launches since profile(True)."""
        ms = (ctypes.c_double * 6)()
        check(lib.b2c_decode_profile_read(self._ctx, ms), self._ctx)
        return {k: float(ms[i]) for i, k in enumerate(self.DECODE_KERNELS)}

    def staged_count(self, n):
        """Of the first n inputs of the most recent decode launch: how many the staged kernels completed."""
        k = ctypes.c_uint32(0)
        check(lib.b2c_decode_staged_count(self._ctx, n, ctypes.byref(k)), self._ctx)
        return int(k.value)

    def decode_device(self, src, src_sizes, src_offsets=None, src_stride=0, dst=None, dst_cap=CHUNK, dst_offsets=None,
                      out_sizes=None, dst_stride=None):
        """src: uint8 CUDA tensor; stream i is src[off_i : off_i + src_sizes[i]] with off_i = src_offsets[i]
        (uint64/int64 CUDA tensor) or i*src_stride.  Output i goes to dst[i*dst_cap ...] (or dst_offsets[i]),
        at most dst_cap bytes.  Returns (dst, out_sizes int64 CUDA tensor: bytes or negative error).  Async."""
        assert src.is_cuda and src.dtype == torch.uint8
        n = src_sizes.numel()
        dev = src.device
        if dst is None:
            dst = torch.empty((n, dst_cap), dtype=torch.uint8, device=dev)
        if out_sizes is None:
            out_sizes = torch.empty((n,), dtype=torch.int64, device=dev)
        stream = torch.cuda.current_stream(dev).cuda_stream
        rc = lib.b2c_zstd_decode_device(
            self._ctx, src.data_ptr(), src_stride, None if src_offsets is None else src_offsets.data_ptr(),
            src_sizes.data_ptr(), dst.data_ptr(), dst_cap if dst_stride is None else dst_stride, None if dst_offsets is None else dst_offsets.data_ptr(),
            dst_cap, out_sizes.data_ptr(), n, ctypes.c_void_p(stream))
        check(rc, self._ctx)
        return dst, out_sizes

    def decode_chunks(self, streams, caps=None):
        """streams: list of bytes-like zstd streams.  Returns (list of bytes or None, list of codes)."""
        n = len(streams)
        if n == 0:
            return [], []
        if caps is None:
            caps = [self.max_decoded] * n
        bufs = [np.frombuffer(bytes(c), dtype=np.uint8) if len(c) else np.zeros(0, dtype=np.uint8) for c in streams]
        outs = [np.empty(max(int(cp), 1), dtype=np.uint8) for cp in caps]
        srcs = (ctypes.c_void_p * n)(*[b.ctypes.data for b in bufs])
        ssz = (ctypes.c_size_t * n)(*[len(c) for c in streams])
        dsts = (ctypes.c_void_p * n)(*[o.ctypes.data for o in outs])
        dcap = (ctypes.c_size_t * n)(*[int(cp) for cp in caps])
        res = (ctypes.c_int64 * n)()
        rc = lib.b2c_zstd_decode_chunks(self._ctx, srcs, ssz, dsts, dcap, res, n)
        check(rc, self._ctx)
        codes = [int(r) for r in res]
        return [outs[i][:codes[i]].tobytes() if codes[i] >= 0 else None for i in range(n)], codes

    def DecodeAll(self, input, dst=None, size_hint=None):
        """DecodeAll decodes a full zstd stream and appends it to dst (zstd/decoder.go:311-385)."""
        cap = self.max_decoded if size_hint is None else size_hint
        outs, codes = self.decode_chunks([input], [cap])
        if codes[0] < 0:
            raise ZstdError(codes[0])
        if dst is not None:
            dst += outs[0]
            return dst
        return outs[0]


# ---- stream reader (zstd.NewReader over an io.Reader) ---------------------------------------------------------------
FRAME_MAGIC = 0xFD2FB528
SKIPPABLE_MAGIC = 0x184D2A50          # .. 0x184D2A5F (zstd/framedec.go:49-50)
MIN_WINDOW = 1 << 10                  # MinWindowSize, zstd/zstd.go
MAX_BLOCK = 128 << 10                 # maxCompressedBlockSize, zstd/blockdec.go:41-45
ErrReservedBit = ErrCorrupt
ErrUnexpectedEOF = -5


HeaderMaxSize = 14 + 3                 # zstd/decodeheader.go:13


class ErrUnexpectedEOFHeader(B2CError):
    """io.ErrUnexpectedEOF from Header.Decode: the input ends inside the header."""


def frame_header_bytes(content_size, window_size=0, single_segment=False, checksum=False, dict_id=0):
    """frameHeader.appendTo (zstd/frameenc.go:25-92): magic, descriptor, window byte unless single segment, dictionary id,
    content size in the shortest of the 0/1/2/4/8-byte forms (frames < 256 bytes store none unless single segment)."""
    fhd = (4 if checksum else 0) | (0x20 if single_segment else 0)
    did = b""
    if dict_id > 0:
        if dict_id < 256:
            fhd |= 1; did = bytes([dict_id])
        elif dict_id < 1 << 16:
            fhd |= 2; did = dict_id.to_bytes(2, "little")
        else:
            fhd |= 3; did = dict_id.to_bytes(4, "little")
    fcs = (content_size >= 256) + (content_size >= 65536 + 256) + (content_size >= 0xFFFFFFFF)
    fhd |= fcs << 6
    out = bytearray(b"\x28\xb5\x2f\xfd")
    out.append(fhd)
    if not single_segment:
        out.append(((max(int(window_size) - 1, 0).bit_length() - 10) << 3) & 0xFF)
    out += did
    if fcs == 0:
        if single_segment:
            out.append(content_size & 0xFF)
    elif fcs == 1:
        out += (content_size - 256).to_bytes(2, "little")
    elif fcs == 2:
        out += content_size.to_bytes(4, "little")
    else:
        out += content_size.to_bytes(8, "little")
    return bytes(out)


def calcSkippableFrame(written, want_multiple):
    """Bytes to add so that `written` becomes a multiple of want_multiple: 0, or a total >= 8 (a skippable frame's header)
    (zstd/frameenc.go:96-116)."""
    if want_multiple <= 0:
        raise ValueError("wantMultiple <= 0")
    if written < 0:
        raise ValueError("written < 0")
    left = written % want_multiple
    if left == 0:
        return 0
    add = want_multiple - left
    while add < 8:
        add += want_multiple
    return add


def skippableFrame(dst, total, fill=None):
    """Append a skippable frame of `total` bytes in all (zstd/frameenc.go:118-137); its content comes from fill(n) -> bytes
    (default os.urandom, the reference's crypto/rand.Reader)."""
    if total == 0:
        return dst
    if total < 8:
        raise ValueError("requested skippable frame (%d) < 8" % total)
    if total > 0xFFFFFFFF:
        raise ValueError("requested skippable frame (%d) > max uint32" % total)
    import os
    body = (fill or os.urandom)(total - 8)
    if len(body) != total - 8:
        raise ErrUnexpectedEOFHeader("short read filling a skippable frame")
    return dst + b"\x50\x2a\x4d\x18" + (total - 8).to_bytes(4, "little") + body


class Header:
    """zstd.Header (zstd/decodeheader.go:15-76): what the first bytes of a frame say, without decoding anything."""

    class Block:
        __slots__ = ("OK", "Last", "Compressed", "DecompressedSize", "CompressedSize")

        def __init__(self):
            self.OK = self.Last = self.Compressed = False
            self.DecompressedSize = self.CompressedSize = 0

    def __init__(self):
        self._clear()

    def _clear(self):
        self.SingleSegment = False
        self.WindowSize = 0
        self.DictionaryID = 0
        self.HasFCS = False
        self.FrameContentSize = 0
        self.Skippable = False
        self.SkippableID = 0
        self.SkippableSize = 0
        self.HeaderSize = 0
        self.FirstBlock = Header.Block()
        self.HasCheckSum = False

    def Decode(self, data):
        """Header.Decode (zstd/decodeheader.go:78-86); at least HeaderMaxSize bytes give every field."""
        self.DecodeAndStrip(data)

    def DecodeAndStrip(self, data):
        """-> the bytes after the header (zstd/decodeheader.go:88-229).  ErrUnexpectedEOFHeader when the input ends inside
        the header, ZstdError(ErrMagicMismatch / ErrReservedBit) as the reference."""
        self._clear()
        b = bytes(data)
        if len(b) < 4:
            raise ErrUnexpectedEOFHeader("unexpected EOF")
        self.HeaderSize = 4
        if b[:4] != b"\x28\xb5\x2f\xfd":
            if b[1:4] != b"\x2a\x4d\x18" or b[0] & 0xF0 != 0x50:
                raise ZstdError(ErrMagicMismatch)
            if len(b) < 8:
                raise ErrUnexpectedEOFHeader("unexpected EOF")
            self.HeaderSize = 8
            self.Skippable = True
            self.SkippableID = b[0] & 0xF
            self.SkippableSize = int.from_bytes(b[4:8], "little")
            return b[8:]
        p = 4
        if len(b) <= p:
            raise ErrUnexpectedEOFHeader("unexpected EOF")
        fhd = b[p]; p += 1
        self.SingleSegment = bool(fhd & 0x20)
        self.HasCheckSum = bool(fhd & 4)
        if fhd & 8:
            raise ZstdError(ErrReservedBit)
        if not self.SingleSegment:
            if len(b) <= p:
                raise ErrUnexpectedEOFHeader("unexpected EOF")
            wd = b[p]; p += 1
            base = 1 << (10 + (wd >> 3))
            self.WindowSize = base + (base // 8) * (wd & 7)
        size = (0, 1, 2, 4)[fhd & 3]
        if size:
            if len(b) - p < size:
                raise ErrUnexpectedEOFHeader("unexpected EOF")
            self.DictionaryID = int.from_bytes(b[p:p + size], "little")
            p += size
        v = fhd >> 6
        fcs = (1 if self.SingleSegment else 0) if v == 0 else 1 << v
        if fcs:
            self.HasFCS = True
            if len(b) - p < fcs:
                raise ErrUnexpectedEOFHeader("unexpected EOF")
            self.FrameContentSize = int.from_bytes(b[p:p + fcs], "little") + (256 if fcs == 2 else 0)
            p += fcs
        self.HeaderSize = p
        rest = b[p:]
        if len(rest) < 3:
            return rest
        bh = rest[0] | rest[1] << 8 | rest[2] << 16
        fb = self.FirstBlock
        fb.Last = bool(bh & 1)
        typ, size = (bh >> 1) & 3, bh >> 3
        if typ == 3:
            return rest
        if typ == 1:
            fb.Compressed, fb.DecompressedSize, fb.CompressedSize = True, size, 1
        elif typ == 2:
            fb.Compressed, fb.CompressedSize = True, size
        else:
            fb.DecompressedSize = fb.CompressedSize = size
        fb.OK = True
        return rest

    def AppendTo(self, dst=b""):
        """The header these fields describe, appended to dst (zstd/decodeheader.go:231-252)."""
        if self.Skippable:
            return dst + bytes([0x50 | (self.SkippableID & 0xF), 0x2A, 0x4D, 0x18]) + (self.SkippableSize & 0xFFFFFFFF).to_bytes(4, "little")
        return dst + frame_header_bytes(self.FrameContentSize, self.WindowSize & 0xFFFFFFFF, self.SingleSegment, self.HasCheckSum,
                                        self.DictionaryID)

    def as_dict(self):
        fb = self.FirstBlock
        return {"SingleSegment": self.SingleSegment, "WindowSize": self.WindowSize, "DictionaryID": self.DictionaryID,
                "HasFCS": self.HasFCS, "FrameContentSize": self.FrameContentSize, "Skippable": self.Skippable,
                "SkippableID": self.SkippableID, "SkippableSize": self.SkippableSize, "HeaderSize": self.HeaderSize,
                "FirstBlock": {"OK": fb.OK, "Last": fb.Last, "Compressed": fb.Compressed, "DecompressedSize": fb.DecompressedSize,
                               "CompressedSize": fb.CompressedSize},
                "HasCheckSum": self.HasCheckSum}


class FrameSpan:
    """One frame of a stream as the host walk sees it: ``length`` compressed bytes; ``content_size`` from the header or None;
    ``bound`` = an upper bound of the decoded size from the block headers; ``skippable`` for 0x184D2A5x frames."""
    __slots__ = ("length", "content_size", "bound", "window", "skippable", "blocks")

    def __init__(self, length, content_size, bound, window, skippable, blocks):
        self.length, self.content_size, self.bound, self.window = length, content_size, bound, window
        self.skippable, self.blocks = skippable, blocks


def frame_span(buf, off=0, max_window=None):
    """Find the frame starting at buf[off] without touching block contents: the frame header fields of frameDec.reset
    (zstd/framedec.go:62-230) and then the 3-byte block headers (zstd/blockdec.go:129-190) up to the last block and the
    optional checksum.  Returns a FrameSpan, or None when buf ends inside the frame (more input needed).  Raises ZstdError for
    what the reference rejects at this level: bad magic, reserved bit, window limits, reserved block type."""
    n = len(buf)
    if n - off < 4:
        return None
    magic = int.from_bytes(buf[off:off + 4], "little")
    if magic & 0xFFFFFFF0 == SKIPPABLE_MAGIC:
        if n - off < 8:
            return None
        ln = 8 + int.from_bytes(buf[off + 4:off + 8], "little")
        return FrameSpan(ln, 0, 0, 0, True, 0) if n - off >= ln else None
    if magic != FRAME_MAGIC:
        raise ZstdError(ErrMagicMismatch)
    p = off + 4
    if p >= n:
        return None
    fhd = buf[p]; p += 1
    if fhd & 8:
        raise ZstdError(ErrReservedBit)
    single = bool(fhd & 0x20)
    window = 0
    if not single:
        if p >= n:
            return None
        wd = buf[p]; p += 1
        base = 1 << (10 + (wd >> 3))
        window = base + (base // 8) * (wd & 7)
    p += (0, 1, 2, 4)[fhd & 3]                       # dictionary id (ignored here; the decoder rejects what it cannot serve)
    flag = fhd >> 6
    fcs_len = (1 if single else 0, 2, 4, 8)[flag]
    if p + fcs_len > n:
        return None
    content = None
    if fcs_len:
        content = int.from_bytes(buf[p:p + fcs_len], "little") + (256 if fcs_len == 2 else 0)
        p += fcs_len
    if single:
        window = content
    elif window < MIN_WINDOW:
        raise ZstdError(ErrWindowSizeExceeded)        # (ErrWindowSizeTooSmall shares the window error class of the C ABI)
    if max_window is not None and window > max_window:
        raise ZstdError(ErrWindowSizeExceeded)
    bound = blocks = 0
    while True:
        if p + 3 > n:
            return None
        bh = buf[p] | buf[p + 1] << 8 | buf[p + 2] << 16
        p += 3
        last, typ, size = bh & 1, (bh >> 1) & 3, bh >> 3
        if typ == 3:
            raise ZstdError(ErrCorrupt)               # ErrReservedBlockType
        if typ == 1:
            p += 1; bound += size
        elif typ == 0:
            p += size; bound += size
        else:
            if size > MAX_BLOCK:
                raise ZstdError(ErrCorrupt)           # ErrCompressedSizeTooBig
            p += size; bound += MAX_BLOCK if not window else min(MAX_BLOCK, max(window, 1))
        blocks += 1
        if last:
            break
    if fhd & 4:
        p += 4
    if p > n:
        return None
    return FrameSpan(p - off, content, bound, window, False, blocks)


class Reader:
    """zstd.NewReader / Decoder.Read / WriteTo / Reset (zstd/decoder.go:84-310) for a stream of frames.  The reference runs a
    three-stage goroutine pipeline over the blocks of one frame at a time (startStreamDecoder, zstd/decoder.go:655-950); on
    the GPU the unit of parallelism is the frame: the reader walks frame and block headers on the host (frame_span), gathers
    complete frames up to ``batch_bytes`` of input and decodes the batch in one call -- every frame its own warp / block set.
    A stream written by this package's Writer (frames of four blocks) is decoded on the staged fast path."""

    def __init__(self, r, device=0, max_window=128 << 20, max_frame=256 << 20, batch_bytes=16 << 20, read_size=1 << 20,
                 decoder=None):
        self._dec = decoder if decoder is not None else Decoder(device=device)
        self._own = decoder is None
        self._max_window, self._max_frame, self._batch, self._rs = max_window, max_frame, batch_bytes, read_size
        self.Reset(r)

    def Reset(self, r):
        """Start over on a new source, keeping the device context (zstd/decoder.go:166-232)."""
        self._r = r
        self._in = bytearray()
        self._out = bytearray()
        self._eof = False
        self._err = None
        self.frames = 0

    def _fill(self, push=False):
        """Decode the next batch of complete frames into the output queue.  Returns False at the clean end of the stream; an
        error is raised once everything decoded before it has been handed out.  push: never read the source -- stop at the
        first incomplete frame."""
        if self._err:
            raise self._err
        spans, pos = [], 0
        while True:
            sp = None
            if pos < len(self._in):
                try:
                    sp = frame_span(self._in, pos, self._max_window)
                except ZstdError as e:
                    self._err = e
                    break
            if sp is None:                                   # the input ends inside a frame (or exactly between frames)
                if push:
                    break
                if self._eof:
                    if pos < len(self._in):
                        self._err = ZstdError(ErrUnexpectedEOF)        # io.ErrUnexpectedEOF
                    break
                if spans and len(self._in) >= self._batch:
                    break                                    # enough for a batch; the partial frame waits for the next call
                chunk = self._r.read(self._rs)
                if chunk:
                    self._in += chunk
                else:
                    self._eof = True
                continue
            if not sp.skippable:
                cap = sp.content_size if sp.content_size is not None else sp.bound
                if cap > self._max_frame:
                    self._err = ZstdError(ErrDecoderSizeExceeded)
                    break
                spans.append((pos, sp.length, cap))
            pos += sp.length
            if pos >= self._batch:
                break
        before = len(self._out)
        if spans:
            view = bytes(self._in[:pos])
            outs, codes = self._dec.decode_chunks([view[o:o + ln] for o, ln, _ in spans], [max(c, 1) for _, _, c in spans])
            for out, code in zip(outs, codes):
                if code < 0:
                    self._err = ZstdError(code)
                    break
                self._out += out
                self.frames += 1
        del self._in[:pos]
        if self._err:
            if len(self._out) > before or self._out:
                return True                                  # hand out what was decoded; the error comes with the next call
            raise self._err
        return bool(spans) or pos > 0 or not self._eof

    def read(self, size=-1):
        """Up to ``size`` decoded bytes (all that remains for size < 0); b"" at the end of the stream."""
        while size < 0 or len(self._out) < size:
            if self._err and self._out:
                break                                        # what precedes an error is delivered first
            if not self._fill():
                break
        if size < 0 or size >= len(self._out):
            out = bytes(self._out); self._out.clear()
            return out
        out = bytes(self._out[:size])
        del self._out[:size]
        return out

    Read = read

    def Feed(self, data):
        """Push form, for callers that are handed the compressed bytes piecewise (a zip reader): append data, decode every
        complete frame now buffered and return the decoded bytes; a partial frame stays pending (see Pending)."""
        self._in += data
        while self._in and not self._err:
            before = len(self._in)
            self._fill(push=True)
            if len(self._in) == before:
                break
        if self._err and not self._out:
            raise self._err
        out = bytes(self._out)
        self._out.clear()
        return out

    def Pending(self):
        """Compressed bytes buffered but not yet decoded (an incomplete frame)."""
        return len(self._in)

    def WriteTo(self, w):
        """Decode everything that remains into w; returns the byte count (zstd/decoder.go:287-310)."""
        total = 0
        while True:
            if self._out:
                total += len(self._out)
                w.write(bytes(self._out)); self._out.clear()
            if not self._fill():
                break
        if self._out:
            total += len(self._out)
            w.write(bytes(self._out)); self._out.clear()
        return total

    def Close(self):
        if self._own and self._dec is not None:
            self._dec.close()
        self._dec = None

    close = Close


# ---- coalescing queue (the shim's batching of concurrent one-block calls) ----------------------------------------
class Queue:
    """Thread-safe, blocking per-block calls batched onto one GPU by a dispatcher thread inside libb200comp.so
    (include/b2c.h, b2c_queue_*): what a cgo shim puts behind concurrent ``Encoder.EncodeAll`` calls
    (zstd/encoder.go:717-729), ``Decoder.DecodeAll`` calls and s2's ``WriterCustomEncoder`` hook
    (s2/writer.go:1052-1064).  ctypes releases the GIL during the call, so Python threads exercise real concurrency."""

    def __init__(self, device=0, max_batch=1024, linger_us=200):
        if not torch.cuda.is_available() or lib.b2c_device_count() == 0:
            raise B2CError("no CUDA device: compress_b200 has no CPU fallback")
        self._q = lib.b2c_queue_create(device, max_batch, linger_us)
        if not self._q:
            raise B2CError("b2c_queue_create failed")

    def close(self):
        if self._q:
            lib.b2c_queue_destroy(self._q)
            self._q = None

    def __del__(self):
        try:
            self.close()
        except Exception:
            pass

    def stats(self):
        calls, batches = ctypes.c_uint64(0), ctypes.c_uint64(0)
        check(lib.b2c_queue_stats(self._q, ctypes.byref(calls), ctypes.byref(batches)))
        return int(calls.value), int(batches.value)

    def _call(self, fn, args, src, cap):
        src = bytes(src)
        out = ctypes.create_string_buffer(max(cap, 1))
        r = fn(self._q, *args, src, len(src), out, cap)
        if r < 0:
            raise ZstdError(r)
        return out.raw[:r]

    def EncodeAll(self, src, level=SpeedFastest, crc=True):
        """EncodeAll for any input size -> one frame (single-block, or multi-block through frame mode); blocks until the
        batch it joined has run."""
        flags = (FLAG_CRC if crc else 0) | FLAG_FRAME
        cap = max(int(lib.b2c_zstd_bound(len(src), level)), int(lib.b2c_zstd_frame_bound(len(src), level))) + 16
        return self._call(lib.b2c_queue_zstd_encode, (level, flags), src, cap)

    def DecodeAll(self, src, max_size=1 << 20):
        return self._call(lib.b2c_queue_zstd_decode, (), src, max_size)

    def S2Encode(self, src, snappy=False):
        """The WriterCustomEncoder contract on one block: the encoded block (this mirror keeps the uvarint length)."""
        cap = int(lib.b2c_s2_bound(len(src)))
        return self._call(lib.b2c_queue_s2_encode, (1, 1 if snappy else 0), src, cap)

    def S2Decode(self, src, max_size=1 << 20):
        return self._call(lib.b2c_queue_s2_decode, (), src, max_size)
