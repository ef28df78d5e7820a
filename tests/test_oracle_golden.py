"""The oracle (oracle/*.c) pinned against the reference's own golden vectors and against the
system libzstd.  CPU only."""
import ctypes
import io
import os
import struct
import zipfile

import numpy as np
import pytest

import helpers as H


def _pairs(zf):
    names = set(zf.namelist())
    for nm in sorted(names):
        if nm.endswith(".zst") and nm[:-4] in names:
            yield nm, zf.read(nm), zf.read(nm[:-4])


def test_decoder_zip_full(oracle_lib):
    # zstd/decoder_test.go:201-216 TestNewDecoder: every zN.zst must decode to zN (all 94 pairs of decoder.zip)
    zf = zipfile.ZipFile(os.path.join(H.GOLDEN, "zstd_decoder.zip"))
    n = 0
    for nm, comp, want in _pairs(zf):
        r, got = H.oracle_decode(comp, len(want) + 1024)
        assert r == len(want) and got == want, nm
        n += 1
    assert n == 94


def test_seqdec_golden(oracle_lib):
    """Test_seqdec_decoder (zstd/seqdec_test.go:199-302): ready-made decoding tables + bitstream -> (matchOffset,
    matchLength, litLength) per sequence and the final repeat offsets, compared with the reference's seqs-want.zip."""
    c = ctypes
    L = oracle_lib
    L.orc_zstd_seqdec_golden.restype = c.c_int
    L.orc_zstd_seqdec_golden.argtypes = [c.c_void_p, c.c_uint, c.c_void_p, c.c_uint, c.c_void_p, c.c_uint, c.c_char_p,
                                         c.c_size_t, c.c_int, c.c_void_p, c.c_uint64, c.c_size_t, c.c_void_p]
    zs = zipfile.ZipFile(os.path.join(H.GOLDEN, "zstd_seqs.zip"))
    zw = zipfile.ZipFile(os.path.join(H.GOLDEN, "zstd_seqs_want.zip"))
    import re
    n_files = 0
    for nm in zs.namelist():
        m = re.fullmatch(r"n-(\d+)-lits-(\d+)-prev-(\d+)-(\d+)-(\d+)-win-(\d+)\.blk", nm)
        assert m, nm
        nseq, nlit, p0, p1, p2, win = map(int, m.groups())
        d = zs.read(nm)
        off, tabs = 0, []
        for _ in range(3):      # readDecoders: litLengths, matchLengths, offsets (fse_decoder.go:186-207 layout)
            dt = np.frombuffer(d, dtype="<u8", count=512, offset=off).copy()
            symlen, tl, maxbits = struct.unpack_from("<HBB", d, off + 4096)
            tabs.append((dt, tl))
            off += 4096 + 4 + 512 + 512 + 1
        bits = d[off:]
        prev = np.array([p0, p1, p2], dtype=np.int64)
        out = np.zeros((nseq, 3), dtype=np.int64)
        r = L.orc_zstd_seqdec_golden(tabs[0][0].ctypes.data, tabs[0][1], tabs[1][0].ctypes.data, tabs[1][1],
                                     tabs[2][0].ctypes.data, tabs[2][1], bits, len(bits), nseq, prev.ctypes.data, win, nlit,
                                     out.ctypes.data)
        assert r == 0, (nm, r)
        rows = [tuple(map(int, ln.split(","))) for ln in zw.read(nm).decode().split()]
        assert tuple(prev) == rows[0], (nm, tuple(prev), rows[0])
        want = np.array(rows[1:], dtype=np.int64)
        assert want.shape == out.shape and (want == out).all(), nm
        n_files += 1
    assert n_files == 14


def test_header_decode_golden(oracle_lib):
    """TestHeader_Decode (zstd/decodeheader_test.go): every entry of headers.zip parses to exactly the Header in
    headers-want.json.zst, or fails when the reference has no entry for it."""
    import json
    c = ctypes
    L = oracle_lib
    L.orc_zstd_header_decode.restype = c.c_int
    L.orc_zstd_header_decode.argtypes = [c.c_char_p, c.c_size_t, c.c_void_p]
    jz = open(os.path.join(H.GOLDEN, "zstd_headers-want.json.zst"), "rb").read()
    golden = json.loads(H.libzstd_decode(jz, 32 << 20))
    zh = zipfile.ZipFile(os.path.join(H.GOLDEN, "zstd_headers.zip"))
    out = np.zeros(16, dtype=np.uint32)
    ok = bad = 0
    for nm in zh.namelist():
        b = zh.read(nm)
        r = L.orc_zstd_header_decode(b, len(b), out.ctypes.data)
        want = golden.get(nm)
        if r != 0:
            assert want is None, (nm, r)
            bad += 1
            continue
        assert want is not None, nm
        o = [int(x) for x in out]
        got = {"SingleSegment": bool(o[0]), "WindowSize": o[1] | (o[2] << 32), "DictionaryID": o[3], "HasFCS": bool(o[4]),
               "FrameContentSize": o[5] | (o[6] << 32), "Skippable": bool(o[7]), "SkippableID": o[8], "SkippableSize": o[9],
               "HeaderSize": o[10],
               "FirstBlock": {"OK": bool(o[11]), "Last": bool(o[12]), "Compressed": bool(o[13] & 1), "DecompressedSize": o[14],
                              "CompressedSize": o[15]},
               "HasCheckSum": bool(o[13] & 2)}
        assert got == want, (nm, got, want)
        ok += 1
    assert ok == len(golden) and ok + bad == len(zh.namelist())


def test_good_zip(oracle_lib):
    # zstd/decoder_test.go:393 TestNewDecoderGood: all must decode; libzstd agrees on the bytes
    zf = zipfile.ZipFile(os.path.join(H.GOLDEN, "zstd_good.zip"))
    n = 0
    for nm in zf.namelist():
        if not nm.endswith(".zst"):
            continue
        comp = zf.read(nm)
        r, got = H.oracle_decode(comp, 64 << 20)
        assert r >= 0, nm
        z = H.libzstd_decode(comp, max(r, 1))
        assert z == got, nm
        n += 1
    assert n == 12


def test_bad_zip(oracle_lib):
    # zstd/decoder_test.go:409-455 TestNewDecoderBad: every file must be rejected (libzstd accepts 2 of them)
    zf = zipfile.ZipFile(os.path.join(H.GOLDEN, "zstd_bad.zip"))
    n = 0
    for nm in zf.namelist():
        if not nm.endswith(".zst"):
            continue
        r, _ = H.oracle_decode(zf.read(nm), 64 << 20)
        assert r < 0, nm
        n += 1
    assert n == 32


# zstd/decoder_test.go:1938-1975 (TestPredefTables), literal-length table: (nextState, nbAddBits, nbBits, baseVal)
_LL_WANT = [
    (0, 0, 4, 0), (16, 0, 4, 0), (32, 0, 5, 1), (0, 0, 5, 3), (0, 0, 5, 4), (0, 0, 5, 6), (0, 0, 5, 7), (0, 0, 5, 9),
    (0, 0, 5, 10), (0, 0, 5, 12), (0, 0, 6, 14), (0, 1, 5, 16), (0, 1, 5, 20), (0, 1, 5, 22), (0, 2, 5, 28),
    (0, 3, 5, 32), (0, 4, 5, 48), (32, 6, 5, 64), (0, 7, 5, 128), (0, 8, 6, 256), (0, 10, 6, 1024), (0, 12, 6, 4096),
    (32, 0, 4, 0), (0, 0, 4, 1), (0, 0, 5, 2), (32, 0, 5, 4), (0, 0, 5, 5), (32, 0, 5, 7), (0, 0, 5, 8), (32, 0, 5, 10),
    (0, 0, 5, 11), (0, 0, 6, 13), (32, 1, 5, 16), (0, 1, 5, 18), (32, 1, 5, 22), (0, 2, 5, 24), (32, 3, 5, 32),
    (0, 3, 5, 40), (0, 6, 4, 64), (16, 6, 4, 64), (32, 7, 5, 128), (0, 9, 6, 512), (0, 11, 6, 2048), (48, 0, 4, 0),
    (16, 0, 4, 1), (32, 0, 5, 2), (32, 0, 5, 3), (32, 0, 5, 5), (32, 0, 5, 6), (32, 0, 5, 8), (32, 0, 5, 9),
    (32, 0, 5, 11), (32, 0, 5, 12), (0, 0, 6, 15), (32, 1, 5, 18), (32, 1, 5, 20), (32, 2, 5, 24), (32, 2, 5, 28),
    (32, 3, 5, 40), (32, 4, 5, 48), (0, 16, 6, 65536), (0, 15, 6, 32768), (0, 14, 6, 16384), (0, 13, 6, 8192),
]


def test_predef_tables(oracle_lib):
    buf = (ctypes.c_uint32 * (4 * 64))()
    assert oracle_lib.orc_zstd_predef_table(0, buf, 64) == 64
    ll = np.frombuffer(buf, dtype=np.uint32).reshape(64, 4)  # nbBits, addBits, newState, baseline
    for i, (ns, ab, nb, base) in enumerate(_LL_WANT):
        assert tuple(int(x) for x in ll[i]) == (nb, ab, ns, base), i
    assert oracle_lib.orc_zstd_predef_table(1, buf, 64) == 32
    assert oracle_lib.orc_zstd_predef_table(2, buf, 64) == 64
    ml = np.frombuffer(buf, dtype=np.uint32).reshape(64, 4).copy()
    # first and last rows of the match-length table (decoder_test.go:2003-2040)
    assert tuple(int(x) for x in ml[0]) == (6, 0, 0, 3)
    assert tuple(int(x) for x in ml[1]) == (4, 0, 0, 4)
    assert tuple(int(x) for x in ml[63]) == (6, 10, 0, 1027)
    assert tuple(int(x) for x in ml[57]) == (6, 16, 0, 65539)


def test_xxh64_kat(oracle_lib):
    # XXH64 reference values (seed 0)
    assert oracle_lib.orc_xxh64(b"", 0, 0) == 0xEF46DB3751D8E999
    assert oracle_lib.orc_xxh64(b"a", 1, 0) == 0xD24EC4F1A98C6E5B
    assert oracle_lib.orc_xxh64(b"abc", 3, 0) == 0x44BC2CF5AD770999
    s = b"Nobody inspects the spammish repetition"
    assert oracle_lib.orc_xxh64(s, len(s), 0) == 0xFBCEA83C8A378BF1


@pytest.mark.parametrize("name", ["twain.txt", "html.txt", "e.txt"])
def test_oracle_encode_roundtrip(oracle_lib, name):
    # encoder tests upstream are round-trip only (zstd/encoder_test.go:68-304); add libzstd as 2nd decoder
    data = H.golden(name)
    r, enc = H.oracle_encode(data)
    assert 0 < r <= oracle_lib.orc_zstd_max_encoded_size(len(data), 1, 1)
    r2, dec = H.oracle_decode(enc, len(data) + 64)
    assert dec == data
    assert H.libzstd_decode(enc, len(data)) == data
    for i in range(0, len(data), 65536):
        c = data[i:i + 65536]
        r, enc = H.oracle_encode(c)
        assert H.libzstd_decode(enc, len(c)) == c


def test_oracle_encode_edge(oracle_lib):
    rng = np.random.Generator(np.random.PCG64(5))
    cases = [b"", b"a", b"ab" * 3, b"a" * 9, b"a" * 10, b"abcdefgh" * 100, bytes(1000), bytes(65536),
             rng.integers(0, 256, 65536, dtype=np.uint8).tobytes(), rng.integers(0, 4, 70000, dtype=np.uint8).tobytes(),
             H.synth_text(200000)]
    for c in cases:
        r, enc = H.oracle_encode(c)
        assert r > 0
        assert H.libzstd_decode(enc, len(c)) == c
        r2, dec = H.oracle_decode(enc, len(c) + 64)
        assert dec == c


def test_huff0_error_classes(oracle_lib):
    # huff0/compress_test.go:20-52: random => ErrIncompressible, single symbol => ErrUseRLE, too big => ErrTooBig
    out = ctypes.create_string_buffer(300000)
    tl = ctypes.c_uint64()
    rng = np.random.Generator(np.random.PCG64(9))
    rnd = rng.integers(0, 256, 100004, dtype=np.uint8).tobytes()
    assert oracle_lib.orc_huf_compress_oneshot(rnd, len(rnd), 1, 0, out, len(out), ctypes.byref(tl)) == -1
    z = bytes(1000)
    assert oracle_lib.orc_huf_compress_oneshot(z, len(z), 1, 0, out, len(out), ctypes.byref(tl)) == -2
    big = bytes(1 << 18)
    assert oracle_lib.orc_huf_compress_oneshot(big, len(big), 1, 0, out, len(out), ctypes.byref(tl)) == -3
    tw = H.golden("twain.txt")[:200000]
    r = oracle_lib.orc_huf_compress_oneshot(tw, len(tw), 1, 0, out, len(out), ctypes.byref(tl))
    # Shannon lower-bound sanity (huff0/compress_test.go:250-253)
    cnt = np.bincount(np.frombuffer(tw, dtype=np.uint8), minlength=256).astype(np.float64)
    pz = cnt[cnt > 0] / len(tw)
    shannon = -(pz * np.log2(pz)).sum() * len(tw) / 8
    assert shannon <= r < len(tw) * 0.7


def test_xxh64_kats(oracle_lib):
    # zstd/internal/xxhash/xxhash_test.go:17-27 (TestAll) and the content digests the encoder tests expect
    # (zstd/encoder_test.go:543-563: Twain, HTML)
    L = H.oracle()
    L.orc_xxh64.restype = ctypes.c_uint64
    L.orc_xxh64.argtypes = [ctypes.c_char_p, ctypes.c_size_t, ctypes.c_uint64]
    kats = [(b"", 0xef46db3751d8e999), (b"a", 0xd24ec4f1a98c6e5b), (b"as", 0x1c330fb2d66be179), (b"asd", 0x631c37ce72a97393),
            (b"asdf", 0x415872f599cea71e),
            (b"Call me Ishmael. Some years ago--never mind how long precisely-", 0x02a2e85470d6fd96)]
    for data, want in kats:
        assert L.orc_xxh64(data, len(data), 0) == want, data
    tw, ht = H.golden("twain.txt"), H.golden("html.txt")
    assert L.orc_xxh64(tw, len(tw), 0) == 0x121f127079371fc6
    assert L.orc_xxh64(ht, len(ht), 0) == 0x35a95c37209ec337
