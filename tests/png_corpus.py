"""Seeded PNG files for the decoder tests (tests/test_png_decode_host_cpu.py, tests/test_gpu_png_decode.py): files written
by cv2 and PIL, hand-built files (a PNG writer with forced filters, chunk splits and raw deflate blocks), corrupt files
with the status the decoder must give, the reference decoders and a ctypes call of ledb200_png_decode_host."""
import ctypes as C
import io
import struct
import zlib

import cv2
import numpy as np
from PIL import Image

from lednet_b200 import lib as LIB, ops

SIG = b'\x89PNG\r\n\x1a\n'
BPP = {0: 1, 2: 3, 3: 1, 4: 2, 6: 4}


# ---- pixels ----------------------------------------------------------------------------------------------------------
def smooth_rgb(h, w, seed=0):
    """a gradient with blocks and some noise: every filter type and match length shows up when encoders pick"""
    rng = np.random.default_rng(seed)
    y, x = np.mgrid[0:h, 0:w]
    base = np.stack([(x * 3 + y) % 256, (y * 5) % 256, ((x // 7 + y // 5) * 37) % 256], -1)
    noise = rng.integers(0, 4, (h, w, 3)) * (rng.random((h, w, 1)) < 0.3)
    return ((base + noise) % 256).astype(np.uint8)


def blocky_labels(h, w, seed=0, k=19, cell=16):
    rng = np.random.default_rng(seed)
    small = rng.integers(0, k, (-(-h // cell), -(-w // cell)))
    lab = np.kron(small, np.ones((cell, cell), np.int64))[:h, :w]
    lab[rng.random((h, w)) < 0.02] = 255
    return lab.astype(np.uint8)


# ---- a PNG writer ------------------------------------------------------------------------------------------------------
def chunk(typ, data):
    return struct.pack('>I', len(data)) + typ + data + struct.pack('>I', zlib.crc32(typ + data))


def ihdr(w, h, ct, depth=8, interlace=0):
    return chunk(b'IHDR', struct.pack('>IIBBBBB', w, h, depth, ct, 0, 0, interlace))


def _paeth(a, b, c):
    p = a + b - c
    pa, pb, pc = np.abs(p - a), np.abs(p - b), np.abs(p - c)
    return np.where((pa <= pb) & (pa <= pc), a, np.where(pb <= pc, b, c))


def filter_rows(px, ct, filters):
    """the scanline stream of pixels px [h, w * bpp] uint8, row y filtered with filters[y % len(filters)]"""
    bpp = BPP[ct]
    h = px.shape[0]
    out = []
    for y in range(h):
        cur = px[y].astype(np.int64)
        prev = px[y - 1].astype(np.int64) if y else np.zeros_like(cur)
        a = np.concatenate([np.zeros(bpp, np.int64), cur[:-bpp]])
        c = np.concatenate([np.zeros(bpp, np.int64), prev[:-bpp]])
        ft = filters[y % len(filters)]
        pred = [0, a, prev, (a + prev) // 2, _paeth(a, prev, c)][ft]
        out.append(bytes([ft]) + ((cur - pred) % 256).astype(np.uint8).tobytes())
    return b''.join(out)


def unfilter(raw, h, w, ct):
    """the pixels [h, w * bpp] of a scanline stream, None when a filter type is invalid or the size is wrong"""
    bpp, s = BPP[ct], 1 + w * BPP[ct]
    if len(raw) != h * s:
        return None
    rows = np.frombuffer(raw, np.uint8).reshape(h, s)
    out = np.zeros((h, s - 1), np.int64)
    for y in range(h):
        ft = rows[y, 0]
        if ft > 4:
            return None
        cur = rows[y, 1:].astype(np.int64)
        prev = out[y - 1] if y else np.zeros(s - 1, np.int64)
        if ft in (0, 2):
            out[y] = (cur + (prev if ft == 2 else 0)) % 256
            continue
        for j in range(s - 1):
            a = out[y, j - bpp] if j >= bpp else 0
            b = prev[j]
            c = prev[j - bpp] if j >= bpp else 0
            p = a if ft == 1 else (a + b) // 2 if ft == 3 else int(_paeth(np.int64(a), np.int64(b), np.int64(c)))
            out[y, j] = (cur[j] + p) % 256
    return out.astype(np.uint8)


def png(px, ct, filters=(0,), level=6, strategy=zlib.Z_DEFAULT_STRATEGY, plte=None, pre=(), post=(), split=None,
        zdata=None):
    """A PNG file of pixels px [h, w, channels] (or [h, w]).  pre / post: extra chunks before the first / after the
    last IDAT; split: IDAT payload sizes (the rest in one chunk; 0 = an empty IDAT); zdata: the zlib stream itself."""
    px = px.reshape(px.shape[0], -1)
    h, w = px.shape[0], px.shape[1] // BPP[ct]
    if zdata is None:
        co = zlib.compressobj(level, zlib.DEFLATED, 15, 9, strategy)
        zdata = co.compress(filter_rows(px, ct, filters)) + co.flush()
    idats, at = [], 0
    for n in (split or ()):
        idats.append(chunk(b'IDAT', zdata[at:at + n]))
        at += n
    idats.append(chunk(b'IDAT', zdata[at:]))
    body = b''.join(pre) + (chunk(b'PLTE', plte) if plte is not None else b'') + b''.join(idats) + b''.join(post)
    return SIG + ihdr(w, h, ct) + body + chunk(b'IEND', b'')


# ---- raw deflate blocks --------------------------------------------------------------------------------------------------
class Bits:
    def __init__(self):
        self.v, self.n = 0, 0

    def put(self, v, k):                       # LSB first
        self.v |= v << self.n
        self.n += k

    def code(self, c, k):                      # Huffman codes MSB first
        self.put(int(f'{c:0{k}b}'[::-1], 2), k)

    def bytes(self):
        return self.v.to_bytes((self.n + 7) // 8, 'little')


def fixed_code(b, sym):
    if sym < 144:
        b.code(0x30 + sym, 8)
    elif sym < 256:
        b.code(0x190 + sym - 144, 9)
    elif sym < 280:
        b.code(sym - 256, 7)
    else:
        b.code(0xc0 + sym - 280, 8)


def zwrap(deflate, raw):
    return b'\x78\x01' + deflate + struct.pack('>I', zlib.adler32(raw))


# ---- reference decoders and the host entry point ------------------------------------------------------------------------
def cv2_ref(b):
    return cv2.imdecode(np.frombuffer(b, np.uint8), cv2.IMREAD_COLOR).transpose(2, 0, 1)


def pil_label_ref(b, reduce_zero_label=False, label_map=None):
    return ops.label_lut(reduce_zero_label, label_map)[np.array(Image.open(io.BytesIO(b)))][None]


def host_decode(files, kind='color', reduce_zero_label=False, label_map=None):
    """ledb200_png_decode_host over the files: (statuses, outputs)"""
    n = len(files)
    srcs = [np.frombuffer(b, np.uint8).copy() for b in files]
    infos = [ops.png_info(b, kind) for b in files]
    ch = 3 if kind == 'color' else 1
    outs = [np.zeros((ch, h, w), np.uint8) for h, w, _ in infos]
    arr = (LIB.PngFile * n)()
    for d, s, o, (h, w, ct) in zip(arr, srcs, outs, infos):
        d.data, d.size, d.out, d.h, d.w, d.color_type = s.ctypes.data, s.size, o.ctypes.data, h, w, ct
    st = (C.c_int32 * n)()
    lut = (C.c_uint8 * 256)(*ops.label_lut(reduce_zero_label, label_map).tolist()) if kind == 'label' else None
    LIB.check(LIB.get().ledb200_png_decode_host(arr, n, LIB.PNG_LABEL if kind == 'label' else LIB.PNG_COLOR, lut, st))
    return list(st), outs


# ---- corpora ----------------------------------------------------------------------------------------------------------
def _pil(img, mode, **kw):
    bio = io.BytesIO()
    Image.fromarray(img).convert(mode).save(bio, format='PNG', **kw)
    return bio.getvalue()


def color_corpus():
    """(name, file) pairs that cv2.imdecode(IMREAD_COLOR) reads"""
    img = smooth_rgb(45, 67, seed=1)
    out = []
    for level in (0, 1, 3, 9):
        for strat in (cv2.IMWRITE_PNG_STRATEGY_DEFAULT, cv2.IMWRITE_PNG_STRATEGY_FILTERED,
                      cv2.IMWRITE_PNG_STRATEGY_HUFFMAN_ONLY, cv2.IMWRITE_PNG_STRATEGY_RLE,
                      cv2.IMWRITE_PNG_STRATEGY_FIXED):
            ok, enc = cv2.imencode('.png', img, [cv2.IMWRITE_PNG_COMPRESSION, level, cv2.IMWRITE_PNG_STRATEGY, strat])
            out.append((f'cv2-l{level}-s{strat}', enc.tobytes()))
    rgb = img[..., ::-1].copy()
    for level in range(10):
        out.append((f'pil-l{level}', _pil(rgb, 'RGB', compress_level=level)))
    for mode in ('L', 'RGB', 'RGBA', 'LA', 'P'):
        out.append((f'pil-opt-{mode}', _pil(rgb, mode, optimize=True)))
    rng = np.random.default_rng(2)
    for ct, ch in ((0, 1), (2, 3), (4, 2), (6, 4)):
        px = rng.integers(0, 256, (9, 13, ch)).astype(np.uint8)
        for ft in range(5):
            out.append((f'filter{ft}-ct{ct}', png(px, ct, filters=(ft,))))
        out.append((f'filters-mixed-ct{ct}', png(px, ct, filters=(4, 0, 1, 2, 3))))
    pal = rng.integers(0, 256, (5, 3)).astype(np.uint8).tobytes()
    idx = rng.integers(0, 5, (11, 7, 1)).astype(np.uint8)
    out.append(('palette-5', png(idx, 3, filters=(4,), plte=pal)))
    out.append(('palette-past-end', png(np.arange(77, dtype=np.uint8).reshape(11, 7, 1) % 9, 3, plte=pal)))
    out.append(('palette-256-trns', png(rng.integers(0, 256, (8, 8, 1)).astype(np.uint8), 3, pre=(
        chunk(b'PLTE', rng.integers(0, 256, 768).astype(np.uint8).tobytes()), chunk(b'tRNS', bytes(range(0, 256, 2)))))))
    px = rng.integers(0, 256, (6, 10, 3)).astype(np.uint8)
    out.append(('gama-trns-text', png(px, 2, pre=(chunk(b'gAMA', struct.pack('>I', 22000)),
                                                  chunk(b'tRNS', b'\x00\x01\x00\x02\x00\x03')),
                                      post=(chunk(b'tEXt', b'Comment\x00seeded'),))))
    out.append(('fixed-huffman', png(smooth_rgb(20, 31, seed=3), 2, strategy=zlib.Z_FIXED)))
    big = smooth_rgb(200, 150, seed=4)                                      # 90,200 scanline bytes: two stored blocks
    out.append(('stored-over-64k', png(big, 2, level=0)))
    row = np.random.default_rng(5).integers(0, 256, (1, 32767, 1)).astype(np.uint8)
    out.append(('len258-dist32768', png(np.repeat(row, 4, 0), 0, level=9)))   # rows of 32768 bytes repeat
    z = zlib.compress(filter_rows(px.reshape(6, -1), 2, (1,)))
    out.append(('idat-1-byte', png(px, 2, filters=(1,), split=[1] * (len(z) - 1))))
    out.append(('idat-empty', png(px, 2, split=[0, 3, 0, 5, 0])))
    for h, w in ((1, 1), (1, 9), (7, 1), (5, 33), (3, 101)):
        out.append((f'size-{h}x{w}', png(rng.integers(0, 256, (h, w, 3)).astype(np.uint8), 2, filters=(4, 3))))
    return out


def label_corpus():
    """(name, file) pairs of grey and palette label maps"""
    lab = blocky_labels(40, 56, seed=6)
    out = []
    for level in range(10):
        bio = io.BytesIO()
        Image.fromarray(lab).save(bio, format='PNG', compress_level=level)
        out.append((f'pil-L-l{level}', bio.getvalue()))
    p = Image.fromarray(lab % 19, 'P')
    p.putpalette(list(np.random.default_rng(7).integers(0, 256, 19 * 3)))
    for opt in (False, True):
        bio = io.BytesIO()
        p.save(bio, format='PNG', optimize=opt)
        out.append((f'pil-P-opt{int(opt)}', bio.getvalue()))
    ok, enc = cv2.imencode('.png', lab)
    out.append(('cv2-grey', enc.tobytes()))
    out.append(('hand-P-short-palette', png(lab[..., None] % 19, 3, filters=(4, 1), plte=bytes(range(57)))))
    return out


def _bad_adler(z):
    return z[:-4] + bytes([z[-4] ^ 1]) + z[-3:]


def corrupt_corpus():
    """(name, file, expected status) of files the decoder must reject; statuses as lib.PNG_STATUS lists them"""
    px = smooth_rgb(6, 10, seed=8)
    raw = filter_rows(px.reshape(6, -1), 2, (0,))
    good = png(px, 2)
    z = zlib.compress(raw)
    idat = good.index(b'IDAT') - 4
    n = struct.unpack('>I', good[idat:idat + 4])[0]
    out = []
    bad = bytearray(good); bad[idat + 8 + n] ^= 0xff
    out.append(('idat-crc', bytes(bad), 3))
    out.append(('file-cut-in-idat', good[:idat + 8 + n // 2], 2))
    out.append(('no-iend', good[:-12], 2))
    out.append(('chunk-length-past-end', good[:idat] + struct.pack('>I', 1 << 30) + good[idat + 4:], 2))
    out.append(('bad-chunk-name', png(px, 2, pre=(chunk(b'a1bC', b'x'),)), 2))
    out.append(('unknown-critical', png(px, 2, pre=(chunk(b'ABCD', b'x'),)), 2))
    split = png(px, 2, split=[5])
    second = split.index(b'IDAT', split.index(b'IDAT') + 4) - 4
    out.append(('idat-split-by-chunk', split[:second] + chunk(b'tEXt', b'a\x00b') + split[second:], 2))
    out.append(('plte-after-idat', split[:-12] + chunk(b'PLTE', b'\x00' * 3) + split[-12:], 2))
    out.append(('exif', png(px, 2, pre=(chunk(b'eXIf', b'MM\x00\x2a\x00\x00\x00\x08\x00\x00'),)), 5))
    pal = bytes(range(30))
    idx = (np.arange(60).reshape(6, 10, 1) % 10).astype(np.uint8)
    out.append(('missing-plte', png(idx, 3), 4))
    out.append(('plte-length', png(idx, 3, plte=pal[:29]), 4))
    good_p = png(idx, 3, plte=pal)
    k = good_p.index(b'PLTE') + 4 + 30
    out.append(('plte-crc', good_p[:k] + bytes([good_p[k] ^ 1]) + good_p[k + 1:], 3))
    out.append(('zlib-method', png(px, 2, zdata=b'\x79' + z[1:]), 6))
    out.append(('zlib-check', png(px, 2, zdata=z[:1] + bytes([z[1] ^ 1]) + z[2:]), 6))
    out.append(('zlib-fdict', png(px, 2, zdata=b'\x78\x20' + z[2:]), 6))     # 0x7820 % 31 == 0, FDICT set
    out.append(('trailing-data', png(px, 2, zdata=z + b'\x00'), 6))
    out.append(('truncated-zlib', png(px, 2, zdata=z[:len(z) // 2]), 8))
    out.append(('no-adler', png(px, 2, zdata=z[:-2]), 8))
    out.append(('bad-adler', png(px, 2, zdata=_bad_adler(z)), 10))
    out.append(('too-few-bytes', png(px, 2, zdata=zlib.compress(raw[:-1])), 9))
    out.append(('too-many-bytes', png(px, 2, zdata=zlib.compress(raw + b'\x00')), 9))
    bad_f = bytes([5]) + raw[1:]
    out.append(('filter-type-5', png(px, 2, zdata=zlib.compress(bad_f)), 11))
    b = Bits(); b.put(1, 1); b.put(3, 2)
    out.append(('block-type-3', png(px, 2, zdata=zwrap(b.bytes(), raw)), 7))
    b = Bits(); b.put(1, 1); b.put(0, 2)                                  # a stored block whose NLEN is wrong
    out.append(('stored-nlen', png(px, 2, zdata=zwrap(b.bytes() + struct.pack('<HH', 40, 40) + raw[:40], raw)), 7))
    b = Bits(); b.put(1, 1); b.put(1, 2); fixed_code(b, 286)
    out.append(('invalid-litlen-symbol', png(px, 2, zdata=zwrap(b.bytes(), raw)), 7))
    b = Bits(); b.put(1, 1); b.put(1, 2); fixed_code(b, 97); fixed_code(b, 257); b.code(1, 5)   # length 3, distance 2
    out.append(('distance-too-far', png(px, 2, zdata=zwrap(b.bytes(), raw)), 7))
    b = Bits(); b.put(1, 1); b.put(1, 2); fixed_code(b, 97); fixed_code(b, 257); b.code(30, 5)
    out.append(('invalid-distance-symbol', png(px, 2, zdata=zwrap(b.bytes(), raw)), 7))
    b = Bits(); b.put(1, 1); b.put(2, 2); b.put(0, 5); b.put(0, 5); b.put(15, 4)
    for _ in range(19):
        b.put(1, 3)                                                       # 19 code-length codes of length 1
    out.append(('oversubscribed', png(px, 2, zdata=zwrap(b.bytes() + b'\x00' * 8, raw)), 7))
    b = Bits(); b.put(1, 1); b.put(2, 2); b.put(0, 5); b.put(0, 5); b.put(0, 4)
    for v in (0, 0, 0, 2):
        b.put(v, 3)                                                       # one code-length code of length 2
    out.append(('incomplete-code-lengths', png(px, 2, zdata=zwrap(b.bytes() + b'\x00' * 8, raw)), 7))
    # a complete code-length code {0: '0', 2: '1'}, then literal / length lengths 0 -> 2, 256 -> 2, the rest 0, and one
    # distance length 2: an incomplete literal / length code of maximum length 2
    b = Bits(); b.put(1, 1); b.put(2, 2); b.put(0, 5); b.put(0, 5); b.put(14, 4)
    order = [16, 17, 18, 0, 8, 7, 9, 6, 10, 5, 11, 4, 12, 3, 13, 2, 14, 1]
    for s in order:
        b.put(1 if s in (0, 2) else 0, 3)
    for s in range(258):
        b.code(1 if s in (0, 256, 257) else 0, 1)
    out.append(('incomplete-litlen', png(px, 2, zdata=zwrap(b.bytes() + b'\x00' * 8, raw)), 7))
    b = Bits(); b.put(1, 1); b.put(2, 2); b.put(0, 5); b.put(0, 5); b.put(14, 4)
    for s in order:
        b.put(1 if s in (0, 2) else 0, 3)
    for s in range(258):
        b.code(1 if s in (0, 257) else 0, 1)                              # no end-of-block code
    out.append(('no-end-of-block', png(px, 2, zdata=zwrap(b.bytes() + b'\x00' * 8, raw)), 7))
    return out


def fuzz_corpus(n=300, seed=0):
    """(file, zlib payload, (h, w, ct)) of seeded mutations of small files' zlib streams; chunk CRCs are recomputed so
    the mutation reaches the inflater"""
    rng = np.random.default_rng(seed)
    out = []
    for i in range(n):
        h, w = int(rng.integers(1, 12)), int(rng.integers(1, 12))
        ct = int(rng.choice([0, 2, 4, 6]))
        px = rng.integers(0, 3, (h, w * BPP[ct])).astype(np.uint8) * 60
        strategy = [zlib.Z_DEFAULT_STRATEGY, zlib.Z_FIXED, zlib.Z_HUFFMAN_ONLY, zlib.Z_RLE][i % 4]
        co = zlib.compressobj(int(rng.integers(0, 10)), zlib.DEFLATED, 15, 9, strategy)
        z = bytearray(co.compress(filter_rows(px, ct, (int(rng.integers(0, 5)),))) + co.flush())
        kind = rng.integers(6)
        if kind == 4:                                                     # unchanged
            pass
        elif kind == 5:                                                   # a flipped bit, then the Adler-32 repaired
            j = int(rng.integers(2, max(3, len(z) - 4)))
            z[j] ^= 1 << int(rng.integers(8))
            try:
                z[-4:] = struct.pack('>I', zlib.adler32(zlib.decompressobj(-15).decompress(bytes(z[2:-4]))))
            except zlib.error:
                pass
        elif kind == 0:                                                     # flip bits
            for _ in range(int(rng.integers(1, 4))):
                j = int(rng.integers(len(z)))
                z[j] ^= 1 << int(rng.integers(8))
        elif kind == 1:                                                   # random bytes
            j = int(rng.integers(len(z)))
            z[j] = int(rng.integers(256))
        elif kind == 2:                                                   # cut
            z = z[:int(rng.integers(len(z)))]
        else:                                                             # flip in the deflate header bits
            z[min(2, len(z) - 1)] ^= 1 << int(rng.integers(3))
        z = bytes(z)
        out.append((png(px, ct, zdata=z), z, (h, w, ct)))
    return out


def fuzz_expect(z, h, w, ct):
    """the pixels [h, w * bpp] zlib and a restated unfilter give for the payload, None when the file is invalid"""
    d = zlib.decompressobj()
    try:
        raw = d.decompress(z)
    except zlib.error:
        return None
    if not d.eof or d.unused_data:
        return None
    return unfilter(raw, h, w, ct)
