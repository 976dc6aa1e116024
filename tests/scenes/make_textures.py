"""Writes the small image files the textured golden scenes read (tests/scenes/textures/), and the OpenEXR reader's
fixtures written by the OpenEXR library (tests/golden/openexr/).  Deterministic; the files are committed, this script
documents how they were made:

    python tests/scenes/make_textures.py
"""
import os
import struct
import zlib

import numpy as np

OUT = os.path.join(os.path.dirname(os.path.abspath(__file__)), "textures")
OUT_OPENEXR = os.path.join(os.path.dirname(os.path.dirname(os.path.abspath(__file__))), "golden", "openexr")


def write_pfm(path, img):
    """img: (h, w) or (h, w, 3) float32, row 0 at the top; PFM stores the bottom row first, little endian (scale -1)."""
    img = np.asarray(img, np.float32)
    h, w = img.shape[:2]
    with open(path, "wb") as f:
        f.write(b"PF\n" if img.ndim == 3 else b"Pf\n")
        f.write(b"%d %d\n-1.0\n" % (w, h))
        f.write(img[::-1].astype("<f4").tobytes())


def write_png(path, rgb8):
    """8-bit RGB, filter type 0 on every scanline except a few with Sub / Up / Paeth so that the reader's filters run."""
    h, w, _ = rgb8.shape
    raw = bytearray()
    prev = np.zeros((w, 3), np.int32)
    for y in range(h):
        cur = rgb8[y].astype(np.int32)
        ft = y % 5
        left = np.vstack([np.zeros((1, 3), np.int32), cur[:-1]])
        upleft = np.vstack([np.zeros((1, 3), np.int32), prev[:-1]])
        if ft == 0:
            pred = 0
        elif ft == 1:
            pred = left
        elif ft == 2:
            pred = prev
        elif ft == 3:
            pred = (left + prev) // 2
        else:
            p = left + prev - upleft
            pa, pb, pc = abs(p - left), abs(p - prev), abs(p - upleft)
            pred = np.where((pa <= pb) & (pa <= pc), left, np.where(pb <= pc, prev, upleft))
        raw.append(ft)
        raw += ((cur - pred) & 255).astype(np.uint8).tobytes()
        prev = cur

    def chunk(tag, data):
        return struct.pack(">I", len(data)) + tag + data + struct.pack(">I", zlib.crc32(tag + data) & 0xffffffff)

    with open(path, "wb") as f:
        f.write(b"\x89PNG\r\n\x1a\n")
        f.write(chunk(b"IHDR", struct.pack(">IIBBBBB", w, h, 8, 2, 0, 0, 0)))
        comp = zlib.compress(bytes(raw), 9)
        f.write(chunk(b"IDAT", comp[:len(comp) // 2]))   # two IDAT chunks: the stream may be split anywhere
        f.write(chunk(b"IDAT", comp[len(comp) // 2:]))
        f.write(chunk(b"IEND", b""))


def write_tga(path, rgb8, rle=True):
    """24-bit true colour, bottom-to-top (the TGA default origin), run-length encoded."""
    h, w, _ = rgb8.shape
    body = bytearray()
    rows = rgb8[::-1, :, ::-1]   # bottom row first, BGR
    if not rle:
        body += rows.tobytes()
    else:
        flat = rows.reshape(-1, 3)
        i = 0
        while i < len(flat):
            run = 1
            while i + run < len(flat) and run < 128 and (flat[i + run] == flat[i]).all():
                run += 1
            if run > 1:
                body.append(128 | (run - 1))
                body += flat[i].tobytes()
                i += run
            else:
                n = 1
                while i + n < len(flat) and n < 128 and not (i + n + 1 < len(flat) and (flat[i + n] == flat[i + n + 1]).all()):
                    n += 1
                body.append(n - 1)
                body += flat[i:i + n].tobytes()
                i += n
    with open(path, "wb") as f:
        f.write(struct.pack("<BBBHHBHHHHBB", 0, 0, 10 if rle else 2, 0, 0, 0, 0, 0, w, h, 24, 0))
        f.write(body)


def write_exr(path, img, compression="zip"):
    """Scan-line OpenEXR, half B / G / R channels (stored alphabetically), ZIP (16 lines per block), ZIPS (1) or NONE."""
    img = np.asarray(img, np.float16)
    h, w, _ = img.shape
    comp = {"none": 0, "zips": 2, "zip": 3}[compression]
    lines_per_block = 16 if comp == 3 else 1

    def attr(name, typ, data):
        return name.encode() + b"\0" + typ.encode() + b"\0" + struct.pack("<i", len(data)) + data

    chlist = b"".join(c + b"\0" + struct.pack("<iB3xii", 1, 0, 1, 1) for c in (b"B", b"G", b"R")) + b"\0"
    box = struct.pack("<4i", 0, 0, w - 1, h - 1)
    header = (struct.pack("<II", 20000630, 2) + attr("channels", "chlist", chlist) + attr("compression", "compression", bytes([comp]))
              + attr("dataWindow", "box2i", box) + attr("displayWindow", "box2i", box) + attr("lineOrder", "lineOrder", b"\0")
              + attr("pixelAspectRatio", "float", struct.pack("<f", 1.0)) + attr("screenWindowCenter", "v2f", struct.pack("<2f", 0, 0))
              + attr("screenWindowWidth", "float", struct.pack("<f", 1.0)) + b"\0")
    chunks = []
    for y0 in range(0, h, lines_per_block):
        raw = b"".join(img[y, :, c].astype("<f2").tobytes() for y in range(y0, min(h, y0 + lines_per_block)) for c in (2, 1, 0))
        data = raw
        if comp:
            a = np.frombuffer(raw, np.uint8)
            t = np.concatenate([a[0::2], a[1::2]]).astype(np.int32)      # even bytes first, then odd bytes
            d = t.copy()
            d[1:] = (t[1:] - t[:-1] + 128 + 256) % 256                   # byte deltas
            z = zlib.compress(d.astype(np.uint8).tobytes(), 9)
            if len(z) < len(raw):
                data = z
        chunks.append(struct.pack("<ii", y0, len(data)) + data)
    offset = len(header) + 8 * len(chunks)
    table = b""
    for c in chunks:
        table += struct.pack("<Q", offset)
        offset += len(c)
    with open(path, "wb") as f:
        f.write(header + table + b"".join(chunks))


def write_exr_openexr(path, img, compression):
    """The same picture written by the OpenEXR library itself (as bundled with OpenCV), for the codecs write_exr does not
    implement and for ZIP / ZIPS as the library compresses them: half B / G / R channels, RLE (1 line per block), ZIPS (1),
    ZIP (16), PIZ (32) or B44 (lossy; the reader must refuse it)."""
    os.environ["OPENCV_IO_ENABLE_OPENEXR"] = "1"
    import cv2
    comp = {"rle": 1, "zips": 2, "zip": 3, "piz": 4, "b44": 6}[compression]
    bgr = np.ascontiguousarray(np.asarray(img, np.float32)[:, :, ::-1])
    assert cv2.imwrite(path, bgr, [cv2.IMWRITE_EXR_TYPE, cv2.IMWRITE_EXR_TYPE_HALF, cv2.IMWRITE_EXR_COMPRESSION, comp])


def with_decreasing_line_order(src, dst):
    """The scan-line file `src` laid out as lineOrder DECREASING_Y: the same blocks stored from the last to the first, the
    offset table still indexed from the first block."""
    data = open(src, "rb").read()
    pos, order_at = 8, None
    while data[pos] != 0:                                   # attributes: name \0 type \0 size data
        name_end = data.index(b"\0", pos)
        type_end = data.index(b"\0", name_end + 1)
        size = struct.unpack_from("<i", data, type_end + 1)[0]
        if data[pos:name_end] == b"lineOrder":
            order_at = type_end + 5
        pos = type_end + 5 + size
    table = pos + 1
    n = (struct.unpack_from("<Q", data, table)[0] - table) // 8
    offsets = list(struct.unpack_from("<%dQ" % n, data, table)) + [len(data)]
    blocks = [data[offsets[i]:offsets[i + 1]] for i in range(n)]
    header = bytearray(data[:table])
    header[order_at] = 1
    new, at = [0] * n, table + 8 * n
    for i in reversed(range(n)):
        new[i], at = at, at + len(blocks[i])
    with open(dst, "wb") as f:
        f.write(bytes(header) + struct.pack("<%dQ" % n, *new) + b"".join(blocks[::-1]))


def pattern(w, h, seed):
    """coloured tiles with a smooth gradient on top: detail at the texel scale and below"""
    rs = np.random.RandomState(seed)
    tiles = rs.uniform(0.05, 0.95, (h // 3 + 1, w // 3 + 1, 3))
    y, x = np.mgrid[0:h, 0:w]
    img = tiles[y // 3, x // 3] * (0.6 + 0.4 * np.sin(0.9 * x + 0.5 * y)[..., None] ** 2)
    return img.astype(np.float32)


def main():
    os.makedirs(OUT, exist_ok=True)
    write_pfm(os.path.join(OUT, "tiles_37x23.pfm"), pattern(37, 23, 1))          # not a power of two: resampled
    write_pfm(os.path.join(OUT, "tiles_64x32.pfm"), pattern(64, 32, 2))
    # alpha mask: blocks of exact zeros (a hit counts unless the bilinear look-up is exactly 0)
    y, x = np.mgrid[0:16, 0:16]
    holes = np.where(((x // 4 + y // 4) % 2 == 0) & (x % 4 < 3) & (y % 4 < 3), 0.0, 1.0).astype(np.float32)
    write_pfm(os.path.join(OUT, "holes_16x16.pfm"), holes)
    stripes = np.where((x // 2) % 3 == 0, 0.0, 1.0).astype(np.float32)
    write_pfm(os.path.join(OUT, "stripes_16x16.pfm"), stripes)
    rs = np.random.RandomState(3)
    write_pfm(os.path.join(OUT, "rough_8x8.pfm"), rs.uniform(0.02, 0.35, (8, 8)).astype(np.float32))
    # a smooth height field for bump mapping (periodic, so that the repeat wrap has no seam)
    yy, xx = np.mgrid[0:32, 0:32] * (2 * np.pi / 32)
    write_pfm(os.path.join(OUT, "bumps_32x32.pfm"), (0.5 + 0.25 * np.sin(3 * xx) * np.cos(2 * yy) + 0.2 * np.sin(xx + 4 * yy)).astype(np.float32))
    rgb8 = (pattern(20, 12, 4) * 255 + 0.5).astype(np.uint8)
    write_png(os.path.join(OUT, "tiles_20x12.png"), rgb8)
    rgb8b = (pattern(24, 10, 5) * 255 + 0.5).astype(np.uint8)
    rgb8b[2:5, 3:15] = rgb8b[2, 3]   # some runs for the run-length packets
    write_tga(os.path.join(OUT, "tiles_24x10.tga"), rgb8b)
    hdr = (pattern(24, 18, 6) * np.float32(3.0)).astype(np.float16)      # 18 lines: a full ZIP block of 16 and a short one
    hdr[3, 5] = [1000.0, 0.001, 0.0]
    write_exr(os.path.join(OUT, "tiles_24x18_zip.exr"), hdr, "zip")
    write_exr(os.path.join(OUT, "tiles_24x18_zips.exr"), hdr, "zips")
    write_exr(os.path.join(OUT, "tiles_24x18_none.exr"), hdr, "none")
    np.savez_compressed(os.path.join(OUT, "decoded_8bit.npz"), png=rgb8, tga=rgb8b, exr=hdr.astype(np.float32))
    # 70 lines: two full PIZ blocks of 32 and a short one
    hdr2 = (pattern(40, 70, 7) * np.float32(3.0)).astype(np.float16)
    hdr2[5, 9] = [2000.0, 0.0004, 0.0]
    os.makedirs(OUT_OPENEXR, exist_ok=True)
    for codec in ("rle", "zips", "zip", "piz", "b44"):
        write_exr_openexr(os.path.join(OUT_OPENEXR, "tiles_40x70_%s.exr" % codec), hdr2, codec)
    with_decreasing_line_order(os.path.join(OUT_OPENEXR, "tiles_40x70_piz.exr"), os.path.join(OUT_OPENEXR, "tiles_40x70_piz_decreasing.exr"))
    np.savez_compressed(os.path.join(OUT_OPENEXR, "decoded.npz"), exr=hdr2.astype(np.float32))


if __name__ == "__main__":
    main()
