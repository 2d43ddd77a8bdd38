"""Minimal HEIF writer for tests: one image item (a grid of hvc1 tiles, or a single hvc1 item) with a chosen list of
transformative properties (clap / irot / imir) in a chosen ipma order.  TEST INFRASTRUCTURE ONLY: no thumbnails, no
auxiliary images, no colour properties; not a product container writer.

Boxes: ftyp, meta (hdlr, pitm, iinf, iref dimg, iloc, idat with the grid descriptor, iprp with hvcC / ispe / clap / irot /
imir) and mdat with the tiles as 4-byte length-prefixed NAL units."""
from __future__ import annotations

import struct


def _box(kind: bytes, payload: bytes) -> bytes:
    return struct.pack(">I4s", 8 + len(payload), kind) + payload


def _fullbox(kind: bytes, version: int, flags: int, payload: bytes) -> bytes:
    return _box(kind, struct.pack(">I", (version << 24) | flags) + payload)


def _hvcc(vps: bytes, sps: bytes, pps: bytes) -> bytes:
    # configurationVersion 1, Main profile fields (not interpreted), lengthSizeMinusOne = 3, three arrays
    rec = bytes([1, 0x01]) + struct.pack(">I", 0x60000000) + bytes(6) + bytes([90]) + struct.pack(">H", 0xF000)
    rec += bytes([0xFC, 0xFD, 0xF8, 0xF8]) + struct.pack(">H", 0) + bytes([0x0F, 3])
    for nal_type, nal in ((32, vps), (33, sps), (34, pps)):
        rec += bytes([0x80 | nal_type]) + struct.pack(">HH", 1, len(nal)) + nal
    return _box(b"hvcC", rec)


def clap(width_n, width_d, height_n, height_d, horiz_off_n, horiz_off_d, vert_off_n, vert_off_d):
    return ("clap", (width_n, width_d, height_n, height_d, horiz_off_n, horiz_off_d, vert_off_n, vert_off_d))


def irot(angle):
    return ("irot", angle)


def imir(axis):
    return ("imir", axis)


def _prop(p) -> bytes:
    kind, v = p
    if kind == "clap":
        return _box(b"clap", struct.pack(">IIIIiIiI", *v))
    if kind == "irot":
        return _box(b"irot", bytes([v & 3]))
    if kind == "imir":
        return _box(b"imir", bytes([v & 1]))
    raise ValueError(kind)


def write_heif(vps: bytes, sps: bytes, pps: bytes, tiles, tile_size, grid=None, canvas=None, props=()) -> bytes:
    """tiles: escaped slice NAL units (2-byte header included), row-major; tile_size: (w, h) for the tiles' ispe.
    grid: (rows, cols) for a grid item, None for a single hvc1 item (one tile).  canvas: (w, h) of the grid.
    props: clap(...) / irot(...) / imir(...) of the image item, in ipma order."""
    tiles = [bytes(t) for t in tiles]
    if grid is None and len(tiles) != 1:
        raise ValueError("a single item has one tile")
    n = len(tiles)
    image_id = 1
    tile_ids = [image_id] if grid is None else list(range(2, 2 + n))

    # ipco: 1 hvcC, 2 ispe of a tile, 3 ispe of the canvas (grid only), then the transformative properties
    ipco = [_hvcc(vps, sps, pps), _fullbox(b"ispe", 0, 0, struct.pack(">II", *tile_size))]
    if grid is not None:
        ipco.append(_fullbox(b"ispe", 0, 0, struct.pack(">II", *canvas)))
    first_tp = len(ipco) + 1
    ipco += [_prop(p) for p in props]
    tp_idx = list(range(first_tp, first_tp + len(props)))
    assoc = []
    if grid is None:
        assoc.append((image_id, [0x81, 2] + tp_idx))
    else:
        assoc.append((image_id, [3] + tp_idx))
        assoc += [(t, [0x81, 2]) for t in tile_ids]
    ipma = struct.pack(">I", len(assoc))
    for item, entries in assoc:
        ipma += struct.pack(">HB", item, len(entries)) + bytes(entries)
    iprp = _box(b"iprp", _box(b"ipco", b"".join(ipco)) + _fullbox(b"ipma", 0, 0, ipma))

    infes = []
    if grid is not None:
        infes.append(_fullbox(b"infe", 2, 0, struct.pack(">HH4s", image_id, 0, b"grid") + b"\0"))
    infes += [_fullbox(b"infe", 2, 1 if grid is not None else 0, struct.pack(">HH4s", t, 0, b"hvc1") + b"\0") for t in tile_ids]
    iinf = _fullbox(b"iinf", 0, 0, struct.pack(">H", len(infes)) + b"".join(infes))
    hdlr = _fullbox(b"hdlr", 0, 0, struct.pack(">I4s", 0, b"pict") + bytes(12) + b"\0")
    pitm = _fullbox(b"pitm", 0, 0, struct.pack(">H", image_id))
    iref = b""
    idat = b""
    if grid is not None:
        iref = _fullbox(b"iref", 0, 0, _box(b"dimg", struct.pack(">HH", image_id, n) + b"".join(struct.pack(">H", t) for t in tile_ids)))
        idat = _box(b"idat", struct.pack(">BBBBHH", 0, 0, grid[0] - 1, grid[1] - 1, canvas[0], canvas[1]))  # 8 bytes
    payloads = [struct.pack(">I", len(t)) + t for t in tiles]

    def meta(mdat_data_start: int) -> bytes:
        entries = []
        if grid is not None:  # construction method 1: the grid descriptor in idat
            entries.append(struct.pack(">HHHHII", image_id, 1, 0, 1, 0, 8))
        off = mdat_data_start
        for t, p in zip(tile_ids, payloads):
            entries.append(struct.pack(">HHHHII", t, 0, 0, 1, off, len(p)))
            off += len(p)
        iloc = _fullbox(b"iloc", 1, 0, bytes([0x44, 0x00]) + struct.pack(">H", len(entries)) + b"".join(entries))
        return _fullbox(b"meta", 0, 0, hdlr + pitm + iinf + iref + iprp + iloc + idat)

    ftyp = _box(b"ftyp", b"heic" + struct.pack(">I", 0) + b"mif1heic")
    start = len(ftyp) + len(meta(0)) + 8  # the meta box's size does not depend on the offsets
    mdat = _box(b"mdat", b"".join(payloads))
    return ftyp + meta(start) + mdat
