"""Film checkpoints (lr_film_save / lr_multi_film_save) read back in numpy, and the noise of their 8x4 tiles as adaptive sampling
(lr_film_render_adaptive) measures it, restated in float64 from the raw sums: for inspecting a checkpoint and for tools and
tests that check the device's selection."""
import struct

import numpy as np

FLOOR = 1e-3                                          # kAdaptiveFloor, csrc/device_scene.h
HEADER = struct.Struct("<8s14iQ")                     # FilmHeader, csrc/api.cpp


def read_checkpoint(path):
    """(magic, spp_done, raw sums (h, w, 3), sums of squares or None, tile counts (tiles_y, tiles_x)) of a film checkpoint."""
    with open(path, "rb") as f:
        raw = f.read()
    h = HEADER.unpack_from(raw)
    magic, (_, _, _, _, cw, ch, _, _, _, _, _, _, spp_done, has_sq), _ = h[0], h[1:15], h[15]
    n = cw * ch * 3
    data = np.frombuffer(raw, dtype=np.float32, count=n * (2 if has_sq else 1), offset=HEADER.size)
    tx, ty = (cw + 7) // 8, (ch + 3) // 4
    if magic == b"LRFILM2\0":
        counts = np.frombuffer(raw, dtype=np.int32, count=tx * ty, offset=HEADER.size + data.nbytes).reshape(ty, tx)
    else:
        if magic != b"LRFILM1\0" or len(raw) != HEADER.size + data.nbytes:
            raise ValueError("%s: not a film checkpoint" % path)
        counts = np.full((ty, tx), spp_done, dtype=np.int32)
    s = data[:n].reshape(ch, cw, 3)
    q = data[n:].reshape(ch, cw, 3) if has_sq else None
    return magic, spp_done, s, q, counts


def tile_errors(s, q, counts):
    """The tile errors and the tiles whose in-crop sums and squares are all finite, in float64 (adaptive_error)."""
    ch, cw, _ = s.shape
    ty, tx = counts.shape
    n = np.repeat(np.repeat(counts, 4, axis=0), 8, axis=1)[:ch, :cw, None].astype(np.float64)
    S, Q = s.astype(np.float64), q.astype(np.float64)
    with np.errstate(all="ignore"):
        m = S / n
        var = np.fmax(0.0, (Q - S * m) / (n - 1.0))
        e = np.sqrt(var / n) / np.fmax(m, FLOOR)
    fin = np.isfinite(s) & np.isfinite(q)
    pad_e = np.full((ty * 4, tx * 8, 3), -np.inf)
    pad_e[:ch, :cw] = e
    pad_f = np.ones((ty * 4, tx * 8, 3), dtype=bool)
    pad_f[:ch, :cw] = fin
    err = np.fmax.reduce(pad_e.reshape(ty, 4, tx, 8, 3).transpose(0, 2, 1, 3, 4).reshape(ty, tx, -1), axis=2)
    finite = pad_f.reshape(ty, 4, tx, 8, 3).transpose(0, 2, 1, 3, 4).reshape(ty, tx, -1).all(axis=2)
    return err, finite
