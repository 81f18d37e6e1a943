"""CPU: the source blocks that the weight pack (sscvae_pack_weights) and the fused clip + SGD + pack of the optimizer
(sscvae_sgd_step_packed) run their jobs from (sscvae_debug_sgd_pack_jobs, a host-only function of the dims), at the
benchmark's dims. The fused update relies on these properties:
  * every element of every weight is updated by exactly one job (the blocks of a weight split its columns);
  * the jobs write the images of the packed layout that the forward, backward and decode kernels read (written out
    below block by block), each from the same source elements;
  * every byte of the packed buffer is written by at most one job, and no padding byte is written.
"""
import ctypes

import numpy as np
import pytest

from sscvae import _lib

(EMB, ATT_IH, ATT_HH, ATT_BIH, ATT_BHH, QP, IP, AVEC, ENC_IH, ENC_HH, ENC_BIH, ENC_BHH, DEC_IH, DEC_HH, DEC_BIH, DEC_BHH,
 FCM_W, FCM_B, FCL_W, FCL_B, OUT_W, OUT_B) = range(22)
PLAIN, TRANS, F32 = 0, 1, 2
F, E, H, A, Z, V = 2048, 600, 900, 768, 150, 10000             # bench.py DIMS


def _pad(x, m=64):
    return (x + m - 1) // m * m


class _D:
    def __init__(self, sv, le, tied):
        self.sv, self.tied = sv, tied
        self.cvar = int(sv == 2)
        self.c = 0 if sv == 0 else (1 if sv == 1 else (1 if le == 1 else Z))
        self.Fp, self.Ep, self.Hp, self.Ap, self.Zp, self.Vp = map(_pad, (F, E, H, A, Z, V))
        self.G = 4 * H
        self.Gp, self.Z2p = _pad(self.G), _pad(2 * Z)
        self.KX = self.Fp + 2 * self.Hp
        self.Cp = _pad(self.c) if self.cvar else 0
        self.ZC = self.Zp + self.Cp
        self.GP = (H + 31) // 32 * 128
        self.NO, self.NOp = (E, self.Ep) if tied else (V, self.Vp)


def _shapes(d):
    G, c = d.G, d.c
    return {EMB: (V, E), ATT_IH: (G, E + F + 2 * H), ATT_HH: (G, H), ATT_BIH: (1, G), ATT_BHH: (1, G), QP: (A, H),
            IP: (A, F), AVEC: (1, A), ENC_IH: (G, F + 2 * H + c), ENC_HH: (G, H), ENC_BIH: (1, G), ENC_BHH: (1, G),
            DEC_IH: (G, F + 2 * H + c + Z), DEC_HH: (G, H), DEC_BIH: (1, G), DEC_BHH: (1, G), FCM_W: (Z, H),
            FCM_B: (1, Z), FCL_W: (Z, H), FCL_B: (1, Z), OUT_W: (d.NO, H), OUT_B: (1, d.NO)}


def _regions(d):
    """Byte offset and size of every region of the packed buffer: in order, each rounded up to 1 KB."""
    b, G = 2, d.G
    sizes = [("w_att_rec", d.GP * 2 * d.Hp * b), ("wq", A * d.Hp * b), ("w_enc_x", d.GP * d.KX * b),
             ("w_enc_hh", d.GP * d.Hp * b)]
    if d.cvar:
        sizes.append(("w_enc_c", d.GP * d.Cp * b))
    sizes += [("w_fc", 2 * Z * d.Hp * b), ("w_dec_x", d.GP * d.KX * b), ("w_dec_z", d.GP * d.ZC * b), ("fwd_end", 0),
              ("w_dec_xzT", (d.KX + d.ZC) * d.Gp * b), ("w_fcT", d.Hp * d.Z2p * b),
              ("w_enc_xhT", (d.KX + d.Hp + d.Cp) * d.Gp * b), ("wqT", d.Hp * d.Ap * b),
              ("w_att_recT", 2 * d.Hp * d.Gp * b), ("bwd_end", 0), ("embb", V * d.Ep * b)]
    if d.tied:
        sizes.append(("embT", E * d.Vp * b))
    sizes += [("w_att_e", d.GP * d.Ep * b), ("w_att_eT", d.Ep * d.Gp * b), ("w_att_f", d.GP * d.Fp * b),
              ("wv", A * d.Fp * b), ("w_out", d.NO * d.Hp * b), ("w_outT", d.Hp * d.NOp * b), ("b_att", G * 4),
              ("b_enc", G * 4), ("b_dec", G * 4), ("scol_enc", G * 4), ("scol_dec", G * 4), ("b_fc", 2 * Z * 4)]
    out, off = {}, 0
    for name, n in sizes:
        out[name] = (off, n)
        off += (n + 1023) // 1024 * 1024
    return out, off


def _reference(d):
    """(weight, fold partner, first column, columns) -> images {(kind, region, element offset, ld, gate_H)}."""
    G, Gp, c = d.G, d.Gp, d.c
    ref = {}

    def add(w, w2, c0, cols, *outs):
        if cols > 0:
            ref[(w, w2, c0, cols)] = set(outs)
    add(EMB, -1, 0, E, (PLAIN, "embb", 0, d.Ep, 0), *([(TRANS, "embT", 0, d.Vp, 0)] if d.tied else []))
    add(ATT_IH, -1, 0, E, (PLAIN, "w_att_e", 0, d.Ep, H), (TRANS, "w_att_eT", 0, Gp, 0))
    add(ATT_IH, -1, E, F, (PLAIN, "w_att_f", 0, d.Fp, H))
    add(ATT_IH, ATT_HH, E + F, H, (PLAIN, "w_att_rec", 0, 2 * d.Hp, H), (TRANS, "w_att_recT", 0, Gp, 0))
    add(ATT_IH, -1, E + F + H, H, (PLAIN, "w_att_rec", d.Hp, 2 * d.Hp, H), (TRANS, "w_att_recT", d.Hp * Gp, Gp, 0))
    add(ATT_BIH, ATT_BHH, 0, G, (F32, "b_att", 0, G, 0))
    add(QP, -1, 0, H, (PLAIN, "wq", 0, d.Hp, 0), (TRANS, "wqT", 0, d.Ap, 0))
    add(IP, -1, 0, F, (PLAIN, "wv", 0, d.Fp, 0))
    add(AVEC, -1, 0, A)
    src, dst = (0, F, F + H), (0, d.Fp, d.Fp + d.Hp)
    for k, width in enumerate((F, H, H)):
        add(ENC_IH, -1, src[k], width, (PLAIN, "w_enc_x", dst[k], d.KX, H), (TRANS, "w_enc_xhT", dst[k] * Gp, Gp, 0))
        add(DEC_IH, DEC_HH if k == 2 else -1, src[k], width, (PLAIN, "w_dec_x", dst[k], d.KX, H),
            (TRANS, "w_dec_xzT", dst[k] * Gp, Gp, 0))
    if d.cvar:
        add(ENC_IH, -1, F + 2 * H, c, (PLAIN, "w_enc_c", 0, d.Cp, H), (TRANS, "w_enc_xhT", (d.KX + d.Hp) * Gp, Gp, 0))
        add(DEC_IH, -1, F + 2 * H, c, (PLAIN, "w_dec_z", d.Zp, d.ZC, H), (TRANS, "w_dec_xzT", (d.KX + d.Zp) * Gp, Gp, 0))
    else:                                                       # the sentiment column stays fp32, one value per gate row
        add(ENC_IH, -1, F + 2 * H, c, (F32, "scol_enc", 0, 1, 0))
        add(DEC_IH, -1, F + 2 * H, c, (F32, "scol_dec", 0, 1, 0))
    add(ENC_HH, -1, 0, H, (PLAIN, "w_enc_hh", 0, d.Hp, H), (TRANS, "w_enc_xhT", d.KX * Gp, Gp, 0))
    add(ENC_BIH, ENC_BHH, 0, G, (F32, "b_enc", 0, G, 0))
    add(DEC_IH, -1, F + 2 * H + c, Z, (PLAIN, "w_dec_z", 0, d.ZC, H), (TRANS, "w_dec_xzT", d.KX * Gp, Gp, 0))
    add(DEC_BIH, DEC_BHH, 0, G, (F32, "b_dec", 0, G, 0))
    add(FCM_W, -1, 0, H, (PLAIN, "w_fc", 0, d.Hp, 0), (TRANS, "w_fcT", 0, d.Z2p, 0))
    add(FCL_W, -1, 0, H, (PLAIN, "w_fc", Z * d.Hp, d.Hp, 0), (TRANS, "w_fcT", Z, d.Z2p, 0))
    add(FCM_B, -1, 0, Z, (F32, "b_fc", 0, Z, 0))
    add(FCL_B, -1, 0, Z, (F32, "b_fc", Z, Z, 0))
    add(OUT_W, -1, 0, H, (PLAIN, "w_out", 0, d.Hp, 0), (TRANS, "w_outT", 0, d.NOp, 0))
    add(OUT_B, -1, 0, d.NO)
    return ref


def _jobs(sv, le, tied):
    L = _lib.lib()
    dims = _lib.SscvaeDims(F, E, H, A, Z, V, 20, sv, 0, tied, 0, 1, 1.0, 0.5, le)
    h = ctypes.c_void_p()
    _lib.check(L.sscvae_create(ctypes.byref(dims), ctypes.byref(h)))
    try:
        out = (ctypes.c_int64 * (16 * 64))()
        n = L.sscvae_debug_sgd_pack_jobs(h, out, 64)
        _lib.check(min(n, 0))
        total = L.sscvae_packed_bytes(h)
    finally:
        L.sscvae_destroy(h)
    return np.array(out[:16 * n], dtype=np.int64).reshape(n, 16), total


def _gate_row(k, j):
    return (j >> 5) * 128 + k * 32 + (j & 31)


@pytest.mark.parametrize("sv,le,tied", [(1, 0, 1), (1, 0, 0), (2, 0, 1), (2, 1, 0), (0, 0, 1)])
def test_source_blocks_partition_the_weights_and_write_the_packed_layout_once(sv, le, tied):
    d = _D(sv, le, tied)
    jobs, total = _jobs(sv, le, tied)
    regions, planned = _regions(d)
    assert total == planned
    shapes = _shapes(d)
    # every element of every weight is updated by exactly one job
    cover = {w: np.zeros(s, np.uint8) for w, s in shapes.items()}
    for w, w2, c0, rows, cols, ld, ld2 in jobs[:, :7]:
        assert (rows, ld) == shapes[w]
        cover[w][:, c0:c0 + cols] += 1
        if w2 >= 0:
            assert (rows, cols) == shapes[w2] and ld2 == shapes[w2][1]
            cover[w2] += 1
    for w, cnt in cover.items():
        assert (cnt == 1).all(), w
    # the jobs' images are the reference layout's, from the same source blocks
    got = {}
    for j in jobs:
        w, w2, c0, rows, cols, ld, ld2, nout = (int(x) for x in j[:8])
        outs = set()
        for k in range(nout):
            kind, off, old, gh = (int(x) for x in j[8 + 4 * k:12 + 4 * k])
            esz = 4 if kind == F32 else 2
            name = max((n for n, (o, _) in regions.items() if o <= off and regions[n][1] > 0), key=lambda n: regions[n][0])
            outs.add((kind, name, (off - regions[name][0]) // esz, old, gh))
        assert (w, w2, c0, cols) not in got
        got[(w, w2, c0, cols)] = outs
    assert got == _reference(d)
    # every byte is written at most once, inside its region's logical extent; padding stays untouched
    count = np.zeros(total // 2, np.uint8)                     # per bf16 element (an fp32 element is two)
    for j in jobs:
        w, w2, c0, rows, cols, ld, ld2, nout = (int(x) for x in j[:8])
        for k in range(nout):
            kind, off, old, gh = (int(x) for x in j[8 + 4 * k:12 + 4 * k])
            name = max((n for n, (o, _) in regions.items() if o <= off and regions[n][1] > 0), key=lambda n: regions[n][0])
            r_off, r_bytes = regions[name]
            if kind == F32:
                e0, n_el = off // 2, rows * cols
                assert off % 4 == 0 and (rows == 1 or old == 1 and cols == 1)
                assert off + 4 * n_el <= r_off + r_bytes
                count[e0:e0 + 2 * n_el] += 1
                continue
            assert off % 2 == 0
            if kind == PLAIN:
                drows = np.array([_gate_row(r // gh, r % gh) for r in range(rows)]) if gh else np.arange(rows)
                dcols = cols
            else:
                drows, dcols = np.arange(cols), rows
            # rows of the image are distinct, and no row runs past the leading dimension into the padding columns
            assert len(np.unique(drows)) == len(drows) and (off - r_off) // 2 % old + dcols <= old
            assert off + 2 * (int(drows.max()) * old + dcols) <= r_off + r_bytes, name
            count[off // 2 + drows[:, None] * old + np.arange(dcols)[None, :]] += 1
    assert count.max() == 1
    images = sum(int(j[3]) * int(j[4]) * (2 if int(j[8 + 4 * k]) == F32 else 1) for j in jobs for k in range(int(j[7])))
    assert int(count.sum()) == images
