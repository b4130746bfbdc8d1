"""Host reference of the in-kernel noise generator (``Philox`` in psld_b200/csrc/phase_space.cu).

Philox4x32-10 is counter based: every normal the device draws is a function of (key, stream, index)
alone, so the host can recompute any subset of a launch's noise and follow single pairs of a
sampler's state pathwise.  The arithmetic mirrors the device:

  counter = (index lo, index hi, stream lo, stream hi), key = (seed lo, seed hi)
  u0 = min((f32(r.x) + 0.5f) 2^-32, 0.99999994f), u1 = f32(r.y) 2^-32  (u2, u3 from r.z, r.w)
  angle = 6.283185307179586f * (u - 0.5f)           (float32, bit-identical to the device)
  z = (ra cos a, ra sin a, rb cos b, rb sin b),  ra = sqrt(-2 log u0)   (float64 here)

What remains is the device's ``logf`` (<= 1 ulp) and ``__sincosf`` (2^-21.41 absolute on [-pi, pi)):
|z_device - z_host| <= ~3.5e-6 at the 6.77-sigma tail.

(stream, index) rule of each entry point (include/psld_b200.h):
  PSLD state kernels (psld_sscs_update, psld_em_update[_guided], psld_prior_sample): the 4-pair
    vector v = b * chw/4 + j/4 draws index 2v for x[j..j+3] and 2v+1 for m[j..j+3];
    SSCS streams: HALF_A 2 step, HALF_B 2 step + 1, HALF_C 2 step + 2; EM: step; prior: 2^64 - 1
  psld_vp_em_update: stream step, index v = flat element / 4
  psld_inpaint_combine: streams (k << 2) | 2^62 | {0, 1, 2} for (z_m0, e_x, e_m), index v = flat / 4
"""
from __future__ import annotations

import numpy as np

M32 = 0xFFFFFFFF
M64 = (1 << 64) - 1
PRIOR_STREAM = M64


def philox4x32_10(counter, key):
    """Philox4x32-10 on uint32 words: ``counter`` four arrays (broadcast), ``key`` two scalars."""
    c0, c1, c2, c3 = np.broadcast_arrays(*(np.asarray(w, dtype=np.uint64) & np.uint64(M32)
                                           for w in counter))
    k0, k1 = int(key[0]) & M32, int(key[1]) & M32
    m0, m1, lo = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57), np.uint64(M32)
    for _ in range(10):
        p0, p1 = c0 * m0, c2 * m1                       # < 2^64: exact in uint64
        c0, c1, c2, c3 = ((p1 >> np.uint64(32)) ^ c1 ^ np.uint64(k0), p1 & lo,
                          (p0 >> np.uint64(32)) ^ c3 ^ np.uint64(k1), p0 & lo)
        k0 = (k0 + 0x9E3779B9) & M32
        k1 = (k1 + 0xBB67AE85) & M32
    return tuple(w.astype(np.uint32) for w in (c0, c1, c2, c3))


def draw(seed, stream, index):
    """Raw 4 x uint32 of one device draw; ``stream`` and ``index`` broadcast (uint64)."""
    idx = np.asarray(index, dtype=np.uint64)
    st = np.asarray(int(stream) & M64 if np.ndim(stream) == 0 else stream, dtype=np.uint64)
    s32 = np.uint64(32)
    seed = int(seed) & M64
    return philox4x32_10((idx, idx >> s32, st, st >> s32), (seed & M32, seed >> 32))


def normal4(seed, stream, index):
    """The device's 4 normals of draw (seed, stream, index) as float64 [..., 4]."""
    r = draw(seed, stream, index)
    k, half = np.float32(2.0 ** -32), np.float32(0.5)
    top, two_pi = np.float32(0.99999994), np.float32(6.283185307179586)
    u0 = np.minimum((r[0].astype(np.float32) + half) * k, top)
    u2 = np.minimum((r[2].astype(np.float32) + half) * k, top)
    a = two_pi * (r[1].astype(np.float32) * k - half)
    b = two_pi * (r[3].astype(np.float32) * k - half)
    ra = np.sqrt(-2.0 * np.log(u0.astype(np.float64)))
    rb = np.sqrt(-2.0 * np.log(u2.astype(np.float64)))
    a, b = a.astype(np.float64), b.astype(np.float64)
    return np.stack([ra * np.cos(a), ra * np.sin(a), rb * np.cos(b), rb * np.sin(b)], -1)


# ---- streams ---------------------------------------------------------------------------
def sscs_stream(step, stage):
    """Stream of an SSCS stage (``"a"``, ``"b"``, ``"c"``) at ``step``."""
    return (2 * int(step) + {"a": 0, "b": 1, "c": 2}[stage]) & M64


def inpaint_stream(k, which):
    """Stream of inpainting draw ``which`` (0: z_m0, 1: e_x, 2: e_m) of combine call ``k``."""
    return ((int(k) << 2) | (1 << 62) | int(which)) & M64


# ---- index rules -----------------------------------------------------------------------
def pair_normals_at(seed, stream, b, j, chw):
    """(z_x, z_m) the PSLD state kernels draw for pair j of sample b (arrays of any shape)."""
    b, j = np.asarray(b, dtype=np.int64), np.asarray(j, dtype=np.int64)
    v = (b * (chw // 4) + j // 4).astype(np.uint64)
    lane = j % 4
    zx = np.take_along_axis(normal4(seed, stream, 2 * v), lane[..., None], -1)[..., 0]
    zm = np.take_along_axis(normal4(seed, stream, 2 * v + 1), lane[..., None], -1)[..., 0]
    return zx, zm


def pair_normals(seed, stream, B, chw):
    """Whole-tensor (z_x, z_m), each float64 [B, chw]."""
    v = np.arange(B * chw // 4, dtype=np.uint64)
    zx = normal4(seed, stream, 2 * v).reshape(B, chw)
    zm = normal4(seed, stream, 2 * v + 1).reshape(B, chw)
    return zx, zm


def flat_normals_at(seed, stream, e):
    """Normal of flat element ``e`` under the flat rule (VP EM, inpainting)."""
    e = np.asarray(e, dtype=np.int64)
    z = normal4(seed, stream, (e // 4).astype(np.uint64))
    return np.take_along_axis(z, (e % 4)[..., None], -1)[..., 0]


def flat_normals(seed, stream, n):
    """Whole-tensor normals of ``n`` flat elements (n % 4 == 0), float64 [n]."""
    return normal4(seed, stream, np.arange(n // 4, dtype=np.uint64)).reshape(n)
