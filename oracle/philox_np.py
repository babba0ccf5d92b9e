"""Host restatement of the project's random numbers: Philox4x32-10, the 24-bit uniforms and Box-Muller.  Oracle: test
infrastructure only.

* ``philox4x32_10``: the counter-based generator of Salmon, Moraes, Dror and Shaw ("Parallel random numbers: as easy as
  1, 2, 3", SC'11), vectorised over numpy ``uint32`` arrays: ten rounds of two 32 x 32 -> 64-bit multiplications by
  0xD2511F53 / 0xCD9E8D57 whose high halves are xor-ed with the other two counter words and the key, the key bumped by the
  Weyl constants 0x9E3779B9 / 0xBB67AE85 between rounds.  ``KAT`` holds Random123's known-answer vectors.
* ``u01`` / ``u01_low_bytes``: ``((float)k + 0.5f) * 2^-24`` in IEEE float32 round-to-nearest-even, bit for bit.  For
  ``k >= 2^23`` the sum ``k + 0.5`` is a tie between two float32 neighbours and rounds to the even one: the uniforms of the
  upper half sit on the 2^-23 grid, and ``k = 2^24 - 1`` gives exactly 1.0.
* ``box_muller_f64``: the float64 Box-Muller normals of those exact float32 uniforms, ``sqrt(-2 ln u1) (cos, sin)(2 pi u2)``,
  with a per-element bound on what the device's ``box_muller`` (csrc/common.cuh: ``__logf``, correctly rounded ``sqrtf``,
  the FP32 angle ``2 pi u2 - pi`` and ``__sincosf``) can return.
* ``mh_words`` / ``draws_f64``: the counters of the samplers' draws and the reference ``dvae_rng_dump`` output built from them.
"""
from __future__ import annotations

import numpy as np

MASK32 = np.uint64(0xFFFFFFFF)
PHILOX_M = (np.uint64(0xD2511F53), np.uint64(0xCD9E8D57))
PHILOX_W = (np.uint32(0x9E3779B9), np.uint32(0xBB67AE85))

# Random123 (kat_vectors): counter, key -> output, Philox4x32 with 10 rounds
KAT = [
    ((0, 0, 0, 0), (0, 0), (0x6627E8D5, 0xE169C58D, 0xBC57AC4C, 0x9B00DBD8)),
    ((0xFFFFFFFF,) * 4, (0xFFFFFFFF,) * 2, (0x408F276D, 0x41C83B0E, 0xA20BC7C6, 0x6D5451FD)),
    ((0x243F6A88, 0x85A308D3, 0x13198A2E, 0x03707344), (0xA4093822, 0x299F31D0),
     (0xD16CFE09, 0x94FDCCEB, 0x5001E420, 0x24126EA1)),
]

U32 = 2.0 ** -24                       # FP32 unit roundoff
LOGF_ABS = 2.0 ** -21.41               # __logf on [0.5, 2]: absolute error (CUDA C++ Programming Guide, intrinsic functions)
LOGF_ULP = 3                           # __logf elsewhere: ulp error
SINF_ABS = 2.0 ** -21.41               # __sinf on [-pi, pi]
COSF_ABS = 2.0 ** -21.19               # __cosf on [-pi, pi]
TWO_PI_F32 = float(np.float32(2 * np.pi))
PI_F32 = float(np.float32(np.pi))


def _u32(x):
    """Integers (any sign, any integer dtype) mod 2^32 as uint32."""
    return (np.asarray(x).astype(np.int64) & 0xFFFFFFFF).astype(np.uint32)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Philox4x32-10 of counter ``(c0, c1, c2, c3)`` under key ``(k0, k1)``; arguments broadcast, integers taken mod 2^32.
    Returns four ``uint32`` arrays."""
    c = [v.astype(np.uint64) for v in np.broadcast_arrays(*[_u32(v) for v in (c0, c1, c2, c3)])]
    k = [np.uint64(int(k0) & 0xFFFFFFFF), np.uint64(int(k1) & 0xFFFFFFFF)]
    w = [np.uint64(PHILOX_W[0]), np.uint64(PHILOX_W[1])]
    for r in range(10):
        if r:
            k = [(k[0] + w[0]) & MASK32, (k[1] + w[1]) & MASK32]
        p0 = PHILOX_M[0] * c[0]                       # < 2^64: exact in uint64
        p1 = PHILOX_M[1] * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k[0], p1 & MASK32, (p0 >> np.uint64(32)) ^ c[3] ^ k[1], p0 & MASK32]
    return tuple(v.astype(np.uint32) for v in c)


def u01(r):
    """``((float)(r >> 8) + 0.5f) * 2^-24`` in float32: in (0, 1], 1.0 for ``r >> 8 == 2^24 - 1``."""
    k = (_u32(r) >> np.uint32(8)).astype(np.float32)
    return (k + np.float32(0.5)) * np.float32(2.0 ** -24)


def u01_low_bytes(x, y, z):
    """The accept uniform: the low bytes of three words as a 24-bit integer, through the same float32 arithmetic as ``u01``."""
    v = (_u32(x) & np.uint32(255)) | ((_u32(y) & np.uint32(255)) << np.uint32(8)) | ((_u32(z) & np.uint32(255)) << np.uint32(16))
    return (v.astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)


def _ulp32(x):
    """One float32 ulp at |x| (float64 in, float64 out); 2^-149 at 0."""
    a = np.abs(np.asarray(x, np.float64)).astype(np.float32)
    return (np.nextafter(a, np.float32(np.inf)) - a).astype(np.float64)


def box_muller_f64(a, b):
    """``(n0, n1, bound0, bound1)`` float64 for the words ``a`` (radius) and ``b`` (angle).

    Centre: ``r (cos t, sin t)`` with ``r = sqrt(-2 ln u1)``, ``t = 2 pi u2``, ``u1, u2`` the exact float32 uniforms.  The bound
    covers the device arithmetic ``n0 = -r' cos(t'), n1 = -r' sin(t')``, ``t' = fl(fl(2 pi) u2 - fl(pi))``:

    * ``L = __logf(u1)``: ``2^-21.41`` absolute on [0.5, 2], 3 ulp elsewhere;
    * ``r' = sqrtf(-2 L)`` correctly rounded.  ``-2 L`` is exact, so ``|r'^2 - r^2| <= 2 |L - ln u1|`` up to the square root's
      rounding, and ``|r' - r| <= min(sqrt(|r'^2 - r^2|), |r'^2 - r^2| / r)``: finite at ``r = 0`` (u1 = 1), where a
      relative error of ``r`` is not;
    * the angle: the float32 constants ``fl(2 pi)``, ``fl(pi)`` and the roundings of the product and the difference (also
      covers an FMA, which rounds once).  ``cos(t' )`` moves by at most ``|t' - (t - pi)|`` (Lipschitz 1);
    * ``__sincosf``: ``2^-21.41`` (sin) and ``2^-21.19`` (cos) absolute on [-pi, pi].  ``u2 = 1`` gives ``t' = fl(pi)``, one
      float32 step past pi; the hardware reduces the argument by a multiplication with 1 / (2 pi), so the bound is taken to
      hold there too (the sweep of every ``u2`` on the device checks it);
    * the FP32 product ``-r' c'``: ``u |n|``.
    """
    u1 = u01(a).astype(np.float64)
    u2 = u01(b).astype(np.float64)
    lnu = np.log(u1)
    r = np.sqrt(-2.0 * lnu)
    t = 2.0 * np.pi * u2
    n0, n1 = r * np.cos(t), r * np.sin(t)
    # __logf
    e_log = np.where((u1 >= 0.5) & (u1 <= 2.0), LOGF_ABS, LOGF_ULP * _ulp32(lnu) * 1.0000001)
    e_sq = 2.0 * e_log                                             # |(-2L) - r^2|
    e_r = np.minimum(np.sqrt(e_sq), e_sq / np.where(r > 0, r, 1.0)) # through r^2
    e_r = np.where(r > 0, e_r, np.sqrt(e_sq))
    e_r = e_r + U32 * (r + e_r)                                    # sqrtf rounding
    # angle t' against t - pi
    prod = TWO_PI_F32 * u2
    e_ang = abs(TWO_PI_F32 - 2 * np.pi) * u2 + abs(PI_F32 - np.pi) + U32 * prod + U32 * (np.abs(prod - PI_F32) + U32 * prod)
    bounds = []
    for n, e_mufu in ((n0, COSF_ABS), (n1, SINF_ABS)):
        trig = np.abs(n) / np.where(r > 0, r, 1.0)                  # |cos t| or |sin t|
        e_trig = e_mufu + e_ang
        e = e_r * (trig + e_trig) + r * e_trig
        e = e + U32 * ((r + e_r) * (trig + e_trig))                  # the FP32 product r' c'
        bounds.append(e + 1e-15 * (r + 1.0))                        # float64 evaluation of the centre
    return n0, n1, bounds[0], bounds[1]


def mh_words(seed, utt, frame_chain, it, block):
    """The four Philox words of a draw block: counter (utterance id, frame | chain << 20, iteration, block), key = seed."""
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    return philox4x32_10(utt, frame_chain, it, block, seed & 0xFFFFFFFF, seed >> 32)


def draws_f64(seed, frame_gid, frame_idx, n_chains, L, n_iter, iter0=0, iter0_frame=None):
    """What ``dvae_rng_dump`` returns, restated: ``(eps [n_iter][NT*C][L] float64, bound [same], u [n_iter][NT*C] float32)``.
    Chain row ``m = frame * C + c`` draws from counter ``(frame_gid, frame_idx | c << 20, iter0(frame) + it mod 2^32, b)``;
    block ``b`` gives normals ``4b .. 4b+3`` (Box-Muller of words (x, y) and (z, w)), block 0 also the accept uniform."""
    gid = _u32(frame_gid)
    idx = _u32(frame_idx)
    NT = len(gid)
    chains = NT * n_chains
    fr = np.repeat(np.arange(NT), n_chains)
    c = np.tile(np.arange(n_chains, dtype=np.uint32), NT)
    base = _u32(np.full(NT, iter0, np.int64) if iter0_frame is None else iter0_frame)
    it = (base[fr][None, :].astype(np.uint64) + np.arange(n_iter, dtype=np.uint64)[:, None]) & MASK32     # [n_iter][chains]
    utt = np.broadcast_to(gid[fr][None, :], it.shape)
    fc = np.broadcast_to((idx[fr] | (c << np.uint32(20)))[None, :], it.shape)
    nb = (L + 3) // 4
    eps = np.empty((n_iter, chains, 4 * nb))
    bnd = np.empty_like(eps)
    u = None
    for blk in range(nb):
        x, y, z, w = mh_words(seed, utt, fc, it.astype(np.uint32), blk)
        if blk == 0:
            u = u01_low_bytes(x, y, z)
        n0, n1, b0, b1 = box_muller_f64(x, y)
        n2, n3, b2, b3 = box_muller_f64(z, w)
        eps[..., 4 * blk:4 * blk + 4] = np.stack([n0, n1, n2, n3], -1)
        bnd[..., 4 * blk:4 * blk + 4] = np.stack([b0, b1, b2, b3], -1)
    return eps[..., :L], bnd[..., :L], u
