"""Host reference of the in-kernel noise (csrc/sampler.cu, struct Philox), in numpy.

Philox4x32-10 (Salmon et al., "Parallel random numbers: as easy as 1, 2, 3", SC'11) vectorised over uint32 arrays, and the
project's layout of its counter and key:

  counter = (quad lo, quad hi, step word, (u32)sid ^ (u32)(sid >> 32) * 0x9E3779B9),   key = (seed lo, seed hi)
  step word = (step + 1) * 8 + draw          (x_T: dmn_randn(step = -1) -> word 0; PC: correctors draw k = 0..n_corr-1, the
                                              predictor draws 7; every other update kernel draws 0)
  quad      = flat NCHW element index over the whole batch / 4   (one quad = 4 consecutive elements)

`normal4` maps a quad to four N(0, 1) values by Box-Muller like the kernel, but evaluates log / sqrt / sincos in float64 from the
float32-rounded uniforms, so the kernel's only departures from it are its fast-math intrinsics (__logf, __sincosf).
"""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint32(0x9E3779B9), np.uint32(0xBB67AE85)
INV_2_32 = np.float32(2.3283064365386963e-10)
MASK32 = np.uint64(0xFFFFFFFF)


def philox4x32_10(c0, c1, c2, c3, k0, k1):
    """Ten rounds of Philox4x32 on uint32 arrays (broadcast together).  Returns four uint32 arrays."""
    c0, c1, c2, c3 = (np.asarray(c).astype(np.uint32) for c in (c0, c1, c2, c3))
    c0, c1, c2, c3 = np.broadcast_arrays(c0, c1, c2, c3)
    k0, k1 = np.uint32(int(k0) & 0xFFFFFFFF), np.uint32(int(k1) & 0xFFFFFFFF)
    with np.errstate(over="ignore"):
        for _ in range(10):
            p0 = M0 * c0.astype(np.uint64)
            p1 = M1 * c2.astype(np.uint64)
            hi0, lo0 = (p0 >> np.uint64(32)).astype(np.uint32), (p0 & MASK32).astype(np.uint32)
            hi1, lo1 = (p1 >> np.uint64(32)).astype(np.uint32), (p1 & MASK32).astype(np.uint32)
            c0, c1, c2, c3 = hi1 ^ c1 ^ k0, lo1, hi0 ^ c3 ^ k1, lo0
            k0, k1 = k0 + W0, k1 + W1
    return c0, c1, c2, c3


def step_word(step: int, draw: int = 0) -> int:
    """Third counter word of step `step` (0-based loop step; -1 = x_T) and draw slot `draw` (0..7)."""
    return ((int(step) + 1) * 8 + int(draw)) & 0xFFFFFFFF


def stream_word(stream_id: int) -> int:
    """Fourth counter word: the 64-bit stream id (the data-parallel rank) folded into 32 bits."""
    sid = int(stream_id) & 0xFFFFFFFFFFFFFFFF
    return ((sid & 0xFFFFFFFF) ^ (((sid >> 32) * 0x9E3779B9) & 0xFFFFFFFF)) & 0xFFFFFFFF


def raw_quads(seed: int, stream_id: int, word: int, quads):
    """uint32 [len(quads), 4] Philox outputs of the given quad indices (int array, may exceed 2^32)."""
    q = np.asarray(quads, dtype=np.uint64)
    seed = int(seed) & 0xFFFFFFFFFFFFFFFF
    r = philox4x32_10((q & MASK32).astype(np.uint32), (q >> np.uint64(32)).astype(np.uint32), np.uint32(word),
                      np.uint32(stream_word(stream_id)), seed & 0xFFFFFFFF, seed >> 32)
    return np.stack(r, axis=-1)


def uniforms(r):
    """The kernel's float32 uniforms of raw quads r [..., 4]: u0 = ((float)r.x + 1) * 2^-32 in (0, 1], u1 = (float)r.y * 2^-32 in
    [0, 1], same for (r.z, r.w).  numpy's uint32 -> float32 cast rounds to nearest like cvt.rn.f32.u32."""
    f = r.astype(np.float32)
    u = np.empty(r.shape, dtype=np.float32)
    u[..., 0::2] = (f[..., 0::2] + np.float32(1.0)) * INV_2_32
    u[..., 1::2] = f[..., 1::2] * INV_2_32
    return u


def box_muller(u):
    """float64 normals of float32 uniforms u [..., 4] in the kernel's output order (ra cos, ra sin, rb cos, rb sin)."""
    u = u.astype(np.float64)
    ra, rb = np.sqrt(-2.0 * np.log(u[..., 0])), np.sqrt(-2.0 * np.log(u[..., 2]))
    # the kernel's angle is 6.283185307179586f * u computed in float32
    a0 = (np.float32(6.283185307179586) * u[..., 1].astype(np.float32)).astype(np.float64)
    a1 = (np.float32(6.283185307179586) * u[..., 3].astype(np.float32)).astype(np.float64)
    return np.stack([ra * np.cos(a0), ra * np.sin(a0), rb * np.cos(a1), rb * np.sin(a1)], axis=-1)


def normal4(seed: int, stream_id: int, word: int, quads):
    """float64 [len(quads), 4] normals of the given quads."""
    return box_muller(uniforms(raw_quads(seed, stream_id, word, quads)))


def randn(seed: int, stream_id: int, step: int, n: int, draw: int = 0, chunk: int = 1 << 22):
    """float64 [n] normals of an n-element (n % 4 == 0) buffer: what dmn_randn(out, n, {seed, stream_id}, step) writes, and what
    every update kernel draws at loop step `step` with draw slot `draw`."""
    assert n % 4 == 0
    word = step_word(step, draw)
    out = np.empty(n, dtype=np.float64)
    for q0 in range(0, n // 4, chunk):
        q = np.arange(q0, min(n // 4, q0 + chunk), dtype=np.uint64)
        out[4 * q0:4 * (q0 + len(q))] = normal4(seed, stream_id, word, q).reshape(-1)
    return out
