"""numpy oracle of the seeded-draw contract (include/nfdpm_b200.h, nfdpm_split_prior_sample_ex): Philox4x32-10 with
key = (lo32(seed), hi32(seed)) and counter = (e >> 2, stream, 0, 0); uniforms fp32((w >> 8) + 0.5) * 2^-24 computed in
fp32 exactly as the kernels do; Box-Muller in fp64 (the kernels' fp32 logf / sincospif differ from it by their rounding)."""
import numpy as np

M0, M1 = np.uint64(0xD2511F53), np.uint64(0xCD9E8D57)
W0, W1 = np.uint64(0x9E3779B9), np.uint64(0xBB67AE85)
MASK = np.uint64(0xFFFFFFFF)
PRIOR_STREAM = 0xFFFFFFFF


def philox4x32_10(ctr, key):
    """ctr [..., 4], key [..., 2] (uint32-valued) -> the four output words [..., 4] as uint32."""
    ctr, key = np.asarray(ctr, dtype=np.uint64), np.asarray(key, dtype=np.uint64)
    c = [ctr[..., i] for i in range(4)]
    k0, k1 = key[..., 0], key[..., 1]
    for _ in range(10):
        p0, p1 = M0 * c[0], M1 * c[2]
        c = [(p1 >> np.uint64(32)) ^ c[1] ^ k0, p1 & MASK, (p0 >> np.uint64(32)) ^ c[3] ^ k1, p0 & MASK]
        k0, k1 = (k0 + W0) & MASK, (k1 + W1) & MASK
    return np.stack(c, -1).astype(np.uint32)


def uniforms(words):
    """fp32((w >> 8) + 0.5) * 2^-24, in fp32 arithmetic like the kernels."""
    return ((words >> np.uint32(8)).astype(np.float32) + np.float32(0.5)) * np.float32(2.0 ** -24)


def normals(seeds, stream: int, n: int) -> np.ndarray:
    """The standard normals of elements e = 0..n-1 of the drawn tensor of each image: [len(seeds), n] float64."""
    s = np.asarray(seeds, dtype=np.int64).view(np.uint64)
    nq = (n + 3) // 4
    q = np.arange(nq, dtype=np.uint64)
    ctr = np.zeros((len(s), nq, 4), dtype=np.uint64)
    ctr[..., 0] = q[None, :]
    ctr[..., 1] = np.uint64(stream)
    key = np.stack([s & MASK, s >> np.uint64(32)], -1)[:, None, :]
    u = uniforms(philox4x32_10(ctr, np.broadcast_to(key, (len(s), nq, 2)))).astype(np.float64)
    r0, r2 = np.sqrt(-2.0 * np.log(u[..., 0])), np.sqrt(-2.0 * np.log(u[..., 2]))
    a1, a3 = 2.0 * np.pi * u[..., 1], 2.0 * np.pi * u[..., 3]
    out = np.stack([r0 * np.cos(a1), r0 * np.sin(a1), r2 * np.cos(a3), r2 * np.sin(a3)], -1)
    return out.reshape(len(s), 4 * nq)[:, :n]
