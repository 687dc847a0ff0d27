"""NumPy restatement of the epoch permutation of `knerf_generate_ray_batch` (include/knerf.h): a 4-round balanced
Feistel network on the smallest even bit width b >= 2 with 2^b >= P, keyed by the splitmix64 finaliser, cycle-walked
until the value is < P."""
import numpy as np

GOLDEN = np.uint64(0x9E3779B97F4A7C15)
ROUNDS = 4
M64 = (1 << 64) - 1


def mix64(z):
    z = np.asarray(z, dtype=np.uint64).copy()
    with np.errstate(over="ignore"):
        z ^= z >> np.uint64(30)
        z *= np.uint64(0xBF58476D1CE4E5B9)
        z ^= z >> np.uint64(27)
        z *= np.uint64(0x94D049BB133111EB)
        z ^= z >> np.uint64(31)
    return z


def epoch_key(perm_seed, epoch):
    a = int(mix64(np.uint64(perm_seed & M64)))
    b = (epoch * 0x9E3779B97F4A7C15 + 0xD1B54A32D192ED03) & M64
    return int(mix64(np.uint64(a ^ b)))


def half_bits(P):
    bits = 2
    while bits < 62 and (1 << bits) < P:
        bits += 2
    return bits // 2


def permute(idx, P, perm_seed, epoch):
    """pi_{seed, epoch}(idx) for positions idx (array-like, each < P) -> uint64 pixel ids"""
    key = np.uint64(epoch_key(perm_seed, epoch))
    half = np.uint64(half_bits(P))
    mask = np.uint64((1 << int(half)) - 1)

    def feistel(v):
        L, R = v >> half, v & mask
        with np.errstate(over="ignore"):
            for r in range(ROUNDS):
                F = mix64(R ^ (key + np.uint64(r) * GOLDEN)) & mask
                L, R = R, L ^ F
        return (L << half) | R

    v = feistel(np.asarray(idx, dtype=np.uint64))
    while True:
        out = v >= np.uint64(P)
        if not out.any():
            return v
        v[out] = feistel(v[out])
