"""Writes tests/golden/reference_vectors.npz: the known answers of the reference's hash functions and frame-of-reference
page codec that tests/test_oracle_golden.py pins the oracle against, so that those tests run on any machine.

Inputs are drawn exactly as the tests drew them when they called the reference libraries (oracle/_ref, built from the
StarRocks tree by `make -C oracle ref`).  Expected values:
  xxh3_64      XXH3_64bits_withSeed of the xxHash library (the `xxhash` Python package; the reference vendors xxhash.h)
  fnv_hash     HashUtil::fnv_hash: h = (byte ^ h) * 0x01000193 per byte (hash_util.hpp:127-134)
  zlib_crc     HashUtil::zlib_crc_hash = zlib crc32(seed, bytes) (hash_util.hpp:34-45)
  crc_hash_32  CRC-32C (Castagnoli, reflected, no pre/post inversion) from the seed, then phmap_mix<4> (hash.h:25-33,96-130)
  FoR pages    the oracle's ForEncoder restatement (no independent implementation exists; the test holds these bytes
               to the reference's own ForEncoder wherever oracle/_ref/libfor_ref.so is built)
Every value is cross-checked against the oracle, and against the reference libraries where oracle/_ref holds them.

    python scripts/make_reference_vectors.py
"""
import os
import sys
import zlib

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)

from oracle import oracle  # noqa: E402
from tests.test_oracle_golden import _for_cases  # noqa: E402

OUT = os.path.join(ROOT, "tests", "golden", "reference_vectors.npz")
M32 = 0xFFFFFFFF


def fnv_hash(b, h):
    for x in b:
        h = ((x ^ h) * 0x01000193) & M32
    return h


def crc_hash_32(b, h):
    for x in b:
        h ^= x
        for _ in range(8):
            h = (h >> 1) ^ (0x82F63B78 if h & 1 else 0)
    m = (h * 0xCC9E2D51) & ((1 << 64) - 1)
    return (m ^ (m >> 32)) & M32


def xxh3_vectors(L, ref):
    import xxhash
    rng = np.random.default_rng(11)
    data, lens, seeds, want = [], [], [], []
    for n in range(1, 17):
        for k in range(200):
            buf = rng.integers(0, 256, n, dtype=np.uint8)
            seed = int(rng.integers(0, 1 << 63)) * 2 + int(rng.integers(0, 2))
            if k % 2:
                seed &= M32          # the exchange feeds 32-bit seeds
            h = xxhash.xxh3_64_intdigest(buf.tobytes(), seed=seed)
            assert L.orc_xxh3_64(buf.ctypes.data, n, seed) == h, (n, seed)
            if ref:
                assert ref.ref_xx_hash3_64(buf.ctypes.data, n, seed) == h, (n, seed)
            data.append(np.pad(buf, (0, 16 - n)))
            lens.append(n)
            seeds.append(seed)
            want.append(h)
    return {"xxh3_data": np.stack(data), "xxh3_len": np.array(lens, dtype=np.int32),
            "xxh3_seed": np.array(seeds, dtype=np.uint64), "xxh3_hash": np.array(want, dtype=np.uint64)}


def hash_vectors(L, ref):
    rng = np.random.default_rng(2)
    bufs, lens, seeds, fnv, zcrc, crc = [], [], [], [], [], []
    for n in list(range(0, 41)) + [100, 1000, 4097]:
        b = rng.integers(0, 256, max(n, 1), dtype=np.uint8)
        bufs.append(b[:n])
        for seed in (0, 0x811C9DC5, 12345):
            raw = b[:n].tobytes()
            got = (fnv_hash(raw, seed), zlib.crc32(raw, seed), crc_hash_32(raw, seed))
            assert got == (L.orc_fnv_hash(b.ctypes.data, n, seed), L.orc_zlib_crc32(b.ctypes.data, n, seed),
                           L.orc_crc_hash_32(b.ctypes.data, n, seed)), (n, seed)
            if ref:
                assert got == (ref.ref_fnv_hash(b.ctypes.data, n, seed), ref.ref_zlib_crc_hash(b.ctypes.data, n, seed),
                               ref.ref_crc_hash_32(b.ctypes.data, n, seed)), (n, seed)
            lens.append(n)
            seeds.append(seed)
            fnv.append(got[0])
            zcrc.append(got[1])
            crc.append(got[2])
    offs = np.cumsum([0] + [len(b) for b in bufs])
    return {"hash_bytes": np.concatenate(bufs), "hash_buf_offset": offs[:-1].repeat(3).astype(np.int64),
            "hash_len": np.array(lens, dtype=np.int32), "hash_seed": np.array(seeds, dtype=np.uint32),
            "fnv_hash": np.array(fnv, dtype=np.uint32), "zlib_crc_hash": np.array(zcrc, dtype=np.uint32),
            "crc_hash_32": np.array(crc, dtype=np.uint32)}


def for_vectors(ref):
    out = {}
    for dt in (np.int32, np.int64):
        for name, v in _for_cases(dt):
            page = oracle.for_encode(v)
            assert (oracle.for_decode(page, dt) == v).all(), name
            if ref:
                enc = ref.ref_for_encode_i32 if dt == np.int32 else ref.ref_for_encode_i64
                buf = np.zeros(len(v) * (v.dtype.itemsize * 8 + 2) + 64, dtype=np.uint8)
                n = enc(v.ctypes.data if len(v) else None, len(v), buf.ctypes.data, len(buf))
                if name in ("random_full_range", "extremes", "ascending_overflow"):   # format 2: the tail is undefined
                    used = v.dtype.itemsize * (1 + len(v))
                    assert page[-7:].tobytes() == buf[n - 7:n].tobytes(), name
                else:
                    used = len(page)
                assert n == len(page) and page[:used].tobytes() == buf[:used].tobytes(), name
            key = f"for_{np.dtype(dt).name}_{name}"
            out[key + "_values"] = v
            out[key + "_page"] = page
    return out


def main():
    L = oracle.lib()
    vec = {}
    vec.update(xxh3_vectors(L, oracle.ref_xxh3()))
    vec.update(hash_vectors(L, oracle.ref_hash()))
    vec.update(for_vectors(oracle.ref_for()))
    os.makedirs(os.path.dirname(OUT), exist_ok=True)
    np.savez_compressed(OUT, **vec)
    print(f"{OUT}: {len(vec)} arrays, {os.path.getsize(OUT)} bytes")


if __name__ == "__main__":
    main()
