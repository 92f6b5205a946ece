"""Public keys of many users for multi-key batches, built from the fixture key: its public key as it is, its relinearisation
key's residues replaced by seeded uniform residues below each limb's modulus (q0, q1, P), written with libzstd level 3 as
SEAL writes it.  oracle.bfv.mul_relin takes any relinearisation key, so every result stays checkable against the oracle."""
from __future__ import annotations

import os

import numpy as np

from oracle import bfv
from oracle import formats as F

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
KEY_MODULI = (0xFFFFEE001, 0xFFFFC4001, 0x1FFFFE0001)  # q0, q1, P


def user_key(seed: int, base: bytes | None = None) -> tuple[bytes, np.ndarray]:
    """(PublicKey bytes, rk [2][2][3][4096] u64) of user `seed`"""
    if base is None:
        base = open(os.path.join(ROOT, "tests/data/public_key.bin"), "rb").read()
    pkf = F.PublicKey.from_bytes(base)
    rel = pkf.relin()
    rng = np.random.default_rng(10_000 + seed)
    for kct in rel.keys[0]:
        data = np.empty((kct.size, kct.coeff_modulus_size, kct.poly_modulus_degree), dtype=np.uint64)
        for l, q in enumerate(KEY_MODULI):
            data[:, l, :] = rng.integers(0, q, size=(kct.size, kct.poly_modulus_degree), dtype=np.uint64)
        kct.data = data.reshape(np.shape(kct.data))
    blob = F.seal_wrap(rel.payload(), F.COMPR_ZSTD, 3)
    pub = F.PublicKey(pkf.public_key, pkf.galois_key, F.WithContext(pkf.relin_key.params, blob)).to_bytes()
    return pub, bfv.rk_array(rel)


def user_keys(k: int) -> list[tuple[bytes, np.ndarray]]:
    base = open(os.path.join(ROOT, "tests/data/public_key.bin"), "rb").read()
    return [user_key(j, base) for j in range(k)]
