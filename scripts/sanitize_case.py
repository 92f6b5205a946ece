"""Small end-to-end case for compute-sanitizer (memcheck / racecheck): every kernel once on a batch of 3."""
import os, sys
import numpy as np, torch
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT); sys.path.insert(0, os.path.join(ROOT, "tests"))
from fhe_precompiles_b200 import device as d
from helpers import KeySet, random_ct, MODULI, N
keys = KeySet.load()
d.init(0)
t = lambda a: torch.from_numpy(np.ascontiguousarray(a).view(np.int64)).cuda()
rng = np.random.default_rng(0)
a, b = t(random_ct(rng, 3)), t(random_ct(rng, 3))
rk, pk, sk = t(keys.net_rk), t(keys.net_pk), t(keys.net_sk)
pl = torch.randint(0, 4096, (3, N), dtype=torch.int16, device="cuda")
out = d.mul_relin(a, b, rk)
d.add(a, b); d.sub(a, b); d.negate(a); d.plain_addsub(a, pl, 3); d.multiply_plain(a, pl)
x = t(rng.integers(0, MODULI[3], size=(6, N), dtype=np.uint64)); d.ntt_(x, [3]); d.ntt_(x, [3], inverse=True)
ct = d.encrypt(pk, pl, torch.arange(3, dtype=torch.int64, device="cuda")); d.decrypt(ct, sk)
torch.cuda.synchronize()
print("sanitize case done", int(out[0,0,0,0]))
