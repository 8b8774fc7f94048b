"""What the original project's own compiled code computed, stored under tests/golden/ (TEST INFRASTRUCTURE).

The tests that compare with the original's CPU library (eigenmat) or CUDA kernels read its results from here, so they
run on any machine.  With CONVNET_B200_RECORD_GOLDEN=1 and oracle/_ref/ built from the original's sources
(`make -C oracle` where they exist), the same tests run the original live instead, compare against its full outputs,
and rewrite the stored file when the module's tests finish.

An output is stored as its values at SAMPLE seeded positions (all of them when it is no larger).  An output that must
match bit for bit is stored as the SHA-256 of all its values, which covers every element, plus the values at every
EXACT_STRIDE-th of those positions for the failure message.  Arrays are numpy (Fortran-ordered cudamat layout) or flat
torch tensors: either way in memory order.
"""
import hashlib
import os
import zlib

import numpy as np

from oracle_lib import Diff

GOLDEN = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
RECORD = os.environ.get("CONVNET_B200_RECORD_GOLDEN") == "1"
SAMPLE = 256
EXACT_STRIDE = 16


def _index(key, n, exact):
    idx = np.arange(n) if n <= SAMPLE else np.sort(np.random.RandomState(zlib.crc32(key.encode())).randint(0, n, SAMPLE))
    return idx[::EXACT_STRIDE] if exact else idx


def _flat(a):
    if isinstance(a, np.ndarray):
        return np.ravel(a, order="K")
    return a.reshape(-1)


def _gather(a, idx):
    a = _flat(a)
    if isinstance(a, np.ndarray):
        return a[idx].astype(np.float32)
    import torch
    return a[torch.from_numpy(idx).to(a.device)].cpu().numpy()


def _digest(a):
    """SHA-256 of the values (-0.0 counted as 0.0, as a comparison of values does); None when one is NaN"""
    a = _flat(a)
    if not isinstance(a, np.ndarray):
        a = a.contiguous().cpu().numpy()
    a = np.ascontiguousarray(a, np.float32) + np.float32(0)
    return None if np.isnan(a).any() else hashlib.sha256(a.tobytes()).digest()


class Stored:
    """the original's output for one key as stored: element count, sampled values, digest (exact outputs only)"""

    def __init__(self, key, n, values, digest):
        self.key, self.n, self.values, self.digest = key, n, values, digest

    def index(self):
        return _index(self.key, self.n, self.digest is not None)


class RefStore:
    """one file of stored outputs: keys, element counts, the samples end to end, and digests (zero bytes: none)"""

    def __init__(self, name):
        self.path = os.path.join(GOLDEN, name + ".npz")
        self.items = {}
        if not RECORD:
            with np.load(self.path) as z:
                starts = z["starts"]
                for i, key in enumerate(z["keys"]):
                    digest = z["sha256"][i].tobytes()
                    self.items[str(key)] = Stored(str(key), int(z["n"][i]), z["values"][starts[i]:starts[i + 1]],
                                                  digest if any(digest) else None)

    def reference(self, key, compute, exact=False):
        """RECORD: run `compute()` (the original, live), keep what is stored of it, return the full output.
        Otherwise: the stored output of `key`."""
        if RECORD:
            full = compute()
            digest = _digest(full) if exact else None
            assert digest is not None or not exact, "%s: the original's output holds NaN" % key
            n = _flat(full).shape[0]
            self.items[key] = Stored(key, n, _gather(full, _index(key, n, exact)), digest)
            return full
        assert key in self.items, "%s: nothing stored for %s (record it with CONVNET_B200_RECORD_GOLDEN=1)" % (self.path, key)
        return self.items[key]

    def save(self):
        if not RECORD:
            return
        items = list(self.items.values())
        np.savez_compressed(self.path, keys=np.array([s.key for s in items]), n=np.array([s.n for s in items], np.int64),
                            starts=np.cumsum([0] + [len(s.values) for s in items]).astype(np.int64),
                            values=np.concatenate([s.values for s in items]).astype(np.float32),
                            sha256=np.array([np.frombuffer(s.digest or bytes(32), np.uint8) for s in items]))


def diff(ours, ref):
    """Diff (py/test_conv.py:382-385) of ours against the original: over every element when `ref` is the live output,
    over the stored sample otherwise"""
    if isinstance(ref, Stored):
        assert _flat(ours).shape[0] == ref.n, (ref.key, _flat(ours).shape[0], ref.n)
        return Diff(_gather(ours, ref.index()), ref.values)
    if isinstance(ref, np.ndarray):
        return Diff(ours, ref)
    import torch
    a, b = _flat(ours), _flat(ref)
    num = (a - b).abs().max().item()
    den = (a + b).abs().mean(dtype=torch.float64).item()
    return num / den if den > 0 else num


def equal(ours, ref):
    """bit-exact equality with the original's output, over every element (the stored digest covers all of them)"""
    if isinstance(ref, Stored):
        assert ref.digest is not None, "%s was stored without a digest" % ref.key
        return (_flat(ours).shape[0] == ref.n and np.array_equal(_gather(ours, ref.index()), ref.values)
                and _digest(ours) == ref.digest)
    if isinstance(ref, np.ndarray):
        return np.array_equal(ours, ref)
    import torch
    return torch.equal(_flat(ours), _flat(ref))
