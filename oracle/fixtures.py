"""Storage of the golden fixtures in tests/golden (TEST INFRASTRUCTURE).

A fixture is a dict whose values are tensors, plain values or dicts of tensors (state_dict, grads, ...).  It is stored
as parts `<name>.<i>.pt` of at most PART_BYTES each, so that no stored file exceeds 1 MB; `load` reassembles the
dict with every key in its original order.
"""
import glob
import os

import torch

PART_BYTES = 900_000
_ENTRY_OVERHEAD = 512          # zip record + pickle bytes torch.save spends per tensor (measured: ~400)


def _nbytes(v):
    return (v.numel() * v.element_size() if torch.is_tensor(v) else 0) + _ENTRY_OVERHEAD


def _parts(directory, name):
    paths = glob.glob(os.path.join(directory, f"{name}.*.pt"))
    return sorted(paths, key=lambda p: int(p.rsplit(".", 2)[1]))


def save(obj, directory, name):
    entries = []          # (key, sub-key or None, value), in dict order
    for k, v in obj.items():
        if isinstance(v, dict):
            entries += [(k, k2, t) for k2, t in v.items()]
        else:
            entries.append((k, None, v))
    parts, cur, size = [], [], 0
    for e in entries:
        n = _nbytes(e[2])
        if n > PART_BYTES:
            raise ValueError(f"fixture {name}: entry {e[0]}/{e[1]} alone exceeds {PART_BYTES} bytes")
        if cur and size + n > PART_BYTES:
            parts.append(cur)
            cur, size = [], 0
        cur.append(e)
        size += n
    parts.append(cur)
    for p in _parts(directory, name):
        os.remove(p)
    for i, part in enumerate(parts):
        path = os.path.join(directory, f"{name}.{i}.pt")
        torch.save({"dicts": sorted({k for k, k2, _ in entries if k2 is not None}), "entries": part}, path)
        assert os.path.getsize(path) < 1_000_000, (path, os.path.getsize(path))


def load(directory, name):
    paths = _parts(directory, name)
    if not paths:
        raise FileNotFoundError(os.path.join(directory, f"{name}.*.pt"))
    out = {}
    for path in paths:
        blob = torch.load(path)
        for k, k2, v in blob["entries"]:
            if k in blob["dicts"]:
                out.setdefault(k, {})[k2] = v
            else:
                out[k] = v
    return out
