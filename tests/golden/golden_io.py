"""On-disk layout of the reference-run golden sets (small_fwd, small_step, modules).

A golden set is a nested dict stored as a directory: one torch.save file per key.  A dict value whose file
would be larger than LIMIT becomes a subdirectory of the same kind, so every stored file stays under 1 MB while
the tests still compare against every value the reference produced.
"""
import io
import os

import torch

LIMIT = 1000000


def save_golden(path, d):
    os.makedirs(path, exist_ok=True)
    for k, v in d.items():
        buf = io.BytesIO()
        torch.save(v, buf)
        if buf.tell() <= LIMIT:
            with open(os.path.join(path, k + ".pt"), "wb") as f:
                f.write(buf.getvalue())
        elif isinstance(v, dict):
            save_golden(os.path.join(path, k), v)
        else:
            raise ValueError("golden value %s is %d bytes: store a dict of smaller parts" % (k, buf.tell()))


def load_golden(path):
    out = {}
    for name in sorted(os.listdir(path)):
        p = os.path.join(path, name)
        if os.path.isdir(p):
            out[name] = load_golden(p)
        elif name.endswith(".pt"):
            out[name[:-3]] = torch.load(p)
    return out
