"""Exact JSON round trip for golden records of the reference's Python objects (tests/golden/*.json.xz).

Plain JSON loses what the differential tests compare: tuples become lists, dict keys become strings and key order
is not part of equality.  `encode` tags dicts (as ordered key/value pairs), tuples and numpy arrays so that
`decode(encode(x)) == x` holds with the same types, keys and insertion order.  Floats round-trip exactly (repr)."""
import hashlib
import json
import lzma

import numpy as np


def encode(x):
    if isinstance(x, dict):
        return {'d': [[encode(k), encode(v)] for k, v in x.items()]}
    if isinstance(x, tuple):
        return {'t': [encode(v) for v in x]}
    if isinstance(x, list):
        return [encode(v) for v in x]
    if isinstance(x, np.ndarray):
        return {'a': x.tolist(), 'dtype': x.dtype.str}
    if isinstance(x, np.generic):
        return x.item()
    assert x is None or isinstance(x, (bool, int, float, str)), type(x)
    return x


def decode(x):
    if isinstance(x, list):
        return [decode(v) for v in x]
    if isinstance(x, dict):
        if 'd' in x:
            return {decode(k): decode(v) for k, v in x['d']}
        if 't' in x:
            return tuple(decode(v) for v in x['t'])
        return np.array(x['a'], dtype=x['dtype'])
    return x


def digest(x):
    """sha256 of the encoded object: a compact stand-in for a record too large to store."""
    return hashlib.sha256(json.dumps(encode(x), separators=(',', ':')).encode()).hexdigest()


def save(path, record):
    with lzma.open(path, 'wb', preset=9) as f:
        f.write(json.dumps(encode(record), separators=(',', ':')).encode())


def load(path):
    with lzma.open(path, 'rb') as f:
        return decode(json.loads(f.read()))
