"""Feature-matrix text files in the spellings np.savetxt and hand-edited files use, and the np.loadtxt path that
Model.from_text must reproduce bit for bit; shared by the host and GPU text-loading tests."""
import os

import numpy as np
import torch

FORMATS = ('%.18e', '%.17g', 'repr', '%.6f', '%g', 'int')


def matrix(rows, cols, seed, fmt):
    rng = np.random.default_rng(seed)
    a = rng.standard_normal((rows, cols)) * 10.0 ** rng.integers(-8, 9, size=(rows, cols))
    if fmt == 'int':
        a = np.round(a * 1000)
    return a


def write(path, a, fmt, seed=0, mess=False):
    """a as text in `fmt`; mess: tabs, CRLF line ends, blank and whitespace-only lines, comment lines and trailing comments"""
    rng = np.random.default_rng(seed)
    spell = (lambda x: repr(float(x))) if fmt == 'repr' else ((lambda x: '%d' % x) if fmt == 'int' else (lambda x: fmt % x))
    out = []
    if mess:
        out.append('# a comment line 1 2 3\n\n')
    for r, row in enumerate(a):
        seps = [rng.choice([' ', '\t', '  ', ' \t']) if mess else ' ' for _ in row]
        line = ''.join((seps[i] if i else ('\t' if mess and r % 3 == 0 else '')) + spell(x) for i, x in enumerate(row))
        if mess and r % 4 == 1:
            line += '  # trailing comment 7'
        out.append(line + ('\r\n' if mess and r % 2 else '\n'))
        if mess and r % 5 == 2:
            out.append(' \t \n' if r % 2 else '\n')
    with open(path, 'w', newline='') as f:
        f.write(''.join(out))
    return path


def case_files(tmp, V, Vd, seed, fmt, mess=False):
    paths = []
    for i, (name, shape) in enumerate((('pmi', (V, V)), ('pmi_w1', (V, V)), ('ed', (V, Vd)), ('ped', (V, Vd)))):
        paths.append(write(os.path.join(str(tmp), name + '.txt'), matrix(shape[0], shape[1], seed + i, fmt), fmt,
                           seed=seed + 10 + i, mess=mess))
    return paths


def loadtxt_model(Model, paths, device):
    """the np.loadtxt path (train.py:589-603 + Model.__init__)"""
    return Model(*[np.loadtxt(p, dtype=np.float64, ndmin=2) for p in paths], device=device)


def bits(x):
    return np.float64(x).view(np.uint64)


def assert_same_model(a, b):
    """planes bit-identical (padding included), ranges equal (NaN where the other is NaN)"""
    for name in ('pmi', 'w1', 'edT', 'pedT'):
        x, y = getattr(a, name), getattr(b, name)
        assert x.shape == y.shape and x.dtype == y.dtype == torch.float32, name
        assert torch.equal(x.cpu().view(torch.int32), y.cpu().view(torch.int32)), name
    for x, y in zip(a.frange + a.ed_range, b.frange + b.ed_range):
        assert (x == y) or (x != x and y != y), (a.frange, a.ed_range, b.frange, b.ed_range)
    assert (a.V, a.Vd, a.ld) == (b.V, b.Vd, b.ld)
