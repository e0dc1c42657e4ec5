"""The text loader behind Model.from_text on the CPU, with the emulated K8 entry point (fake_text_kernels.py): chunk
carry-over at tiny chunk sizes, hard-field patching, every fall-back to np.loadtxt, and bit identity with the np.loadtxt path.  The last test compiles the
field conversion of csrc/parse.cu for the host and checks it against float()."""
import decimal
import os
import random
import shutil
import struct
import subprocess
import sys

import numpy as np
import pytest

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

from fake_kernels import FakeKernels  # noqa: E402
from fake_text_kernels import TextKernels  # noqa: E402
from text_load_cases import FORMATS, assert_same_model, case_files, loadtxt_model, write  # noqa: E402

from macaronicusermodeling_b200 import textload  # noqa: E402
from macaronicusermodeling_b200.engine import Model  # noqa: E402


def from_text(paths, V, Vd, chunk_bytes=None):
    """Model.from_text's GPU path (textload.model_from_text) on the emulated parser"""
    return textload.model_from_text(Model, paths, V, Vd, TextKernels(), chunk_bytes)


def _fallbacks(m):
    return getattr(m, 'load_stats', {'fallback': ['np.loadtxt path']})['fallback']


def test_back_end_without_gpu_takes_the_loadtxt_path(tmp_path):
    """Model.from_text with kernels whose device is the CPU (no GPU to parse on): np.loadtxt and Model(), no parser call"""
    paths = case_files(tmp_path, 5, 3, 8, '%.17g', mess=True)
    k = FakeKernels()
    m = Model.from_text(*paths, 5, 3, kernels=k)
    assert 'mlbp_parse_float_text' not in k.calls and not hasattr(m, 'load_stats')
    assert_same_model(m, loadtxt_model(Model, paths, 'cpu'))


@pytest.mark.parametrize('fmt', FORMATS)
@pytest.mark.parametrize('mess', [False, True])
def test_formats_bit_identical(tmp_path, fmt, mess):
    for V, Vd in ((1, 1), (1, 6), (9, 1), (13, 7)):
        paths = case_files(tmp_path, V, Vd, 11, fmt, mess)
        m = from_text(paths, V, Vd, chunk_bytes=4093)
        assert not _fallbacks(m)
        assert_same_model(m, loadtxt_model(Model, paths, 'cpu'))


def test_chunk_carry_at_tiny_chunks(tmp_path):
    paths = case_files(tmp_path, 3, 2, 5, '%.18e', mess=True)
    want = loadtxt_model(Model, paths, 'cpu')
    for cb in range(1, 65):
        m = from_text(paths, 3, 2, chunk_bytes=cb)
        assert not _fallbacks(m), cb
        assert_same_model(m, want)
        assert m.load_stats['bytes'] == sum(os.path.getsize(p) for p in paths)


def _halfway_strings(n, seed, digits=(20, 25, 40)):
    """decimal strings exactly halfway between adjacent doubles (and one unit of the last digit either side)"""
    decimal.getcontext().prec = 1200
    rng = random.Random(seed)
    out = []
    while len(out) < n:
        x = rng.uniform(0.5, 2.0) * 10.0 ** rng.randint(-300, 300)
        mid = (decimal.Decimal(x) + decimal.Decimal(float(np.nextafter(x, np.inf)))) / 2
        for nd in digits:
            s = format(mid, '.%de' % (nd - 1))
            m, e = s.split('e')
            ulp = decimal.Decimal(1).scaleb(-(nd - 1))
            out += [s, str(decimal.Decimal(m) + ulp) + 'e' + e, str(decimal.Decimal(m) - ulp) + 'e' + e]
    return out[:n]


def test_hard_fields_are_patched(tmp_path):
    V, Vd = 8, 5
    paths = case_files(tmp_path, V, Vd, 2, '%.17g')
    vals = _halfway_strings(V * V, 1)
    with open(paths[0], 'w') as f:
        for r in range(V):
            f.write(' '.join(vals[r * V:(r + 1) * V]) + '\n')
    m = from_text(paths, V, Vd, chunk_bytes=100)
    assert not _fallbacks(m)
    assert m.load_stats['hard_fields'] > 0
    assert_same_model(m, loadtxt_model(Model, paths, 'cpu'))


def test_too_many_hard_fields_fall_back(tmp_path, monkeypatch):
    V, Vd = 4, 3
    paths = case_files(tmp_path, V, Vd, 2, '%g')
    with open(paths[1], 'w') as f:
        vals = _halfway_strings(V * V, 2, digits=(40,))
        f.write('\n'.join(' '.join(vals[r * V:(r + 1) * V]) for r in range(V)) + '\n')
    monkeypatch.setattr(textload, 'HARD_CAP', 1)
    with pytest.warns(RuntimeWarning, match='significant digits'):
        m = from_text(paths, V, Vd)
    assert len(_fallbacks(m)) == 1
    assert_same_model(m, loadtxt_model(Model, paths, 'cpu'))


def _replace(path, text):
    with open(path, 'wb') as f:
        f.write(text)


@pytest.mark.parametrize('kind, text, why', [
    ('non-ASCII comment', b'1 2\n3 4  # caf\xc3\xa9\n', 'byte outside'),
    ('file separator byte', b'1\x1c2\n3 4\n', 'first line'),
    ('lone carriage return', b'1 2\r3 4\n', 'first line'),         # a line break to np.loadtxt's universal newlines
    ('vertical tab and form feed', None, None),
])
def test_fallback_loads_what_numpy_loads(tmp_path, kind, text, why):
    paths = case_files(tmp_path, 2, 3, 4, '%.6f')
    if text is None:                                       # \v and \f are separators on the device too: no fall-back
        _replace(paths[0], b'1\x0b2\n3\x0c4\n')
        m = from_text(paths, 2, 3)
        assert not _fallbacks(m)
    else:
        _replace(paths[0], text)
        with pytest.warns(RuntimeWarning, match=why):
            m = from_text(paths, 2, 3)
        assert len(_fallbacks(m)) == 1
    assert_same_model(m, loadtxt_model(Model, paths, 'cpu'))


@pytest.mark.parametrize('text', [b'1 2\n3\n', b'1 2\n3 4 5\n', b'1_000 2\n3 4\n', b'0x10 2\n3 4\n', b'1d5 2\n3 4\n',
                                  b'1e 2\n3 4\n', b'. 2\n3 4\n', b'1,2 3\n3 4\n', b'infin 2\n3 4\n'])
def test_invalid_file_raises_numpys_error(tmp_path, text):
    paths = case_files(tmp_path, 2, 3, 4, '%.6f')
    _replace(paths[0], text)
    with pytest.raises(Exception) as want:
        loadtxt_model(Model, paths, 'cpu')
    with pytest.warns(RuntimeWarning):
        with pytest.raises(want.type) as got:
            from_text(paths, 2, 3)
    assert str(got.value) == str(want.value)


@pytest.mark.parametrize('V, Vd', [(3, 2), (2, 4), (1, 2)])
def test_shape_other_than_vocabularies_takes_the_loadtxt_path(tmp_path, V, Vd):
    """the matrices are 2 x 3 / 2 x 2: vocabularies of another size send every file through np.loadtxt and Model()"""
    paths = case_files(tmp_path, 2, 3, 4, '%.6f')
    with pytest.warns(RuntimeWarning):
        m = from_text(paths, V, Vd)
    assert_same_model(m, loadtxt_model(Model, paths, 'cpu'))


def test_extra_rows_fall_back(tmp_path):
    paths = case_files(tmp_path, 2, 3, 4, '%.6f')
    with open(paths[2], 'a') as f:
        f.write('1 2 3\n')
    with pytest.raises(AssertionError):                   # Model() refuses ed of 3 rows with pmi of 2, as before
        loadtxt_model(Model, paths, 'cpu')
    with pytest.warns(RuntimeWarning, match='more rows'):
        with pytest.raises(AssertionError):
            from_text(paths, 2, 3)


def test_field_conversion_matches_float(tmp_path):
    """parse_field / eisel_lemire of csrc/parse.cu, compiled for the host, against CPython's correctly rounded float()"""
    nvcc = os.environ.get('NVCC', '/usr/local/cuda/bin/nvcc')
    if not os.path.exists(nvcc) and not shutil.which('nvcc'):
        pytest.skip('no nvcc')
    csrc = os.path.join(os.path.dirname(HERE), 'macaronicusermodeling_b200', 'csrc')
    src = tmp_path / 'fields.cu'
    src.write_text('#include <stdint.h>\n#include <iostream>\n#include <string>\n'
                   'namespace mlbp { void set_error(const char *, ...) {} }\n'
                   '#include "%s/parse.cu"\n'
                   'int main() { std::string s; while (std::getline(std::cin, s)) {\n'
                   '  const unsigned char *p = (const unsigned char *)s.data(); Field f = parse_field(p, p + s.size());\n'
                   '  printf("%%d %%016llx\\n", f.status, (unsigned long long)f.bits); } }\n' % csrc)
    exe = str(tmp_path / 'fields')
    subprocess.check_call([nvcc, '-gencode', 'arch=compute_100a,code=sm_100a', '-std=c++17', '-O2', str(src), '-o', exe])
    rng = random.Random(7)
    S = []
    for _ in range(20000):
        x = struct.unpack('<d', struct.pack('<Q', rng.getrandbits(64)))[0]
        if x != x or abs(x) == float('inf'):
            continue
        y = rng.uniform(-100, 100) * 10.0 ** rng.randint(-12, 12)
        S += [repr(x), '%.18e' % x, '%.17g' % x, '%.6f' % y, '%g' % y, '%.18e' % y, str(rng.randint(-10 ** 19, 10 ** 19))]
    S += _halfway_strings(30000, 3, digits=(17, 18, 19, 20, 25, 40))
    S += ['4.9406564584124654e-324', '2.4703282292062327e-324', '2.4703282292062328e-324', '2.2250738585072011e-308',
          '2.2250738585072014e-308', '1.7976931348623157e308', '1.7976931348623159e308', '1e309', '1e-400', '-1e-400',
          '9007199254740993', '0.' + '0' * 330 + '1', '1' * 400, '-0', '+.5', '5.', 'inf', '-Infinity', 'NaN', '-nan']
    out = subprocess.run([exe], input='\n'.join(S) + '\n', capture_output=True, text=True, check=True).stdout.split()
    hard = 0
    for i, s in enumerate(S):
        status, b = int(out[2 * i]), int(out[2 * i + 1], 16)
        if status == 2:
            hard += 1
            continue
        assert status == 0, s
        assert b == struct.unpack('<Q', struct.pack('<d', float(s)))[0], s
    assert hard < len(S) // 4
    bad = ['1_000', '0x10', '1d5', '1e', '.', '1,2', 'infin', 'nan(1)', '+-1', '1e+', 'e5', '+.', '1..2', '--1', '']
    out = subprocess.run([exe], input='\n'.join(bad) + '\n', capture_output=True, text=True, check=True).stdout.split()
    assert [int(out[2 * i]) for i in range(len(bad))] == [1] * len(bad)
