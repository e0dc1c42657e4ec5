"""K8 on the B200: Model.from_text against the np.loadtxt path, bit for bit -- the grammar, correctly rounded conversion of
hard decimal strings, random matrices in the spellings np.savetxt writes at chunk sizes that cut numbers and lines, the
fall-backs, and a command-line run whose output bytes equal a run with np.loadtxt."""
import os
import sys

import numpy as np
import pytest
import torch

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

from text_load_cases import FORMATS, assert_same_model, case_files, loadtxt_model  # noqa: E402
from test_text_load_host import _halfway_strings  # noqa: E402

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def Model():
    from macaronicusermodeling_b200 import build
    build.build()
    from macaronicusermodeling_b200.engine import Model
    torch.cuda.set_device(0)
    return Model


def _parse_row(tmp_path, fields, chunk_bytes=None):
    """one line of fields through the device parser: (fp32 bits, (min, max), hard count), or the failure text"""
    from macaronicusermodeling_b200.engine import Kernels
    from macaronicusermodeling_b200.textload import TextLoader
    p = str(tmp_path / 'row.txt')
    with open(p, 'w') as f:
        f.write(' '.join(fields) + '\n')
    loader = TextLoader(Kernels(), chunk_bytes)
    out = torch.zeros((1, len(fields)), dtype=torch.float32, device='cuda')
    r = loader.parse(p, 1, len(fields), out, len(fields))
    return (r if isinstance(r, str) else (out.cpu().numpy().view(np.uint32)[0], r)), loader.stats['hard_fields'], p


def _check_row(tmp_path, fields, chunk_bytes=None):
    got, hard, p = _parse_row(tmp_path, fields, chunk_bytes)
    assert not isinstance(got, str), got
    a = np.loadtxt(p, dtype=np.float64, ndmin=2)
    want = np.ascontiguousarray(a, dtype=np.float32).view(np.uint32)[0]
    bad = np.flatnonzero(got[0] != want)
    assert len(bad) == 0, [(fields[i], hex(got[0][i]), hex(want[i])) for i in bad[:10]]
    lo, hi = got[1]
    for x, y in ((lo, float(a.min())), (hi, float(a.max()))):
        assert (x != x and y != y) or np.float64(x).view(np.uint64) == np.float64(y).view(np.uint64) or x == y == 0.0
    return hard


ACCEPTED = ['1', '+1', '-2', '1.', '.5', '-.5e-3', '1e+5', '1E-5', '0e999999', '-0', 'inf', '-INF', 'iNf', 'Infinity',
            '-infinity', 'nan', '-NaN', '+nan', '1e1000000000000', '00012.5000', '1e309', '-1e309', '1e-400', '-1e-400']
REJECTED = ['1_000', '0x10', '1d5', '1e', '.', '1,2', 'infin', 'nan(1)', '+-1', '1e+', 'e5', '+.', '1..2']


def test_grammar_accepted(Model, tmp_path):
    for s in ACCEPTED:
        _check_row(tmp_path, [s])
    _check_row(tmp_path, [s for s in ACCEPTED if 'nan' not in s.lower()])


@pytest.mark.parametrize('s', REJECTED)
def test_grammar_rejected_raises_numpys_error(Model, tmp_path, s):
    paths = case_files(tmp_path, 1, 1, 3, '%g')
    with open(paths[0], 'w') as f:
        f.write(s + '\n')
    with pytest.raises(Exception) as want:
        loadtxt_model(Model, paths, 'cuda')
    with pytest.warns(RuntimeWarning, match='malformed'):
        with pytest.raises(want.type) as got:
            Model.from_text(*paths, 1, 1, 'cuda')
    assert str(got.value) == str(want.value)


def test_rounding(Model, tmp_path):
    f32 = np.finfo(np.float32)
    tie32 = []                                     # float64 values halfway between adjacent floats: the fp32 rounding is a tie
    for x in np.float32([1.0, 3.0, 1e-30, 7e20, f32.tiny, 1e-45 * 3]):
        nx = np.nextafter(x, np.float32(np.inf))
        mid = (np.float64(x) + np.float64(nx)) / 2
        tie32 += [repr(float(v)) for v in (mid, -mid, np.nextafter(mid, 0.0), np.nextafter(mid, np.inf))]
    fields = (_halfway_strings(3000, 5, digits=(17, 18, 19, 20, 25, 40)) +
              ['4.9406564584124654e-324', '2.4703282292062327e-324', '2.4703282292062328e-324', '2.2250738585072011e-308',
               '2.2250738585072014e-308', '2.2250738585072009e-308', '1.7976931348623157e308', '1.7976931348623159e308',
               '1e309', '1e-400', '3.4028235677973366e38', '3.4028235677973362e38', '1.401298464324817e-45',
               '7.006492321624085e-46', '7.006492321624087e-46'] + tie32)
    hard = _check_row(tmp_path, fields)
    hard += _check_row(tmp_path, fields, chunk_bytes=4093)
    print('hard fields: %d of %d' % (hard, 2 * len(fields)))


def test_numpy_formats_have_no_hard_fields(Model, tmp_path):
    rng = np.random.default_rng(3)
    x = rng.standard_normal(20000) * 10.0 ** rng.integers(-300, 300, size=20000)
    for fmt in ('%.18e', '%.17g', 'repr'):
        fields = [repr(float(v)) if fmt == 'repr' else fmt % v for v in x]
        assert _check_row(tmp_path, fields) == 0


SHAPES = [(1, 1), (1, 37), (41, 1), (67, 203), (1001, 64)]


@pytest.mark.parametrize('V, Vd', SHAPES)
@pytest.mark.parametrize('fmt', FORMATS)
def test_random_matrices(Model, tmp_path, V, Vd, fmt):
    for k, (mess, chunk) in enumerate(((True, 1024), (False, 4093), (True, None))):
        if V == 1001 and chunk == 1024 and fmt != '%.18e':
            continue                                   # 1 KB chunks of a 25 MB file: one format is enough
        d = tmp_path / str(k)
        d.mkdir()
        paths = case_files(d, V, Vd, 100 + V + k, fmt, mess=mess)
        m = Model.from_text(*paths, V, Vd, 'cuda', chunk_bytes=chunk)
        assert not m.load_stats['fallback']
        assert_same_model(m, loadtxt_model(Model, paths, 'cuda'))


def test_fallbacks(Model, tmp_path):
    paths = case_files(tmp_path, 3, 2, 9, '%.6f')
    with open(paths[1], 'ab') as f:
        f.write(b'# caf\xc3\xa9\n')
    with pytest.warns(RuntimeWarning, match='byte outside'):
        m = Model.from_text(*paths, 3, 2, 'cuda')
    assert len(m.load_stats['fallback']) == 1
    assert_same_model(m, loadtxt_model(Model, paths, 'cuda'))
    with open(paths[2], 'a') as f:
        f.write('1\n')
    with pytest.raises(ValueError) as want:
        loadtxt_model(Model, paths, 'cuda')
    with pytest.warns(RuntimeWarning):
        with pytest.raises(ValueError) as got:
            Model.from_text(*paths, 3, 2, 'cuda')
    assert str(got.value) == str(want.value)


def test_cli_output_bytes_equal_loadtxt_run(Model, tmp_path, monkeypatch):
    from macaronicusermodeling_b200 import synth, train_cli
    from predict_cases import write_case
    model = synth.make_model(300, 40, seed=4)
    outs = {}
    for arm in ('device', 'loadtxt'):
        d = tmp_path / arm
        d.mkdir()
        base = write_case(d, model, 40, seed=6)
        if arm == 'loadtxt':
            monkeypatch.setattr(Model, 'from_text', classmethod(
                lambda cls, a, b, c, e, V, Vd, *r, **k: loadtxt_model(cls, (a, b, c, e), 'cuda')))
        i = base.index('--load_params')
        train = base[:i] + base[i + 2:] + ['--save_params', str(d / 'trained.params'), '--epochs', '1']
        assert train_cli.main(train) == 0
        assert train_cli.main(base[:i] + ['--load_params', str(d / 'trained.params'), '--save_predictions', str(d / 'out.pred')]
                               + base[i + 2:]) == 0
        outs[arm] = [open(str(d / n), 'rb').read() for n in ('trained.params', 'out.pred', 'out.pred.dist')]
    for a, b in zip(outs['device'], outs['loadtxt']):
        assert a == b
