"""GPU tier: the .dist text made on the device (mlbp_format_log_rows) and prediction sharded over ranks.

* every non-negative float32, the specials and negative inputs against NumPy's log and CPython's '%0.6f';
* whole rows (with zeros, padded row stride) byte-identical to the reference's expression, n_rows = 0, refused arguments;
* a prediction at V = 10 000 byte-identical to the host formatting it replaces;
* two torchrun ranks writing the files of one rank (when the box has two GPUs)."""
import ctypes
import decimal
import os
import random
import subprocess
import sys

import numpy as np
import pytest
import torch

from macaronicusermodeling_b200 import _lib, build, synth, train_cli
from macaronicusermodeling_b200.engine import Engine

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
from predict_cases import THETA_ED, THETA_EE, dist_numbers, write_case  # noqa: E402

pytestmark = pytest.mark.gpu

NAN, INF, NINF, BAD = -1, -2, -3, -4     # codes of the non-numeric strings (and of a malformed one)


def _fmt(X, V, n_rows, ldx, out_bytes=None):
    """mlbp_format_log_rows on a device fp32 matrix: (rc, text tensor, offsets tensor)"""
    lib = _lib.require_device()
    out_bytes = 12 * V * n_rows if out_bytes is None else out_bytes
    text = torch.full((max(out_bytes, 1),), 7, dtype=torch.uint8, device='cuda')
    off = torch.full((n_rows + 1,), -5, dtype=torch.int64, device='cuda')
    rc = lib.mlbp_format_log_rows(ctypes.c_void_p(X.data_ptr()) if X is not None else None, ldx, V, n_rows,
                                  ctypes.c_void_p(text.data_ptr()), out_bytes, ctypes.c_void_p(off.data_ptr()),
                                  ctypes.c_void_p(torch.cuda.current_stream().cuda_stream))
    torch.cuda.synchronize()
    return rc, text, off


def _codes(text, off, n_rows, W):
    """parse W numbers per row on the device: 2 * round(|log x| * 1e6) + (1 if negative), or NAN / INF / NINF / BAD"""
    t = text[:int(off[-1])]
    sep = torch.nonzero(t == 32).squeeze(1)
    assert sep.numel() == n_rows * (W - 1)
    ends = torch.empty((n_rows, W), dtype=torch.int64, device=t.device)
    ends[:, :W - 1] = sep.view(n_rows, W - 1)
    ends[:, W - 1] = off[1:]
    starts = torch.empty_like(ends)
    starts[:, 0] = off[:-1]
    starts[:, 1:] = ends[:, :-1] + 1
    s, e = starts.reshape(-1), ends.reshape(-1)
    first = t[s].long()
    neg = first == ord('-')
    frac = torch.zeros_like(s)
    ok = (e - s >= 8) & (t[(e - 7).clamp(min=0)] == ord('.'))
    for j in range(1, 7):
        d = t[(e - j).clamp(min=0)].long() - 48
        ok &= (d >= 0) & (d <= 9)
        frac += d * 10 ** (j - 1)
    nd = e - 7 - s - neg.long()
    ok &= (nd >= 1) & (nd <= 3)
    ip = torch.zeros_like(s)
    for j in range(1, 4):
        d = t[(e - 7 - j).clamp(min=0)].long() - 48
        use = nd >= j
        ok &= ~use | ((d >= 0) & (d <= 9))
        ip += torch.where(use, d, torch.zeros_like(d)) * 10 ** (j - 1)
    code = (ip * 1000000 + frac) * 2 + neg.long()
    L = e - s
    second = t[(s + 1).clamp(max=t.numel() - 1)].long()
    code = torch.where(ok, code, torch.full_like(code, BAD))
    code = torch.where((L == 3) & (first == ord('n')), torch.full_like(code, NAN), code)
    code = torch.where((L == 3) & (first == ord('i')), torch.full_like(code, INF), code)
    code = torch.where((L == 4) & neg & (second == ord('i')), torch.full_like(code, NINF), code)
    return code.cpu().numpy()


def _code_of(s):
    if s in ('nan', 'inf', '-inf'):
        return {'nan': NAN, 'inf': INF, '-inf': NINF}[s]
    neg = s.startswith('-')
    ip, fp = s.lstrip('-').split('.')
    return (int(ip) * 1000000 + int(fp)) * 2 + (1 if neg else 0)


def _host_codes(x32):
    """what '%0.6f' % np.log(float64(x)) prints, as codes: a vectorised float round where |log x| * 1e6 is more than 1e-3 from a
    half-integer (exact there: its rounding error is below 1e-7), CPython's formatting for the near-ties"""
    with np.errstate(divide='ignore', invalid='ignore'):
        y = np.log(x32.astype(np.float64))
        t = np.abs(y) * 1e6
        code = np.rint(t) * 2 + (y < 0)
        code = np.where(np.isnan(y), NAN, np.where(y == np.inf, INF, np.where(y == -np.inf, NINF, code)))
        near = np.isfinite(y) & (np.abs(t - np.floor(t) - 0.5) <= 1e-3)
    idx = np.nonzero(near)[0]
    code[idx] = [_code_of('%0.6f' % v) for v in y[idx]]
    return code.astype(np.int64), len(idx)


def _correct_log(x):
    """the correctly rounded float64 log of a float (40 significant digits, then rounded once)"""
    with decimal.localcontext() as ctx:
        ctx.prec = 40
        return float(decimal.Decimal(float(x)).ln())


def test_every_nonnegative_float32():
    build.build()
    W, chunk = 4096, 1 << 26
    n_near = 0
    differ = []
    for lo in range(0, 1 << 31, chunk):
        bits = torch.arange(lo, lo + chunk, dtype=torch.int64, device='cuda').to(torch.int32)
        X = bits.view(torch.float32).view(chunk // W, W)
        rc, text, off = _fmt(X, W, chunk // W, W)
        assert rc == 0
        got = _codes(text, off, chunk // W, W)
        del text, off
        x32 = np.arange(lo, lo + chunk, dtype=np.uint32).view(np.float32)
        want, nn = _host_codes(x32)
        n_near += nn
        assert (got != BAD).all()
        for i in np.nonzero(got != want)[0]:
            differ.append((x32[i], int(got[i]), int(want[i])))
    # every string that differs is one where NumPy's log is not the correctly rounded value and the kernel prints the
    # correctly rounded one
    for x, g, w in differ:
        cr = _correct_log(x)
        with np.errstate(divide='ignore'):
            assert np.log(np.float64(x)) != cr, (x, g, w)
        assert g == _code_of('%0.6f' % cr), (x, g, w)
    print('\nformat_log_rows: 2^31 non-negative float32 inputs, %d near-ties checked with %%0.6f, %d strings differ from '
          'NumPy (each one a NumPy log that is not correctly rounded): %s' % (n_near, len(differ), differ[:20]))


def test_specials_and_negative_inputs():
    build.build()
    rng = np.random.default_rng(1)
    neg = rng.integers(0x80000000, 0xffffffff, size=50000, dtype=np.uint32).view(np.float32)
    spec = np.array([0.0, -0.0, 1.0, np.inf, -np.inf, np.nan, -np.nan, 1.401298464324817e-45, 3.4028234663852886e+38,
                     np.nextafter(np.float32(1), np.float32(0)), np.nextafter(np.float32(1), np.float32(2)),
                     0.99999994, 0.9999999, 0.9999995], dtype=np.float32)
    xs = np.concatenate([spec, neg])
    rc, text, off = _fmt(torch.from_numpy(xs).cuda().view(-1, 1), 1, len(xs), 1)
    assert rc == 0
    text, off = text.cpu().numpy().tobytes(), off.cpu().numpy()
    for r, x in enumerate(xs):
        assert text[off[r]:off[r + 1]] == dist_numbers([x]), (x, text[off[r]:off[r + 1]])
    words = [text[off[r]:off[r + 1]] for r in range(len(spec))]
    assert words[:10] == [b'-inf', b'-inf', b'0.000000', b'inf', b'nan', b'nan', b'nan', b'-103.278930', b'88.722839',
                          b'-0.000000']                            # a negative log that rounds to zero keeps its sign


@pytest.mark.parametrize('V', [1, 7, 120, 10000, 50000])
def test_rows_match_the_host_expression(V):
    build.build()
    rng = np.random.default_rng(V)
    n_rows, ldx = 6, (V + 63) // 64 * 64 + 64
    X = np.full((n_rows, ldx), np.nan, dtype=np.float32)                # padding must not be read
    vals = np.exp(rng.uniform(-105.0, 0.0, size=(n_rows, V))).astype(np.float32)
    vals[rng.random((n_rows, V)) < 0.05] = 0.0
    vals[rng.random((n_rows, V)) < 0.01] = 1.0
    vals[0] /= vals[0].sum()                                            # one belief-like row
    X[:, :V] = vals
    rc, text, off = _fmt(torch.from_numpy(X).cuda(), V, n_rows, ldx)
    assert rc == 0
    text, off = text.cpu().numpy().tobytes(), off.cpu().numpy()
    assert off[0] == 0
    for r in range(n_rows):
        assert text[off[r]:off[r + 1]] == dist_numbers(vals[r]), r
    assert len(text) >= 12 * V * n_rows and off[-1] <= 12 * V * n_rows


def test_empty_and_refused_calls():
    build.build()
    X = torch.ones((4, 64), dtype=torch.float32, device='cuda')
    rc, text, off = _fmt(X, 50, 0, 64)
    assert rc == 0 and off.cpu().tolist() == [0]
    # too small a buffer, a row stride below V, V = 0, no input: refused on the host, nothing launched (buffers untouched)
    for k, args in enumerate(((X, 50, 4, 64, 12 * 50 * 4 - 1), (X, 50, 4, 40, None), (X, 0, 4, 64, 100),
                              (None, 50, 4, 64, None), (X, 50, -1, 64, 100))):
        rc, text, off = _fmt(*args)
        assert rc == 1, args                                           # MLBP_ERR_INVALID
        assert (text == 7).all() and (off == -5).all(), args
        if k == 0:
            assert b'text buffer' in _lib.load().mlbp_last_error()


def _prediction_case(n_sent, V, seed):
    model = synth.make_model_large(V, 400, seed=seed)
    rng = np.random.default_rng(seed)
    raw = [synth.make_sentence(model, ''.join(rng.choice(['p', 'p', 'g', 'r'], size=int(rng.integers(2, 9)))) + 'p',
                               seed=seed * 1000 + i, n_history=4, sent_id=i) for i in range(n_sent)]
    return model, raw, [synth.sentence_to_arrays(r) for r in raw]


def test_cli_prediction_bytes_equal_host_formatting(tmp_path, monkeypatch):
    """the CLI's prediction pass at V = 10 000 (history features, two 64-sentence chunks) with the device formatter and with the
    host loop it replaces: byte-identical .pred and .dist files"""
    build.build()
    V = 10000
    model, raw, sents = _prediction_case(80, V, seed=21)
    eng = Engine(model)
    en = [synth.en_word(i) for i in range(V)]
    opts = train_cli.parse(['--ti', 'x'])
    units = train_cli.prediction_units(len(sents))

    def run(path):
        eng.set_theta(THETA_EE, THETA_ED, with_grad=True)
        out = train_cli.predict(eng, units, sents, raw, en, opts, random.Random(5), False, None, str(path))
        assert eng.pass_stats()['peak_flag'] == 0
        return out

    new = run(tmp_path / 'new.pred')

    def host_dist_text(engine, beliefs, pinned):                      # the pre-change loop: log and '%0.6f' on the host
        B = beliefs.cpu().numpy()[:, :engine.V]
        rows = [dist_numbers(b) for b in B]
        return np.frombuffer(b''.join(rows), dtype=np.uint8), np.concatenate([[0], np.cumsum([len(r) for r in rows])])

    monkeypatch.setattr(train_cli, 'dist_text', host_dist_text)
    old = run(tmp_path / 'old.pred')
    assert new == old
    for s in ('', '.dist'):
        a, b = (open(str(tmp_path / (n + '.pred' + s)), 'rb').read() for n in ('new', 'old'))
        assert a == b, s
    lines = open(str(tmp_path / 'new.pred.dist'), 'rb').read().split(b'\n')
    assert len(lines[0].split(b' ||| ')[2].split(b' ')) == V
    assert sorted(os.listdir(str(tmp_path))) == ['new.pred', 'new.pred.dist', 'old.pred', 'old.pred.dist']


@pytest.mark.parametrize('mode', [[], ['--user_adapt']], ids=['plain', 'user_adapt'])
def test_two_rank_torchrun_prediction_equals_one_rank(tmp_path, mode):
    if torch.cuda.device_count() < 2:
        pytest.skip('needs 2 GPUs for a 2-rank torchrun prediction; this box has %d' % torch.cuda.device_count())
    build.build()
    base = write_case(tmp_path, synth.make_model(120, 24, seed=47), 140, seed=9)
    one, two = tmp_path / 'one', tmp_path / 'two'
    one.mkdir(); two.mkdir()
    assert train_cli.main(base + mode + ['--save_predictions', str(one / 'out.pred')]) == 0
    env = dict(os.environ, PYTHONPATH=os.path.dirname(HERE) + os.pathsep + os.environ.get('PYTHONPATH', ''))
    subprocess.check_call([sys.executable, '-m', 'torch.distributed.run', '--standalone', '--nproc_per_node', '2', '-m',
                           'macaronicusermodeling_b200.train_cli'] + base + mode + ['--save_predictions', str(two / 'out.pred')],
                          env=env, cwd=str(tmp_path))
    for name in ('out.pred', 'out.pred.dist'):
        assert open(str(one / name), 'rb').read() == open(str(two / name), 'rb').read(), name
    assert sorted(os.listdir(str(two))) == ['out.pred', 'out.pred.dist']
