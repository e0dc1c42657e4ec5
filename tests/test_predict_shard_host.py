"""Prediction sharded over torchrun ranks, on the CPU: two gloo ranks on the emulated kernels write .pred / .dist files
byte-identical to one process, in plain and --user_adapt mode, leave no part files behind, and the statistics of a
sharded evaluation pass (the --tune pass of training) equal the single-process ones."""
import os
import random
import sys

import numpy as np
import torch
import torch.distributed as dist
import torch.multiprocessing as mp

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, HERE)
sys.path.insert(0, os.path.dirname(HERE))

from fake_kernels import FakeKernels, _arr  # noqa: E402
from predict_cases import dist_numbers, write_case  # noqa: E402

N_SENT = 140                      # three 64-sentence chunks in plain mode, five (user, chunk) units with --user_adapt


class FormatKernels(FakeKernels):
    """FakeKernels plus mlbp_format_log_rows, emulated with the reference's host expression"""

    def mlbp_format_log_rows(self, X, ldx, V, n_rows, out, out_bytes, offsets):
        assert out_bytes >= 12 * V * n_rows
        O = _arr(offsets, np.int64, n_rows + 1)
        O[0] = 0
        if n_rows == 0:
            return
        Xm = _arr(X, np.float32, n_rows * ldx).reshape(n_rows, ldx)
        buf = _arr(out, np.uint8, out_bytes)
        for r in range(n_rows):
            s = dist_numbers(Xm[r, :V])
            buf[O[r]:O[r] + len(s)] = np.frombuffer(s, dtype=np.uint8)
            O[r + 1] = O[r] + len(s)


def _model():
    from macaronicusermodeling_b200 import synth
    return synth.make_model(64, 16, seed=5)


def _run_cli(argv):
    from macaronicusermodeling_b200 import engine, train_cli
    engine.Kernels = FormatKernels
    assert train_cli.main(argv) == 0


def _worker(rank, world, port, argv):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port), RANK=str(rank), LOCAL_RANK=str(rank),
                      WORLD_SIZE=str(world))
    _run_cli(argv)
    dist.destroy_process_group()


def _read(path):
    with open(path, 'rb') as f:
        return f.read()


def test_two_rank_prediction_files_equal_one_rank(tmp_path):
    from macaronicusermodeling_b200 import build
    build.build()
    base = write_case(tmp_path, _model(), N_SENT, seed=3)
    for k, mode in enumerate(([], ['--user_adapt'])):
        one, two = tmp_path / ('one%d' % k), tmp_path / ('two%d' % k)
        one.mkdir(); two.mkdir()
        _run_cli(base + mode + ['--save_predictions', str(one / 'out.pred')])
        port = 29700 + k + 2 * (os.getpid() % 1000)
        mp.spawn(_worker, args=(2, port, base + mode + ['--save_predictions', str(two / 'out.pred')]), nprocs=2, join=True)
        for name in ('out.pred', 'out.pred.dist'):
            a, b = _read(one / name), _read(two / name)
            assert a == b, (mode, name)
        assert sorted(os.listdir(two)) == ['out.pred', 'out.pred.dist']        # the part files are merged and removed
        assert sorted(os.listdir(one)) == ['out.pred', 'out.pred.dist']
        assert _read(one / 'out.pred').count(b'*SENT_ID:') == N_SENT


def _tune_stats(world_rank=None):
    """one --tune evaluation pass (statistics only) at a fixed theta"""
    from macaronicusermodeling_b200 import synth, train_cli
    from macaronicusermodeling_b200.engine import Engine
    model = _model()
    rng = np.random.default_rng(8)
    raw = [synth.make_sentence(model, ''.join(rng.choice(['p', 'g'], size=5)) + 'p', seed=90 + i, sent_id=i) for i in range(150)]
    sents = [synth.sentence_to_arrays(r) for r in raw]
    eng = Engine(model, kernels=FormatKernels())
    eng.set_theta([0.4, -0.3, 0.1], [0.8, -0.5, 0.6, 0.4, 0.3, -0.2])
    opts = train_cli.parse(['--ti', 'x'])
    rng = random.Random(11)
    lp, counts = train_cli.predict(eng, train_cli.prediction_units(len(sents)), sents, raw,
                                   [synth.en_word(i) for i in range(model['V'])], opts, rng, True)
    return [lp] + list(counts) + [rng.random()]   # every rank draws the roots of all sentences: the training rng stays in step


def _tune_worker(rank, world, port, out):
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    dist.init_process_group('gloo', rank=rank, world_size=world)
    out[rank] = _tune_stats()
    dist.destroy_process_group()


def test_two_rank_tune_statistics_equal_one_rank():
    from macaronicusermodeling_b200 import build
    build.build()
    want = _tune_stats()
    assert want[4] > 0
    out = mp.Manager().dict()
    mp.spawn(_tune_worker, args=(2, 31700 + (os.getpid() % 1000), out), nprocs=2, join=True)
    for r in (0, 1):
        assert out[r] == want                     # the same log-posterior sum (same order) and the same P@0/25/50 counts
