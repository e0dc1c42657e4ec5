"""Prediction throughput (sentences/s) through the command line's prediction pass, train_cli.predict, three ways in one process:

  host    the .dist numbers formatted on the host: the belief rows copied back and np.log + '%0.6f' per number (the loop
          train_cli used before mlbp_format_log_rows; kept here for comparison only)
  device  the .dist numbers formatted on the device (mlbp_format_log_rows), copied back once per 64-sentence chunk
  infer   inference alone (--quick_predict: no beliefs read back, no files): the ceiling

at V = 10 000 (1 024 sentences, k = 20 predicted tokens) and at V = 50 000 (BASELINE C5 feature sizes, 64 sentences).  The
sentences are written as TrainingInstance lines and read back through the CLI's reader; the feature planes are generated
in memory with the same seed (np.loadtxt of a 10 000 x 10 000 text matrix alone takes minutes).  Output files go to a
temporary directory (page cache: no fsync, as the CLI).  The device run also reports where its time goes: inference, the
format kernel, the device-to-host copy of the text, and the host remainder (.pred lines, file writes, merge).  With more
than one GPU the device variant is also run sharded over all of them (one NCCL rank per GPU).  The card's name and power
limit are printed with the numbers.

    python scripts/predict_throughput.py [--out profiles/predict_throughput.jsonl] [--cases 10000 50000]
"""
import argparse
import json
import os
import random
import shutil
import subprocess
import sys
import tempfile
import time

import numpy as np
import torch

sys.path.insert(0, os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
from macaronicusermodeling_b200 import build, synth, train_cli  # noqa: E402
from macaronicusermodeling_b200.engine import Engine  # noqa: E402

CASES = {10000: dict(V=10000, Vd=2000, n=1024, k=20, n_host=64), 50000: dict(V=50000, Vd=2000, n=64, k=20, n_host=8)}
THETA_EE, THETA_ED = [0.8, 0.5, -0.3], [1.0, -0.6, 0.5, 0.3, 0.4, -0.2]


def host_dist_text(engine, beliefs, pinned):
    """the pre-device loop: every belief row to the host, np.log and '%0.6f' per number"""
    B = beliefs.cpu().numpy()[:, :engine.V].astype(np.float64)
    with np.errstate(divide='ignore'):
        rows = [' '.join('%0.6f' % x for x in np.log(b)).encode() for b in B]
    return np.frombuffer(b''.join(rows), dtype=np.uint8), np.concatenate([[0], np.cumsum([len(r) for r in rows])])


def card():
    q = subprocess.run(['nvidia-smi', '--query-gpu=name,power.limit,clocks.max.sm', '--format=csv,noheader'],
                       capture_output=True, text=True)
    return {'card': torch.cuda.get_device_name(), 'nvidia_smi': q.stdout.strip().split('\n')}


def make_case(c, tmp):
    """(model, sentences, raw JSON, en vocabulary): the corpus goes through the CLI's file format and reader"""
    model = synth.make_model_large(c['V'], c['Vd'], seed=1234)
    ti = os.path.join(tmp, 'test.json')
    with open(ti, 'w') as f:
        for i in range(c['n']):
            f.write(json.dumps(synth.make_sentence(model, 'p' * c['k'], seed=7000 + i, n_history=3, sent_id=i)) + '\n')
    lines = [l for l in open(ti).readlines() if l.strip()]
    en = [synth.en_word(i) for i in range(c['V'])]
    opts = train_cli.parse(['--ti', ti, '--history', '--session_history'])
    sents = train_cli.lower(lines, opts, dict((e, i) for i, e in enumerate(en)),
                            dict((synth.de_word(i), i) for i in range(c['Vd'])))
    return model, sents, [json.loads(l) for l in lines], en, opts


def timed_predict(eng, sents, raw, en, opts, qp, out):
    eng.set_theta(THETA_EE, THETA_ED, with_grad=True)
    torch.cuda.synchronize()
    t0 = time.perf_counter()
    train_cli.predict(eng, train_cli.prediction_units(len(sents)), sents, raw, en, opts, random.Random(3), qp, None, out)
    torch.cuda.synchronize()
    return time.perf_counter() - t0


def run_case(V, tmp, log):
    c = CASES[V]
    model, sents, raw, en, opts = make_case(c, tmp)
    eng = Engine(model)
    out = os.path.join(tmp, 'out.pred')
    timed_predict(eng, sents[:64], raw[:64], en, opts, False, out)                 # warm-up: modules, allocator, page cache
    res = {'V': V, 'Vd': c['Vd'], 'k': c['k'], 'sweeps': 3}
    t_inf = timed_predict(eng, sents, raw, en, opts, True, None)
    res['infer'] = {'sentences': len(sents), 'seconds': t_inf, 'sentences_per_s': len(sents) / t_inf}
    # device formatting, with the time of the format kernel and of the copy
    acc = {'kernel': 0.0, 'copy': 0.0}
    orig = train_cli.dist_text

    def split_dist_text(engine, beliefs, pinned):
        torch.cuda.synchronize()
        t0 = time.perf_counter()
        engine.format_log_rows(beliefs)
        torch.cuda.synchronize()
        t1 = time.perf_counter()
        r = orig(engine, beliefs, pinned)                      # formats again, then copies back (synchronous)
        t2 = time.perf_counter()
        acc['kernel'] += t1 - t0
        acc['copy'] += max(t2 - t1 - (t1 - t0), 0.0)
        return r
    t_dev = timed_predict(eng, sents, raw, en, opts, False, out)
    nbytes = os.path.getsize(out + '.dist') + os.path.getsize(out)
    train_cli.dist_text = split_dist_text
    try:
        t_split = timed_predict(eng, sents, raw, en, opts, False, out)
    finally:
        train_cli.dist_text = orig
    # the instrumented run formats every chunk twice (once alone, timed); 'inference' is the --quick_predict run's time
    res['device'] = {'sentences': len(sents), 'seconds': t_dev, 'sentences_per_s': len(sents) / t_dev, 'bytes_written': nbytes,
                     'breakdown_s': {'inference': t_inf, 'format_kernel': acc['kernel'], 'd2h_copy': acc['copy'],
                                     'host_pred_lines_file_writes': t_split - 2 * acc['kernel'] - acc['copy'] - t_inf,
                                     'instrumented_total': t_split}}
    os.remove(out); os.remove(out + '.dist')
    nh = c['n_host']
    train_cli.dist_text = host_dist_text
    try:
        t_host = timed_predict(eng, sents[:nh], raw[:nh], en, opts, False, out)
    finally:
        train_cli.dist_text = orig
    res['host'] = {'sentences': nh, 'seconds': t_host, 'sentences_per_s': nh / t_host}
    os.remove(out); os.remove(out + '.dist')
    res['pass_stats'] = eng.pass_stats()
    log(res)
    del eng
    torch.cuda.empty_cache()
    return res


def _rank(rank, world, port, V, tmp, q):
    import torch.distributed as dist
    os.environ.update(MASTER_ADDR='127.0.0.1', MASTER_PORT=str(port))
    torch.cuda.set_device(rank)
    dist.init_process_group('nccl', rank=rank, world_size=world)
    model, sents, raw, en, opts = make_case(CASES[V], os.path.join(tmp, 'r%d' % rank))
    eng = Engine(model)
    out = os.path.join(tmp, 'out.pred')
    timed_predict(eng, sents[:64 * world], raw[:64 * world], en, opts, False, out)
    dist.barrier()
    t = timed_predict(eng, sents, raw, en, opts, False, out)
    dist.barrier()
    if rank == 0:
        q.put({'V': V, 'ranks': world, 'sentences': len(sents), 'seconds': t, 'sentences_per_s': len(sents) / t})
    dist.destroy_process_group()


def main():
    ap = argparse.ArgumentParser()
    ap.add_argument('--out', default='')
    ap.add_argument('--cases', type=int, nargs='+', default=[10000, 50000])
    a = ap.parse_args()
    if not torch.cuda.is_available():
        raise SystemExit('predict_throughput.py measures the GPU path: no CUDA device')
    build.build()
    info = card()

    def log(rec):
        rec = dict(rec, **info)
        line = json.dumps(rec)
        print(line, flush=True)
        if a.out:
            with open(a.out, 'a') as f:
                f.write(line + '\n')
    for V in a.cases:
        tmp = tempfile.mkdtemp(prefix='predict_tp_')
        try:
            run_case(V, tmp, log)
            n = torch.cuda.device_count()
            if n > 1:
                import torch.multiprocessing as mp
                q = mp.get_context('spawn').SimpleQueue()
                for r in range(n):
                    os.makedirs(os.path.join(tmp, 'r%d' % r), exist_ok=True)
                mp.spawn(_rank, args=(n, 29600 + os.getpid() % 1000, V, tmp, q), nprocs=n, join=True)
                log(dict(q.get(), sharded=True))
        finally:
            shutil.rmtree(tmp, ignore_errors=True)


if __name__ == '__main__':
    main()
