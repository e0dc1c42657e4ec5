"""Command-line trainer / predictor with the reference's flags (train.py:437-462, train_mp.py:457,463) on the batched
B200 engine -- the real-data front end: TrainingInstance JSON lines, vocabulary files, np.loadtxt feature matrices
(train.py:551-610), text parameter checkpoints (train.py:46-99) and the prediction / .dist files eval.py and get_corr.py
read (LBP.py:109-143).

    python -m macaronicusermodeling_b200.train_cli --ti train.json --end en.vocab --ded de.vocab \
        --phi_pmi pmi.mat --phi_pmi_w1 pmi_w1.mat --phi_ed ed.mat --phi_ped ped.mat --save_params model.params
    python -m macaronicusermodeling_b200.train_cli --ti test.json ... --load_params model.params --save_predictions out.pred

Where train_mp.py hands sentences to `--cpu N` pool workers that each see a theta about N sentences old
(train_mp.py:634-649), this trainer takes synchronous minibatches of `--minibatch` sentences (default: the value of
--cpu, 4) that all see the same theta; `--minibatch 1` is train.py's exact per-sentence SGD.  Under torchrun the
minibatch is sharded over the ranks and the gradient all-reduced (trainer.Trainer); prediction (and the --tune pass)
shares its 64-sentence chunks out over the ranks and writes the files one process writes (predict).
"""
import argparse
import codecs
import json
import random
import sys

import numpy as np

from . import synth
from .train_compat import F_EN_DE_NAMES, F_EN_EN_NAMES, read_params, save_params


def parse(argv=None):
    opt = argparse.ArgumentParser(description='batched B200 trainer for the macaronic user model')
    opt.add_argument('--ti', dest='training_instances', default='')
    opt.add_argument('--tune', dest='tuning_instances', default='')
    opt.add_argument('--end', dest='en_domain', default='')
    opt.add_argument('--ded', dest='de_domain', default='')
    opt.add_argument('--phi_pmi', dest='phi_pmi', default='')
    opt.add_argument('--phi_pmi_w1', dest='phi_pmi_w1', default='')
    opt.add_argument('--phi_ed', dest='phi_ed', default='')
    opt.add_argument('--phi_ped', dest='phi_ped', default='')
    opt.add_argument('--cpu', dest='cpus', default='')
    opt.add_argument('--minibatch', dest='minibatch', type=int, default=0)
    opt.add_argument('--epochs', dest='epochs', type=int, default=3)                  # train_mp.py:629
    opt.add_argument('--reg_param', dest='reg_param', default='0.2')
    opt.add_argument('--reg_param_ua_scale', dest='reg_param_ua_scale', default='1.0')
    opt.add_argument('--save_params', dest='save_params_file', default='')
    opt.add_argument('--load_params', dest='load_params_file', default='')
    opt.add_argument('--save_predictions', dest='save_predictions_file', default='')
    opt.add_argument('--history', dest='history', default=False, action='store_true')  # train_mp.py:463
    opt.add_argument('--session_history', dest='session_history', default=False, action='store_true')
    opt.add_argument('--user_adapt', dest='user_adapt', default=False, action='store_true')
    opt.add_argument('--experience_adapt', dest='experience_adapt', default=False, action='store_true')
    opt.add_argument('--quick_predict', dest='quick_predict', default=False, action='store_true')
    opt.add_argument('--use_approx_inference', dest='use_approx_inference', default=False, action='store_true')
    opt.add_argument('--use_approx_beliefs', dest='use_approx_beliefs', default=False, action='store_true')
    opt.add_argument('--report_times', dest='report_times', default=False, action='store_true')
    opt.add_argument('--use_correct_feat', dest='use_correct_feat', default=True, action='store_true')
    opt.add_argument('--seed', dest='seed', type=int, default=1234)                   # train.py:436
    # not a reference flag: also report each sentence's joint log-likelihood of its labels (Bethe estimate, Engine.run want_joint)
    opt.add_argument('--joint_likelihood', dest='joint_likelihood', default=False, action='store_true')
    # not a reference flag: also decode each sentence's most probable joint guess (max-product BP, Engine.run max_product)
    opt.add_argument('--map_decode', dest='map_decode', default=False, action='store_true')
    return opt.parse_args(argv)


def gather_domain_thetas(tr, owner, rank, world):
    """Domain thetas never leave the rank that owns the domain during training; before a checkpoint is written rank 0
    collects every owner's current values (no-op on one rank)."""
    if world <= 1:
        return
    import torch.distributed as dist
    mine = dict((d, t) for d, t in tr.domain2theta.items() if owner.get(d, 0) == rank)
    parts = [None] * world
    dist.all_gather_object(parts, mine)
    for part in parts:
        tr.domain2theta.update(part)


def error_msg():
    sys.stderr.write('Usage: python -m macaronicusermodeling_b200.train_cli\n  --ti [training instance file]\n  --tune [dev set]\n'
                     '  --end [en domain file]\n  --ded [de domain file]\n  --phi_pmi [pmi file]\n  --phi_pmi_w1 [pmi w1 file]\n'
                     '  --phi_ed [ed file]\n  --phi_ped [ped file]\n  --save_params [file] or --load_params [file] --save_predictions [file]\n')


def load_inputs(options):
    from .engine import Model
    de_domain = [i.strip() for i in codecs.open(options.de_domain, 'r', 'utf8').readlines()]       # train.py:582-585
    en_domain = [i.strip() for i in codecs.open(options.en_domain, 'r', 'utf8').readlines()]
    en2id = dict((e, idx) for idx, e in enumerate(en_domain))
    de2id = dict((d, idx) for idx, d in enumerate(de_domain))
    # train.py:589-603 np.loadtxt's the four matrices; they are parsed on the device into the same planes (textload.py)
    model = Model.from_text(options.phi_pmi, options.phi_pmi_w1, options.phi_ed, options.phi_ped, len(en_domain), len(de_domain))
    return en_domain, de_domain, en2id, de2id, model


def lower(lines, options, en2id, de2id):
    return [synth.sentence_to_arrays(json.loads(l), en2id, de2id, history=options.history,
                                     session_history=options.session_history, use_correct_feat=options.use_correct_feat)
            for l in lines if l.strip()]


def domain_of(raw, options):
    """adaptation domain of a training instance: the user (train.py:160-164) or the experience level (:165-169)"""
    if options.user_adapt:
        return str(raw['user_id'])
    return str(len(raw.get('past_sentences_seen', [])))


def read_domains(options):
    """train.py:488-505: <ti>.users / <ti>.experience list the adaptation domains"""
    ext = '.users' if options.user_adapt else '.experience'
    try:
        return [d.strip() for d in codecs.open(options.training_instances + ext).readlines() if d.strip()]
    except IOError:
        sys.stderr.write('%s option can not find %s file. (looked for: %s)\n'
                         % ('user_adapt' if options.user_adapt else 'experience_adapt', ext, options.training_instances + ext))
        raise SystemExit(1)


def adapt_ext(options):
    return '.user_adapt' if options.user_adapt else ('.exp_adapt' if options.experience_adapt else '')


def read_params_adapt(path, options):
    """train.py:524-531: try <file><ext>, then <file>"""
    for cand in (path + adapt_ext(options), path):
        try:
            print('trying to read:', cand)
            return read_params(cand)
        except IOError:
            continue
    raise IOError('no parameter file: ' + path)


def d2t_arrays(tr):
    """AdaptTrainer.domain2theta -> the reference's {('en_en', d): (1,3), ('en_de', d): (1,6)} dict (save_params)"""
    d2t = {}
    for d, (te, td) in tr.domain2theta.items():
        d2t['en_en', d] = np.asarray(te, dtype=np.float64).reshape(1, -1)
        d2t['en_de', d] = np.asarray(td, dtype=np.float64).reshape(1, -1)
    return d2t


def draw_roots(corpus, sweeps, rng):
    k = np.diff(corpus.var_off)
    return np.array([[rng.randrange(int(kk)) for _ in range(1 + sweeps)] for kk in k], dtype=np.int32)


def prediction_units(n_sents, doms=None, batch=64):
    """The engine calls of a prediction pass in the order one process makes them: (domain, sentence indices) per chunk of
    `batch` sentences -- of the whole file, or (--user_adapt / --experience_adapt) of each domain's sentences, domains sorted.
    Under torchrun the ranks share out these units, so every chunk is the same engine call whatever the number of ranks."""
    if doms is None:
        return [(None, list(range(lo, min(lo + batch, n_sents)))) for lo in range(0, n_sents, batch)]
    units = []
    for d in sorted(set(doms)):
        idx = [i for i, x in enumerate(doms) if x == d]
        units += [(d, idx[lo:lo + batch]) for lo in range(0, len(idx), batch)]
    return units


def dist_text(engine, beliefs, pinned):
    """The .dist numbers of a chunk's belief rows, formatted on the device (mlbp_format_log_rows) and copied back at once into
    the pinned buffer pinned[0] (grown as needed): (uint8 array, int64 row offsets [n + 1]) on the host."""
    import torch
    text, off = engine.format_log_rows(beliefs)
    off = off.cpu().numpy()
    total = int(off[-1])
    if pinned[0] is None or pinned[0].numel() < total:
        pinned[0] = None
        pinned[0] = torch.empty(total + total // 4 + 1, dtype=torch.uint8, pin_memory=engine.device.type == 'cuda')
    host = pinned[0][:total]
    host.copy_(text[:total])
    return host.numpy(), off


def merge_parts(path, parts, spans):
    """The final file from the ranks' part files: spans[i] = (rank, offset, length) of sentence i, in file order.  The part
    files are removed."""
    import os
    runs = []
    for rk, off, ln in spans:
        if runs and runs[-1][0] == rk and runs[-1][1] + runs[-1][2] == off:
            runs[-1][2] += ln
        else:
            runs.append([rk, off, ln])
    if len(runs) == 1 and runs[0][1] == 0 and runs[0][2] == os.path.getsize(parts[runs[0][0]]):
        os.replace(parts[runs[0][0]], path)                    # one part holds the whole file in order: no copy
    else:
        srcs = [open(p, 'rb') for p in parts]
        try:
            with open(path, 'wb') as w:
                for rk, off, ln in runs:
                    srcs[rk].seek(off)
                    while ln > 0:
                        b = srcs[rk].read(min(ln, 1 << 24))
                        if not b:
                            raise IOError('%s is shorter than the spans written to it' % parts[rk])
                        w.write(b)
                        ln -= len(b)
        finally:
            for f in srcs:
                f.close()
    for p in parts:
        if os.path.exists(p):
            os.remove(p)


def predict(engine, units, sents, raw, en_domain, options, rng, qp, thetas=None, out_path=None, joint=False, map_decode=False):
    """train.py:308-338 batched and sharded over the torchrun ranks.  `units`: prediction_units(); `thetas`: domain ->
    (theta_ee, theta_ed) for the adaptation modes (else the engine's current theta is used).  The roots of every sentence are
    drawn from `rng` in unit order before the units are shared out, so a sentence gets the same roots on any number of ranks.
    Rank r runs units r, r + world, ...; with `out_path` (and not qp) each rank writes its sentences' .pred / .dist text
    to part files next to the output, and after a barrier rank 0 merges them in file order.  Returns the all-reduced
    (sum log-posterior, (p0, p25, p50, total)) on every rank, summed in the order one process sums them.
    `joint`: also the sum of the sentences' joint log-likelihoods (Engine.run want_joint) as a third result, and with `out_path`
    the file <out_path>.joint, one line  sent_id TAB joint TAB sum of marginal logp  per sentence in file order.
    `map_decode`: every unit also runs max-product inference with the same roots (no further draws from `rng`); one more result
    (tokens whose decoded word is the label, sentences decoded entirely right), and with `out_path` the file <out_path>.map, one
    line  sent_id TAB decoded words in position order TAB map_score TAB label_score  per sentence in file order."""
    import torch
    from .engine import Corpus
    from .trainer import dist_info
    rank, world = dist_info()
    V = len(en_domain)
    corpora = [Corpus([sents[i] for i in idx]) for _, idx in units]
    roots = [draw_roots(c, 3, rng) for c in corpora]
    # per unit: sum logp, #rank == 0, < 26, < 50, variables, sum joint, MAP tokens right, MAP sentences right
    stats = np.zeros((len(units), 8))
    write = bool(out_path) and not qp
    if write:
        parts = [out_path + '.rank%d.part' % r for r in range(world)]
        dparts = [out_path + '.dist.rank%d.part' % r for r in range(world)]
        wp, wd = open(parts[rank], 'wb'), open(dparts[rank], 'wb')
        spans, p_off, d_off = [], 0, 0                          # (sentence, .pred offset, length, .dist offset, length)
    write_joint = bool(out_path) and joint
    if write_joint:
        jparts = [out_path + '.joint.rank%d.part' % r for r in range(world)]
        wj = open(jparts[rank], 'wb')
        jspans, j_off = [], 0                                   # (sentence, .joint offset, length)
    write_map = bool(out_path) and map_decode
    if write_map:
        mparts = [out_path + '.map.rank%d.part' % r for r in range(world)]
        wm = open(mparts[rank], 'wb')
        mspans, m_off = [], 0                                   # (sentence, .map offset, length)
    pinned = [None]
    cur = object()
    for u in range(rank, len(units), world):
        dom, idx = units[u]
        if thetas is not None and dom != cur:
            engine.set_theta(thetas[dom][0], thetas[dom][1], with_grad=True)
            cur = dom
        corpus = corpora[u]
        r = engine.run(corpus, roots[u], 3, want_grad=False, want_marg=True, want_beliefs=not qp,
                       approx_inference=options.use_approx_inference, want_topk=0 if qp else min(50, V - 1), want_joint=joint)
        rk = r.rank.cpu().numpy()
        stats[u, :5] = (float(r.logp.sum().item()), int((rk == 0).sum()), int((rk < 26).sum()), int((rk < 50).sum()), len(rk))
        if joint:
            lj = r.logp_joint.cpu().numpy()
            stats[u, 5] = float(lj.sum())
        if write_joint:
            lm = r.logp.cpu().numpy()
            for si, i in enumerate(idx):
                nodes = sorted(raw[i]['current_sent'], key=lambda n: int(n['position']))
                j_len = wj.write(('%s\t%r\t%r\n' % (nodes[0]['sent_id'], float(lj[si]), float(lm[si]))).encode('utf8'))
                jspans.append((i, j_off, j_len))
                j_off += j_len
        if map_decode:
            rm = engine.run(corpus, roots[u], 3, want_grad=False, want_marg=True, max_product=True)
            dec, lab = rm.top1.cpu().numpy(), corpus.var_label
            ok = dec == lab
            stats[u, 6] = int(ok.sum())
            stats[u, 7] = sum(1 for si in range(len(idx)) if ok[corpus.var_off[si]:corpus.var_off[si + 1]].all())
            if write_map:
                ms, ls = rm.map_score.cpu().numpy(), rm.label_score.cpu().numpy()
                for si, i in enumerate(idx):
                    nodes = sorted(raw[i]['current_sent'], key=lambda n: int(n['position']))
                    words = ' '.join(en_domain[int(e)] for e in dec[corpus.var_off[si]:corpus.var_off[si + 1]])
                    m_len = wm.write(('%s\t%s\t%r\t%r\n' % (nodes[0]['sent_id'], words, float(ms[si]), float(ls[si]))).encode('utf8'))
                    mspans.append((i, m_off, m_len))
                    m_off += m_len
        if not write:
            continue
        text, toff = dist_text(engine, r.beliefs, pinned)
        B = r.beliefs.cpu().numpy()[:, :V].astype(np.float64)
        TI, _, TT = (x.cpu().numpy() for x in r.topk)        # the 50 best words per variable, listed on the device (mlbp_topk_rows)
        for si, i in enumerate(idx):
            s, ti = sents[i], raw[i]
            nodes = sorted(ti['current_sent'], key=lambda n: int(n['position']))
            lines = ['*SENT_ID:' + str(nodes[0]['sent_id'])]
            vi = int(corpus.var_off[si])
            d_len = 0
            for p, n in enumerate(nodes):                                            # FactorGraph.to_string, LBP.py:109-123
                if s.kind[p] == 1:
                    b = B[vi]
                    vi += 1
                    top = min(50, V - 1)
                    if TT[vi - 1] == 0:
                        idx_top = TI[vi - 1]
                    else:                                    # exact ties: the reference's order is NumPy's (LBP.py:405-406)
                        idx_top = np.argpartition(b, -top)[-top:]
                        idx_top = idx_top[np.argsort(b[idx_top])][::-1]
                    with np.errstate(divide='ignore'):
                        lb = np.log(b)
                    sl = en_domain[int(s.label[p])]
                    pred = ' '.join(en_domain[e] + ' ' + '%0.4f' % lb[e] for e in idx_top)
                    lines.append(' '.join([n['l2_word'], sl, '%0.4f' % lb[int(s.label[p])], pred]))
                    truth = n['l1_parent'].lower().replace("'", "") if n.get('l1_parent') else 'None'
                    # to_dist, LBP.py:125-143: "truth ||| label ||| " + the numbers made on the device
                    head = ('\n' if d_len else '') + ' ||| '.join([truth, sl, ''])
                    d_len += wd.write(head.encode('utf8')) + wd.write(text[toff[vi - 1]:toff[vi]])
                else:
                    lines.append(' '.join(['', en_domain[int(s.label[p])], '']))
            d_len += wd.write(b'\n')
            p_len = wp.write(('\n'.join(lines) + '\n').encode('utf8'))
            spans.append((i, p_off, p_len, d_off, d_len))
            p_off += p_len
            d_off += d_len
    if world > 1:
        import torch.distributed as dist
        red = torch.from_numpy(stats).to(engine.device)        # every unit is non-zero on exactly one rank: the sums are exact
        dist.all_reduce(red, op=dist.ReduceOp.SUM)
        stats = red.cpu().numpy()
    if write:
        wp.close()
        wd.close()
        every = [spans]
        if world > 1:
            every = [None] * world
            dist.all_gather_object(every, spans)
            dist.barrier()                                      # every part file is closed
        if rank == 0:
            where = [None] * len(sents)
            for rr, sp in enumerate(every):
                for i, po, pl, do, dl in sp:
                    where[i] = (rr, po, pl, do, dl)
            merge_parts(out_path, parts, [(w[0], w[1], w[2]) for w in where])
            merge_parts(out_path + '.dist', dparts, [(w[0], w[3], w[4]) for w in where])
    if write_joint:
        wj.close()
        every = [jspans]
        if world > 1:
            every = [None] * world
            dist.all_gather_object(every, jspans)
            dist.barrier()
        if rank == 0:
            where = [None] * len(sents)
            for rr, sp in enumerate(every):
                for i, jo, jl in sp:
                    where[i] = (rr, jo, jl)
            merge_parts(out_path + '.joint', jparts, where)
    if write_map:
        wm.close()
        every = [mspans]
        if world > 1:
            every = [None] * world
            dist.all_gather_object(every, mspans)
            dist.barrier()
        if rank == 0:
            where = [None] * len(sents)
            for rr, sp in enumerate(every):
                for i, mo, ml in sp:
                    where[i] = (rr, mo, ml)
            merge_parts(out_path + '.map', mparts, where)
    sums = []
    for col in (0, 5):
        total, k = 0.0, 0
        while k < len(units):                                   # one partial sum per domain, as the single-process loop
            part, d = 0.0, units[k][0]
            while k < len(units) and units[k][0] == d:
                part += float(stats[k, col])
                k += 1
            total += part
        sums.append(total)
    c = stats[:, 1:5].sum(axis=0) if len(units) else np.zeros(4)
    out = (sums[0], tuple(int(x) for x in c))
    if joint:
        out += (sums[1],)
    if map_decode:
        out += (tuple(int(x) for x in stats[:, 6:8].sum(axis=0)),)
    return out


def print_map(prefix, counts, n_tokens, n_sents):
    """the two --map_decode lines: decoded word == label over predicted tokens (compare P@0), and whole sentences right"""
    print(prefix + 'prediction MAP token accuracy:', '%0.2f' % (float(100 * counts[0]) / float(max(n_tokens, 1))), 'total:', n_tokens)
    print(prefix + 'prediction MAP sentence accuracy:', '%0.2f' % (float(100 * counts[1]) / float(max(n_sents, 1))), 'total:',
          n_sents)


def main(argv=None):
    options = parse(argv)
    need = [options.training_instances, options.en_domain, options.de_domain, options.phi_pmi_w1, options.phi_pmi,
            options.phi_ed, options.phi_ped]
    if '' in need or (options.save_params_file == '' and options.load_params_file == '' and options.save_predictions_file == ''):
        error_msg()
        return 1
    if options.user_adapt and options.experience_adapt:
        sys.stderr.write('Currently only supports 1 type of adaptation.')                  # train.py:489-491
        return 1
    if options.map_decode and (options.use_approx_inference or options.use_approx_beliefs):
        sys.stderr.write('--map_decode decodes with exact max-product inference: it does not combine with --use_approx_inference '
                         'or --use_approx_beliefs\n')
        return 1
    adapt = options.user_adapt or options.experience_adapt
    import os
    import torch
    from .engine import Corpus, Engine
    from .trainer import AdaptTrainer, Trainer, dist_info
    # one process per GPU under torchrun: rank / world from the environment, NCCL over NVLink for the 16 x f64 all-reduce
    if int(os.environ.get('WORLD_SIZE', '1')) > 1:
        import torch.distributed as dist
        if torch.cuda.is_available():
            torch.cuda.set_device(int(os.environ.get('LOCAL_RANK', '0')))
        if not dist.is_initialized():
            os.environ.setdefault('MASTER_ADDR', '127.0.0.1')
            dist.init_process_group('nccl' if torch.cuda.is_available() else 'gloo')
    # the reference trains AND predicts with these flags (train.py:155-156 -> LBP.py:506-516, :554-563)
    approx_kw = dict(approx_inference=options.use_approx_inference, approx_beliefs=options.use_approx_beliefs)
    random.seed(options.seed)
    rng = random.Random(options.seed + 1)
    en_domain, de_domain, en2id, de2id, model = load_inputs(options)
    print(len(en_domain), len(de_domain))
    train_lines = [l for l in codecs.open(options.training_instances, 'r', 'utf8').readlines() if l.strip()]
    tune_lines = ([l for l in codecs.open(options.tuning_instances, 'r', 'utf8').readlines() if l.strip()]
                  if options.tuning_instances else None)
    engine = Engine(model)
    mode = 'training' if options.save_predictions_file == '' else 'predicting'
    f_en_en_names, f_en_de_names = list(F_EN_EN_NAMES), list(F_EN_DE_NAMES)
    theta_ee, theta_ed = np.zeros((1, 3)), np.zeros((1, 6))
    d2t_loaded = {}
    if options.load_params_file:
        f_en_en_names, theta_ee, f_en_de_names, theta_ed, d2t_loaded = read_params_adapt(options.load_params_file, options)
    rank, world = dist_info()
    if mode == 'training' and adapt:
        # --user_adapt / --experience_adapt (train.py:160-173, :224-245, :379-390, :402-409): the sentences of a minibatch are
        # grouped by domain; each domain's theta builds its own potentials and stays on the rank that owns the domain
        domains = read_domains(options)
        raws = [json.loads(l) for l in train_lines]
        sents = lower(train_lines, options, en2id, de2id)
        doms = [domain_of(r, options) for r in raws]
        for d in doms:
            if d not in domains:
                domains.append(d)
        owner = dict((d, i % world) for i, d in enumerate(domains))
        mb = options.minibatch or (4 if options.cpus.strip() == '' else int(options.cpus))
        tr = AdaptTrainer(engine, domains, reg_param=float(options.reg_param), ua_scale=float(options.reg_param_ua_scale),
                          N=len(train_lines))
        tr.theta_ee, tr.theta_ed = theta_ee.reshape(-1).copy(), theta_ed.reshape(-1).copy()
        for (ft, d), t in d2t_loaded.items():
            te, td = tr.domain2theta.get(d, (np.zeros(3), np.zeros(6)))
            tr.domain2theta[d] = (t.reshape(-1).copy(), td) if ft == 'en_en' else (te, t.reshape(-1).copy())
        order = list(range(len(sents)))
        ext = adapt_ext(options)
        for epoch in range(options.epochs):
            lr = tr.lr(epoch)
            random.shuffle(order)
            logp = 0.0
            for lo in range(0, len(order), mb):
                groups = {}
                for i in order[lo:lo + mb]:
                    if owner[doms[i]] == rank:
                        groups.setdefault(doms[i], []).append(sents[i])
                batches = []
                for d in sorted(groups):
                    c = Corpus(groups[d])
                    batches.append((d, c, draw_roots(c, 3, rng)))
                red = tr.step_domains(batches, lr, **approx_kw)
                logp += tr.apply(red, lr)[9]
            print('\nepoch:', epoch)
            print(f_en_en_names, tr.theta_ee)
            print(f_en_de_names, tr.theta_ed)
            print('\ntrain prediction probs:', logp / float(len(sents)))
            if options.save_params_file:
                gather_domain_thetas(tr, owner, rank, world)              # a domain's theta lives on the rank that owns it
            if rank == 0 and options.save_params_file:
                save_params(codecs.open(options.save_params_file + ext + '.iter' + str(epoch), 'w', 'utf8'),
                            tr.theta_ee.reshape(1, -1), tr.theta_ed.reshape(1, -1), f_en_en_names, f_en_de_names, d2t_arrays(tr))
                print('saved params')
        print('\ntheta final:', tr.theta_ee, tr.theta_ed)
        if options.save_params_file:
            gather_domain_thetas(tr, owner, rank, world)
        if rank == 0 and options.save_params_file:
            save_params(codecs.open(options.save_params_file + ext, 'w', 'utf8'), tr.theta_ee.reshape(1, -1),
                        tr.theta_ed.reshape(1, -1), f_en_en_names, f_en_de_names, d2t_arrays(tr))
        return 0
    if mode == 'training':
        mb = options.minibatch or (4 if options.cpus.strip() == '' else int(options.cpus))     # train_mp.py:493
        tr = Trainer(engine, reg_param=float(options.reg_param), N=len(train_lines))
        tr.theta_ee, tr.theta_ed = theta_ee.reshape(-1).copy(), theta_ed.reshape(-1).copy()
        sents = lower(train_lines, options, en2id, de2id)
        order = list(range(len(sents)))
        for epoch in range(options.epochs):
            lr = tr.lr(epoch)
            random.shuffle(order)                                                          # train.py:624
            logp = 0.0
            for lo in range(0, len(order), mb):
                batch = [sents[i] for i in order[lo:lo + mb]][rank::world]
                corpus = Corpus(batch)                  # an empty shard contributes a zero vector to the all-reduce
                red = tr.step(corpus, draw_roots(corpus, 3, rng), lr, **approx_kw)
                logp += tr.apply(red, lr)[9]
            print('\nepoch:', epoch)
            print(f_en_en_names, tr.theta_ee)
            print(f_en_de_names, tr.theta_ed)
            print('\ntrain prediction probs:', logp / float(len(sents)))
            if rank == 0 and options.save_params_file:
                save_params(codecs.open(options.save_params_file + '.iter' + str(epoch), 'w', 'utf8'), tr.theta_ee.reshape(1, -1),
                            tr.theta_ed.reshape(1, -1), f_en_en_names, f_en_de_names, {})
                print('saved params')
            if tune_lines is not None:
                engine.set_theta(tr.theta_ee, tr.theta_ed, with_grad=True)
                tune_sents = lower(tune_lines, options, en2id, de2id)
                res = predict(engine, prediction_units(len(tune_sents)), tune_sents, [json.loads(l) for l in tune_lines],
                              en_domain, options, rng, True, joint=options.joint_likelihood, map_decode=options.map_decode)
                lp, (p0, p25, p50, tot) = res[:2]
                if rank == 0:
                    print('\ntune prediction probs:', lp / float(len(tune_lines)))
                    for name, p in (('Prec at 0:', p0), ('prec at 25:', p25), ('prec at 50:', p50)):
                        print(name, '%0.2f' % (float(100 * p) / float(max(tot, 1))), 'total:', tot)
                    if options.joint_likelihood:
                        print('tune prediction joint log-likelihood:', res[2] / float(len(tune_lines)))
                    if options.map_decode:
                        print_map('tune ', res[-1], tot, len(tune_sents))
        print('\ntheta final:', tr.theta_ee, tr.theta_ed)
        if rank == 0 and options.save_params_file:
            save_params(codecs.open(options.save_params_file, 'w', 'utf8'), tr.theta_ee.reshape(1, -1), tr.theta_ed.reshape(1, -1),
                        f_en_en_names, f_en_de_names, {})
        return 0
    # ---- predicting (train.py:678-757)
    raw = [json.loads(l) for l in train_lines]
    all_sents = lower(train_lines, options, en2id, de2id)
    if adapt:
        # every sentence is scored with its domain's theta (train.py:224-245 via create_factor_graph); results keep file order
        doms = [domain_of(r, options) for r in raw]
        thetas = dict((d, (d2t_loaded['en_en', d].reshape(-1), d2t_loaded['en_de', d].reshape(-1))) for d in set(doms))
        units = prediction_units(len(all_sents), doms)
    else:
        engine.set_theta(theta_ee.reshape(-1), theta_ed.reshape(-1), with_grad=True)
        thetas, units = None, prediction_units(len(all_sents))
    res = predict(engine, units, all_sents, raw, en_domain, options, rng, options.quick_predict, thetas,
                  options.save_predictions_file, joint=options.joint_likelihood, map_decode=options.map_decode)
    lp, (p0, p25, p50, tot) = res[:2]
    if rank == 0:
        print('\nprediction probs:', lp / float(len(train_lines)))
        for name, p in (('Prec at 0:', p0), ('prec at 25:', p25), ('prec at 50:', p50)):
            print(name, '%0.2f' % (float(100 * p) / float(max(tot, 1))), 'total:', tot)
        if options.joint_likelihood:
            print('prediction joint log-likelihood:', res[2] / float(len(train_lines)))
        if options.map_decode:
            print_map('', res[-1], tot, len(all_sents))
    if torch.cuda.is_available():
        torch.cuda.synchronize()
    return 0


if __name__ == '__main__':
    sys.exit(main())
