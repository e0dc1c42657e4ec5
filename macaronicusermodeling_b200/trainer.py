"""Trainer-level semantics of train.py / train_mp.py on top of the batched engine.

Reference (one sentence per step, train.py:357-416, :617-638):
    g_ee, g_ed = fg.return_gradient()       # lr * (g - (reg_param / N) * theta)        LBP.py:293-299, :322-327
    theta += g                              # in place, before the next sentence      train.py:404-405
train_mp.py ships sentences to a multiprocessing.Pool and sums the returned gradients under a lock
(:405-424, :634-649) -- asynchronous SGD with stale theta.  Here a *minibatch* of sentences sees the same theta,
per-GPU partial sums are all-reduced (one NCCL all-reduce of 16 float64 per step) and every rank applies the
identical update
    theta += lr * (sum_s g_s - n * (reg_param / N) * theta)
which for a minibatch of one sentence on one GPU is exactly train.py's step (tests/test_gpu_trainer.py).
"""
import ctypes

import numpy as np
import torch

from .engine import Corpus, Engine


def dist_info():
    import torch.distributed as dist
    if dist.is_available() and dist.is_initialized():
        return dist.get_rank(), dist.get_world_size()
    return 0, 1


class Trainer(object):
    def __init__(self, engine, reg_param=0.2, N=None, sweeps=3, init_lr=0.1, objective='lbp'):
        if objective not in ('lbp', 'pl'):
            raise ValueError("objective must be 'lbp' (the reference's loopy-BP gradient) or 'pl' (the pseudo-likelihood)")
        self.engine = engine
        # 'pl': step() follows the exact gradient of the pseudo-likelihood (Engine.pseudo_likelihood, K13) instead of BP's;
        # the 16-vector, the all-reduce and apply() are the same, eval_step() stays BP prediction
        self.objective = objective
        self.reg_param = float(reg_param)
        self.N = N                                  # len(training_instances), train.py:619 (reg = reg_param / N, :158)
        self.sweeps = sweeps
        self.init_lr = init_lr
        self.theta_ee = np.zeros(3)                 # train.py:511
        self.theta_ed = np.zeros(6)                 # train.py:514
        self._red = None

    def lr(self, epoch):
        return self.init_lr / float(1.0 + epoch * 0.3)           # train.py:621

    def step(self, parts_or_corpus, roots, lr, all_reduce=True, next_roots=None, **kw):
        """One synchronous minibatch SGD step over this rank's sentences.  Returns the 16-vector
        [g_ee(3), g_ed(6), sum logp, p@0, p@25, p@50, n_vars, n_sent, peaked] summed over all ranks (device tensor);
        `peaked` counts the ranks whose var->factor kernel saw a peaked message (their message GEMMs ran three passes).
        `next_roots` (with prepared parts): the roots of the NEXT step over the same parts -- its first micro-batch's schedule
        is compiled in the background while the host waits for this step's result (Engine.precompile)."""
        return self._reduce(parts_or_corpus, roots, True, all_reduce, next_roots, **kw)

    def eval_step(self, parts_or_corpus, roots, all_reduce=True, next_roots=None, **kw):
        """batch_predictions (train.py:308-338) for this rank's sentences: inference only; same 16-vector, gradient slots 0"""
        return self._reduce(parts_or_corpus, roots, False, all_reduce, next_roots, **kw)

    def _reduce(self, parts_or_corpus, roots, want_grad, all_reduce, next_roots=None, **kw):
        eng = self.engine
        pl = want_grad and self.objective == 'pl'
        if pl and not isinstance(parts_or_corpus, Corpus):
            raise ValueError("objective='pl' steps take a Corpus: prepared BP parts carry BP's micro-batching, not K13's")
        if pl and any(kw.values()):
            raise ValueError("objective='pl' steps run exact conditionals: BP options (%s) do not apply"
                             % ', '.join(k for k, v in kw.items() if v))
        eng.set_theta(self.theta_ee, self.theta_ed, with_grad=want_grad)
        if self._red is None:
            self._red = torch.zeros(16, dtype=torch.float64, device=eng.device)
        red = self._red                                        # the all-reduce buffer: every micro-batch is added on the device
        eng.k.call('mlbp_zero_words', ctypes.c_void_p(red.data_ptr()), 32)
        if pl:                                                 # no roots: the pseudo-likelihood has no schedule
            eng.pseudo_likelihood(parts_or_corpus, want_grad=True, reduce_into=red)
        else:
            fn = eng.run_many if isinstance(parts_or_corpus, Corpus) else eng.run_prepared
            fn(parts_or_corpus, roots, self.sweeps, want_grad, True, reduce_into=red, collect=False, **kw)
        if next_roots is not None and not isinstance(parts_or_corpus, Corpus) and parts_or_corpus:
            lo, hi, c = parts_or_corpus[0]                          # everything of this step is enqueued: the host is free
            eng.precompile(c, np.ascontiguousarray(next_roots, dtype=np.int32)[lo:hi], self.sweeps, want_grad, True,
                           **{k: v for k, v in kw.items() if k in ('approx_inference', 'approx_beliefs')})
        if all_reduce and dist_info()[1] > 1:
            import torch.distributed as dist
            dist.all_reduce(red, op=dist.ReduceOp.SUM)
        return red

    def apply(self, red, lr):
        """theta update from the reduced vector (the only host<-device read of a step)"""
        h = red.cpu().numpy()
        n = h[14]
        reg = self.reg_param / float(self.N if self.N else n)
        self.theta_ee = self.theta_ee + lr * (h[0:3] - n * reg * self.theta_ee)
        self.theta_ed = self.theta_ed + lr * (h[3:9] - n * reg * self.theta_ed)
        if not (np.isfinite(self.theta_ee).all() and np.isfinite(self.theta_ed).all()):
            raise FloatingPointError('theta diverged (learning rate too large for a summed minibatch gradient?)')
        return h


def batch_sgd_many(engine, sentences, theta_ee, theta_ed, lr, roots_pos, reg_param=0.2, N=None, sweeps=3):
    """train.batch_sgd (train.py:357-397) for MANY sentences at one theta: returns the reference's result list
    [sent_id, logp, g_en_en (1,3), g_en_de (1,6), None] per sentence (gradients already lr * (g - reg * theta))."""
    corpus = Corpus(sentences)
    engine.set_theta(theta_ee, theta_ed)
    roots = corpus.roots_from_positions(roots_pos)
    grad, logp, _, _ = engine.run_many(corpus, roots, sweeps, True, True)
    g, lp = grad.cpu().numpy(), logp.cpu().numpy()
    reg = float(reg_param) / float(N if N else len(sentences))
    te = np.asarray(theta_ee, dtype=np.float64).reshape(1, 3)
    td = np.asarray(theta_ed, dtype=np.float64).reshape(1, 6)
    out = []
    for i, s in enumerate(sentences):
        out.append([s.sent_id, float(lp[i]), lr * (g[i:i + 1, :3] - reg * te), lr * (g[i:i + 1, 3:] - reg * td), None])
    return out


class AdaptTrainer(Trainer):
    """--user_adapt / --experience_adapt (train.py:160-173, :224-245, :379-390, :402-409), batched per domain.

    Each adaptation domain d (a user, or an experience level) owns a theta pair that REPLACES the base theta when that
    domain's potentials are built, so the sentences of a domain form their own batch with their own table planes.  One
    step = for every domain of this rank: K2 for theta_d, one engine pass over the domain's sentences, then
        theta_d    += lr * (sum g - n_d * reg * ua_scale * theta_d)          (stays on this rank: no collective)
        theta_base += lr * (sum over all domains and ranks of g - n * reg * theta_base)   (the 16 x f64 all-reduce)
    With one sentence per domain batch this is train.py's update, sentence by sentence."""

    def __init__(self, engine, domains, reg_param=0.2, ua_scale=1.0, N=None, sweeps=3, init_lr=0.1):
        Trainer.__init__(self, engine, reg_param, N, sweeps, init_lr)
        self.ua_scale = float(ua_scale)
        self.domain2theta = {d: (np.zeros(3), np.zeros(6)) for d in domains}

    def step_domains(self, batches, lr, **kw):
        """batches: list of (domain, Corpus, roots).  Returns the reduced 16-vector like Trainer.step.  `kw`: Engine.run options
        (approx_inference, approx_beliefs, topk: the reference trains with them too, train.py:155-156).  A domain appears at most
        once per call (its sentences of this minibatch form ONE batch): every batch sees the theta its domain had before the call."""
        if len(set(d for d, _, _ in batches)) != len(batches):
            raise ValueError('step_domains: one batch per domain and call')
        eng = self.engine
        # one row of sums per domain, all on the device: a domain's theta only needs ITS row, so nothing is read back before every
        # domain is enqueued -- the host compiles the next domain's schedule while the GPU works on this one (a read-back per
        # domain, as in round 1, left the GPU idle for one schedule compile per user: 16 % of a 64-user pass)
        doms = torch.zeros((max(len(batches), 1), 16), dtype=torch.float64, device=eng.device)
        reg = self.reg_param / float(self.N if self.N else sum(c.n_sent for _, c, _ in batches))
        for i, (d, corpus, roots) in enumerate(batches):
            te, td = self.domain2theta[d]
            eng.set_theta(te, td)
            eng.run_many(corpus, roots, self.sweeps, True, True, reduce_into=doms[i], collect=False, **kw)
        total = doms.sum(dim=0)
        hd = doms.cpu().numpy()                                     # the step's only device -> host read before the all-reduce
        for i, (d, corpus, roots) in enumerate(batches):
            te, td = self.domain2theta[d]
            n = corpus.n_sent
            self.domain2theta[d] = (te + lr * (hd[i, :3] - n * reg * self.ua_scale * te),
                                    td + lr * (hd[i, 3:9] - n * reg * self.ua_scale * td))
        total[15] = (total[15] > 0).to(total.dtype)
        if dist_info()[1] > 1:
            import torch.distributed as dist
            dist.all_reduce(total, op=dist.ReduceOp.SUM)
        return total
