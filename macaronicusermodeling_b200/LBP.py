"""Drop-in for the reference's ``LBP.py``: same classes, constructor orders, attribute and method names, return
shapes and exceptions (SURVEY.md §8(b)), executed by the batched B200 engine instead of per-message NumPy calls.

How it runs.  The object graph built through ``add_varset_with_potentials`` / ``add_factor`` is only RECORDED.
``initialize()`` and ``treelike_inference(n)`` record the BFS roots they draw from the global ``random`` (the
same one draw per call site as LBP.py:176 and :223).  The first method that needs numbers (marginals, gradient,
log-posterior, ``graph.messages[...]``) lowers the recorded graph + roots to index arrays, lets the C++ schedule
compiler reproduce the reference's sequential update order exactly, and executes everything on the GPU in one go.
Asking for more sweeps later re-runs from the uniform initial messages with the longer root list (inference is a
deterministic function of the roots).

Supported graphs: the macaronic model the reference's callers build (train.py:255-297): factors with
``factor_type`` 'en_de' (unary, observed German word) or 'en_en' (unary with an observed English word, or pairwise),
tables selected by ``gap`` like FactorNode.get_pot (LBP.py:456-467), features as stacked by train.py:594-609
(phi_en_en = [pmi, 0, 1], phi_en_en_w1 = [pmi, pmi_w1, 1], phi_en_de = [ed, ped, correct, full_history,
hit_history, 1]).

Eager mode.  The reference's one-message-at-a-time API -- ``VariableNode.update_message_to(fc)`` /
``FactorNode.update_message_to(var)`` (LBP.py:377-389, :490-526) -- and graphs built from explicit
``PotentialTable(table=...)`` arrays (run.py / toy style) bypass the batched engine: ``graph.messages`` becomes the
state, each update is the same ``au`` call the reference makes (a device kernel per pointwise product, dot product and
normalisation), ``treelike_inference`` walks the schedule literally, marginals and gradients are computed factor by
factor.  It is the reference's cost model (one launch per tiny op) and exists for API completeness and debugging; the
fast path is the lazy batched mode above.  There is no CPU fallback: without libmlbp.so and a B200 the first
computation raises.
"""
import random
import sys
import time

import numpy as np
from numpy import float64 as DTYPE

from .array_utils import c_array_utils as au

VAR_TYPE_PREDICTED = 'var_type_predicted'
VAR_TYPE_GIVEN = 'var_type_given'
VAR_TYPE_LATENT = 'var_type_latent'
UNARY_FACTOR = 'unary_factor'
BINARY_FACTOR = 'binary_factor'

_ENGINES = {}      # (id(phi_en_en), id(phi_en_en_w1), id(phi_en_de)) -> Engine : feature planes stay resident
_DOMAIN_INDEX = {}  # id(domain list) -> {word: index}
_KERNELS_FACTORY = None   # test hook: the CPU test tier injects an emulation of the device kernels here


def _engine_for(graph):
    from .engine import Engine, Model
    key = (id(graph.phi_en_en), id(graph.phi_en_en_w1), id(graph.phi_en_de))
    ent = _ENGINES.get(key)
    if ent is None or ent[1] is not graph.phi_en_en:
        ee, ee1, ed = graph.phi_en_en, graph.phi_en_en_w1, graph.phi_en_de
        if ee.ndim != 3 or ee.shape[2] != 3 or ee1.shape != ee.shape or ed.ndim != 3 or ed.shape[2] != 6:
            raise NotImplementedError('feature tensors must be the (V,V,3) / (V,Vd,6) stacks of train.py:594-609')
        from .engine import Kernels
        k = _KERNELS_FACTORY() if _KERNELS_FACTORY is not None else Kernels()
        model = Model(ee[:, :, 0], ee1[:, :, 1], ed[:, :, 0], ed[:, :, 1], k.device)
        _ENGINES.clear()                     # one resident model at a time (V x V planes are large)
        ent = (Engine(model, kernels=k), ee)
        _ENGINES[key] = ent
    return ent[0]


def _index_of(domain, label):
    d = _DOMAIN_INDEX.get(id(domain))
    if d is None or d[0] is not domain:
        d = (domain, dict((w, i) for i, w in reversed(list(enumerate(domain)))))
        if len(_DOMAIN_INDEX) > 8:
            _DOMAIN_INDEX.clear()
        _DOMAIN_INDEX[id(domain)] = d
    return d[1].get(label)


class FactorGraph():
    def __init__(self,
                 theta_en_en_names,
                 theta_en_de_names,
                 theta_en_en,
                 theta_en_de,
                 phi_en_en_w1,
                 phi_en_en,
                 phi_en_de):
        self.theta_en_en = theta_en_en
        self.theta_en_de = theta_en_de
        self.theta_en_en_names = theta_en_en_names
        self.theta_en_de_names = theta_en_de_names
        self.phi_en_en = phi_en_en
        self.phi_en_en_w1 = phi_en_en_w1
        self.phi_en_de = phi_en_de
        self.pot_en_en = None
        self.pot_en_en_w1 = None
        self.pot_en_de = None
        self.variables = {}
        self.factors = []
        self.normalize_messages = True
        self.isLoopy = None
        self.regularization_param = 0.01
        self.learning_rate = 0.1
        self.report_times = False
        self.bb_times = []
        self.ub_times = []
        self.it_times = []
        self.gg_times = []
        self.sgg_times = []
        self.active_domains = {}
        self.use_approx_inference = False
        self.use_approx_beliefs = False
        if isinstance(self.theta_en_en_names, tuple):
            self.theta_en_en_names = self.theta_en_en_names[0]
        if isinstance(self.theta_en_de_names, tuple):
            self.theta_en_de_names = self.theta_en_de_names[0]
        # --user_adapt / --experience_adapt: train.py:224-229, :242-245 build the potentials from the active domain's
        # theta INSTEAD of theta_en_en / theta_en_de (which still regularise and receive the update); None = no adaptation
        self.pot_theta_en_en = None
        self.pot_theta_en_de = None
        # recorder state
        self._roots = []          # [has_loops draw, sweep roots...] as variable ids
        self._sweeps = 0
        self._initialized = False
        self._res = None          # cached engine outputs for (_sweeps, theta snapshot)
        self._joint = None        # (key, get_joint_log_likelihood())
        self._messages = None
        # Eager mode: the reference's one-message-at-a-time API (VariableNode / FactorNode.update_message_to) and
        # graphs with explicit PotentialTable(table=...) arrays.  graph.messages then IS the state, every update is
        # one `au` device op exactly where the reference calls au (LBP.py:377-389, :490-526), and the batched engine
        # is bypassed.  None = lazy batched mode (the fast path).
        self._eager = None
        self._explicit = False

    # ------------------------------------------------------------------ reference API: bookkeeping
    def display_timing_info(self):
        if self.report_times:
            for name, ts in (('ubtimes', self.ub_times), ('bbtimes', self.bb_times), ('ggtimes', self.gg_times),
                             ('sggtimes', self.sgg_times), ('it_times', self.it_times)):
                if len(ts) > 0:
                    print(name.ljust(11) + ':', np.sum(ts) / len(ts), 'total', np.sum(ts), 'len', len(ts))
            print('num vars   :', len(self.variables))
        return True

    def add_factor(self, fac):
        if __debug__: assert fac not in self.factors
        self.factors.append(fac)
        fac.graph = self
        for v in fac.varset:
            if v.id not in self.variables:
                self.variables[v.id] = v
                v.graph = self
        self._res = self._joint = None

    def get_message_schedule(self, root):
        """The (child, parent) edge list one sweep walks (reference: LBP.py:155-172).  Breadth-first from `root` with the
        reference's visiting rule: a node only counts as visited once it has been taken OFF the queue, so in a loopy graph a
        node is queued -- and scheduled -- once for every neighbour that reaches it before its own turn comes.  Neighbours are
        taken in attach order (facset / varset).  csrc/plan.cpp `schedule` is the batched twin of this walk."""
        from collections import deque
        if __debug__: assert isinstance(root, VariableNode)
        done, edges, queue = set(), [], deque([root])
        while queue:
            node = queue.popleft()
            if str(node) in done:
                continue
            done.add(str(node))
            if isinstance(node, VariableNode):
                around = node.facset
            elif isinstance(node, FactorNode):
                around = node.varset
            else:
                raise NotImplementedError("Only handles 2 kinds of nodes, variables and factors")
            fresh = [nb for nb in around if str(nb) not in done]
            edges += [(nb, node) for nb in fresh]
            queue.extend(fresh)
        return edges

    def _draw_root(self):
        return random.sample(sorted(self.variables.keys()), 1)[0]

    def has_loops(self, _root_id=None):
        """True when a depth-first walk from one randomly drawn variable (the reference's single RNG draw, LBP.py:174-190)
        meets a node twice without walking an edge straight back.  `_root_id` (not in the reference) pins the draw."""
        start = self._draw_root() if _root_id is None else _root_id
        self._last_loop_root = start
        reached, todo = set(), [(self.variables[start], None)]
        while todo:
            node, came_from = todo.pop()
            if str(node) in reached:
                return True
            reached.add(str(node))
            if isinstance(node, VariableNode):
                around = node.facset
            elif isinstance(node, FactorNode):
                around = node.varset
            else:
                raise NotImplementedError("Only handles 2 kinds of nodes, variables and factors")
            todo.extend((nb, node) for nb in around if nb is not came_from)
        return False

    def initialize(self, root=None):
        """LBP.py:192-216.  ``root`` (optional, not in the reference) pins the has_loops draw."""
        if __debug__: assert len(self.variables) > 0
        if __debug__: assert len(self.factors) > 0
        fs = sorted([(f.id, f) for f in self.factors], key=lambda t: t[0])
        self.factors = [f for fid, f in fs]
        self.isLoopy = self.has_loops(root)
        self._explicit = False
        for f in self.factors:
            if __debug__: assert len(f.potential_table.var_id2dim) == len(f.varset)
            if f.potential_table.explicit:
                self._explicit = True
            # The batched schedule compiler walks a pairwise factor's variables in TABLE order (dim 0, dim 1); the reference's
            # BFS walks f.varset (LBP.py:165-171).  create_factor_graph attaches them in table order (train.py:273-275); a graph
            # that does not is run one message at a time, where the walk is the reference's own
            if len(f.varset) == 2 and f.potential_table.var_id2dim.get(f.varset[0].id) != 0:
                self._explicit = True
        self._roots = [self._last_loop_root]
        self._sweeps = 0
        self._initialized = True
        self._res = self._joint = None
        self._messages = None
        self._eager = self._uniform_messages() if self._explicit else None

    def _uniform_messages(self):
        """LBP.py:200-216: unary factors only send, pairwise factors exchange messages in both directions"""
        msgs = {}
        for f in self.factors:
            if len(f.varset) == 1:
                v = f.varset[0]
                msgs[str(f), str(v)] = Message.new_message(v.domain, 1.0 / len(v.domain))
            else:
                for v in f.varset:
                    msgs[str(v), str(f)] = Message.new_message(v.domain, 1.0 / len(v.domain))
                    msgs[str(f), str(v)] = Message.new_message(v.domain, 1.0 / len(v.domain))
        return msgs

    def _enter_eager(self):
        """Switch to the one-message-at-a-time mode, starting from the current messages (the batched result of the
        sweeps recorded so far, or the uniform initial messages)."""
        if self._eager is None:
            if not self._initialized:
                raise KeyError('messages are not initialised: call initialize() first')
            self._eager = self._uniform_messages() if self._sweeps == 0 else dict(self.messages)
            self._res = self._joint = None
            self._messages = None
        return self._eager

    def treelike_inference(self, iterations, roots=None):
        """LBP.py:218-245.  ``roots`` (optional, not in the reference) pins the per-sweep BFS roots."""
        if not self._initialized:
            raise KeyError('messages are not initialised: call initialize() first')
        iterations = iterations if self.isLoopy else 1
        for i in range(iterations):
            if self.report_times: it = time.time()
            root = self._draw_root() if roots is None else roots[i]
            self._roots.append(root)
            self._sweeps += 1
            if self._eager is not None:                  # LBP.py:225-243, one update at a time
                _schedule = self.get_message_schedule(self.variables[root])
                for frm, to in reversed(_schedule):
                    if not (isinstance(to, FactorNode) and len(to.varset) < 2):
                        frm.update_message_to(to)
                for to, frm in _schedule:
                    if not (isinstance(to, FactorNode) and len(to.varset) < 2):
                        frm.update_message_to(to)
            if self.report_times: self.it_times.append(time.time() - it)
        self._res = self._joint = None
        self._messages = None
        return True

    # ------------------------------------------------------------------ lowering + execution
    def _pot_thetas(self):
        te = self.theta_en_en if self.pot_theta_en_en is None else self.pot_theta_en_en
        td = self.theta_en_de if self.pot_theta_en_de is None else self.pot_theta_en_de
        return np.asarray(te, dtype=np.float64).reshape(-1), np.asarray(td, dtype=np.float64).reshape(-1)

    def _theta_key(self):
        te, td = self._pot_thetas()
        return (te.tobytes(), td.tobytes())

    def _lower(self):
        """recorded object graph -> engine Corpus (one sentence).  Pairwise factors in attach order (facset order)."""
        from .engine import Corpus
        vids = sorted(self.variables.keys())
        local = dict((vid, i) for i, vid in enumerate(vids))
        var_de, var_label = [-1] * len(vids), [0] * len(vids)
        giv = [[] for _ in vids]
        ed_factor = [None] * len(vids)
        pairs = []
        for f in self.factors:
            if len(f.varset) == 1:
                v = f.varset[0]
                od = f.potential_table.observed_dim
                if f.factor_type == 'en_de':
                    if var_de[local[v.id]] != -1:
                        raise NotImplementedError('more than one en_de factor on a variable')
                    var_de[local[v.id]] = int(od)
                    ed_factor[local[v.id]] = f
                elif f.factor_type == 'en_en':
                    giv[local[v.id]].append((int(od), 1 if self._gap_class(f) else 0))
                else:
                    raise BaseException('only 2 kinds of factors allowed...')
            elif len(f.varset) == 2:
                if f.factor_type != 'en_en':
                    raise BaseException("only two kinds of potentials are supported...")
                d = f.potential_table.var_id2dim
                a, b = sorted(f.varset, key=lambda v: d[v.id])
                pairs.append((f._attach_seq, local[a.id], local[b.id], 1 if self._gap_class(f) else 0, f))
            else:
                raise BaseException("only unary or binary factors are supported...")
        pairs.sort(key=lambda t: t[0])
        sp_off, sp_en, sp_feat, sp_val = [0], [], [], []
        for i, vid in enumerate(vids):
            var_label[i] = int(self.variables[vid].supervised_label_index)
            d = var_de[i]
            if d >= 0:                                   # train.py:176-215 wrote the dynamic features into phi_en_de in place;
                for e, feat, val in self._sparse_for(ed_factor[i]):     # the list is the snapshot slice_potentials() took
                    sp_en.append(e); sp_feat.append(feat); sp_val.append(val)
            sp_off.append(len(sp_en))
        giv_off, giv_label, giv_gap1 = [0], [], []
        for g in giv:
            for od, g1 in g:
                giv_label.append(od); giv_gap1.append(g1)
            giv_off.append(len(giv_label))
        i32 = lambda x: np.asarray(x, dtype=np.int32)
        corpus = Corpus(var_off=i32([0, len(vids)]), var_de=i32(var_de), var_label=i32(var_label), var_pos=i32(vids),
                        sp_off=i32(sp_off), sp_en=i32(sp_en), sp_feat=i32(sp_feat), sp_val=np.asarray(sp_val, dtype=np.float32),
                        giv_off=i32(giv_off), giv_label=i32(giv_label), giv_gap1=i32(giv_gap1),
                        pair_off=i32([0, len(pairs)]), pair_v0=i32([p[1] for p in pairs]), pair_v1=i32([p[2] for p in pairs]),
                        pair_gap1=i32([p[3] for p in pairs]))
        return corpus, vids, [p[4] for p in pairs]

    @staticmethod
    def _gap_class(f):
        if f.gap is None:
            raise TypeError("'>' not supported between instances of 'NoneType' and 'int'")
        if f.gap > 1:
            return False
        elif f.gap == 1:
            return True
        raise BaseException("only 2 kinds of distances are supported ...")

    def _run(self):
        if self._res is not None and self._res['key'] == (self._sweeps, self._theta_key(), bool(self.use_approx_inference),
                                                          bool(self.use_approx_beliefs)):
            return self._res
        if not self._initialized:
            raise KeyError('messages are not initialised: call initialize() first')
        eng = _engine_for(self)
        corpus, vids, pair_factors = self._lower()
        eng.set_theta(*self._pot_thetas())
        roots = corpus.roots_from_positions([list(self._roots)])
        r = eng.run(corpus, roots, self._sweeps, want_grad=True, want_marg=True, want_beliefs=True, want_messages=True,
                    approx_inference=bool(self.use_approx_inference), approx_beliefs=bool(self.use_approx_beliefs),
                    want_topk=min(50, eng.V))                 # get_max_vocab(50) lists (LBP.py:87, :115) made on the device
        V = eng.V
        # name the final pairwise messages like the reference's dict keys
        final = {}
        local = dict((vid, i) for i, vid in enumerate(vids))
        uni = np.full(V, 1.0 / V)
        slot = dict((i, 0) for i in range(len(vids)))
        for p, f in enumerate(pair_factors):                  # attach order == facset order of every variable
            d = f.potential_table.var_id2dim
            a, b = sorted(f.varset, key=lambda v: d[v.id])
            final[str(a), str(f)], final[str(b), str(f)] = r.messages['v2f'][p]
            for v in (a, b):
                m = r.messages['f2v'][local[v.id]][slot[local[v.id]]]
                final[str(f), str(v)] = uni.copy() if m is None else m
                slot[local[v.id]] += 1
        self._res = {'key': (self._sweeps, self._theta_key(), bool(self.use_approx_inference), bool(self.use_approx_beliefs)),
                     'vids': vids, 'pairs': pair_factors,
                     'beliefs': r.beliefs.cpu().numpy()[:, :V].astype(np.float64), 'grad': r.grad.cpu().numpy()[0],
                     'logp_var': r.logp_var.cpu().numpy(), 'top1': r.top1.cpu().numpy(), 'rank': r.rank.cpu().numpy(),
                     'topk': tuple(x.cpu().numpy() for x in r.topk), 'final': final}
        return self._res

    @property
    def messages(self):
        """graph.messages[(str(src), str(dst))] -> Message, like the dict the reference keeps (LBP.py:40)"""
        if self._eager is not None:
            return self._eager
        if self._messages is None:
            res = self._run()
            msgs = {}
            fin = res['final']
            for (a, b), m in fin.items():
                msgs[a, b] = Message(m.reshape(-1, 1))
            eng = _engine_for(self)
            for f in self.factors:                        # unary factor -> variable: normalize(copy(table)), LBP.py:492-498
                if len(f.varset) == 1:
                    msgs[str(f), str(f.varset[0])] = Message(eng.unary_message(f.factor_type, f.potential_table.observed_dim,
                                                                             self._gap_class(f) if f.factor_type == 'en_en' else False,
                                                                             self._sparse_for(f)).reshape(-1, 1))
            self._messages = msgs
        return self._messages

    def _sparse_now(self, observed_dim):
        col = self.phi_en_de[:, observed_dim, 2:5]
        e_idx, k_idx = np.nonzero(col)
        return [(int(e), 2 + int(k), float(col[e, k])) for e, k in zip(e_idx, k_idx)]

    def _sparse_for(self, f):
        """COO list of the dynamic features (train.py:176-215) of an en_de factor: the snapshot slice_potentials() took, else
        (a table attached without slice_potentials) the planes as they are now"""
        if f.factor_type != 'en_de':
            return []
        snap = getattr(f.potential_table, 'sparse', None)
        return snap if snap is not None else self._sparse_now(f.potential_table.observed_dim)

    # ------------------------------------------------------------------ reference API: results
    def get_posterior_probs(self):
        """LBP.py:247-259"""
        log_posterior = 0.0
        if self._eager is not None:
            for v_key, v in self.variables.items():
                p = v.get_marginal().m[v.supervised_label_index]
                with np.errstate(divide='ignore'):
                    _l = np.log(p)
                if _l == float('-inf'):
                    sys.stderr.write('err -inf' + str(p))
                    log_posterior += -99.99
                else:
                    log_posterior += np.sum(_l)
            return log_posterior
        res = self._run()
        for _l in res['logp_var']:
            if _l <= -99.99:
                sys.stderr.write('err -inf' + str(0.0))
            log_posterior += float(_l)
        return log_posterior

    def get_joint_log_likelihood(self):
        """Not in the reference: the joint log-likelihood of the supervised labels, log p(y) with
        p(y) ~ prod U_i(y_i) prod T_F(y_i, y_j), as loopy BP estimates it (Bethe free energy at the final messages; exact on
        trees).  get_posterior_probs is the sum of per-variable MARGINAL log-probabilities instead.  -inf when a label has
        belief 0.  Lazy batched mode only; the approximate modes are refused (ValueError)."""
        if self._eager is not None or self._explicit:
            raise NotImplementedError('the joint log-likelihood is computed on the device from the batched run: not available '
                                      'with explicit potential tables or once messages were set or updated by hand')
        if self.use_approx_inference or self.use_approx_beliefs:
            raise ValueError('the joint log-likelihood is not defined for the approximate modes')
        key = (self._sweeps, self._theta_key(), tuple(self._roots))
        if self._joint is None or self._joint[0] != key:
            if not self._initialized:
                raise KeyError('messages are not initialised: call initialize() first')
            eng = _engine_for(self)
            corpus, _, _ = self._lower()
            eng.set_theta(*self._pot_thetas())
            r = eng.run(corpus, corpus.roots_from_positions([list(self._roots)]), self._sweeps, want_grad=False,
                        want_marg=True, want_joint=True)
            self._joint = (key, float(r.logp_joint[0].item()))
        return self._joint[1]

    def get_max_postior_label(self, top=10):
        label_guesses = []
        for v_key, v in self.variables.items():
            s, sp, g = v.get_max_vocab(top)
            g_str = ' '.join([i + ' ' + p for i, p in g])
            label_guesses.append(s + ' ' + sp + ' ' + g_str)
        return label_guesses

    def _positioned(self):
        """factors that carry a sentence position, by position (ties keep factor-id order: the lines they produce are equal)"""
        return sorted((f for f in self.factors if f.position is not None), key=lambda f: f.position)

    def get_precision_counts(self):
        """(P@0, P@25, P@50, n) over the en_de factors' variables: where the supervised label sits in the 50 most probable
        words -- first / among the first 26 / listed at all (reference: LBP.py:80-106)."""
        hits = [0, 0, 0]
        n = 0
        for f in self.factors:
            if f.factor_type != 'en_de':
                continue
            n += 1
            label, _, top = f.varset[0].get_max_vocab(50)
            words = [w for w, _ in top]
            if label in words:
                place = words.index(label)
                for i, bound in enumerate((1, 26, 51)):
                    hits[i] += 1 if place < bound else 0
        return hits[0], hits[1], hits[2], n

    def to_string(self):
        """One prediction line per sentence position (reference: LBP.py:109-123): for a predicted token
        `<de word> <label> <log p(label)> <word log p> x 50`, for a given token ` <word> `."""
        lines = {}
        for f in self._positioned():
            if f.factor_type == 'en_de':
                label, label_logp, top = f.varset[0].get_max_vocab(50)
                lines[f.position] = ' '.join([f.word_label, label, label_logp] + ['%s %s' % wp for wp in top])
            elif f.factor_type == 'en_en':
                lines[f.position] = ' %s ' % f.word_label
        return [lines[pos] for pos in sorted(lines)]

    def to_dist(self):
        """One `.dist` line per predicted token (reference: LBP.py:125-143): `truth ||| guess ||| log-marginal x V`, 6 decimals."""
        out = []
        for f in self._positioned():
            if f.factor_type != 'en_de':
                continue
            v = f.varset[0]
            with np.errstate(divide='ignore'):
                logs = np.log(v.get_marginal().m).reshape(-1)
            out.append(' ||| '.join(['None' if v.truth_label is None else v.truth_label,
                                     'None' if v.supervised_label is None else v.supervised_label,
                                     ' '.join('%0.6f' % x for x in logs)]))
        return '\n'.join(out)

    def hw_inf(self, iterations):
        raise BaseException("This method assumes self.variables is a list.. depricated...")

    def get_unregularized_gradeint(self):
        """LBP.py:301-320 -> (grad_en_en (1,3), grad_en_de (1,6))"""
        for f in self.factors:
            if f.factor_type not in ('en_en', 'en_de'):
                raise BaseException('only 2 kinds of factors allowed...')
        grad_en_en = np.zeros_like(self.theta_en_en, dtype=DTYPE)
        grad_en_de = np.zeros_like(self.theta_en_de, dtype=DTYPE)
        if self._eager is not None:                      # LBP.py:304-319, factor by factor
            for f in self.factors:
                g = f.get_gradient()
                if f.factor_type == 'en_en':
                    grad_en_en += g
                else:
                    grad_en_de += g
            return grad_en_en, grad_en_de
        g = self._run()['grad']
        grad_en_en += g[:3].reshape(grad_en_en.shape)
        grad_en_de += g[3:].reshape(grad_en_de.shape)
        return grad_en_en, grad_en_de

    def get_gradient(self):
        """LBP.py:293-299 -> (grad_en_de, grad_en_en)   [sic: note the order]"""
        grad_en_en, grad_en_de = self.get_unregularized_gradeint()
        grad_en_en -= self.regularization_param * self.theta_en_en
        grad_en_de -= self.regularization_param * self.theta_en_de
        return grad_en_de, grad_en_en

    def return_gradient(self):
        """LBP.py:322-327 -> (lr * g_en_en, lr * g_en_de)"""
        grad_en_de, grad_en_en = self.get_gradient()
        return self.learning_rate * grad_en_en, self.learning_rate * grad_en_de

    def update_theta(self):
        """LBP.py:329-333 (in place, like the reference)"""
        grad_en_de, grad_en_en = self.get_gradient()
        self.theta_en_en += (self.learning_rate * grad_en_en)
        self.theta_en_de += (self.learning_rate * grad_en_de)
        return self.theta_en_en, self.theta_en_de


class VariableNode():
    def __init__(self, id, var_type, domain_type, domain, supervised_label):
        if not isinstance(id, int):
            print('id ', id, 'not an int')
        idx = _index_of(domain, supervised_label)
        if idx is None:
            print(supervised_label, 'not in', 'domain of size %d' % len(domain))
            exit(-1)
        self.id = id
        self.var_type = var_type
        self.domain = domain
        self.facset = []
        self.graph = None
        self.supervised_label = supervised_label
        self.supervised_label_index = idx
        self.domain_type = domain_type
        self.truth_label = None
        self.truth_label_index = None

    def set_truth_label(self, tl):
        self.truth_label = tl

    def __str__(self):
        return "X_" + str(self.id)

    def __eq__(self, other):
        return isinstance(other, VariableNode) and self.id == other.id

    __hash__ = None

    def display(self, m):
        raise NotImplementedError()

    def add_factor(self, fc):
        if __debug__: assert isinstance(fc, FactorNode)
        self.facset.append(fc)

    def init_message_to(self, fc, init_m):
        raise AttributeError("VariableNode instance has no attribute 'messages'")      # LBP.py:375 is broken the same way

    def update_message_to(self, fc):
        """LBP.py:377-389: leave-one-out product of the incoming factor messages, one au.pointwise_multiply (device) per
        message, then renormalise.  Switches the graph to eager mode."""
        if __debug__: assert isinstance(fc, FactorNode)
        if __debug__: assert fc in self.facset
        msgs = self.graph._enter_eager()
        new_m = Message.new_message(self.domain, 1.0 / len(self.domain))
        for other_fc in self.facset:
            if other_fc is not fc:
                m = msgs[str(other_fc), str(self)]
                new_m = pointwise_multiply(m, new_m)
                if __debug__: assert np.shape(new_m.m) == np.shape(m.m)
        if self.graph.normalize_messages:
            new_m.renormalize()
        msgs[str(self), str(fc)] = new_m

    def get_marginal(self):
        """LBP.py:392-400"""
        if self.graph._eager is not None:
            new_m = Message.new_message(self.domain, 1.0 / len(self.domain))
            for fc in self.facset:
                new_m = pointwise_multiply(self.graph._eager[str(fc), str(self)], new_m)
            if self.graph.normalize_messages:
                new_m.renormalize()
            return new_m
        res = self.graph._run()
        return Message(res['beliefs'][res['vids'].index(self.id)].reshape(-1, 1))

    def get_max_vocab(self, top):
        """(label, '%0.4f' % log p(label), [(word, '%0.4f' % log p)] for the `top` most probable words, best first)
        (reference: LBP.py:402-411; the same argpartition + argsort calls, so exact ties order alike)"""
        belief = self.get_marginal().m.reshape(-1)
        best = None
        if self.graph._eager is None:
            # the list mlbp_topk_rows made on the device (descending probability); rows whose order exact ties leave open are
            # re-listed with the reference's own calls, whose order among equal values is NumPy's
            res = self.graph._run()
            idx, _, ties = res['topk']
            row = res['vids'].index(self.id)
            if top <= idx.shape[1] and ties[row] == 0:
                best = idx[row, :top]
        if best is None:
            best = np.argpartition(belief, -top)[-top:]
            best = best[np.argsort(belief[best])][::-1]
        with np.errstate(divide='ignore'):
            logs = np.log(belief)
        return (self.supervised_label, '%0.4f' % logs[self.supervised_label_index],
                [(self.domain[i], '%0.4f' % logs[i]) for i in best])


class FactorNode():
    _seq = [0]

    def __init__(self, id, factor_type=None, observed_domain_type=None, observed_value=None, observed_domain_size=None):
        if __debug__: assert isinstance(id, int)
        self.id = id
        self.varset = []
        self.potential_table = None
        self.factor_type = factor_type
        self.graph = None
        self.observed_domain_type = observed_domain_type
        self.observed_value = observed_value
        self.observed_domain_size = observed_domain_size
        self.position = None
        self.word_label = None
        self.gap = None
        self.connect_type = None
        self._attach_seq = -1

    def __str__(self):
        return 'F_' + str(self.id)

    def __eq__(self, other):
        return isinstance(other, FactorNode) and self.id == other.id

    __hash__ = None

    def init_message_to(self, var, init_m):
        raise NotImplementedError('messages live on the GPU; initialize() resets them to uniform')

    def add_varset_with_potentials(self, varset, ptable):
        if __debug__: assert isinstance(ptable, PotentialTable)
        if len(varset) == 2:
            if __debug__: assert varset[0] != varset[1]
        if __debug__: assert len(varset) == len(ptable.var_id2dim)
        if len(varset) > 2:
            raise NotImplementedError("Currently supporting unary and pairwise factors...")
        for v in varset:
            if __debug__: assert v not in self.varset
            self.varset.append(v)
            v.add_factor(self)
        ptable.add_factor(self)
        self.potential_table = ptable
        FactorNode._seq[0] += 1
        self._attach_seq = FactorNode._seq[0]

    def _table_kind(self, what):
        """which of the graph's three tables this factor uses: en_de, or en_en by gap (== 1: the *_w1 table, > 1: the plain
        one; reference: LBP.py:456-480)"""
        if self.factor_type == 'en_de':
            return 'en_de'
        if self.factor_type == 'en_en':
            if self.gap > 1:
                return 'en_en'
            if self.gap == 1:
                return 'en_en_w1'
            raise BaseException("only 2 kinds of distances are supported ..." if what == 'pot' else
                                "only 2 distances supported at the moment")
        raise BaseException("only two kinds of potentials are supported..." if what == 'pot' else
                            "only 2 feature value types are supported right now..")

    def get_pot(self):
        return getattr(self.graph, 'pot_' + self._table_kind('pot'))

    def get_phi(self):
        return getattr(self.graph, 'phi_' + self._table_kind('phi'))

    def get_shape(self):
        """(rows, columns) of the potential table: a unary factor's second axis is its observed domain (LBP.py:482-488)"""
        if len(self.varset) not in (1, 2):
            raise BaseException("only unary or binary factors are supported...")
        rows = len(self.varset[0].domain)
        return rows, (self.observed_domain_size if len(self.varset) == 1 else len(self.varset[1].domain))

    def update_message_to(self, var):
        """LBP.py:490-526: unary -> normalize(copy(table)); pairwise -> T.m or m'.T through au.dense_dot (device), or
        au.sparse_vec_mat_dot with use_approx_inference; then renormalise.  Switches the graph to eager mode."""
        msgs = self.graph._enter_eager()
        other_vars = [v for v in self.varset if v.id != var.id]
        if len(other_vars) == 0:
            new_m = Message(np.copy(self._table()))
        else:
            o_var = other_vars[0]
            o_var_dim = self.potential_table.var_id2dim[o_var.id]
            msg = msgs[str(o_var), str(self)]
            table = np.ascontiguousarray(self._table())
            if o_var_dim == 1:
                if self.graph.use_approx_inference:
                    marginalized = au.sparse_vec_mat_dot(msg.m, table)
                else:
                    marginalized = au.dense_dot(table, msg.m)
            else:
                if self.graph.use_approx_inference:
                    marginalized = au.sparse_vec_mat_dot(np.ascontiguousarray(msg.m.T), table)
                else:
                    marginalized = au.dense_dot(np.ascontiguousarray(msg.m.T), table)
            new_m = Message(marginalized)
        if self.graph.normalize_messages:
            new_m.renormalize()
        if __debug__: assert np.shape(new_m.m) == np.shape(msgs[str(self), str(var)].m)
        msgs[str(self), str(var)] = new_m

    def _table(self):
        """the factor's potential table as a float64 array: the explicit array of PotentialTable(table=...), else
        computed on the GPU from theta and the features"""
        if self.potential_table.explicit:
            return self.potential_table.table
        from . import LBP as _self  # noqa: F401
        eng = _engine_for(self.graph)
        g = self.graph
        eng.set_theta(*g._pot_thetas())
        if len(self.varset) == 1:
            gap1 = FactorGraph._gap_class(self) if self.factor_type == 'en_en' else False
            return eng.unary_message(self.factor_type, self.potential_table.observed_dim, gap1, g._sparse_for(self),
                                     normalized=False).reshape(-1, 1)
        return eng.dense_table(FactorGraph._gap_class(self))

    def get_factor_beliefs(self):
        """LBP.py:528-574: unary -> normalize(table) (incoming messages ignored); pairwise -> normalize((c r') o T)"""
        if len(self.varset) == 1:
            if self.graph.report_times: ub = time.time()
            beliefs = au.normalize(self._table())
            if self.graph.report_times: self.graph.ub_times.append(time.time() - ub)
            return beliefs
        if self.graph.report_times: bb = time.time()
        r = c = None
        for v in self.varset:
            vd = self.potential_table.var_id2dim[v.id]
            m = self.graph.messages[str(v), str(self)]
            if vd == 0:
                c = np.reshape(m.m, (np.size(m.m), 1))
            elif vd == 1:
                r = np.reshape(m.m, (1, np.size(m.m)))
            else:
                raise NotImplementedError("only supports pairwise factors..")
        c, r = np.ascontiguousarray(c), np.ascontiguousarray(r)
        if self.graph.use_approx_beliefs and np.size(c) > au.K:   # LBP.py:554-563: the top-K x top-K block only
            approx_marginals, c_idx, r_idx = au.sparse_dot(c, r)
            beliefs = au.sparse_pointwise_multiply(approx_marginals, c_idx, r_idx, self._table())
            beliefs = au.sparse_normalize(beliefs, c_idx, r_idx)
        else:
            marginals = au.dense_dot(c, r)
            beliefs = au.normalize(au.dense_pointwise_multiply(marginals, self._table()))
        if self.graph.report_times: self.graph.bb_times.append(time.time() - bb)
        return beliefs

    def get_observed_factor_as_array(self):
        cell = sorted([(self.potential_table.var_id2dim[v.id], v.supervised_label_index) for v in self.varset])
        return [tuple([o for d, o in cell])]

    def get_observed_factor(self):
        """LBP.py:584-589"""
        shape = (len(self.varset[0].domain), 1) if len(self.varset) == 1 else self.get_shape()
        of = np.zeros(shape, dtype=DTYPE)
        cell = sorted([(self.potential_table.var_id2dim[v.id], v.supervised_label_index) for v in self.varset])
        cell = tuple([o for d, o in cell])
        of[cell if len(cell) == 2 else (cell[0], 0)] = 1.0
        return of

    def cell_gradient(self):
        return self.get_observed_factor() - self.get_factor_beliefs()

    def cell_gradient_alt(self):
        d = -self.get_factor_beliefs()
        for c in self.get_observed_factor_as_array():
            d[c if len(c) == 2 else (c[0], 0)] = 1.0 + d[c if len(c) == 2 else (c[0], 0)]
        return d

    def get_gradient(self):
        """LBP.py:592-613 -> (1, F)"""
        g = self.cell_gradient()
        if self.graph.report_times: gg = time.time()
        if self.potential_table.observed_dim is not None:
            phi_g = self.get_phi()[:, self.potential_table.observed_dim, :]
            grad = au.dense_dot(np.ascontiguousarray(g.T), np.ascontiguousarray(phi_g, dtype=np.float64))
        else:
            phi = self.get_phi()
            grad = np.array([float(au.dense_dot(np.ascontiguousarray(g.reshape(1, -1)),
                                                np.ascontiguousarray(phi[:, :, k].reshape(-1, 1), dtype=np.float64))[0, 0])
                             for k in range(phi.shape[2])])
        grad = np.reshape(grad, (1, np.size(grad)))
        if self.graph.report_times: self.graph.gg_times.append(time.time() - gg)
        return grad


class ObservedFactor(FactorNode):
    def __init__(self, id, observed_domain_type, observed_value):
        FactorNode.__init__(self, id, factor_type=UNARY_FACTOR)
        self.observed_domain_type = observed_domain_type
        self.observed_value = observed_value


class Message():
    def __init__(self, m):
        if __debug__: assert isinstance(m, np.ndarray)
        if __debug__: assert np.size(m[m < 0.0]) == 0
        if np.shape(m) != (np.size(m), 1):
            self.m = np.reshape(m, (np.size(m), 1))
        else:
            self.m = m

    def __str__(self):
        return np.array_str(self.m)

    def renormalize(self):
        """LBP.py:649-659"""
        s = np.sum(self.m)
        if s > 0:
            self.m = au.normalize(self.m)
        else:
            e = np.empty_like(self.m)
            e.fill(1.0 / np.size(self.m))
            self.m = e
        if __debug__: assert np.size(self.m[self.m < 0.0]) == 0
        if __debug__: assert np.abs(np.sum(self.m) - 1.0) < 1e-10

    @staticmethod
    def new_message(domain, init):
        m = np.empty((len(domain), 1))
        m.fill(init)
        if m.dtype != DTYPE:
            m = m.astype(DTYPE)
        return Message(m)


class PotentialTable():
    def __init__(self, v_id2dim, table=None, observed_dim=None):
        self.factor = None
        self.observed_dim = observed_dim
        self.var_id2dim = v_id2dim
        self.explicit = table is not None
        self.table = None
        if table is not None:
            if __debug__: assert isinstance(table, np.ndarray)
            if observed_dim is not None:
                if __debug__: assert len(v_id2dim) == 1
                if v_id2dim[list(v_id2dim.keys())[0]] == 0:
                    self.table = np.reshape(table[:, observed_dim], (np.shape(table)[0], 1))
                else:
                    raise NotImplementedError("a unary factor should always be a column vector")
            else:
                self.table = table
            if self.table.dtype != DTYPE:
                self.table = self.table.astype(DTYPE)

    def slice_potentials(self):
        """LBP.py:695-710.  When the caller computed graph.pot_* (train.py:251-253) the table is sliced from it like the
        reference does (a view / column copy, no arithmetic); the GPU engine never reads it -- it rebuilds the potentials
        from theta and the features."""
        # the per-sentence (dynamic) features of an en_de factor are fixed HERE, like the reference's potentials are
        # (train.py:239-250 computes them right before this call): graphs built from one PhiWrapper one after the other must
        # not see each other's history features when they are evaluated later
        g = getattr(self.factor, 'graph', None)
        if g is not None and self.factor.factor_type == 'en_de' and self.observed_dim is not None and not self.explicit:
            self.sparse = g._sparse_now(self.observed_dim)
        table = self.factor.get_pot()
        if table is None:
            self.table = None
            return
        table = np.reshape(table, self.factor.get_shape())
        if self.observed_dim is not None:
            table = np.reshape(table[:, self.observed_dim], (np.shape(table)[0], 1))
        self.table = table
        if self.table.dtype != DTYPE:
            self.table = self.table.astype(DTYPE)

    def add_factor(self, factor):
        if __debug__: assert isinstance(factor, FactorNode)
        if __debug__: assert self.factor is None
        self.factor = factor


def pointwise_multiply(m1, m2):
    """LBP.py:717-730"""
    if __debug__: assert isinstance(m1, Message)
    if __debug__: assert isinstance(m2, Message)
    if m2 is None:
        return m1
    elif m1 is None:
        return m2
    else:
        if __debug__: assert np.shape(m1.m) == np.shape(m2.m)
        new_m = au.pointwise_multiply(m1.m, m2.m)
        new_m = np.nan_to_num(new_m)
    return Message(new_m)


class PhiWrapper:
    def __init__(self, phi_en_en, phi_en_en_w1, phi_en_de):
        self.phi_en_en = phi_en_en
        self.phi_en_en_w1 = phi_en_en_w1
        self.phi_en_de = phi_en_de


class ThetaWrapper(object):
    def __init__(self, theta_en_en_names, theta_en_en, theta_en_de_names, theta_en_de):
        self.theta_en_en_names = theta_en_en_names
        self.theta_en_de_names = theta_en_de_names
        self.theta_en_en = theta_en_en
        self.theta_en_de = theta_en_de
