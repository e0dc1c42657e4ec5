"""Batched LBP executor: many sentence graphs -> level-batched sm_100a kernels behind the C ABI (include/mlbp.h).

Replaces, for a whole batch of sentences at once, the reference's per-sentence sequence
    create_factor_graph (train.py:133-305) -> fg.initialize (LBP.py:192-216) -> fg.treelike_inference (:218-245)
    -> fg.get_unregularized_gradeint (:301-320) -> fg.get_posterior_probs (:247-259) -> get_precision_counts (:80-106)

Data layout in HBM (all rows padded to ld = roundup(V, 64) elements):
    Model   pmi, pmi_w1 [V, ld] fp32; edT, pedT [Vd, ld] fp32 (de-major)            resident, like weights
    Tables  planes [14, V, ld] fp16 (hi/lo operand planes), colsums [5, V], edstats  rebuilt once per theta (K2)
    U       [NV, ld] fp32   product of each variable's unary messages (K1)
    A_hi/lo [RA, ld] fp16   variable->factor messages, one row per GEMM row that reads them (K3 -> K4)
    D       [RD, ld] fp32   factor->variable messages, one row per GEMM row (K4 -> K3/K5/K6)
PyTorch is used for device memory and streams only; all arithmetic is in libmlbp.so.
"""
import contextlib
import ctypes
import math
import os

import numpy as np
import torch

from . import _lib

# plan blob header (csrc/plan.cpp)
(H_NLEVELS, H_LEVELS_OFF, H_INIT_N, H_INIT_OFF, H_NPAIR, H_PAIR_C, H_PAIR_U0, H_PAIR_U1, H_PAIR_U2, H_PAIR_GAP1,
 H_PAIR_V0, H_PAIR_V1, H_NGRAD_GEMM, H_GRAD_GEMM_OFF, H_MARG_N, H_MARG_U, H_MARG_OFF, H_MARG_IN, H_NGRAPHS,
 H_A_ROWS, H_D_ROWS, H_MAX_IN, H_NVARS, H_PAIR_R, H_PAIR_Z, H_MSG_BLK_N, H_MSG_BLK_OFF, H_MSG_ROWS, H_SPK_BLK_N, H_PAIR_M0,
 H_PAIR_M1) = range(31)
H_WORDS, LEV_WORDS, GEMM_WORDS = 32, 10, 4
(PLAN_BLOB_WORDS, PLAN_A_ROWS, PLAN_D_ROWS, PLAN_N_LEVELS, PLAN_N_PAIR, PLAN_N_GEMM_ROWS, PLAN_MAX_IN, PLAN_HDR_WORDS,
 PLAN_N_DEAD, PLAN_TMPL_HITS, PLAN_TMPL_MISSES) = range(11)
A_SCALE_LOG2 = 14
GEMM_A_HI_ONLY = 256          # include/mlbp.h MLBP_GEMM_A_HI_ONLY
GEMM_B_HI_ONLY = 512          # include/mlbp.h MLBP_GEMM_B_HI_ONLY
N_PLANES = 20
TRANSPOSED_TABLE = {0: 1, 1: 0, 2: 3, 3: 2, 4: 7, 5: 8, 6: 9}   # include/mlbp.h MLBP_TABLE_*: where a table's columns are rows
N_SUMS = 7
D_CONST_ROWS = 5
# Engine._flags (device int32 words): the peak flag of the var->factor kernel (sticky per theta), the flagged-variable count of
# one marginals launch, and the re-score counters (mlbp_rescore_candidates)
FLAG_PEAK, FLAG_NFLAGGED, FLAG_MAXBITS, FLAG_SPIKE, FLAG_NSPIKY, FLAG_COUNTERS, FLAG_WORDS = 0, 1, 2, 3, 4, 8, 16
SPIKE_SLOTS = 4               # include/mlbp.h MLBP_SPIKE_SLOTS
FMT_MAX_BYTES = 12            # include/mlbp.h MLBP_FMT_MAX_BYTES: text bytes per number that mlbp_format_log_rows may need


def round_up(x, m):
    return (x + m - 1) // m * m


def _p(t, word_off=0):
    """device (or host) pointer of a tensor, optionally offset by int32 words"""
    if t is None:
        return None
    return ctypes.c_void_p(t.data_ptr() + 4 * word_off)


def _hp(a):
    return a.ctypes.data_as(ctypes.c_void_p)


class Kernels(object):
    """The product back end: libmlbp.so on the current CUDA device.  Constructing it without a B200 raises."""

    def __init__(self):
        self.lib = _lib.require_device()
        self.device = torch.device('cuda', torch.cuda.current_device())

    @staticmethod
    def stream():
        return ctypes.c_void_p(torch.cuda.current_stream().cuda_stream)

    def call(self, name, *args):
        _lib.check(getattr(self.lib, name)(*args, self.stream()))


class Model(object):
    """Feature planes resident on the device (what train.py:589-612 loads once and wraps in PhiWrapper)."""

    def __init__(self, pmi, pmi_w1, ed, ped, device):
        pmi, pmi_w1, ed, ped = (np.asarray(x) for x in (pmi, pmi_w1, ed, ped))
        V, Vd = ed.shape
        assert pmi.shape == (V, V) and pmi_w1.shape == (V, V) and ped.shape == (V, Vd)
        self.V, self.Vd, self.ld = V, Vd, round_up(V, 64)
        self.device = device

        def padded(a):
            t = torch.zeros((a.shape[0], self.ld), dtype=torch.float32)
            t[:, :V] = torch.from_numpy(np.ascontiguousarray(a, dtype=np.float32))
            return t.to(device)

        self.pmi, self.w1 = padded(pmi), padded(pmi_w1)
        self.edT, self.pedT = padded(ed.T), padded(ped.T)
        self.frange = (float(pmi.min()), float(pmi.max()), float(pmi_w1.min()), float(pmi_w1.max()))
        self.ed_range = (float(ed.max() - ed.min()), float(ped.max() - ped.min()))

    @classmethod
    def from_dict(cls, m, device):
        return cls(m['pmi'], m['pmi_w1'], m['ed'], m['ped'], device)

    @classmethod
    def from_text(cls, pmi, pmi_w1, ed, ped, V, Vd, device=None, chunk_bytes=None, kernels=None):
        """The model that Model(*[np.loadtxt(p, dtype=np.float64, ndmin=2) for p in (pmi, pmi_w1, ed, ped)], device) builds,
        with the text parsed on the GPU (textload.py, K8): pmi / pmi_w1 [V, V] and ed / ped [V, Vd] text files.  A file
        that is not a clean V-row matrix in the device grammar is read with np.loadtxt instead (one RuntimeWarning).
        chunk_bytes: size of the two pinned read buffers (default 256 MB).  A back end whose device is not a GPU (the
        emulated kernels of the CPU test tier) has nothing to parse on: it gets the np.loadtxt path."""
        from . import textload
        paths = (pmi, pmi_w1, ed, ped)
        cuda = device is not None and torch.device(device).type == 'cuda'
        with torch.cuda.device(torch.device(device)) if cuda else contextlib.nullcontext():
            k = kernels or Kernels()
            if k.device.type != 'cuda':
                return cls(*[np.loadtxt(p, dtype=np.float64, ndmin=2) for p in paths], device=k.device)
            return textload.model_from_text(cls, paths, V, Vd, k, chunk_bytes)


class Corpus(object):
    """Sentences lowered to the flat integer arrays the kernels index (host numpy + lazily cached device copy).

    Restates train.py:255-297: one variable per PREDICTED position (sentence order), one en_de unary factor per
    variable, a unary en_en factor per (predicted, given) pair and a pairwise en_en factor per predicted pair,
    gap = |i - j| (gap == 1 selects pot_en_en_w1, LBP.py:456-463).  Sparse per-sentence en_de features
    (train.py:176-215) are kept only where their German index equals the variable's observed word: the only
    column of phi_en_de the variable's factor ever reads (LBP.py:602, :702-703)."""

    MAX_PREDICTED = 49          # 48 pairwise factors per variable (mlbp_var_to_factor), 64 in mlbp_marginals

    FIELDS = ('var_off', 'var_de', 'var_label', 'var_pos', 'sp_off', 'sp_en', 'sp_feat', 'sp_val', 'giv_off',
              'giv_label', 'giv_gap1', 'pair_off', 'pair_v0', 'pair_v1', 'pair_gap1')

    def __init__(self, sentences=None, **arrays):
        if sentences is None:
            for k in self.FIELDS:
                setattr(self, k, arrays[k])
        else:
            self._build(sentences)
        self._dev = {}

    def _build(self, sentences):
        var_off, var_de, var_label, var_pos = [0], [], [], []
        sp_off, sp_en, sp_feat, sp_val = [0], [], [], []
        giv_off, giv_label, giv_gap1 = [0], [], []
        pair_off, pair_v0, pair_v1, pair_gap1 = [0], [], [], []
        for s in sentences:
            kind, label, de = s.kind, s.label, s.de
            pred = [p for p in range(len(kind)) if kind[p] == 1]
            given = [p for p in range(len(kind)) if kind[p] == 0]
            if not pred:
                raise ValueError('sentence without predicted tokens has no factor graph (LBP.py:193)')
            if len(pred) > self.MAX_PREDICTED:
                # the reference has no limit; the leave-one-out kernel (K3) handles at most 48 pairwise messages per variable.
                # Raised HERE, when the batch is lowered, not from a kernel launch in the middle of an epoch.
                raise ValueError('sentence with %d predicted tokens: at most %d are supported' % (len(pred), self.MAX_PREDICTED))
            for p in pred:
                var_de.append(int(de[p])); var_label.append(int(label[p])); var_pos.append(p)
                for e, d, f, val in s.sparse:
                    if int(d) == int(de[p]):
                        sp_en.append(int(e)); sp_feat.append(int(f)); sp_val.append(float(val))
                sp_off.append(len(sp_en))
                for q in given:
                    giv_label.append(int(label[q])); giv_gap1.append(1 if abs(p - q) == 1 else 0)
                giv_off.append(len(giv_label))
            for a in range(len(pred)):
                for b in range(a + 1, len(pred)):
                    pair_v0.append(a); pair_v1.append(b); pair_gap1.append(1 if pred[b] - pred[a] == 1 else 0)
            var_off.append(len(var_de)); pair_off.append(len(pair_v0))
        i32 = lambda x: np.asarray(x, dtype=np.int32)
        self.var_off, self.var_de, self.var_label, self.var_pos = i32(var_off), i32(var_de), i32(var_label), i32(var_pos)
        self.sp_off, self.sp_en, self.sp_feat = i32(sp_off), i32(sp_en), i32(sp_feat)
        self.sp_val = np.asarray(sp_val, dtype=np.float32)
        self.giv_off, self.giv_label, self.giv_gap1 = i32(giv_off), i32(giv_label), i32(giv_gap1)
        self.pair_off, self.pair_v0, self.pair_v1, self.pair_gap1 = i32(pair_off), i32(pair_v0), i32(pair_v1), i32(pair_gap1)

    @property
    def n_sent(self):
        return len(self.var_off) - 1

    @property
    def n_vars(self):
        return int(self.var_off[-1])

    @property
    def n_pairs(self):
        return int(self.pair_off[-1])

    def slice(self, lo, hi):
        """sentences [lo, hi) as a Corpus with rebased offsets"""
        v0, v1 = int(self.var_off[lo]), int(self.var_off[hi])
        p0, p1 = int(self.pair_off[lo]), int(self.pair_off[hi])
        s0, s1 = int(self.sp_off[v0]), int(self.sp_off[v1])
        g0, g1 = int(self.giv_off[v0]), int(self.giv_off[v1])
        return Corpus(var_off=self.var_off[lo:hi + 1] - v0, var_de=self.var_de[v0:v1], var_label=self.var_label[v0:v1],
                      var_pos=self.var_pos[v0:v1], sp_off=self.sp_off[v0:v1 + 1] - s0, sp_en=self.sp_en[s0:s1],
                      sp_feat=self.sp_feat[s0:s1], sp_val=self.sp_val[s0:s1], giv_off=self.giv_off[v0:v1 + 1] - g0,
                      giv_label=self.giv_label[g0:g1], giv_gap1=self.giv_gap1[g0:g1],
                      pair_off=self.pair_off[lo:hi + 1] - p0, pair_v0=self.pair_v0[p0:p1], pair_v1=self.pair_v1[p0:p1],
                      pair_gap1=self.pair_gap1[p0:p1])

    def roots_from_positions(self, roots_pos):
        """reference roots are variable ids = sentence positions; the plan wants indices local to the sentence"""
        out = np.zeros((self.n_sent, len(roots_pos[0])), dtype=np.int32)
        for s in range(self.n_sent):
            pos = self.var_pos[self.var_off[s]:self.var_off[s + 1]].tolist()
            out[s] = [pos.index(int(r)) for r in roots_pos[s]]
        return out

    def gemm_rows_estimate(self, sweeps, grad):
        k = np.diff(self.var_off).astype(np.int64)
        rows = sweeps * k * (k - 1) + (3 * k * (k - 1) // 2 + k * (k - 1) // 2 if grad else 0)
        return rows

    def dev(self, name, device):
        key = (name, str(device))
        if key not in self._dev:
            a = getattr(self, name)
            t = torch.from_numpy(np.ascontiguousarray(a))
            if len(a) == 0:
                t = torch.zeros(1, dtype=t.dtype)          # keep a valid pointer for empty CSR payloads
            self.h2d_bytes = getattr(self, 'h2d_bytes', 0) + t.numel() * t.element_size()
            if torch.device(device).type == 'cuda':
                t = t.pin_memory()                        # asynchronous H2D: the host does not wait for queued GPU work
            self._dev[key] = t.to(device, non_blocking=True)
        return self._dev[key]


class Result(object):
    """Outputs of one Engine.run: tensors stay on the device until read."""

    def __init__(self, grad, logp, logp_var, top1, rank, beliefs, stats, messages=None, topk=None, logp_joint=None,
                 map_score=None, label_score=None):
        self.grad, self.logp, self.logp_var, self.top1, self.rank, self.beliefs, self.stats = \
            grad, logp, logp_var, top1, rank, beliefs, stats
        # want_joint: [n_sent] float64, each sentence's joint log-likelihood of its labels, the Bethe estimate at the final
        # messages (mlbp_joint_logp); -inf where a label has belief 0.  `logp` is the sum of MARGINAL log-probabilities.
        self.logp_joint = logp_joint
        # max_product: [n_sent] float64, the log of the unnormalised joint potential of the decoded assignment (top1) and of the
        # labels (mlbp_assignment_score); map_score - label_score is the log-odds of the model's best joint guess against the labels
        self.map_score, self.label_score = map_score, label_score
        self.messages = messages     # final pairwise messages (want_messages): see Engine.run
        # want_topk = K: (idx [n_vars, K] int32, prob [n_vars, K] float32, n_ties [n_vars] int32), best first, made on the
        # device by mlbp_topk_rows (VariableNode.get_max_vocab, LBP.py:402-411)
        self.topk = topk

    def precision_counts(self):
        """FactorGraph.get_precision_counts (LBP.py:80-106) summed over the batch: (p@0, p@25, p@50, total)"""
        r = self.rank
        return int((r == 0).sum()), int((r < 26).sum()), int((r < 50).sum()), int(r.numel())


class Engine(object):
    def __init__(self, model, kernels=None, workspace_bytes=24 << 30, gemm_impl=0, grad_a_terms=1, grad_b_terms=1,
                 gemm_slice_pairs=None, msg_passes=None, tau=None, tau_label=None, peak_mult=16.0, one_pass_min_v=4096,
                 gemm_k_chunks=None):
        self.k = kernels if kernels is not None else Kernels()
        self.device = self.k.device
        self.model = model if isinstance(model, Model) else Model.from_dict(model, self.device)
        self.V, self.Vd, self.ld = self.model.V, self.model.Vd, self.model.ld
        self.workspace_bytes = int(workspace_bytes)
        self.gemm_impl = gemm_impl
        # Gradient-stage GEMM rows multiply only the hi half of the message r (2 tensor-core passes instead of 3): the
        # expectation N/Z is a ratio of two rows built from the same r, so its 2^-12 rounding largely cancels (<= 2e-7
        # relative on a sentence's gradient, measured against the float64 oracle).  2 = all three passes.
        self.grad_a_terms = int(grad_a_terms)
        self.grad_b_terms = int(grad_b_terms)     # 1: the table's lo half is dropped too where grad_one_pass_ok (set_theta)
        self.gemm_slice_rows = self._gemm_slice_rows(gemm_slice_pairs)
        # K ranges of one GEMM launch (elements, multiples of 64): a long contraction can be issued as several launches that add
        # into D (mlbp_factor_to_var_gemm_gated k0 / k_len).  The idea -- a kernel boundary re-aligns CTA pairs that drifted
        # apart in K, as the row slices above do -- was MEASURED at V = 50 000 (782 k-blocks in four launches of 196) and did
        # not pay: C5 25.8 vs 27.5 sentences/s, 970 vs 1 045 TFLOP/s executed (profiles/r2a_bench_c5_ab_k_ranges.txt): four
        # epilogues and read-modify-writes of D per tile cost more than the re-alignment saves.  Off unless asked for.
        n_k = int(gemm_k_chunks or 1)
        step = round_up(-(-self.V // n_k), 64)
        self.gemm_k_ranges = [(k0, min(step, self.V - k0)) for k0 in range(0, self.V, step)] if n_k > 1 else [(0, 0)]
        # Message rows with REDUCED tensor-core passes plus an exact re-score of every near-tied decision (csrc/rescore.cu).
        #   two passes  A_hi . (B_hi + B_lo): the lo half of the message is dropped;
        #   ONE pass    A_hi . B_hi         : the lo half of the table is dropped too (the default at V >= 8192, see msg_passes).
        # Why this is safe: a rounding error upstream is damped by every later contraction (a message D = T a averages V terms,
        # and K2 rounds the table's hi halves stochastically, so equal entries do not share one error), so the only error that
        # reaches a belief undamped is the rounding of the LAST hop -- measured on the ratio of two candidates' beliefs at
        # V = 10 000 in the bench's trained regime: 2.5e-7 relative (mean absolute) with two passes, 2.2e-5 with one -- and that
        # hop is recomputed from the full 22-bit operands for every candidate within `tau` of the arg-max (or within
        # `tau_label` of the label while its rank can matter): the bands are ~15x that error.  Against the float64 oracle with
        # one pass (profiles/r2c_*): 0 top-1 mismatches, beliefs 4e-8 abs (contract 1e-4), gradients 2e-6 relative at C3 size and
        # 6e-6 on the hostile cases of tests/test_gpu_gates.py (contract 1e-4), log-posterior 3e-6 relative.
        # Guards: (i) the potentials span at most e^3 (set_theta); (ii) spikes: an element that carries more than peak_mult / V
        # of a message's mass does not average its rounding away, so mlbp_spike_scan files it and mlbp_spike_correct restores
        # the dropped terms of that element exactly after the GEMM (a few AXPYs per spiky row: its lo part times the full table
        # row and, with one pass, its hi part times the table row's lo half); a row with more spikes than slots raises a flag
        # ON THE DEVICE that switches all later message GEMMs of this theta to three passes (mlbp_factor_to_var_gemm_gated; no
        # host synchronisation).  The one-pass gradient rows are gated the same way: once any spike was seen they keep the lo
        # half of the table planes (a peaked belief does not average the fp16 rounding of T o PMI away: tests/test_gpu_gates.py).
        # msg_passes: None = one pass where V >= 8192, two where 4096 <= V < 8192 (the rounding noise of the un-spiky remainder of
        # a message shrinks like 1 / sqrt(V); worst belief error seen with ONE pass on the hostile cases at V = 4608: 1.3e-5
        # absolute against the contract's 1e-4, ten times the two-pass figure, so the smaller vocabularies keep the second
        # pass); 1 / 2 = one / two passes at any V; 3 = never reduced.  MLBP_MSG_PASSES in the environment overrides None (A/B runs of whole suites).
        if msg_passes is None and os.environ.get('MLBP_MSG_PASSES'):
            msg_passes = int(os.environ['MLBP_MSG_PASSES'])
        self.msg_passes = msg_passes
        self.one_pass_min_v = int(one_pass_min_v)   # one-pass gradient rows from this vocabulary size on (tests lower it)
        # bands of the near-tie detection: defaults 4e-4 / 2e-4 with one-pass message rows, 2e-4 / 1e-4 with two
        self.msg_one_pass_min_v = 8192
        one = self.msg_passes == 1 or (self.msg_passes is None and self.V >= self.msg_one_pass_min_v)
        self.msg_one_pass = one                     # (only while msg_two_pass_ok: set_theta's gate on the potentials' span)
        # ONE-pass rows multiply the hi half of R = T - tbar (tbar = the table at phi = 0) and add tbar * sum(message) back as
        # a constant: the fp16 rounding of the table is then relative to |T - tbar| -- zero under the zeros of a sparse feature
        # plane, small everywhere once the pairwise weights are small (the regime SGD drives the bench into) -- instead of to T.
        # Measured against the float64 oracle in that regime at V = 10 000 (profiles/r2h_*, r2i_*): worst belief error 1.3e-5 ->
        # 6.4e-8 absolute, log-posterior 2e-6 -> 8e-9, decisions moved by the re-score 1 405 -> 6 per 82 k variables; hostile sparse
        # case at V = 4 608: 1.3e-5 -> 3.9e-6.  Price: 3.5 % of the step (same-box A/B 3 496 vs 3 632 sentences/s,
        # profiles/r2j_bench_c3_ab_residual_planes.txt): the kernels are the same, but residuals spread over many binades toggle
        # more bits in the tensor cores than table entries that share two exponents, and the step is power-capped -- the SM clock
        # drops from 1 631 to 1 603 MHz and the untouched gradient rows slow down with the message rows.
        # MLBP_MSG_RESIDUAL=0: plain T_hi operands (A/B runs).
        self.msg_residual = os.environ.get('MLBP_MSG_RESIDUAL', '1') != '0'
        self.tau = float(tau) if tau is not None else (4e-4 if one else 2e-4)
        self.tau_label = float(tau_label) if tau_label is not None else (2e-4 if one else 1e-4)
        self.peak_mult = float(peak_mult)
        self.msg_two_pass_ok = False
        self._flags = torch.zeros(FLAG_WORDS, dtype=torch.int32, device=self.device)
        self.theta_ee = None
        self.theta_ed = None
        self.planes = None
        self.colsums = torch.zeros((N_SUMS, self.V), dtype=torch.float64, device=self.device)
        self.const_rows = None      # factor->variable messages of a pairwise factor fed the uniform initial message
        self.map_const_rows = None  # the same for max-product messages (K10), built on first use after each set_theta
        self.map_const_ok = False
        self.edstats = torch.zeros((self.Vd, 3), dtype=torch.float64, device=self.device)
        self.with_grad_planes = False
        self._A = self._D = self._U = None
        self._blob_host = None
        self._blob_dev = None
        self._blob_event = None     # H2D copy of the previous plan blob (the pinned buffer is reused)
        self.launches = 0           # kernels launched by this engine (bench.py's gpu_launches)
        self.gemm_rows = 0          # GEMM rows executed (algorithmic GEMV count)
        self.gemm_launches = 0
        self.blob_bytes = 0         # schedule bytes uploaded (H2D) so far
        self.profile_gemm = False   # record a CUDA-event pair around every K4 launch (bench.py roofline)
        self.gemm_events = []
        self.profile_kernels = False  # same for the HBM-bound kernels: (name, event, event, algorithmic bytes)
        self.kernel_events = []
        self.event_tag = 0          # copied into every gemm_events record (bench.py: which step a launch belongs to)
        self._tbar = np.zeros(1, dtype=np.float32)
        self.tbar = 0.0
        self.r_plane0 = N_PLANES
        self.plan_seconds = 0.0     # host time spent in the schedule compiler (mlbp_plan_compile + export)
        self.plan_template_hits = self.plan_template_misses = 0   # graphs served from / added to the template cache (csrc/plan.cpp)
        self._pre = {}              # schedules being compiled ahead of their run() call: key -> (thread, result box)
        self.plan_prefetched = 0    # run() calls that found their schedule precompiled

    def _gemm_slice_rows(self, pairs):
        """Rows per K4 launch of the three-pass message GEMMs (0 = never slice).  The CTA pairs of one launch start in step and
        share A / B slabs in L2, but drift apart in K from wave to wave (ncu: 1.5x the wave-ideal DRAM bytes after 5 waves, 1.9x
        after 40) and the re-reads cost power under the cap; a kernel boundary re-aligns them.  Measured at 87 552 rows, V = 10 000
        (profiles/r1f_gemm_probe_split.txt): slices of 11-37 M-pairs are 4-6 % faster than one launch.  The slice is the pair count
        worth 8 to 24 waves of the resident pairs whose tiles fill whole waves best (V = 10 000 on 148 SMs: 37 pairs = exactly 20
        waves)."""
        if pairs is not None:
            return int(pairs) * 256
        if self.V <= 2048 or self.device.type != 'cuda':
            return 0
        resident = max(torch.cuda.get_device_properties(self.device).multi_processor_count // 2, 1)
        n_tiles = (self.V + 255) // 256
        waste = lambda p: -(-p * n_tiles // resident) * resident / float(p * n_tiles)
        lo, hi = max(-(-8 * resident // n_tiles), 1), max(24 * resident // n_tiles, 1)
        return 256 * min(range(lo, max(hi, lo) + 1), key=lambda p: (round(waste(p), 4), -p))

    def _timed(self, name, nbytes, fn):
        """launch through fn(); with profile_kernels the launch is bracketed by CUDA events on the launching stream and
        recorded with its ALGORITHMIC bytes (each input and output counted once; `nbytes` may be a callable)"""
        if not self.profile_kernels:
            return fn()
        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
        e0.record()
        fn()
        e1.record()
        self.kernel_events.append((name, e0, e1, float(nbytes() if callable(nbytes) else nbytes)))

    # ------------------------------------------------------------------ theta -> tables (K2)
    def set_theta(self, theta_ee, theta_ed, with_grad=True):
        te = np.ascontiguousarray(np.asarray(theta_ee, dtype=np.float64).reshape(3))
        td = np.ascontiguousarray(np.asarray(theta_ed, dtype=np.float64).reshape(6))
        self.theta_ee, self.theta_ed = te, td
        pmin, pmax, wmin, wmax = self.model.frange
        zmax = te[2] + max(te[0] * pmin, te[0] * pmax) + max(te[1] * wmin, te[1] * wmax, 0.0)
        fabs = max(1.0, abs(pmin), abs(pmax), abs(wmin), abs(wmax))
        self.scale_exp = 13 - int(math.ceil((zmax / math.log(2.0)) + math.log2(fabs)))
        # log2 range of the factor->variable messages: D[r, a] is a convex combination of T[a, .], so after the
        # power-of-two centring folded into the GEMM's alpha every element lies within 2^(+-half_range_log2)
        zmin = te[2] + min(te[0] * pmin, te[0] * pmax) + min(te[1] * wmin, te[1] * wmax, 0.0)
        self.centre_exp = int(round((zmin + zmax) / 2.0 / math.log(2.0)))
        self.half_range_log2 = (zmax - zmin) / 2.0 / math.log(2.0) + 0.5
        if zmax - zmin > 12.0:
            import warnings
            warnings.warn('pairwise potentials span e^%.1f: entries more than 2^18 below the largest lose relative '
                          'precision in the fp16 hi/lo operand planes (absolute error stays 2^-38 of the maximum)' % (zmax - zmin))
        erange, prange = self.model.ed_range
        # two-pass gradient rows (grad_a_terms == 1) only while the potentials are moderately peaked: the error of one
        # expectation is bounded by 2^-12 x the belief's mean absolute deviation of the feature, measured 2e-7 relative
        # on a sentence's gradient at log-ranges ~1.5 and 9e-6 at ~6.5; beyond e^3 the third pass is kept
        self.grad_hi_only_ok = (zmax - zmin) <= 3.0 and (abs(td[0]) * erange + abs(td[1]) * prange) <= 3.0
        # ... and ONE pass (plain fp16 x fp16, fp32 accumulate) when, in addition, the vocabulary is large: the fp16 rounding of
        # the table entries is random per entry and averages over the ~V^2 entries a belief spreads over (measured on a
        # sentence's gradient against the float64 oracle: <= 3.2e-6 relative over 24 sentences at V = 10 000, 3e-6 at V = 2 000)
        self.grad_one_pass_ok = self.grad_hi_only_ok and self.V >= self.one_pass_min_v
        self.msg_two_pass_ok = (zmax - zmin) <= 3.0 and (self.msg_passes in (1, 2) or (self.msg_passes is None and self.V >= 4096)) \
            and (self.gemm_impl & 0xff) != 1                      # the SIMT cross-check kernel has no device-side gate
        self.k.call('mlbp_zero_words', _p(self._flags), FLAG_WORDS)   # the peak flag is sticky per theta
        self.unary_range_log2 = (abs(td[0]) * erange + abs(td[1]) * prange + 4.0 * (abs(td[2]) + abs(td[3]) + abs(td[4]))) / math.log(2.0)
        n_planes = N_PLANES if with_grad else 8
        # + 4 residual planes R = T - tbar (hi halves only), the operand of the ONE-pass message rows (include/mlbp.h, K2)
        self.r_plane0 = n_planes
        if self.planes is None or self.planes.shape[0] < n_planes + 4:
            self.planes = torch.zeros((n_planes + 4, self.V, self.ld), dtype=torch.float16, device=self.device)
        self.with_grad_planes = with_grad
        m = self.model
        # tbar: 0 = the entry point's default, the table at phi = 0.  (The smallest possible entry, exp(zmin) -- every residual
        # non-negative -- was measured too: same accuracy, same speed: profiles/r2j_bench_c3_ab_residual_planes.txt.)
        self._tbar[0] = 0.0
        self._timed('K2 build_pairwise_tables', 2.0 * self.V * self.V * 4 + (n_planes + 4) * self.V * self.V * 2.0,
                    lambda: self.k.call('mlbp_build_pairwise_tables', _p(m.pmi), _p(m.w1), self.V, self.ld, _hp(te),
                                        self.scale_exp, _p(self.planes), self.V * self.ld, self.ld, _p(self.colsums),
                                        1 if with_grad else 0, _p(self.planes[self.r_plane0]), _hp(self._tbar)))
        self.tbar = float(self._tbar[0])                          # 2^scale_exp * exp(theta_bias): written by the entry point on the host
        self.k.call('mlbp_build_unary_tables', _p(m.edT), _p(m.pedT), self.V, self.Vd, self.ld, _hp(td), _p(self.edstats))
        self.launches += 2
        # D rows 0..4: the constant-one row and the constant messages by table id (T: row sums, Tt: column sums, T1, T1t),
        # mean-one scaled (messages are scale-free); copied into every micro-batch's D buffer (device-to-device memcpy)
        if self.const_rows is None:
            self.const_rows = torch.empty((D_CONST_ROWS, self.ld), dtype=torch.float32, device=self.device)
        self.k.call('mlbp_const_rows', _p(self.colsums), self.V, self.ld, _p(self.const_rows))
        self.launches += 1
        self.map_const_ok = False

    def maxprod_rows(self, A_hi, A_lo, a_rows_total, a_row0, n_rows, table, D, d_row0):
        """K10: max-product factor->variable messages of A rows [a_row0, a_row0 + n_rows) into D rows d_row0 .. under the current
        theta, row-normalised by each row's max and centred like the sum-product rows (mlbp_factor_to_var_maxprod)"""
        m = self.model
        self._timed('K10 maxprod', lambda: n_rows * self.V * 8.0 + (2 if table in (2, 3) else 1) * self.V * self.V * 4.0,
                    lambda: self.k.call('mlbp_factor_to_var_maxprod', _p(A_hi), _p(A_lo), int(a_rows_total), int(a_row0),
                                        int(n_rows), int(table), _p(m.pmi), _p(m.w1), self.V, self.ld, self.ld,
                                        _hp(self.theta_ee), self.centre_exp, _p(D), int(d_row0), int(D.shape[1])))
        self.launches += 1

    def _map_const(self):
        """D rows 0..4 of a max-product run: the constant-one row and, per message table, K10 of the uniform message -- the row
        (T, T1) or column (Tt, T1t) maxima of the centred table"""
        if self.map_const_ok:
            return self.map_const_rows
        if self.map_const_rows is None:
            self.map_const_rows = torch.zeros((D_CONST_ROWS, self.ld), dtype=torch.float32, device=self.device)
            self._map_uniform = torch.zeros((2, 1, self.ld), dtype=torch.float16, device=self.device)
            rows = torch.zeros(1, dtype=torch.int32, device=self.device)
            self.k.call('mlbp_fill_uniform_rows', _p(self._map_uniform[0]), _p(self._map_uniform[1]), self.ld, self.V, _p(rows), 1,
                        None)
            self.launches += 1
        self.map_const_rows[0].copy_(self.const_rows[0])
        for t in range(4):
            self.maxprod_rows(self._map_uniform[0], self._map_uniform[1], 1, 0, 1, t, self.map_const_rows, 1 + t)
        self.map_const_ok = True
        return self.map_const_rows

    def pass_stats(self):
        """Host copy of the device-side decisions since the last set_theta (one small D2H read): whether a peaked message
        switched the message GEMMs back to three passes, and what the exact re-score did."""
        f = self._flags.cpu().numpy()
        c = f[FLAG_COUNTERS:FLAG_COUNTERS + 5]
        return {'msg_two_pass': bool(self.msg_two_pass_ok),       # (name kept from the two-pass build: "reduced-pass message rows")
                'msg_passes': (1 if self.msg_one_pass else 2) if self.msg_two_pass_ok else 3, 'peak_flag': int(f[FLAG_PEAK]), 'spike_flag': int(f[FLAG_SPIKE]),
                'spiky_rows_last_batch': int(f[FLAG_NSPIKY]),
                'max_message_prob': float(f[FLAG_MAXBITS:FLAG_MAXBITS + 1].view(np.float32)[0]) * 2.0 ** -A_SCALE_LOG2, 'rescored': int(c[0]),
                'skipped_mass_tie': int(c[1]), 'skipped_degenerate': int(c[2]), 'top1_changed': int(c[3]),
                'rank_changed': int(c[4])}

    def plane(self, table, lo):
        return self.planes[2 * table + (1 if lo else 0)]

    def r_plane(self, table):
        """residual plane (T - tbar, hi half) of message table 0..3 (T, Tt, T1, T1t)"""
        assert 0 <= table < 4
        return self.planes[self.r_plane0 + table]

    # ------------------------------------------------------------------ API read-back helpers (LBP.py drop-in)
    def unary_message(self, factor_type, observed_dim, gap1=False, sparse=(), normalized=True):
        """Message / table column of ONE unary factor as float64 [V] (LBP.py:492-498, :702-703), computed by K1 on a
        pseudo-variable that owns only this factor."""
        en_de = factor_type == 'en_de'
        i32 = lambda x: np.asarray(x, dtype=np.int32)
        sp = list(sparse) if en_de else []
        c = Corpus(var_off=i32([0, 1]), var_de=i32([observed_dim if en_de else -1]), var_label=i32([0]), var_pos=i32([0]),
                   sp_off=i32([0, len(sp)]), sp_en=i32([x[0] for x in sp]), sp_feat=i32([x[1] for x in sp]),
                   sp_val=np.asarray([x[2] for x in sp], dtype=np.float32), giv_off=i32([0, 0 if en_de else 1]),
                   giv_label=i32([] if en_de else [observed_dim]), giv_gap1=i32([] if en_de else [1 if gap1 else 0]),
                   pair_off=i32([0, 0]), pair_v0=i32([]), pair_v1=i32([]), pair_gap1=i32([]))
        dev, ld, V, m = self.device, self.ld, self.V, self.model
        d = lambda name: _p(c.dev(name, dev))
        inv_sigma = torch.empty(1, dtype=torch.float64, device=dev)
        g_unary = torch.empty((1, 9), dtype=torch.float64, device=dev)
        U = torch.empty((1, ld), dtype=torch.float32, device=dev)
        self.k.call('mlbp_unary_stats', 1, d('var_de'), d('var_label'), d('sp_off'), d('sp_en'), d('sp_feat'), d('sp_val'),
                    d('giv_off'), d('giv_label'), d('giv_gap1'), _p(m.pmi), _p(m.w1), _p(m.edT), _p(m.pedT), V, ld,
                    _hp(self.theta_ed), _p(self.edstats), _p(self.colsums), _p(inv_sigma), _p(g_unary))
        self.k.call('mlbp_unary_products', 1, d('var_de'), d('sp_off'), d('sp_en'), d('sp_feat'), d('sp_val'), d('giv_off'),
                    d('giv_label'), d('giv_gap1'), _p(m.edT), _p(m.pedT), V, ld, _hp(self.theta_ed), _p(inv_sigma),
                    _p(self.planes), V * ld, ld, self.scale_exp, _p(self.colsums), _p(U))
        self.launches += 2
        u = U[0, :V].double() / V                                        # normalised message
        if not normalized:
            norm = (1.0 / inv_sigma[0]) if en_de else self.colsums[1 if gap1 else 0, observed_dim]
            u = u * norm
        return u.cpu().numpy()

    def dense_table(self, gap1):
        """pot_en_en (gap > 1) or pot_en_en_w1 (gap == 1) as float64 [V, V], from the operand planes (22 bits)"""
        t = 2 if gap1 else 0
        T = (self.plane(t, 0)[:, :self.V].double() + self.plane(t, 1)[:, :self.V].double()) * (2.0 ** -self.scale_exp)
        return T.cpu().numpy()

    # ------------------------------------------------------------------ workspace
    def rows_budget(self):
        """GEMM rows (A and D rows) that fit the workspace: 4 bytes (A hi+lo) + 4 bytes (D) per element"""
        return max(1024, self.workspace_bytes // (8 * self.ld))

    def _ensure(self, a_rows, d_rows, n_vars, blob_words):
        ld, dev = self.ld, self.device
        if self._A is None or self._A.shape[1] < a_rows:
            cap = max(a_rows, 0 if self._A is None else int(self._A.shape[1] * 1.25))
            self._A = None
            self._A = torch.empty((2, cap, ld), dtype=torch.float16, device=dev)
        d_rows = max(d_rows, D_CONST_ROWS)
        if self._D is None or self._D.shape[0] < d_rows:
            cap = max(d_rows, 0 if self._D is None else int(self._D.shape[0] * 1.25))
            self._D = None
            self._D = torch.empty((cap, ld), dtype=torch.float32, device=dev)
        if self._U is None or self._U.shape[0] < n_vars:
            self._U = torch.empty((max(n_vars, 0 if self._U is None else int(self._U.shape[0] * 1.25)), ld),
                                  dtype=torch.float32, device=dev)
        if self._blob_host is None or self._blob_host.numel() < blob_words:
            n = int(blob_words * 1.25) + 1024
            pin = self.device.type == 'cuda'
            self._blob_host = torch.empty(n, dtype=torch.int32, pin_memory=pin)
            self._blob_dev = torch.empty(n, dtype=torch.int32, device=dev)

    # ------------------------------------------------------------------ one microbatch
    @staticmethod
    def _compile_raw(corpus, roots, sweeps, flags):
        handle = ctypes.c_void_p()
        lib = _lib.load()
        _lib.check(lib.mlbp_plan_compile(corpus.n_sent, _hp(corpus.var_off), _hp(corpus.pair_off), _hp(corpus.pair_v0),
                                         _hp(corpus.pair_v1), _hp(corpus.pair_gap1), _hp(roots), sweeps, flags,
                                         ctypes.byref(handle)))
        sizes = np.zeros(16, dtype=np.int64)
        _lib.check(lib.mlbp_plan_sizes(handle, _hp(sizes)))
        return handle, sizes

    @staticmethod
    def _plan_key(corpus, roots, sweeps, flags):
        return (id(corpus), corpus.n_sent, int(corpus.var_off[-1]), int(corpus.pair_off[-1]), int(sweeps), int(flags), roots.tobytes())

    def _plan_flags(self, want_grad, want_marg, approx_inference=False, approx_beliefs=False, want_joint=False):
        """mlbp_plan_compile flags of a run() call under the CURRENT theta (the reduced-pass gates of set_theta decide reuse_z)"""
        approx = approx_inference or approx_beliefs
        grad_hi_only = self.grad_a_terms == 1 and self.grad_hi_only_ok and not approx
        two_pass = self.msg_two_pass_ok and not approx
        fold, reuse_z = not approx_inference, (not approx and not grad_hi_only and not two_pass)
        return (1 if (want_grad or want_joint) else 0) | (2 if want_marg else 0) | (0 if fold else 4) | (0 if reuse_z else 8) | \
            (16 if want_joint else 0)

    def compile(self, corpus, roots, sweeps, want_grad, want_marg, fold=True, reuse_z=True, want_joint=False):
        """want_joint: plan the gradient stage and the per-factor rows of mlbp_joint_logp (flag bit 4)"""
        roots = np.ascontiguousarray(roots, dtype=np.int32)
        assert roots.shape[0] == corpus.n_sent and roots.shape[1] >= 1 + sweeps, roots.shape
        roots = np.ascontiguousarray(roots[:, :1 + sweeps])
        flags = (1 if (want_grad or want_joint) else 0) | (2 if want_marg else 0) | (0 if fold else 4) | (0 if reuse_z else 8) | \
            (16 if want_joint else 0)
        pre = self._pre.pop(self._plan_key(corpus, roots, sweeps, flags), None) if self._pre else None
        if pre is not None:                                       # compiled ahead by precompile(): wait for it, take it
            pre[0].join()
            if 'error' in pre[1]:
                raise pre[1]['error']
            handle, sizes = pre[1]['plan']
            self.plan_prefetched += 1
        else:
            handle, sizes = self._compile_raw(corpus, roots, sweeps, flags)
        self.plan_template_hits += int(sizes[PLAN_TMPL_HITS])
        self.plan_template_misses += int(sizes[PLAN_TMPL_MISSES])
        return handle, sizes

    def precompile(self, corpus, roots, sweeps=3, want_grad=True, want_marg=True, approx_inference=False, approx_beliefs=False,
                   want_joint=False):
        """Start compiling the schedule of a LATER run(corpus, roots, ...) call in a background thread (mlbp_plan_compile keeps
        no Python state and ctypes releases the GIL): the roots of the next SGD step do not depend on theta, so the host can
        compile its first micro-batch while it waits for the GPU to finish the current step.  run() picks the plan up when it
        is called with the same Corpus object, roots and options; a plan nobody picks up (theta moved across a reduced-pass
        gate and changed the flags, say) is dropped by the next precompile() / drop_precompiled()."""
        import threading
        self.drop_precompiled()
        roots = np.ascontiguousarray(roots, dtype=np.int32)
        roots = np.ascontiguousarray(roots[:, :1 + sweeps])
        flags = self._plan_flags(want_grad, want_marg, approx_inference, approx_beliefs, want_joint)
        box = {}

        def work():
            try:
                box['plan'] = self._compile_raw(corpus, roots, sweeps, flags)
            except Exception as e:                                # re-raised by the run() that picks the plan up
                box['error'] = e

        t = threading.Thread(target=work, daemon=True)
        t.start()
        self._pre[self._plan_key(corpus, roots, sweeps, flags)] = (t, box)

    def drop_precompiled(self):
        for t, box in self._pre.values():
            t.join()
            if 'plan' in box:
                _lib.load().mlbp_plan_destroy(box['plan'][0])
        self._pre = {}

    def run(self, corpus, roots, sweeps=3, want_grad=True, want_marg=True, want_beliefs=False, want_messages=False,
            approx_inference=False, approx_beliefs=False, topk=100, reduce_into=None, want_topk=0, want_joint=False,
            max_product=False):
        """All sentences of `corpus` (must fit the workspace; use run_many to micro-batch).  `roots`: int
        [n_sent, 1 + sweeps] variable indices local to each sentence (draw 0 = has_loops, LBP.py:176).
        `reduce_into`: optional device tensor of 16 float64 that this call's sums are ADDED to (mlbp_batch_reduce: the
        vector trainer.Trainer all-reduces).
        `want_joint`: also Result.logp_joint, the joint log-likelihood of each sentence's labels (Bethe estimate, K9).  It
        needs the normaliser Z of every pairwise belief, so the gradient-stage rows run as with want_grad; `grad` is still
        only the unary part unless want_grad.  Needs want_marg and a set_theta(with_grad=True); not defined for the
        approximate modes (ValueError).
        `max_product`: max-product BP instead of sum-product (K10 replaces every pairwise message row, on the same plan).
        `top1` is then the decoded assignment -- the arg-max of each variable's max-marginal, first index on ties --, and
        `beliefs`, `logp_var`, `logp` and `rank` are K5's usual outputs computed on the normalised MAX-marginals.
        Result.map_score / label_score: the log-potential of the decoded assignment and of the labels (K11).  Inference only:
        ValueError with want_grad, want_joint, the approximate modes or without want_marg.  Synchronises the stream (K11
        checks the assignments on the host)."""
        assert self.theta_ee is not None, 'set_theta first'
        if max_product and (want_grad or want_joint or approx_inference or approx_beliefs or not want_marg):
            raise ValueError('max_product is inference only: it needs want_marg and does not combine with want_grad, want_joint '
                             'or the approximate modes (approx_inference / approx_beliefs)')
        if want_joint and (approx_inference or approx_beliefs):
            raise ValueError('the joint log-likelihood is not defined for the approximate modes (approx_inference / approx_beliefs)')
        if want_joint and not want_marg:
            raise ValueError('want_joint needs want_marg: the joint is built around the per-variable log-marginals')
        grad_stage = want_grad or want_joint
        assert not grad_stage or self.with_grad_planes
        if corpus.n_sent == 0:                                    # empty batch: nothing to launch
            dev = self.device
            z = lambda *shape, dt=torch.float64: torch.zeros(shape, dtype=dt, device=dev)
            return Result(z(0, 9), z(0), z(0), z(0, dt=torch.int32), z(0, dt=torch.int32),
                          z(0, self.ld, dt=torch.float32) if want_beliefs else None,
                          {'a_rows': 0, 'd_rows': 0, 'levels': 0, 'gemm_rows': 0, 'dead': 0, 'blob_words': 0},
                          {'v2f': [], 'f2v': []} if want_messages else None, logp_joint=z(0) if want_joint else None,
                          map_score=z(0) if max_product else None, label_score=z(0) if max_product else None)
        lib = _lib.load()
        # masked (top-K) message rows: the pairwise normaliser Z must come from its own GEMM row of the final messages
        approx = approx_inference or approx_beliefs
        grad_hi_only = self.grad_a_terms == 1 and self.grad_hi_only_ok and not approx
        # Z = c'Tr may reuse the D row of a message update only if that row was built from the same operand as the
        # numerator rows: not with masked (top-K) messages, not when the gradient rows drop the lo half of r, and not when
        # the message rows do (two-pass message rows)
        import time as _time
        t_plan = _time.perf_counter()
        two_pass = self.msg_two_pass_ok and not approx
        msg_one_pass = two_pass and self.msg_one_pass            # message rows as A_hi . B_hi (see __init__)
        handle, sizes = self.compile(corpus, roots, sweeps, want_grad, want_marg, fold=not approx_inference,
                                     reuse_z=not approx and not grad_hi_only and not two_pass, want_joint=want_joint)
        self.plan_seconds += _time.perf_counter() - t_plan
        try:
            words = int(sizes[PLAN_BLOB_WORDS])
            nv = corpus.n_vars
            if self._blob_event is not None:
                self._blob_event.synchronize()
            self._ensure(int(sizes[PLAN_A_ROWS]), int(sizes[PLAN_D_ROWS]), nv, words)
            t_plan = _time.perf_counter()
            _lib.check(lib.mlbp_plan_export(handle, ctypes.c_void_p(self._blob_host.data_ptr())))
            self.plan_seconds += _time.perf_counter() - t_plan   # (the wait for the previous blob's upload is not counted)
        finally:
            lib.mlbp_plan_destroy(handle)
        blob = self._blob_host.numpy()[:words]
        self._blob_dev[:words].copy_(self._blob_host[:words], non_blocking=True)
        self.blob_bytes += 4 * words
        if self.device.type == 'cuda':
            self._blob_event = torch.cuda.Event()
            self._blob_event.record()
        bd = self._blob_dev
        dev, ld, V, k, m = self.device, self.ld, self.V, self.k, self.model
        if max_product:
            # the spike scan and compensation, the device gates and the K5b re-score exist only to make reduced-pass GEMM rows safe
            two_pass = msg_one_pass = False
        A_hi, A_lo, D, U = self._A[0], self._A[1], self._D, self._U
        a_cap = int(self._A.shape[1])
        td = self.theta_ed
        c = lambda name: _p(corpus.dev(name, dev))
        # one-pass gradient rows (A_hi . B_hi) and two-pass message rows both rely on the spike lists of the var->factor kernel
        one_pass = grad_stage and grad_hi_only and self.grad_one_pass_ok and self.grad_a_terms == 1 and self.grad_b_terms == 1 \
            and (self.gemm_impl & 0xff) != 1
        track = two_pass or one_pass
        peak_flag = _p(self._flags, FLAG_PEAK) if track else None
        n_spk = max(int(sizes[PLAN_A_ROWS]), 1)
        spk_cnt = spk_ent = spk_rows = None
        if track:                                                 # spike bookkeeping of this batch's A rows
            spk_cnt = torch.empty(n_spk, dtype=torch.int32, device=dev)
            spk_ent = torch.empty((n_spk, SPIKE_SLOTS, 2), dtype=torch.int32, device=dev)
            spk_rows = torch.empty(n_spk, dtype=torch.int32, device=dev)
            n_blk = int(blob[H_SPK_BLK_N])
            blk_host = blob[int(blob[H_MSG_BLK_OFF]):int(blob[H_MSG_BLK_OFF]) + GEMM_WORDS * n_blk].reshape(-1, GEMM_WORDS)
            blk_of = dict((int(r[1]), i) for i, r in enumerate(blk_host))     # first A row of a block -> its index
            spk_blk = torch.empty(max(n_blk, 1), dtype=torch.int32, device=dev)
            k.call('mlbp_zero_words', _p(spk_blk), max(n_blk, 1))
            k.call('mlbp_zero_words', _p(self._flags, FLAG_NSPIKY), 1)

        D[:D_CONST_ROWS].copy_(self._map_const() if max_product else self.const_rows)   # row 0: the constant-one row
        inv_sigma = torch.empty(max(nv, 1), dtype=torch.float64, device=dev)
        g_unary = torch.empty((max(nv, 1), 9), dtype=torch.float64, device=dev)
        k.call('mlbp_unary_stats', nv, c('var_de'), c('var_label'), c('sp_off'), c('sp_en'), c('sp_feat'), c('sp_val'),
               c('giv_off'), c('giv_label'), c('giv_gap1'), _p(m.pmi), _p(m.w1), _p(m.edT), _p(m.pedT), V, ld, _hp(td),
               _p(self.edstats), _p(self.colsums), _p(inv_sigma), _p(g_unary))
        self._timed('K1 unary_products', lambda: (3.0 * nv + len(corpus.giv_label)) * V * 4,
                    lambda: k.call('mlbp_unary_products', nv, c('var_de'), c('sp_off'), c('sp_en'), c('sp_feat'),
                                   c('sp_val'), c('giv_off'), c('giv_label'), c('giv_gap1'), _p(m.edT), _p(m.pedT), V, ld,
                                   _hp(td), _p(inv_sigma), _p(self.planes), V * ld, ld, self.scale_exp,
                                   _p(self.colsums), _p(U)))
        self.launches += 2
        if blob[H_INIT_N]:
            keep = None
            if (approx_inference or approx_beliefs) and topk < V:
                # The reference takes the top-K of the still-uniform initial message too; which K of the V equal entries
                # survive is decided by NumPy's argpartition (pyx:198, :203).  Ask the same NumPy (indices only, no arithmetic).
                km = np.zeros(V, dtype=np.uint8)
                km[np.argpartition(-np.full(V, 1.0 / V), topk - 1)[:topk]] = 1
                keep = torch.from_numpy(km).to(dev)
            k.call('mlbp_fill_uniform_rows', _p(A_hi), _p(A_lo), ld, V, _p(bd, int(blob[H_INIT_OFF])), int(blob[H_INIT_N]),
                   _p(keep))
            self.launches += 1
        max_in = int(blob[H_MAX_IN])
        alpha = float(2.0 ** (-(A_SCALE_LOG2 + self.scale_exp + self.centre_exp)))
        # one-pass message rows contract with the residual planes; every message row sums to 2^14, so the dropped constant is
        # the same for every element of the product (K4's add_const)
        msg_residual = msg_one_pass and self.msg_residual and len(self.gemm_k_ranges) == 1
        msg_const = float(alpha * (2.0 ** A_SCALE_LOG2) * self.tbar)
        g_max = int(np.diff(corpus.giv_off).max()) if corpus.n_vars else 0
        range_log2 = float((max_in + 2 * g_max) * self.half_range_log2 + self.unary_range_log2)

        def spike_scan(a0, rows, listed=True):
            """file the spikes of A rows [a0, a0 + rows) -- one GEMM block -- before its GEMM (mlbp_spike_scan)"""
            self._timed('K4a spike_scan', rows * V * 2.0,
                        lambda: k.call('mlbp_spike_scan', _p(A_hi), _p(A_lo), ld, V, a0, rows, self.peak_mult / V, peak_flag, _p(spk_cnt),
                                       _p(spk_ent), _p(spk_rows, a0) if listed else None, _p(spk_blk, blk_of[a0]) if listed else None))
            self.launches += 1

        def spike_correct(t, a0, d0, rows, block_a0, one_pass_rows=False):
            """restore what the dropped lo half of A contributed at the spikes of rows [a0, a0 + rows) (block starting at block_a0);
            one_pass_rows: the block also dropped the lo half of the table, restored at the spikes as well"""
            b = blk_of[block_a0]
            tt = TRANSPOSED_TABLE[t]
            self._timed('K4b spike_correct', 0.0,                # bytes depend on the data (spikes found on the device)
                        lambda: k.call('mlbp_spike_correct', peak_flag, _p(spk_cnt), _p(spk_ent), _p(spk_rows, block_a0), _p(spk_blk, b),
                                       a0, rows, _p(self.plane(tt, 0)), _p(self.plane(tt, 1)), V, ld, _p(D), d0, ld, alpha,
                                       _p(A_hi) if one_pass_rows else None,
                                       _p(self.r_plane(tt)) if (one_pass_rows and msg_residual and t < 4) else None, self.tbar))
            self.launches += 1

        def gemm_calls(off, n, mask, impl_flags=0, gated=False, role='message', residual=False):
            masked = set()
            for i in range(n):
                t, a0, d0, rows = (int(x) for x in blob[off + GEMM_WORDS * i: off + GEMM_WORDS * (i + 1)])
                if mask and (a0, rows) not in masked:             # reference's top-K approximations (pyx:193-205)
                    k.call('mlbp_topk_mask_rows', _p(A_hi), _p(A_lo), ld, V, a0, rows, topk)
                    masked.add((a0, rows))
                    self.launches += 1
                passes = 3 - (1 if impl_flags & GEMM_A_HI_ONLY else 0) - (1 if impl_flags & GEMM_B_HI_ONLY else 0)
                # one-pass rows are L2-bandwidth-bound, not power-bound: slicing does not help them (measured)
                step = self.gemm_slice_rows if (self.gemm_slice_rows and passes > 1) else rows
                for r0 in range(0, rows, max(step, 1)):
                    n = min(step, rows - r0)
                    if self.profile_gemm:
                        e0, e1 = torch.cuda.Event(enable_timing=True), torch.cuda.Event(enable_timing=True)
                        e0.record()
                    if gated:
                        # decided on the device: the reduced-pass variant while the gate word is clear, else the fallback
                        gate, fallback = gated if isinstance(gated, tuple) else (peak_flag, 0)
                        for k0, k_len in self.gemm_k_ranges:
                            for fl, run_if_set in ((impl_flags, 0), (fallback, 1)):
                                # residual: the reduced (one-pass) variant contracts with R = T - tbar and adds the constant
                                res = residual and run_if_set == 0
                                k.call('mlbp_factor_to_var_gemm_gated', _p(A_hi), _p(A_lo), a_cap, a0 + r0, n,
                                       _p(self.r_plane(t) if res else self.plane(t, 0)), _p(self.plane(t, 1)), V, ld, _p(D), d0 + r0, ld,
                                       alpha, self.gemm_impl | fl, gate, run_if_set, k0, k_len, msg_const if res else 0.0)
                            self.launches += 2
                        self.launches -= 1
                    elif len(self.gemm_k_ranges) > 1:
                        for k0, k_len in self.gemm_k_ranges:
                            k.call('mlbp_factor_to_var_gemm_gated', _p(A_hi), _p(A_lo), a_cap, a0 + r0, n, _p(self.plane(t, 0)),
                                   _p(self.plane(t, 1)), V, ld, _p(D), d0 + r0, ld, alpha, self.gemm_impl | impl_flags, None, 0, k0, k_len, 0.0)
                            self.launches += 1
                        self.launches -= 1
                    else:
                        k.call('mlbp_factor_to_var_gemm', _p(A_hi), _p(A_lo), a_cap, a0 + r0, n, _p(self.plane(t, 0)),
                               _p(self.plane(t, 1)), V, ld, _p(D), d0 + r0, ld, alpha, self.gemm_impl | impl_flags)
                    if self.profile_gemm:
                        e1.record()
                        self.gemm_events.append((e0, e1, n, passes, (2 if isinstance(gated, tuple) else 1) if gated else 0, self.event_tag, role))
                    self.launches += 1
                    self.gemm_launches += 1
                self.gemm_rows += rows

        for L in range(int(blob[H_NLEVELS])):
            rec = blob[H_WORDS + LEV_WORDS * L: H_WORDS + LEV_WORDS * (L + 1)]
            if rec[0]:
                def k3_bytes(rec=rec):
                    ng = int(rec[0])
                    n_in = int(blob[int(rec[2]) + ng])
                    present = int((blob[int(rec[3]):int(rec[3]) + n_in] >= 0).sum())
                    n_dest = int(blob[int(rec[4]) + n_in])
                    return (ng + present + n_dest) * V * 4.0           # U row + D rows read (fp32), A hi+lo rows written
                self._timed('K3 var_to_factor', k3_bytes,
                            lambda: k.call('mlbp_var_to_factor', int(rec[0]), _p(bd, int(rec[1])), _p(bd, int(rec[2])),
                                           _p(bd, int(rec[3])), _p(bd, int(rec[4])), _p(bd, int(rec[5])), _p(bd, int(rec[8])), _p(bd, int(rec[9])),
                                           _p(U), _p(D), ld,
                                           V, _p(A_hi), _p(A_lo), max_in, range_log2))
                self.launches += 1
            if track:                                             # spikes of this level's GEMM blocks, before their GEMMs
                for i in range(int(rec[6])):
                    t, a0, d0, rows = (int(x) for x in blob[int(rec[7]) + GEMM_WORDS * i: int(rec[7]) + GEMM_WORDS * (i + 1)])
                    if two_pass:
                        spike_scan(a0, rows)
            if max_product:
                for i in range(int(rec[6])):
                    t, a0, d0, rows = (int(x) for x in blob[int(rec[7]) + GEMM_WORDS * i: int(rec[7]) + GEMM_WORDS * (i + 1)])
                    self.maxprod_rows(A_hi, A_lo, a_cap, a0, rows, t, D, d0)
                    self.gemm_rows += rows
            elif two_pass:
                gemm_calls(int(rec[7]), int(rec[6]), False, GEMM_A_HI_ONLY | (GEMM_B_HI_ONLY if msg_one_pass else 0), gated=True,
                           residual=msg_residual)
                for i in range(int(rec[6])):                      # restore what the dropped lo half of the spikes contributed
                    t, a0, d0, rows = (int(x) for x in blob[int(rec[7]) + GEMM_WORDS * i: int(rec[7]) + GEMM_WORDS * (i + 1)])
                    spike_correct(t, a0, d0, rows, a0, msg_one_pass)
            else:
                gemm_calls(int(rec[7]), int(rec[6]), approx_inference)

        n_pair = int(blob[H_NPAIR])
        pair_stats = torch.empty((max(n_pair, 1), 3), dtype=torch.float64, device=dev)   # every entry is written by K6a
        v2f_rows = None
        if want_messages and n_pair:                              # before any gradient-stage masking
            oc, orr = int(blob[H_PAIR_C]), int(blob[H_PAIR_R])
            rows = torch.cat([bd[oc:oc + n_pair], bd[orr:orr + n_pair]]).long()
            v2f_rows = (A_hi[rows, :V].double() + A_lo[rows, :V].double()) * (2.0 ** -A_SCALE_LOG2)
        if grad_stage and n_pair:
            if one_pass and not want_grad:
                # rows run for the joint alone: their spike words go to a copy, so that a gradient-stage row with more spikes
                # than slots does not switch the later message rows of this theta to three passes (beliefs stay as without it)
                joint_words = self._flags[:FLAG_COUNTERS].clone()
                peak_flag = _p(joint_words)
            if one_pass:
                # spikes of the gradient stage's r rows (two ranges, listed for the AXPY below) and c rows (cells only)
                for i in range(int(blob[H_MSG_BLK_N]), int(blob[H_SPK_BLK_N])):
                    spike_scan(int(blk_host[i][1]), int(blk_host[i][3]))
                spike_scan(int(blob[int(blob[H_PAIR_C])]), n_pair, listed=False)
                # one pass (r_hi . B_hi); the cells where BOTH messages of a factor have a spike -- the only ones whose fp16
                # table rounding does not average away -- are restored in mlbp_pair_expectations from the spike lists.  A row
                # with more spikes than slots (PEAK word, device gate) switches these rows to two passes instead.
                gemm_calls(int(blob[H_GRAD_GEMM_OFF]), int(blob[H_NGRAD_GEMM]), False, GEMM_A_HI_ONLY | GEMM_B_HI_ONLY,
                           gated=(peak_flag, GEMM_A_HI_ONLY), role='gradient')
                # ... and the lo part of r at its spikes (the rows drop A_lo): without it the rounding of a spike that Z contains
                # but the numerator does not (a zero of a sparse feature plane under the spike) shows up undamped in N / Z
                go = int(blob[H_GRAD_GEMM_OFF])
                for i in range(int(blob[H_NGRAD_GEMM])):
                    t, a0, d0, rows = (int(x) for x in blob[go + GEMM_WORDS * i: go + GEMM_WORDS * (i + 1)])
                    spike_correct(t, a0, d0, rows, a0)
            else:
                gemm_calls(int(blob[H_GRAD_GEMM_OFF]), int(blob[H_NGRAD_GEMM]), approx_beliefs,
                           (GEMM_A_HI_ONLY | (GEMM_B_HI_ONLY if one_pass else 0)) if grad_hi_only else 0, role='gradient')
            if approx_beliefs:                                    # the c rows follow the r rows in the A buffer
                c0 = int(blob[int(blob[H_PAIR_C])])
                k.call('mlbp_topk_mask_rows', _p(A_hi), _p(A_lo), ld, V, c0, n_pair, topk)
                self.launches += 1
            def k6_bytes():
                o = lambda h: blob[int(blob[h]):int(blob[h]) + n_pair]
                rows = 3 * n_pair + int((o(H_PAIR_U2) >= 0).sum()) + int((o(H_PAIR_Z) != o(H_PAIR_C)).sum())
                return rows * V * 4.0                                  # c (hi+lo), u0, u1 [, u2] [, z] rows read
            self._timed('K6a pair_expectations', k6_bytes,
                        lambda: k.call('mlbp_pair_expectations', n_pair, _p(bd, int(blob[H_PAIR_C])),
                                       _p(bd, int(blob[H_PAIR_Z])), _p(bd, int(blob[H_PAIR_U0])),
                                       _p(bd, int(blob[H_PAIR_U1])), _p(bd, int(blob[H_PAIR_U2])), _p(A_hi), _p(A_lo),
                                       _p(D), ld, V, _p(pair_stats), _p(bd, int(blob[H_PAIR_R])), _p(bd, int(blob[H_PAIR_GAP1])),
                                       peak_flag if one_pass else None, _p(spk_cnt), _p(spk_ent),
                                       _p(self.planes), V * ld, alpha))
            self.launches += 1
        logp_var = top1 = rank = beliefs = None
        if want_marg:
            n_m = int(blob[H_MARG_N])
            logp_var = torch.empty(n_m, dtype=torch.float64, device=dev)
            top1 = torch.empty(n_m, dtype=torch.int32, device=dev)
            rank = torch.empty(n_m, dtype=torch.int32, device=dev)
            beliefs = torch.empty((n_m, ld), dtype=torch.float32, device=dev) if (want_beliefs or want_topk) else None
            def k5_bytes():
                mo, mi = int(blob[H_MARG_OFF]), int(blob[H_MARG_IN])
                n_in = int(blob[mo + n_m])
                return (n_m + int((blob[mi:mi + n_in] >= 0).sum()) + (n_m if want_beliefs else 0)) * V * 4.0
            aux = cnts = vflags = flagged = None
            if two_pass:                                          # near-tie detection + exact re-score (csrc/rescore.cu)
                aux = torch.empty((n_m, 2), dtype=torch.float64, device=dev)
                cnts = torch.empty((n_m, 2), dtype=torch.int32, device=dev)
                vflags = torch.empty(n_m, dtype=torch.int32, device=dev)
                flagged = torch.empty(n_m, dtype=torch.int32, device=dev)
                k.call('mlbp_zero_words', _p(self._flags, FLAG_NFLAGGED), 1)
            self._timed('K5 marginals', k5_bytes,
                        lambda: k.call('mlbp_marginals', n_m, _p(bd, int(blob[H_MARG_U])), _p(bd, int(blob[H_MARG_OFF])),
                                       _p(bd, int(blob[H_MARG_IN])), c('var_label'), _p(U), _p(D), ld, V, _p(logp_var),
                                       _p(top1), _p(rank), _p(beliefs), range_log2 + self.half_range_log2, max_in,
                                       self.tau, self.tau_label, _p(aux), _p(cnts), _p(vflags), _p(flagged),
                                       _p(self._flags, FLAG_NFLAGGED) if two_pass else None))
            self.launches += 1
            if two_pass:
                self._timed('K5b rescore', 0.0,                   # bytes depend on the data (variables flagged on the device)
                            lambda: k.call('mlbp_rescore_candidates', n_m, _p(flagged), _p(self._flags, FLAG_NFLAGGED), _p(vflags),
                                           _p(bd, int(blob[H_MARG_U])), _p(bd, int(blob[H_MARG_OFF])), _p(bd, int(blob[H_MARG_IN])),
                                           c('var_label'), _p(U), _p(D), ld, V, _p(A_hi), _p(A_lo), _p(self.planes), V * ld,
                                           _p(bd, int(blob[H_MSG_BLK_OFF])), int(blob[H_MSG_BLK_N]), int(blob[H_MSG_ROWS]),
                                           _p(aux), _p(cnts), self.tau, self.tau_label, range_log2 + self.half_range_log2,
                                           _p(top1), _p(rank), _p(self._flags, FLAG_COUNTERS)))
                self.launches += 2
        logp_joint = None
        if want_joint:                                            # K9: the Bethe estimate of the joint at the final messages
            logp_joint = torch.empty(corpus.n_sent, dtype=torch.float64, device=dev)
            pair_term = torch.empty(max(n_pair, 1), dtype=torch.float64, device=dev)
            oc, orr, om0, om1 = (int(blob[h]) for h in (H_PAIR_C, H_PAIR_R, H_PAIR_M0, H_PAIR_M1))
            self._timed('K9 joint_logp', 16.0 * n_pair * V,     # c and r rows (hi + lo fp16), the two mu rows (fp32)
                        lambda: k.call('mlbp_joint_logp', corpus.n_sent, n_pair, c('var_off'), c('pair_off'), _p(logp_var),
                                       _p(bd, oc), _p(bd, orr), _p(bd, om0), _p(bd, om1), _p(bd, int(blob[H_PAIR_V0])),
                                       _p(bd, int(blob[H_PAIR_V1])), c('var_label'), _p(bd, int(blob[H_PAIR_GAP1])),
                                       _p(pair_stats), _p(A_hi), _p(A_lo), _p(D), ld, V, _p(m.pmi), _p(m.w1), ld,
                                       _hp(self.theta_ee), -(A_SCALE_LOG2 + self.centre_exp), _p(pair_term), _p(logp_joint)))
            self.launches += 1
        map_score = label_score = None
        if max_product:                                           # K11 on the decoded assignment and on the labels
            map_score = torch.empty(corpus.n_sent, dtype=torch.float64, device=dev)
            label_score = torch.empty(corpus.n_sent, dtype=torch.float64, device=dev)
            for x, out in ((_p(top1), map_score), (c('var_label'), label_score)):
                self._timed('K11 assignment_score', 4.0 * (nv + len(corpus.giv_label) + 2 * corpus.n_pairs),
                            lambda x=x, out=out: k.call('mlbp_assignment_score', corpus.n_sent, nv, len(corpus.giv_label),
                                                        c('var_off'), x, c('var_de'), c('sp_off'), c('sp_en'), c('sp_feat'),
                                                        c('sp_val'), c('giv_off'), c('giv_label'), c('giv_gap1'), c('pair_off'),
                                                        c('pair_v0'), c('pair_v1'), c('pair_gap1'), _p(m.pmi), _p(m.w1),
                                                        _p(m.edT), _p(m.pedT), V, ld, _hp(self.theta_ee), _hp(td), _p(out)))
                self.launches += 1
        top_words = None
        if want_marg and want_topk:                               # after the re-score: K5b only moves top1 / rank, not beliefs
            top_words = self.topk_rows(beliefs, min(int(want_topk), V))
        grad = torch.empty((corpus.n_sent, 9), dtype=torch.float64, device=dev)
        logp = torch.empty(corpus.n_sent, dtype=torch.float64, device=dev)
        # per-sentence segmented sums (deterministic, no atomics); without the gradient stage only log-posteriors matter
        use_pairs = want_grad and n_pair > 0
        k.call('mlbp_gradient_reduce', corpus.n_sent, c('var_off'), c('pair_off') if use_pairs else None,
               _p(g_unary), _p(pair_stats), _p(bd, int(blob[H_PAIR_V0])) if use_pairs else None,
               _p(bd, int(blob[H_PAIR_V1])) if use_pairs else None, c('var_label'),
               _p(bd, int(blob[H_PAIR_GAP1])) if use_pairs else None,
               _p(m.pmi), _p(m.w1), ld, _p(logp_var), _p(grad), _p(logp))
        self.launches += 1
        if reduce_into is not None:                                # batch level: this micro-batch into the all-reduce buffer
            k.call('mlbp_batch_reduce', corpus.n_sent, _p(grad), _p(logp), int(blob[H_MARG_N]) if want_marg else 0, _p(rank),
                   _p(self._flags, FLAG_PEAK), _p(reduce_into))
            self.launches += 1
        messages = None
        if want_messages:
            # final pairwise messages, normalised, float64 on the host (API read-back for LBP.FactorGraph.messages):
            #   'v2f'[p] = (message of the dim-0 variable, message of the dim-1 variable) into pairwise factor p
            #   'f2v'[v] = factor->variable messages of variable v in facset (attach) order; None = still uniform
            assert want_grad and want_marg
            messages = {'v2f': [], 'f2v': []}
            if n_pair:
                m = v2f_rows.cpu().numpy()
                messages['v2f'] = [(m[i], m[n_pair + i]) for i in range(n_pair)]
            mo, mi = int(blob[H_MARG_OFF]), int(blob[H_MARG_IN])
            n_m = int(blob[H_MARG_N])
            off = blob[mo:mo + n_m + 1]
            rows = blob[mi:mi + int(off[-1])]
            if len(rows):
                dr = D[torch.from_numpy(np.maximum(rows, 0).astype(np.int64)).to(dev), :V].double()
                dr = (dr / dr.sum(dim=1, keepdim=True)).cpu().numpy()
            for v in range(n_m):
                messages['f2v'].append([dr[j] if rows[j] >= 0 else None for j in range(int(off[v]), int(off[v + 1]))])
        stats = {'a_rows': int(sizes[PLAN_A_ROWS]), 'd_rows': int(sizes[PLAN_D_ROWS]), 'levels': int(sizes[PLAN_N_LEVELS]),
                 'gemm_rows': int(sizes[PLAN_N_GEMM_ROWS]), 'dead': int(sizes[PLAN_N_DEAD]), 'blob_words': words,
                 'msg_two_pass': bool(two_pass), 'msg_passes': 1 if msg_one_pass else (2 if two_pass else 3)}
        return Result(grad, logp, logp_var, top1, rank, beliefs, stats, messages, top_words, logp_joint, map_score, label_score)

    def topk_rows(self, X, K):
        """the K largest entries of every row of the fp32 device matrix X[:, :V], best first: (idx, value, n_ties) device
        tensors (mlbp_topk_rows; get_max_vocab, LBP.py:402-411).  n_ties[r] > 0: the order of row r is not decided by the
        values alone (exact ties) -- NumPy's order for those is an implementation detail of its introselect."""
        n = int(X.shape[0])
        idx = torch.empty((n, K), dtype=torch.int32, device=self.device)
        val = torch.empty((n, K), dtype=torch.float32, device=self.device)
        ties = torch.empty(n, dtype=torch.int32, device=self.device)
        self._timed('K5c topk_rows', n * self.V * 4.0,
                    lambda: self.k.call('mlbp_topk_rows', _p(X), int(X.stride(0)), self.V, n, int(K), _p(idx), _p(val), _p(ties)))
        self.launches += 1
        return idx, val, ties

    def format_log_rows(self, X):
        """The .dist numbers of every row of the fp32 device matrix X[:, :V] as text, made on the device (mlbp_format_log_rows;
        FactorGraph.to_dist, LBP.py:125-143): (text uint8, offsets int64 [n + 1]) device tensors, row r is
        text[offsets[r]:offsets[r + 1]] = ' '.join('%0.6f' % x for x in np.log(row.astype(np.float64)))."""
        n = int(X.shape[0])
        text = torch.empty(max(FMT_MAX_BYTES * self.V * n, 1), dtype=torch.uint8, device=self.device)
        offsets = torch.empty(n + 1, dtype=torch.int64, device=self.device)
        self._timed('K7 format_log_rows', n * self.V * 4.0,
                    lambda: self.k.call('mlbp_format_log_rows', _p(X), int(X.stride(0)), self.V, n, _p(text), int(text.numel()),
                                        _p(offsets)))
        self.launches += 1
        return text, offsets

    # ------------------------------------------------------------------ micro-batching
    def microbatches(self, corpus, sweeps, want_grad):
        """split [0, n_sent) so that each piece's GEMM rows fit the workspace"""
        rows = corpus.gemm_rows_estimate(sweeps, want_grad) + 2 * np.diff(corpus.pair_off) + 8
        budget = self.rows_budget()
        out, lo, acc = [], 0, 0
        for s in range(corpus.n_sent):
            if acc + rows[s] > budget and s > lo:
                out.append((lo, s))
                lo, acc = s, 0
            acc += int(rows[s])
        out.append((lo, corpus.n_sent))
        return out

    def prepare(self, corpus, sweeps=3, want_grad=True):
        """Micro-batch slices of `corpus` with their index arrays already resident on the device (want_grad: sized for the
        gradient-stage rows, which run_prepared(want_joint=True) runs too)."""
        parts = []
        for lo, hi in self.microbatches(corpus, sweeps, want_grad):
            c = corpus.slice(lo, hi) if (lo, hi) != (0, corpus.n_sent) else corpus
            for name in Corpus.FIELDS:
                if name != 'var_pos':
                    c.dev(name, self.device)
            parts.append((lo, hi, c))
        return parts

    def run_prepared(self, parts, roots, sweeps=3, want_grad=True, want_marg=True, reduce_into=None, collect=True,
                     want_joint=False, **kw):
        """`collect` = False (with reduce_into): only the batch-level sums are wanted, nothing is concatenated.
        want_joint: a fifth result, logp_joint [B] (see run)"""
        roots = np.ascontiguousarray(roots, dtype=np.int32)
        grads, logps, top1s, ranks, joints = [], [], [], [], []
        for lo, hi, c in parts:
            r = self.run(c, roots[lo:hi], sweeps, want_grad, want_marg, reduce_into=reduce_into, want_joint=want_joint, **kw)
            if not collect:
                continue
            grads.append(r.grad); logps.append(r.logp); joints.append(r.logp_joint)
            if want_marg:
                top1s.append(r.top1); ranks.append(r.rank)
        return self._collected(collect, want_joint, grads, logps, top1s, ranks, joints)

    @staticmethod
    def _collected(collect, want_joint, grads, logps, top1s, ranks, joints):
        out = (None, None, None, None)
        if collect:
            cat = lambda xs: xs[0] if len(xs) == 1 else torch.cat(xs)
            out = (cat(grads), cat(logps), (cat(top1s) if top1s else None), (cat(ranks) if ranks else None))
        return out + ((cat(joints) if collect else None),) if want_joint else out

    def run_many(self, corpus, roots, sweeps=3, want_grad=True, want_marg=True, reduce_into=None, collect=True,
                 want_joint=False, **kw):
        """Micro-batched run over a large corpus; returns (grad [B, 9], logp [B], top1 [NV], rank [NV]) on device, and
        logp_joint [B] as a fifth entry with want_joint (see run).
        Launches are asynchronous: the host compiles the next micro-batch's schedule while the GPU works."""
        roots = np.ascontiguousarray(roots, dtype=np.int32)
        grads, logps, top1s, ranks, joints = [], [], [], [], []
        for lo, hi in self.microbatches(corpus, sweeps, want_grad or want_joint):
            r = self.run(corpus.slice(lo, hi) if (lo, hi) != (0, corpus.n_sent) else corpus, roots[lo:hi], sweeps,
                         want_grad, want_marg, reduce_into=reduce_into, want_joint=want_joint, **kw)
            if not collect:
                continue
            grads.append(r.grad); logps.append(r.logp); joints.append(r.logp_joint)
            if want_marg:
                top1s.append(r.top1); ranks.append(r.rank)
        return self._collected(collect, want_joint, grads, logps, top1s, ranks, joints)
