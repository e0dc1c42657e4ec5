"""Seeded prediction runs in the command line's file formats (vocabularies, feature matrices, TrainingInstance lines, a
parameter file with per-user thetas), shared by the prediction tests, and the reference's host formatting of .dist numbers."""
import codecs
import json

import numpy as np

from macaronicusermodeling_b200 import synth
from macaronicusermodeling_b200.train_compat import F_EN_DE_NAMES, F_EN_EN_NAMES, save_params

THETA_EE = [0.4, -0.3, 0.1]
THETA_ED = [0.8, -0.5, 0.6, 0.4, 0.3, -0.2]


def dist_numbers(row):
    """FactorGraph.to_dist's numbers (LBP.py:125-143) as the host wrote them before the device formatter"""
    with np.errstate(divide='ignore', invalid='ignore'):
        return ' '.join('%0.6f' % x for x in np.log(np.asarray(row, dtype=np.float32).astype(np.float64))).encode()


def write_case(tmp, model, n_sent, seed, users=('ua', 'ub', 'uc')):
    """n_sent sentences with history features, users assigned round-robin; returns the argv of a prediction run (without
    --save_predictions).  Add --user_adapt for the per-user thetas of the parameter file."""
    V, Vd = model['V'], model['Vd']
    rng = np.random.default_rng(seed)
    p = {}
    for name, words in (('en', [synth.en_word(i) for i in range(V)]), ('de', [synth.de_word(i) for i in range(Vd)])):
        p[name] = str(tmp / (name + '.vocab'))
        with codecs.open(p[name], 'w', 'utf8') as f:
            f.write('\n'.join(words) + '\n')
    for k in ('pmi', 'pmi_w1', 'ed', 'ped'):
        p[k] = str(tmp / (k + '.mat'))
        np.savetxt(p[k], model[k], fmt='%.9g')
    ti = str(tmp / 'test.json')
    with codecs.open(ti, 'w', 'utf8') as f:
        for i in range(n_sent):
            layout = ''.join(rng.choice(['p', 'p', 'g', 'r'], size=int(rng.integers(2, 8)))) + 'p'
            f.write(json.dumps(synth.make_sentence(model, layout, seed=seed * 1000 + i, n_history=3, sent_id=i,
                                                   user_id=users[i % len(users)])) + '\n')
    with codecs.open(ti + '.users', 'w', 'utf8') as f:
        f.write('\n'.join(users) + '\n')
    d2t = {}
    for j, u in enumerate(users):
        d2t['en_en', u] = np.array([THETA_EE]) * (1.0 + 0.2 * j)
        d2t['en_de', u] = np.array([THETA_ED]) * (1.0 - 0.1 * j)
    params = str(tmp / 'model.params')
    with codecs.open(params, 'w', 'utf8') as w:
        save_params(w, np.array([THETA_EE]), np.array([THETA_ED]), list(F_EN_EN_NAMES), list(F_EN_DE_NAMES), d2t)
    return ['--ti', ti, '--end', p['en'], '--ded', p['de'], '--phi_pmi', p['pmi'], '--phi_pmi_w1', p['pmi_w1'],
            '--phi_ed', p['ed'], '--phi_ped', p['ped'], '--history', '--session_history', '--load_params', params]
