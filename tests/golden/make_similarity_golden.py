"""Generates tests/golden/similarity_ref.npz:

    python tests/golden/make_similarity_golden.py

The nearest issue chosen by the reference notebook's own one-shot labeler (Kubeflow-FewShotLearning.ipynb cell 46,
oneshotlabeler.query) for golden encoder outputs (the encoder fixtures written by make_golden.py).  Only data is
stored: the row numbers and their f32 cosines.
"""
import os

import numpy as np
import torch

HERE = os.path.dirname(os.path.abspath(__file__))


SIMILARITY_INDEX = 'encoder_r4_b256_t512.npz'
SIMILARITY_QUERIES = ('encoder_r4_varlen.npz', 'encoder_r4_t1024.npz')
NOTEBOOK = '/root/reference/Issue_Embeddings/notebooks/scratch/Kubeflow-FewShotLearning.ipynb'


def similarity_fixture():
    """The nearest issue chosen by the reference notebook's OWN one-shot labeler (oneshotlabeler.query, cell 46 of
    Kubeflow-FewShotLearning.ipynb, source read from the notebook now) with golden encoder outputs as `vecs`: the cell
    scores with the global `cs = CosineSimilarity()` it actually uses, argsorts descending and renders the nearest
    issue's labels through display(Markdown(...)); `display` / `Markdown` are stand-ins that capture that text, and each
    reference issue's labels are its own row number.  Stores the chosen row and its f32 cosine per query."""
    import json
    import re
    import pandas as pd
    cells = json.load(open(NOTEBOOK))['cells']
    src = ''.join(cells[46]['source'])
    assert src.startswith('class oneshotlabeler')
    shown = []
    ns = {'json': json, 'CosineSimilarity': torch.nn.CosineSimilarity, 'cs': torch.nn.CosineSimilarity(),
          'Markdown': lambda text: text, 'display': shown.append}
    exec(compile(src, 'Kubeflow-FewShotLearning.ipynb:cell46', 'exec'), ns)
    vecs = np.load(os.path.join(HERE, SIMILARITY_INDEX))['expected']
    refdf = pd.DataFrame({'labels': [json.dumps([i]) for i in range(len(vecs))],
                          'url': [json.dumps(f'issue/{i}') for i in range(len(vecs))],
                          'title': [''] * len(vecs), 'body': [''] * len(vecs)})
    labeler = ns['oneshotlabeler'](torch.from_numpy(vecs), refdf)
    queries = np.concatenate([np.load(os.path.join(HERE, q))['expected'] for q in SIMILARITY_QUERIES])
    top1, sims = [], []
    for q in queries:
        labeler.query(torch.from_numpy(q))
        top1.append(json.loads(re.search(r'\*\*Predicted Labels\*\*: (\[.*?\])', shown[-1]).group(1))[0])
        sims.append(float(ns['cs'].forward(torch.from_numpy(q)[None], torch.from_numpy(vecs[top1[-1]][None]))[0]))
    np.savez_compressed(os.path.join(HERE, 'similarity_ref.npz'), index_source=np.array(SIMILARITY_INDEX),
                        query_sources=np.array(SIMILARITY_QUERIES), top1=np.array(top1, dtype=np.int64),
                        top1_cos=np.array(sims, dtype=np.float32))
    print('similarity', len(top1), 'queries; distinct nearest rows', len(set(top1)))


if __name__ == '__main__':
    similarity_fixture()
