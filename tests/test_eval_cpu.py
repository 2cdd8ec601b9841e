"""CPU test of the evaluation-loop mirror (imagecaptioning.pytorch_b200/eval_utils.py): the same stub model / loader driven through the
mirror must give the predictions and loss the UNMODIFIED reference eval_split gave (tests/golden/eval_split.json, made by
oracle/make_golden.py: gen_eval_split)."""
import json
import os

import numpy as np
import pytest
import torch


class _StubLoader:
    """The slice of captioning/data/dataloader.py's API eval_split uses: reset_iterator, get_batch -> dict with infos / bounds."""

    def __init__(self, n_images, batch, T, V1, seed=0):
        g = torch.Generator().manual_seed(seed)
        self.n, self.batch, self.pos = n_images, batch, 0
        self.fc = torch.randn(n_images, 8, generator=g)
        self.att = torch.randn(n_images, 3, 8, generator=g)
        self.labels = torch.randint(1, V1, (n_images, 1, T + 2), generator=g)
        self.labels[:, :, 0] = 0
        self.labels[:, :, -1] = 0
        self.masks = torch.ones(n_images, 1, T + 2)
        self.calls = 0

    def reset_iterator(self, split):
        self.pos = 0

    def get_batch(self, split):
        self.calls += 1
        ix = [(self.pos + i) % self.n for i in range(self.batch)]
        wrapped = self.pos + self.batch >= self.n
        self.pos = (self.pos + self.batch) % self.n
        return {'fc_feats': self.fc[ix], 'att_feats': self.att[ix], 'labels': self.labels[ix], 'masks': self.masks[ix], 'att_masks': None,
                'infos': [{'id': i, 'file_path': 'img%d.jpg' % i} for i in ix], 'bounds': {'it_pos_now': self.pos, 'it_max': self.n, 'wrapped': wrapped}}


class _StubModel(torch.nn.Module):
    """Deterministic fake captioner: log-probs are a fixed function of the features, seq = argmax (the surfaces eval_split touches)."""

    def __init__(self, T, V1):
        super().__init__()
        self.T, self.V1 = T, V1
        self.vocab = {str(i): 'w%d' % i for i in range(1, V1)}
        self.w = torch.nn.Parameter(torch.randn(8, T * V1, generator=torch.Generator().manual_seed(1)))
        self.done_beams = []

    def forward(self, fc_feats, att_feats, third, *rest, **kw):
        lp = torch.log_softmax((fc_feats @ self.w).view(-1, self.T, self.V1) * 3, 2)
        if kw.get('mode', 'forward') == 'sample':
            opt = kw.get('opt', {})
            n, beam = opt.get('sample_n', 1), opt.get('beam_size', 1)
            if n > 1:                                       # sample_n captions per image: the j-th is the (j+1)-th best word at every step
                lp = lp.repeat_interleave(n, 0)
                seq = torch.stack([lp[i].topk(n, 1).indices[:, i % n] for i in range(lp.shape[0])])
            else:
                seq = lp.argmax(2)
            ended = (seq == 0).cumsum(1) > 0
            seq = seq.masked_fill(ended, 0)
            if beam > 1:                                    # done_beams[i][j]['seq']: j-th candidate of image i
                cand = lp.topk(beam, 2).indices             # [B, T, beam]
                self.done_beams = [[{'seq': cand[i, :, j]} for j in range(beam)] for i in range(lp.shape[0])]
            return seq, lp
        return lp[:, :third.shape[-1]]            # teacher forcing: third = labels[..., :-1]


def _crit(lp, target, mask):
    target, mask = target.reshape(-1, target.shape[-1])[:, :lp.shape[1]], mask.reshape(-1, mask.shape[-1])[:, :lp.shape[1]]
    return -(lp.gather(2, target.unsqueeze(2)).squeeze(2) * mask).sum() / mask.sum()


T, V1 = 6, 12
EVAL_KWARGS = {'verbose': False, 'verbose_loss': 1, 'split': 'val', 'language_eval': 0, 'dataset': 'coco', 'beam_size': 1, 'sample_n': 1,
               'device': 'cpu', 'id': 'stub', 'num_images': -1}
N_METHODS = ['sample', 'bs', 'top3']


def eval_n_kwargs(method):
    return dict(EVAL_KWARGS, sample_n=3, sample_n_method=method, id='stubn')


def _golden(golden_dir, name):
    with open(os.path.join(golden_dir, 'eval_split.json')) as f:
        return json.load(f)[name]


def test_eval_split_matches_the_reference_loop(tmp_path, monkeypatch, golden_dir):
    from imagecaptioning.pytorch_b200 import eval_utils as EU
    model = _StubModel(T, V1)
    monkeypatch.chdir(tmp_path)
    loss, preds, stats = EU.eval_split(model, _crit, _StubLoader(10, 4, T, V1), dict(EVAL_KWARGS))
    assert stats is None and len(preds) == 10 and [p['image_id'] for p in preds] == list(range(10))
    assert model.training                                     # switched back (eval_utils.py:212)
    ref = _golden(golden_dir, 'n1')
    rpreds = ref['predictions']
    assert abs(loss - ref['loss']) < 1e-6
    assert [p['caption'] for p in preds] == [p['caption'] for p in rpreds]
    assert np.allclose([p['perplexity'] for p in preds], [p['perplexity'] for p in rpreds], atol=1e-5)
    assert np.allclose([p['entropy'] for p in preds], [p['entropy'] for p in rpreds], atol=1e-5)


def test_prefetch_loader_is_one_batch_ahead_and_stops_at_wrap():
    from imagecaptioning.pytorch_b200.eval_utils import PrefetchLoader
    loader = _StubLoader(10, 4, 5, 9)
    seen = [d['infos'][0]['id'] for d in PrefetchLoader(loader, 'val', 'cpu')]
    assert seen == [0, 4, 8] and loader.calls == 3             # the wrapped batch is the last one fetched


@pytest.mark.parametrize('method', N_METHODS)
def test_eval_split_n_matches_the_reference_loop(tmp_path, monkeypatch, golden_dir, method):
    """sample_n > 1 (eval_utils.py:196-197 -> eval_split_n): sample_n captions per image through 'bs' (the best beams) and the sampling
    methods, n_predictions sorted by perplexity and saved beside the predictions like the reference does."""
    from imagecaptioning.pytorch_b200 import eval_utils as EU
    monkeypatch.chdir(tmp_path)
    loss, preds, _ = EU.eval_split(_StubModel(T, V1), _crit, _StubLoader(10, 4, T, V1), eval_n_kwargs(method))
    saved_preds, saved_n = torch.load(os.path.join('eval_results', '.saved_pred_stubn_val.pth'), weights_only=False)
    assert len(saved_preds) == 10 and len(saved_n) == 3 * 12          # three batches of four images reach eval_split_n (the loop's own bookkeeping)
    if method != 'bs':
        ps = [e['perplexity'] for e in saved_n]
        assert ps == sorted(ps)
    ref = _golden(golden_dir, method)
    rpreds, rn = ref['predictions'], ref['n_predictions']
    assert abs(loss - ref['loss']) < 1e-6 and [p['caption'] for p in preds] == [p['caption'] for p in rpreds]
    assert [(e['image_id'], e['caption']) for e in saved_n] == [(e['image_id'], e['caption']) for e in rn]
    if method != 'bs':
        assert np.allclose([e['perplexity'] for e in saved_n], [e['perplexity'] for e in rn], atol=1e-5)
