"""Generate tests/golden/*.npz by running the LIVE reference (build container only; /root/reference is read-only).

    python oracle/make_golden.py            # needs /root/reference; writes tests/golden/

The reference modules are imported unmodified from /root/reference with a scratch cwd that holds the
``cider`` / ``coco-caption`` symlinks and a writable ``data/<name>.p`` document-frequency pickle, because
captioning/utils/rewards.py:12,15 and cider/pyciderevalcap/ciderD/ciderD_scorer.py:109 use cwd-relative paths.
Synthetic weights come from oracle.caption_oracle.make_weights (seeded) and are loaded into the reference's own
nn.Modules with load_state_dict, so each golden file records what the reference computes on exactly the inputs the
tests regenerate from the same seeds.  Nothing here is imported at test time on the GPU box.
"""
from __future__ import annotations

import argparse
import os
import pickle
import sys
import tempfile

import numpy as np
import torch

REPO = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
REF = '/root/reference'
sys.path.insert(0, REPO)

from oracle import caption_oracle as co          # noqa: E402
from oracle import ciderd_oracle as cdo          # noqa: E402


def _enter_scratch():
    d = tempfile.mkdtemp(prefix='refcwd_')
    os.symlink(os.path.join(REF, 'cider'), os.path.join(d, 'cider'))
    os.symlink(os.path.join(REF, 'coco-caption'), os.path.join(d, 'coco-caption'))
    os.makedirs(os.path.join(d, 'data'))
    os.chdir(d)
    sys.path.insert(0, REF)
    sys.dont_write_bytecode = True
    return d


def ref_model(family, V, E, H, A, F_fc, F_att, T, W, **extra):
    import captioning.models as M
    opt = argparse.Namespace(vocab_size=V, input_encoding_size=E, rnn_size=H, num_layers=1, drop_prob_lm=0.5,
                             max_length=T, seq_length=T, fc_feat_size=F_fc, att_feat_size=F_att, att_hid_size=A,
                             vocab={str(i): 'w%d' % i for i in range(1, V + 1)}, caption_model=family, use_bn=0,
                             logit_layers=1)
    for k, v in extra.items():
        setattr(opt, k, v)
    m = M.setup(opt)
    missing = m.load_state_dict(W, strict=True)
    m.eval()
    return m


def beams_to_arrays(done_beams, b, T):
    B = len(done_beams)
    seqs = np.zeros((B, b, T), np.int64)
    lens = np.zeros((B, b), np.int64)
    ps = np.zeros((B, b), np.float64)
    for i, lst in enumerate(done_beams):
        for j, rec in enumerate(lst):
            L = rec['seq'].shape[0]
            seqs[i, j, :L] = rec['seq'].numpy()
            lens[i, j] = L
            ps[i, j] = rec['p']
    return seqs, lens, ps


def gen_updown_small(out_dir):
    cfg = dict(V=60, E=32, H=32, A=16, F_fc=48, F_att=48, T=8)
    B, R, b = 4, 7, 3
    W = co.make_weights('updown', cfg['V'], cfg['E'], cfg['H'], cfg['A'], cfg['F_fc'], cfg['F_att'], seed=11, logit_scale=20.0)
    fc, att = co.make_inputs(B, R, cfg['F_fc'], cfg['F_att'], seed=11)
    m = ref_model('updown', W=W, **cfg)
    res = {}
    with torch.no_grad():
        seq, lp = m(fc, att, None, opt={'sample_method': 'greedy', 'beam_size': 1}, mode='sample')
        res['greedy_seq'], res['greedy_lp'] = seq.numpy(), lp.numpy()
        seq, lp = m(fc, att, None, opt={'beam_size': b, 'sample_n': 1}, mode='sample')
        res['beam_seq'], res['beam_lp'] = seq.numpy(), lp.numpy()
        res['done_seq'], res['done_len'], res['done_p'] = beams_to_arrays(m.done_beams, b, cfg['T'])
        seq, lp = m(fc, att, None, opt={'beam_size': b, 'sample_n': b}, mode='sample')
        res['beamn_seq'] = seq.numpy()
        # variable region counts (prefix masks)
        masks = torch.ones(B, R)
        masks[1, 5:] = 0
        masks[3, 3:] = 0
        seq, lp = m(fc, att, masks, opt={'sample_method': 'greedy', 'beam_size': 1}, mode='sample')
        res['masked_greedy_seq'], res['masked_greedy_lp'] = seq.numpy(), lp.numpy()
        seq, lp = m(fc, att, masks, opt={'beam_size': b, 'sample_n': 1}, mode='sample')
        res['masked_beam_seq'] = seq.numpy()
        res['masks'] = masks.numpy()
        # teacher forcing on the greedy result, 2 captions per image
        labels = torch.from_numpy(np.concatenate([np.zeros((B, 1), np.int64), res['greedy_seq'][:, :-1]], 1))
        labels2 = torch.stack([labels, labels.flip(0)], 1)                      # [B, 2, T]
        res['teacher_in'] = labels2.numpy()
        res['teacher_lp'] = m(fc, att, labels2, None).numpy()
        # sampled run, replayed by the oracle with forced tokens
        torch.manual_seed(5)
        seq, lp = m(fc, att, None, opt={'sample_method': 'sample', 'beam_size': 1, 'sample_n': 3, 'temperature': 1.0}, mode='sample')
        res['sample_seq'], res['sample_lp'] = seq.numpy(), lp.numpy()
    np.savez_compressed(os.path.join(out_dir, 'updown_small.npz'), cfg=np.array([cfg[k] for k in ('V', 'E', 'H', 'A', 'F_fc', 'F_att', 'T')]),
                        meta=np.array([B, R, b, 11]), **res)
    print('updown_small', {k: v.shape for k, v in res.items()})


def gen_updown_penalty(out_dir):
    """Beam search with the length penalties of misc.penalty_builder (:133-158) on the small UpDown configuration."""
    cfg = dict(V=60, E=32, H=32, A=16, F_fc=48, F_att=48, T=8)
    B, R, b = 4, 7, 3
    W = co.make_weights('updown', cfg['V'], cfg['E'], cfg['H'], cfg['A'], cfg['F_fc'], cfg['F_att'], seed=11, logit_scale=20.0)
    fc, att = co.make_inputs(B, R, cfg['F_fc'], cfg['F_att'], seed=11)
    m = ref_model('updown', W=W, **cfg)
    res = {}
    with torch.no_grad():
        for tag, pen in (('wu', 'wu_0.5'), ('avg', 'avg_0'), ('wu2', 'wu_1.5')):
            seq, lp = m(fc, att, None, opt={'beam_size': b, 'sample_n': 1, 'length_penalty': pen}, mode='sample')
            res[tag + '_seq'], res[tag + '_lp'] = seq.numpy(), lp.numpy()
            res[tag + '_done_seq'], res[tag + '_done_len'], res[tag + '_done_p'] = beams_to_arrays(m.done_beams, b, cfg['T'])
    np.savez_compressed(os.path.join(out_dir, 'updown_penalty.npz'), cfg=np.array([cfg[k] for k in ('V', 'E', 'H', 'A', 'F_fc', 'F_att', 'T')]),
                        meta=np.array([B, R, b, 11]), **res)
    print('updown_penalty', res['wu_seq'][0].tolist(), res['avg_seq'][0].tolist(), np.round(res['wu2_done_p'][0], 3).tolist())


def gen_newfc(out_dir):
    """BASELINE.json configs[0]: newfc greedy, batch 4, 2048-d fc feats, seq_len 16 (opts.py defaults E=H=512)."""
    cfg = dict(V=9487, E=512, H=512, A=512, F_fc=2048, F_att=2048, T=16)
    B = 4
    W = co.make_weights('newfc', cfg['V'], cfg['E'], cfg['H'], cfg['A'], cfg['F_fc'], cfg['F_att'], seed=1234, logit_scale=12.0)
    fc, att = co.make_inputs(B, 1, cfg['F_fc'], cfg['F_att'], seed=1234)
    m = ref_model('newfc', W=W, **cfg)
    with torch.no_grad():
        seq, lp = m(fc, att, None, opt={'sample_method': 'greedy', 'beam_size': 1}, mode='sample')
        seqb, lpb = m(fc, att, None, opt={'beam_size': 3, 'sample_n': 1}, mode='sample')
    picked = lp.gather(2, seq.unsqueeze(2)).squeeze(2)
    top2 = lp.topk(2, dim=2).values
    np.savez_compressed(os.path.join(out_dir, 'newfc_cfg1.npz'), cfg=np.array([cfg[k] for k in ('V', 'E', 'H', 'A', 'F_fc', 'F_att', 'T')]),
                        meta=np.array([B, 1, 1, 1234]), greedy_seq=seq.numpy(), greedy_picked_lp=picked.numpy(),
                        greedy_margin=(top2[..., 0] - top2[..., 1]).numpy(), greedy_row_sum=lp.sum(2).numpy(),
                        beam_seq=seqb.numpy(), done_p=beams_to_arrays(m.done_beams, 3, cfg['T'])[2])
    print('newfc_cfg1 greedy', seq[0].tolist())


def gen_updown_full(out_dir):
    """Full model dimensions of configs/updown/updown.yml (E=H=1000, A=512, V=9487), small batch; weights are
    regenerated from the seed at test time, only outputs are stored."""
    cfg = dict(V=9487, E=1000, H=1000, A=512, F_fc=2048, F_att=2048, T=20)
    B, R, b = 6, 36, 5
    W = co.make_weights('updown', cfg['V'], cfg['E'], cfg['H'], cfg['A'], cfg['F_fc'], cfg['F_att'], seed=1234, logit_scale=12.0)
    fc, att = co.make_inputs(B, R, cfg['F_fc'], cfg['F_att'], seed=1234)
    m = ref_model('updown', W=W, **cfg)
    with torch.no_grad():
        seq, lp = m(fc, att, None, opt={'sample_method': 'greedy', 'beam_size': 1}, mode='sample')
        picked = lp.gather(2, seq.unsqueeze(2)).squeeze(2)
        top2 = lp.topk(2, dim=2).values
        seqb, lpb = m(fc, att, None, opt={'beam_size': b, 'sample_n': 1}, mode='sample')
        pickedb = lpb.gather(2, seqb.unsqueeze(2)).squeeze(2)
        dseq, dlen, dp = beams_to_arrays(m.done_beams, b, cfg['T'])
    np.savez_compressed(os.path.join(out_dir, 'updown_full.npz'), cfg=np.array([cfg[k] for k in ('V', 'E', 'H', 'A', 'F_fc', 'F_att', 'T')]),
                        meta=np.array([B, R, b, 1234]), greedy_seq=seq.numpy(), greedy_picked_lp=picked.numpy(),
                        greedy_margin=(top2[..., 0] - top2[..., 1]).numpy(), beam_seq=seqb.numpy(), beam_picked_lp=pickedb.numpy(),
                        done_seq=dseq, done_len=dlen, done_p=dp)
    print('updown_full greedy', seq[0].tolist(), 'beam', seqb[0].tolist())


def gen_ciderd(out_dir, scratch):
    """CIDEr-D scores and the self-critical reward from the reference's own scorer (df from a pickle)."""
    from captioning.utils import rewards as R
    V, B, n, T = 40, 6, 5, 12
    df_imgs = cdo.make_refs(300, V, seed=3)
    df, ref_len = cdo.build_document_frequency(df_imgs)
    # pickle in the prepro_ngrams.py format: keys are tuples of *strings*
    from collections import defaultdict
    dd = defaultdict(float)                              # the reference indexes a defaultdict (ciderD_scorer.py:169)
    dd.update({tuple(str(t) for t in k): v for k, v in df.items()})
    pk = {'document_frequency': dd, 'ref_len': ref_len}
    with open(os.path.join(scratch, 'data', 'golden-df.p'), 'wb') as f:
        pickle.dump(pk, f, protocol=2)
    # cross-check the DF builder against the reference's CiderScorer.compute_doc_freq
    sys.path.append('cider')
    from pyciderevalcap.ciderD.ciderD_scorer import CiderScorer
    cs = CiderScorer(df_mode='corpus')
    for rows in df_imgs:
        cs.cook_append(None, [R.array_to_str(r) for r in rows])
    cs.compute_doc_freq()
    assert {tuple(int(t) for t in k): v for k, v in cs.document_frequency.items()} == df
    R.init_scorer('golden-df')
    gts = cdo.make_refs(B, V, seed=9)
    rng = np.random.RandomState(1)

    def hyp_rows(nrows):
        rows = np.zeros((nrows, T), np.int64)
        for i in range(nrows):
            ln = rng.randint(0, T + 1)
            rows[i, :ln] = np.minimum(rng.zipf(1.3, size=ln), V)
        return rows
    sampled = hyp_rows(B * n)
    greedy = hyp_rows(B)
    # make some hypotheses copy pieces of their references so the scores are not all ~0
    for i in range(B):
        sampled[i * n, :8] = gts[i][0][:8]
        greedy[i, :6] = gts[i][1][:6]
    sampled[3] = 0                                      # empty caption (just EOS)
    opt = argparse.Namespace(cider_reward_weight=1.0, bleu_reward_weight=0.0)
    reward = R.get_self_critical_reward(torch.from_numpy(greedy), gts, torch.from_numpy(sampled), opt)
    # raw scores through the scorer API
    res_ = [{'image_id': i, 'caption': [R.array_to_str(sampled[i])]} for i in range(B * n)]
    gts_ = {i: [R.array_to_str(r) for r in gts[i // n]] for i in range(B * n)}
    _, scores = R.CiderD_scorer.compute_score(gts_, res_)
    keys = np.array([list(k) + [-1] * (4 - len(k)) for k in df.keys()], np.int64)
    vals = np.array(list(df.values()), np.float64)
    np.savez_compressed(os.path.join(out_dir, 'ciderd.npz'), df_keys=keys, df_vals=vals, ref_len=np.array(ref_len),
                        gts=np.stack(gts), sampled=sampled, greedy=greedy, reward=reward, sample_scores=scores,
                        meta=np.array([V, B, n, T]))
    print('ciderd scores', np.round(scores[:6], 4), 'reward', np.round(reward[:3, 0], 4))


def gen_xe_struct(out_dir, scratch):
    """LanguageModelCriterion, LabelSmoothing and StructureLosses('new_self_critical') of the live reference on fixed inputs, plus the XE
    loss and a few parameter gradients of the reference UpDown model (train mode, drop_prob_lm = 0 so no RNG is involved)."""
    from captioning.modules import losses as RL
    from captioning.utils import rewards as R
    g = torch.Generator().manual_seed(8)
    res = {}
    # (1) criteria on random log-probs; labels [N, L+1] with EOS padding, masks through the EOS
    N, L, V1 = 9, 7, 31
    lp = torch.log_softmax(torch.randn(N, L, V1, generator=g) * 2, 2)
    labels = torch.zeros(N, L + 1, dtype=torch.long)
    masks = torch.zeros(N, L + 1)
    for i in range(N):
        ln = int(torch.randint(1, L, (1,), generator=g))
        labels[i, 1:1 + ln] = torch.randint(1, V1, (ln,), generator=g)
        masks[i, :ln + 2] = 1
    for name, crit in (('lm', RL.LanguageModelCriterion()), ('ls', RL.LabelSmoothing(smoothing=0.2))):
        x = lp.clone().requires_grad_(True)
        loss = crit(x, labels[:, 1:], masks[:, 1:])
        loss.backward()
        res[name + '_loss'], res[name + '_grad'] = loss.detach().numpy(), x.grad.numpy()
        res[name + '_loss_none'] = crit(lp, labels[:, 1:], masks[:, 1:], reduction='none').numpy()
    res['crit_lp'], res['crit_labels'], res['crit_masks'] = lp.numpy(), labels.numpy(), masks.numpy()
    # (2) structure loss with the scorer of the ciderd golden (same document-frequency pickle and hypotheses)
    z = np.load(os.path.join(out_dir, 'ciderd.npz'))
    V, B, n, T = [int(v) for v in z['meta']]
    R.init_scorer('golden-df')
    gts = [z['gts'][i] for i in range(B)]
    sampled = torch.from_numpy(z['sampled'])
    opt = argparse.Namespace(structure_loss_type='new_self_critical', train_sample_n=n, cider_reward_weight=1.0, bleu_reward_weight=0.0,
                             entropy_reward_weight=0.0, self_cider_reward_weight=0.0)
    slp = torch.log_softmax(torch.randn(B * n, T, V + 1, generator=g), 2).requires_grad_(True)
    out = RL.StructureLosses(opt)(slp, sampled, gts)
    out['loss'].backward()
    res['struc_lp'], res['struc_loss'], res['struc_grad'], res['struc_reward'] = slp.detach().numpy(), out['loss'].detach().numpy(), slp.grad.numpy(), \
        out['reward'].numpy()
    res['struc_scores'] = R.get_scores(gts, sampled, opt)
    # (3) XE step of the reference UpDown model
    cfg = dict(V=60, E=32, H=32, A=16, F_fc=48, F_att=48, T=8)
    Bm, Rm, spi = 4, 7, 2
    W = co.make_weights('updown', cfg['V'], cfg['E'], cfg['H'], cfg['A'], cfg['F_fc'], cfg['F_att'], seed=11, logit_scale=20.0)
    fc, att = co.make_inputs(Bm, Rm, cfg['F_fc'], cfg['F_att'], seed=11)
    m = ref_model('updown', W=W, **cfg)
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
    m.drop_prob_lm = 0.0
    m.core.drop_prob_lm = 0.0                         # F.dropout on the core output (AttModel.py:637)
    m.train()
    xl = torch.zeros(Bm, spi, cfg['T'] + 2, dtype=torch.long)
    xm = torch.zeros(Bm, spi, cfg['T'] + 2)
    for i in range(Bm):
        for j in range(spi):
            ln = int(torch.randint(2, cfg['T'] - 1, (1,), generator=g))          # every caption ends before the last column: early break
            xl[i, j, 1:1 + ln] = torch.randint(1, cfg['V'] + 1, (ln,), generator=g)
            xm[i, j, :ln + 2] = 1
    for name, crit in (('xe', RL.LanguageModelCriterion()), ('xels', RL.LabelSmoothing(smoothing=0.1))):
        m.zero_grad()
        lpm = m(fc, att, xl[..., :-1], None)
        loss = crit(lpm, xl[..., 1:].reshape(Bm * spi, -1), xm[..., 1:].reshape(Bm * spi, -1))
        loss.backward()
        res[name + '_loss'] = loss.detach().numpy()
        sd = dict(m.named_parameters())
        for k in ('logit.weight', 'core.att_lstm.weight_ih', 'core.lang_lstm.weight_hh', 'embed.0.weight', 'att_embed.0.weight', 'core.attention.alpha_net.bias',
                  'ctx2att.weight', 'fc_embed.0.bias'):
            res[name + '_grad_' + k] = sd[k].grad.numpy().copy()
        if name == 'xe':
            res['xe_logprobs'] = lpm.detach().numpy()
    res['xe_labels'], res['xe_masks'] = xl.numpy(), xm.numpy()
    res['xe_cfg'] = np.array([cfg[k] for k in ('V', 'E', 'H', 'A', 'F_fc', 'F_att', 'T')] + [Bm, Rm, spi, 11])
    np.savez_compressed(os.path.join(out_dir, 'xe_struct.npz'), **res)
    print('xe_struct: lm', float(res['lm_loss']), 'ls', float(res['ls_loss']), 'struc', float(res['struc_loss']), 'xe', float(res['xe_loss']),
          'xels', float(res['xels_loss']))


def gen_decode_sequence(out_dir):
    """captioning/utils/misc.py:62-84 on random id rows (with bad endings, BPE pieces, empty rows), with and without REMOVE_BAD_ENDINGS."""
    import json
    import captioning.utils.misc as M
    rng = np.random.RandomState(3)
    words = ['with', 'in', 'on', 'of', 'a', 'at', 'to', 'for', 'an', 'this', 'his', 'her', 'that', 'the', 'dog', 'cat@@', 's', 'runn@@', 'ing', 'man',
             'sits', 'table', 'red', 'two']
    vocab = {str(i + 1): w for i, w in enumerate(words)}
    seq = np.zeros((40, 9), np.int64)
    for i in range(40):
        ln = rng.randint(0, 10)
        seq[i, :ln] = rng.randint(1, len(words) + 1, size=ln)
    seq[5, :3] = [1, 2, 3]                 # only bad endings
    seq[6, :4] = [15, 21, 3, 14]           # ends with two bad endings
    res = {}
    for flag in ('0', '1'):
        os.environ['REMOVE_BAD_ENDINGS'] = flag
        res[flag] = M.decode_sequence(vocab, torch.from_numpy(seq))
    os.environ.pop('REMOVE_BAD_ENDINGS', None)
    json.dump({'vocab': vocab, 'seq': seq.tolist(), 'out': res}, open(os.path.join(out_dir, 'decode_sequence.json'), 'w'))
    print('decode_sequence', res['0'][6], '|', res['1'][6])


def gen_ciderd_pascal(out_dir, scratch):
    """CIDEr-D of the live reference scorer on REAL captions: the first 60 images of cider/data/pascal50S.json (50 references each) and
    their candidates from pascal_candsB.json, lower-cased and split on non-alphanumerics, words mapped to ids 1..V; the document
    frequencies come from the reference's own compute_doc_freq over those references."""
    import json
    import re
    from collections import defaultdict, OrderedDict
    from captioning.utils import rewards as R
    sys.path.append('cider')
    from pyciderevalcap.ciderD.ciderD_scorer import CiderScorer
    refs_all = json.load(open(os.path.join(REF, 'cider', 'data', 'pascal50S.json')))
    cands_all = json.load(open(os.path.join(REF, 'cider', 'data', 'pascal_candsB.json')))
    tok = lambda t: [w for w in re.split(r'[^a-z0-9]+', t.lower()) if w]
    by_img = OrderedDict()
    for r in refs_all:
        by_img.setdefault(r['image_id'], []).append(tok(r['caption']))
    imgs = [k for k in by_img][:60]
    cand_of = {c['image_id']: tok(c['caption']) for c in cands_all}
    imgs = [k for k in imgs if k in cand_of and cand_of[k]][:60]
    vocab = {}
    def ids(words):
        return [vocab.setdefault(w, len(vocab) + 1) for w in words]
    L = 40
    refs = np.zeros((len(imgs), 50, L), np.int32)
    cands = np.zeros((len(imgs), L), np.int64)
    for i, k in enumerate(imgs):
        for j, words in enumerate(by_img[k][:50]):
            w = ids(words)[:L - 1]
            refs[i, j, :len(w)] = w
        w = ids(cand_of[k])[:L - 1]
        cands[i, :len(w)] = w
    cs = CiderScorer(df_mode='corpus')
    for i in range(len(imgs)):
        cs.cook_append(None, [R.array_to_str(r) for r in refs[i]])
    cs.compute_doc_freq()
    dd = defaultdict(float)
    dd.update(cs.document_frequency)
    with open(os.path.join(scratch, 'data', 'pascal-df.p'), 'wb') as f:
        pickle.dump({'document_frequency': dd, 'ref_len': float(len(imgs))}, f, protocol=2)
    R.CiderD_scorer = None
    R.init_scorer('pascal-df')
    res_ = [{'image_id': i, 'caption': [R.array_to_str(cands[i])]} for i in range(len(imgs))]
    gts_ = {i: [R.array_to_str(r) for r in refs[i]] for i in range(len(imgs))}
    mean, scores = R.CiderD_scorer.compute_score(gts_, res_)
    keys = np.array([[int(t) for t in k] + [-1] * (4 - len(k)) for k in cs.document_frequency.keys()], np.int32)
    vals = np.array(list(cs.document_frequency.values()), np.float64)
    np.savez_compressed(os.path.join(out_dir, 'ciderd_pascal.npz'), df_keys=keys, df_vals=vals, ref_len=np.array(float(len(imgs))), refs=refs.astype(np.int16),
                        cands=cands.astype(np.int16), scores=np.asarray(scores), mean=np.array(mean))
    R.CiderD_scorer = None
    print('ciderd_pascal: %d images, %d n-grams, vocabulary %d, mean CIDEr-D %.4f' % (len(imgs), len(keys), len(vocab), mean))


def gen_reward_criterion(out_dir):
    from captioning.modules.losses import RewardCriterion
    g = torch.Generator().manual_seed(3)
    N, L, V1 = 10, 7, 23
    lp = torch.log_softmax(torch.randn(N, L, V1, generator=g), 2).requires_grad_(True)
    seq = torch.randint(1, V1, (N, L), generator=g)
    seq[0, 3:] = 0
    seq[4, 0:] = 0
    seq[7, 6:] = 0
    reward = torch.randn(N, 1, generator=g).expand(N, L).contiguous()
    crit = RewardCriterion()
    loss = crit(lp, seq, reward)
    loss.backward()
    loss_none = crit(lp.detach(), seq, reward, reduction='none')
    np.savez_compressed(os.path.join(out_dir, 'reward_criterion.npz'), lp=lp.detach().numpy(), seq=seq.numpy(), reward=reward.numpy(),
                        loss=loss.detach().numpy(), grad=lp.grad.numpy(), loss_none=loss_none.numpy())
    print('reward_criterion loss', float(loss))


def _gen_family_small(out_dir, family, name, cfg, extra, heads, logit_scale):
    """greedy / beam / masks / teacher forcing / sampled replay of a small model through the live reference."""
    B, R, b, seed = 4, 7, 3, 17
    W = co.make_weights(family, cfg['V'], cfg['E'], cfg['H'], cfg['A'], cfg['F_fc'], cfg['F_att'], seed=seed, logit_scale=logit_scale)
    fc, att = co.make_inputs(B, R, cfg['F_fc'], cfg['F_att'], seed=seed)
    m = ref_model(family, W=W, **cfg, **extra)
    res = {}
    with torch.no_grad():
        seq, lp = m(fc, att, None, opt={'sample_method': 'greedy', 'beam_size': 1}, mode='sample')
        res['greedy_seq'], res['greedy_lp'] = seq.numpy(), lp.numpy()
        seq, lp = m(fc, att, None, opt={'beam_size': b, 'sample_n': 1}, mode='sample')
        res['beam_seq'], res['beam_lp'] = seq.numpy(), lp.numpy()
        res['done_seq'], res['done_len'], res['done_p'] = beams_to_arrays(m.done_beams, b, cfg['T'])
        masks = torch.ones(B, R)
        masks[1, 5:] = 0
        masks[3, 3:] = 0
        seq, lp = m(fc, att, masks, opt={'sample_method': 'greedy', 'beam_size': 1}, mode='sample')
        res['masked_greedy_seq'], res['masked_greedy_lp'] = seq.numpy(), lp.numpy()
        seq, lp = m(fc, att, masks, opt={'beam_size': b, 'sample_n': 1}, mode='sample')
        res['masked_beam_seq'] = seq.numpy()
        res['masks'] = masks.numpy()
        labels = torch.from_numpy(np.concatenate([np.zeros((B, 1), np.int64), res['greedy_seq'][:, :-1]], 1))
        labels2 = torch.stack([labels, labels.flip(0)], 1)
        res['teacher_in'] = labels2.numpy()
        res['teacher_lp'] = m(fc, att, labels2, None).numpy()
        torch.manual_seed(5)
        seq, lp = m(fc, att, None, opt={'sample_method': 'sample', 'beam_size': 1, 'sample_n': 3, 'temperature': 1.0}, mode='sample')
        res['sample_seq'], res['sample_lp'] = seq.numpy(), lp.numpy()
    np.savez_compressed(os.path.join(out_dir, name), cfg=np.array([cfg[k] for k in ('V', 'E', 'H', 'A', 'F_fc', 'F_att', 'T')]),
                        meta=np.array([B, R, b, seed, heads]), **res)
    print(name, 'greedy', res['greedy_seq'][0].tolist(), 'beam', res['beam_seq'][0].tolist())


def gen_transformer_small(out_dir):
    # make_weights('transformer'): E = d_model, H = d_ff, A = layers per stack
    cfg = dict(V=60, E=32, H=64, A=2, F_fc=48, F_att=48, T=8)
    _gen_family_small(out_dir, 'transformer', 'transformer_small.npz', cfg, dict(num_layers=2, N_enc=2, N_dec=2, d_model=32, d_ff=64,
                                                                                 num_att_heads=4, dropout=0.1), 4, 10.0)


def gen_aoa_small(out_dir):
    cfg = dict(V=60, E=32, H=32, A=16, F_fc=48, F_att=48, T=8)
    _gen_family_small(out_dir, 'aoa', 'aoa_small.npz', cfg, dict(num_layers=2, refine=1, refine_aoa=1, use_ff=0, decoder_type='AoA', use_multi_head=2,
                                                                  num_heads=4, multi_head_scale=1, mean_feats=1, ctx_drop=1, dropout_aoa=0.3), 4, 20.0)


def gen_updown_b256(out_dir):
    """BASELINE.json configs[1] at its own shape: UpDown full dimensions, batch 256, beam 5, through the live reference.  Stores the winning
    ids, their log-probs, the finished-beam scores, and (from the oracle port on the same inputs) each image's smallest candidate gap so
    the GPU test can demand bit-exact ids wherever the decision is not a numerical tie."""
    cfg = dict(V=9487, E=1000, H=1000, A=512, F_fc=2048, F_att=2048, T=20)
    B, R, b = 256, 36, 5
    W = co.make_weights('updown', cfg['V'], cfg['E'], cfg['H'], cfg['A'], cfg['F_fc'], cfg['F_att'], seed=1234, logit_scale=12.0)
    fc, att = co.make_inputs(B, R, cfg['F_fc'], cfg['F_att'], seed=1234)
    m = ref_model('updown', W=W, **cfg)
    with torch.no_grad():
        seqb, lpb = m(fc, att, None, opt={'beam_size': b, 'sample_n': 1}, mode='sample')
        pickedb = lpb.gather(2, seqb.unsqueeze(2)).squeeze(2)
        dseq, dlen, dp = beams_to_arrays(m.done_beams, b, cfg['T'])
        rows = []
        oseq, olp, _ = co.sample_beam(co.Family('updown', W, cfg['T']), fc, att, beam_size=b, margin_rows=rows)
    margin = torch.stack(rows, 1).min(1).values.numpy()
    agree = (oseq == seqb).all(1).numpy()
    np.savez_compressed(os.path.join(out_dir, 'updown_b256.npz'), cfg=np.array([cfg[k] for k in ('V', 'E', 'H', 'A', 'F_fc', 'F_att', 'T')]),
                        meta=np.array([B, R, b, 1234]), beam_seq=seqb.numpy().astype(np.int16), beam_picked_lp=pickedb.numpy(),
                        done_len=dlen.astype(np.int8), done_p=dp, done_seq=dseq.astype(np.int16), image_margin=margin)
    print('updown_b256: oracle port agrees with the reference on %d / %d images; smallest margin %.3g; %d images below 1e-3' %
          (int(agree.sum()), B, float(margin.min()), int((margin < 1e-3).sum())))


def gen_transformer_b64(out_dir):
    """BASELINE.json configs[2] at its per-GPU shape: Transformer 6+6 / d_model 512 / d_ff 2048 / 8 heads, batch 64, beam 5 and greedy,
    through the live reference (which re-runs the whole decoder every step, TransformerModel.py:351-363)."""
    cfg = dict(V=9487, E=512, H=2048, A=6, F_fc=2048, F_att=2048, T=20)
    B, R, b = 64, 36, 5
    W = co.make_weights('transformer', cfg['V'], cfg['E'], cfg['H'], cfg['A'], cfg['F_fc'], cfg['F_att'], seed=1234, logit_scale=3.0)
    fc, att = co.make_inputs(B, R, cfg['F_fc'], cfg['F_att'], seed=1234)
    m = ref_model('transformer', W=W, **cfg, num_layers=6, N_enc=6, N_dec=6, d_model=512, d_ff=2048, num_att_heads=8, dropout=0.1)
    with torch.no_grad():
        seq, lp = m(fc, att, None, opt={'sample_method': 'greedy', 'beam_size': 1}, mode='sample')
        picked = lp.gather(2, seq.unsqueeze(2)).squeeze(2)
        top2 = lp.topk(2, dim=2).values
        gmargin = (top2[..., 0] - top2[..., 1])
        live = torch.cat([torch.ones(B, 1, dtype=torch.bool), (seq[:, :-1] > 0)], 1)
        gmargin = torch.where(live, gmargin, torch.full_like(gmargin, 1e9)).min(1).values
        seqb, lpb = m(fc, att, None, opt={'beam_size': b, 'sample_n': 1}, mode='sample')
        pickedb = lpb.gather(2, seqb.unsqueeze(2)).squeeze(2)
        dseq, dlen, dp = beams_to_arrays(m.done_beams, b, cfg['T'])
        rows = []
        oseq, _, _ = co.sample_beam(co.Family('transformer', W, cfg['T'], heads=8), fc, att, beam_size=b, margin_rows=rows)
    margin = torch.stack(rows, 1).min(1).values.numpy()
    np.savez_compressed(os.path.join(out_dir, 'transformer_b64.npz'), cfg=np.array([cfg[k] for k in ('V', 'E', 'H', 'A', 'F_fc', 'F_att', 'T')]),
                        meta=np.array([B, R, b, 1234, 8]), greedy_seq=seq.numpy().astype(np.int16), greedy_picked_lp=picked.numpy(),
                        greedy_margin=gmargin.numpy(), beam_seq=seqb.numpy().astype(np.int16), beam_picked_lp=pickedb.numpy(), done_len=dlen.astype(np.int8),
                        done_p=dp, image_margin=margin)
    print('transformer_b64: oracle port agrees on %d / %d images; smallest beam margin %.3g, smallest greedy margin %.3g' %
          (int((oseq == seqb).all(1).sum()), B, float(margin.min()), float(gmargin.min())))


def _subsample(t, grid=(96, 80), whole=8192):
    """Compact fingerprint of a gradient tensor: every entry when small, else a strided sub-grid; plus sum / abs-sum / Frobenius norm."""
    a = t.detach().numpy()
    if a.size <= whole:
        sub, step = a.copy(), (1, 1)
    elif a.ndim == 1:
        sub, step = a[::7].copy(), (7, 1)
    else:
        sr, sc = max(1, a.shape[0] // grid[0]), max(1, a.shape[1] // grid[1])
        sub, step = a[::sr, ::sc].copy(), (sr, sc)
    stats = np.array([a.sum(dtype=np.float64), np.abs(a).sum(dtype=np.float64), np.sqrt((a.astype(np.float64) ** 2).sum()), np.abs(a).max()])
    return sub, np.array(step), stats


def gen_aoa_scst_full(out_dir, scratch):
    """BASELINE.json configs[3] at its own shape: AoANet (configs/aoa.yml: E = H = 1024, 8 heads, 6 refiner layers), V = 9487, per-GPU batch 10,
    train_sample_n 5, one LossWrapper(sc_flag=True) step + loss.backward() of the LIVE reference (loss_wrapper.py:56-73).  Every dropout
    probability is set to 0 so no RNG stream has to be shared; the reference's own multinomial samples are stored and the engine replays them
    as forced tokens.  Gradients: a fingerprint (sub-grid + sums + norm) of every parameter."""
    from captioning.modules.loss_wrapper import LossWrapper
    from captioning.utils import rewards as R
    cfg = dict(V=9487, E=1024, H=1024, A=512, F_fc=2048, F_att=2048, T=20)
    B, Rr, n, heads = 10, 36, 5, 8
    W = co.make_weights('aoa', cfg['V'], cfg['E'], cfg['H'], cfg['A'], cfg['F_fc'], cfg['F_att'], seed=1234, logit_scale=6.0)
    fc, att = co.make_inputs(B, Rr, cfg['F_fc'], cfg['F_att'], seed=1234)
    extra = dict(num_layers=2, refine=1, refine_aoa=1, use_ff=0, decoder_type='AoA', use_multi_head=2, num_heads=heads, multi_head_scale=1, mean_feats=1,
                 ctx_drop=1, dropout_aoa=0.3)
    m = ref_model('aoa', W=W, **cfg, **extra)
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
        if isinstance(getattr(mod, 'drop_prob_lm', None), float):
            mod.drop_prob_lm = 0.0
    # Random references share no n-grams with the model's captions at V = 9487 (all rewards ~ 0).  The references are therefore corrupted
    # copies of the model's own greedy caption of each image (30 % of the tokens replaced, three of the five truncated), which gives CIDEr-D
    # scores of O(1) for the greedy baseline and a spread of rewards for the samples.
    with torch.no_grad():
        g0, _ = m(fc, att, None, opt={'sample_method': 'greedy', 'beam_size': 1}, mode='sample')
    rng = np.random.RandomState(5)
    gts = []
    for i in range(B):
        rows = np.zeros((5, 16), np.int64)
        for j in range(5):
            ln = 16 if j < 2 else int(rng.randint(6, 15))
            row = g0[i, :ln].numpy().copy()
            flip = rng.rand(ln) < 0.3
            row[flip] = rng.randint(1, cfg['V'] + 1, size=int(flip.sum()))
            rows[j, :ln] = row
        gts.append(rows)
    df, ref_len = cdo.build_document_frequency(cdo.make_refs(1000, cfg['V'], seed=4) + gts)
    from collections import defaultdict
    dd = defaultdict(float)
    dd.update({tuple(str(t) for t in k): v for k, v in df.items()})
    with open(os.path.join(scratch, 'data', 'aoa-full-df.p'), 'wb') as f:
        pickle.dump({'document_frequency': dd, 'ref_len': ref_len}, f, protocol=2)
    R.CiderD_scorer = None
    R.Cider_scorer = None
    R.init_scorer('aoa-full-df')
    opt = argparse.Namespace(label_smoothing=0, structure_loss_type='seqnll', structure_loss_weight=1, train_sample_method='sample', train_beam_size=1,
                             train_sample_n=n, sc_sample_method='greedy', sc_beam_size=1, cider_reward_weight=1.0, bleu_reward_weight=0.0, use_ppo=0,
                             struc_use_logsoftmax=1)
    lw = LossWrapper(m, opt)
    captured = {}
    orig = m._sample

    def spy(*a, **k):
        out = orig(*a, **k)
        captured.setdefault('calls', []).append(out[0].detach().clone())
        return out
    m._sample = spy
    torch.manual_seed(77)
    m.zero_grad()
    out = lw(fc, att, None, None, None, gts, torch.arange(B), True, False, False)
    out['loss'].backward()
    greedy_seq, sample_seq = captured['calls'][0], captured['calls'][1]
    assert greedy_seq.shape == (B, cfg['T']) and sample_seq.shape == (B * n, cfg['T'])
    reward = R.get_self_critical_reward(greedy_seq, gts, sample_seq, opt)
    res = {'greedy_seq': greedy_seq.numpy().astype(np.int16), 'sample_seq': sample_seq.numpy().astype(np.int16), 'loss': out['loss'].detach().numpy(),
           'reward_mean': out['reward'].numpy(), 'reward': reward[:, 0].astype(np.float64), 'gts': np.stack(gts).astype(np.int16)}
    names = []
    for k, prm in m.named_parameters():
        sub, step, stats = _subsample(prm.grad)
        res['g_' + k], res['s_' + k], res['t_' + k] = sub, step, stats
        names.append(k)
    keys = np.array([list(k) + [-1] * (4 - len(k)) for k in df.keys()], np.int32)
    vals = np.array(list(df.values()), np.float64)
    np.savez_compressed(os.path.join(out_dir, 'aoa_scst_full.npz'), cfg=np.array([cfg[k] for k in ('V', 'E', 'H', 'A', 'F_fc', 'F_att', 'T')]),
                        meta=np.array([B, Rr, n, 1234, heads]), df_keys=keys, df_vals=vals, ref_len=np.array(ref_len), names=np.array(names), **res)
    print('aoa_scst_full: loss %.6g, mean reward %.4g, max |reward| %.4g, %d gradient tensors, sample lengths %s' %
          (float(out['loss']), float(out['reward']), float(np.abs(reward).max()), len(names), (sample_seq > 0).sum(1)[:8].tolist()))


def _gen_transformer_train(out_dir, scratch, name, cfg, layers, heads, B, Rr, n, spi, logit_scale, seed, full_grads):
    """Transformer under the LIVE reference's LossWrapper: (a) the XE branch (teacher-forced _forward + LanguageModelCriterion / LabelSmoothing) and
    (b) the sc branch (greedy baseline, train-mode multinomial samples, CIDEr-D reward, RewardCriterion), each followed by loss.backward().
    Every dropout probability is 0 (no RNG stream to share); the reference's own samples are stored and the engine replays them as forced
    tokens.  Gradients: every tensor in full for the small model, a fingerprint (sub-grid + sums + norm) at BASELINE size."""
    from captioning.modules.loss_wrapper import LossWrapper
    from captioning.modules import losses as RL
    from captioning.utils import rewards as R
    T, V = cfg['T'], cfg['V']
    W = co.make_weights('transformer', V, cfg['E'], cfg['H'], cfg['A'], cfg['F_fc'], cfg['F_att'], seed=seed, logit_scale=logit_scale)
    fc, att = co.make_inputs(B, Rr, cfg['F_fc'], cfg['F_att'], seed=seed)
    m = ref_model('transformer', W=W, **cfg, num_layers=layers, N_enc=layers, N_dec=layers, d_model=cfg['E'], d_ff=cfg['H'], num_att_heads=heads, dropout=0.0)
    for mod in m.modules():
        if isinstance(mod, torch.nn.Dropout):
            mod.p = 0.0
    res = {}

    def store(prefix):
        for k, prm in m.named_parameters():
            if full_grads:
                res[prefix + 'g_' + k] = prm.grad.numpy().copy()
            else:
                res[prefix + 'g_' + k], res[prefix + 's_' + k], res[prefix + 't_' + k] = _subsample(prm.grad, grid=(40, 32), whole=2048)

    # ---- (a) XE: labels [B, spi, T + 2]: BOS, words, EOS / padding; captions of different lengths, some ending early
    g = torch.Generator().manual_seed(seed + 1)
    xl = torch.zeros(B, spi, T + 2, dtype=torch.long)
    xm = torch.zeros(B, spi, T + 2)
    for i in range(B):
        for j in range(spi):
            ln = int(torch.randint(2, T + 1, (1,), generator=g))
            xl[i, j, 1:1 + ln] = torch.randint(1, V + 1, (ln,), generator=g)
            xm[i, j, :ln + 2] = 1
    m.train()
    for tag, crit in (('xe_', RL.LanguageModelCriterion()), ('xels_', RL.LabelSmoothing(smoothing=0.1))):
        if tag == 'xels_' and not full_grads:
            res['xels_loss'] = np.array(0.0)
            continue                                # the BASELINE-size fixture stays small: one XE criterion
        m.zero_grad()
        lpm = m(fc, att, xl[..., :-1], None)
        loss = crit(lpm, xl[..., 1:].reshape(B * spi, -1), xm[..., 1:].reshape(B * spi, -1))
        loss.backward()
        res[tag + 'loss'] = loss.detach().numpy()
        store(tag)
        if tag == 'xe_' and full_grads:
            res['xe_logprobs'] = lpm.detach().numpy()
    res['xe_labels'], res['xe_masks'] = xl.numpy().astype(np.int16), xm.numpy()
    # ---- (b) SCST; references = corrupted copies of the greedy captions (see gen_aoa_scst_full)
    m.eval()
    with torch.no_grad():
        g0, _ = m(fc, att, None, opt={'sample_method': 'greedy', 'beam_size': 1}, mode='sample')
    rng = np.random.RandomState(seed + 2)
    gts = []
    Lr = min(16, T)
    for i in range(B):
        rows = np.zeros((5, Lr), np.int64)
        for j in range(5):
            ln = Lr if j < 2 else int(rng.randint(max(2, Lr // 3), Lr))
            row = g0[i, :ln].numpy().copy()
            flip = rng.rand(ln) < 0.3
            row[flip] = rng.randint(1, V + 1, size=int(flip.sum()))
            rows[j, :ln] = row
        gts.append(rows)
    df, ref_len = cdo.build_document_frequency(cdo.make_refs(300 if full_grads else 1000, V, seed=4) + gts)
    from collections import defaultdict
    dd = defaultdict(float)
    dd.update({tuple(str(t) for t in k): v for k, v in df.items()})
    dfname = 'tfm-train-df-%s' % name.replace('.npz', '')
    with open(os.path.join(scratch, 'data', dfname + '.p'), 'wb') as f:
        pickle.dump({'document_frequency': dd, 'ref_len': ref_len}, f, protocol=2)
    R.CiderD_scorer = None
    R.Cider_scorer = None
    R.init_scorer(dfname)
    opt = argparse.Namespace(label_smoothing=0, structure_loss_type='seqnll', structure_loss_weight=1, train_sample_method='sample', train_beam_size=1,
                             train_sample_n=n, sc_sample_method='greedy', sc_beam_size=1, cider_reward_weight=1.0, bleu_reward_weight=0.0, use_ppo=0,
                             struc_use_logsoftmax=1)
    lw = LossWrapper(m, opt)
    captured = {}
    orig = m._sample

    def spy(*a, **k):
        out = orig(*a, **k)
        captured.setdefault('calls', []).append(out[0].detach().clone())
        return out
    m._sample = spy
    m.train()
    torch.manual_seed(77)
    m.zero_grad()
    out = lw(fc, att, None, None, None, gts, torch.arange(B), True, False, False)
    out['loss'].backward()
    greedy_seq, sample_seq = captured['calls'][0], captured['calls'][1]
    assert greedy_seq.shape == (B, T) and sample_seq.shape == (B * n, T)
    reward = R.get_self_critical_reward(greedy_seq, gts, sample_seq, opt)
    res.update({'greedy_seq': greedy_seq.numpy().astype(np.int16), 'sample_seq': sample_seq.numpy().astype(np.int16), 'sc_loss': out['loss'].detach().numpy(),
                'reward_mean': out['reward'].numpy(), 'reward': reward[:, 0].astype(np.float64), 'gts': np.stack(gts).astype(np.int16)})
    store('sc_')
    names = [k for k, _ in m.named_parameters()]
    keys = np.array([list(k) + [-1] * (4 - len(k)) for k in df.keys()], np.int32)
    vals = np.array(list(df.values()), np.float64)
    np.savez_compressed(os.path.join(out_dir, name), cfg=np.array([cfg[k] for k in ('V', 'E', 'H', 'A', 'F_fc', 'F_att', 'T')]),
                        meta=np.array([B, Rr, n, seed, heads, spi, int(full_grads)]), logit_scale=np.array(logit_scale), df_keys=keys, df_vals=vals,
                        ref_len=np.array(ref_len), names=np.array(names), **res)
    print('%s: xe %.6g, xels %.6g, sc loss %.6g, mean reward %.4g, max |reward| %.4g, %d gradient tensors, sample lengths %s' %
          (name, float(res['xe_loss']), float(res['xels_loss']), float(out['loss']), float(out['reward']), float(np.abs(reward).max()), len(names),
           (sample_seq > 0).sum(1)[:8].tolist()))


def gen_transformer_train(out_dir, scratch):
    _gen_transformer_train(out_dir, scratch, 'transformer_train_small.npz', dict(V=60, E=32, H=64, A=2, F_fc=48, F_att=48, T=8), 2, 4, B=3, Rr=7, n=3, spi=2,
                           logit_scale=10.0, seed=23, full_grads=True)


def gen_transformer_train_full(out_dir, scratch):
    """BASELINE.json configs[2]'s architecture (6+6 layers, d_model 512, d_ff 2048, 8 heads, V = 9487) at configs[3]'s training shape (10 images x 5)."""
    _gen_transformer_train(out_dir, scratch, 'transformer_train_full.npz', dict(V=9487, E=512, H=2048, A=6, F_fc=2048, F_att=2048, T=20), 6, 8, B=10, Rr=36, n=5,
                           spi=5, logit_scale=3.0, seed=1234, full_grads=False)


def gen_updown_options(out_dir):
    """Decode options of the reference on the small UpDown configuration: decoding_constraint, remove_bad_endings, block_trigrams (greedy
    _sample, AttModel.py:294-332) and suppress_UNK / decoding_constraint / remove_bad_endings / temperature in beam search
    (CaptionModel.py:118-120,154-162,204).  The vocabulary carries 'UNK' as its last word and a few bad-ending words."""
    cfg = dict(V=60, E=32, H=32, A=16, F_fc=48, F_att=48, T=10)
    B, R, b = 5, 7, 3
    W = co.make_weights('updown', cfg['V'], cfg['E'], cfg['H'], cfg['A'], cfg['F_fc'], cfg['F_att'], seed=23, logit_scale=8.0)
    fc, att = co.make_inputs(B, R, cfg['F_fc'], cfg['F_att'], seed=23)
    m = ref_model('updown', W=W, **cfg)
    vocab = {str(i): 'w%d' % i for i in range(1, cfg['V'] + 1)}
    vocab[str(cfg['V'])] = 'UNK'
    # make the model's favourite words bad endings so that the option changes something
    with torch.no_grad():
        g0, _ = m(fc, att, None, opt={'sample_method': 'greedy', 'beam_size': 1}, mode='sample')
    fav = [int(t) for t in torch.bincount(g0[g0 > 0].flatten(), minlength=cfg['V'] + 1).argsort(descending=True)[:3] if int(t) != cfg['V']]
    for w, name in zip(fav, ('the', 'a', 'with')):
        vocab[str(w)] = name
    m.vocab = vocab
    m.bad_endings_ix = [int(k) for k, v in vocab.items() if v in ('a', 'an', 'the', 'in', 'for', 'at', 'of', 'with', 'before', 'after', 'on', 'upon', 'near', 'to', 'is', 'are', 'am')]
    res = {'bad_words': np.array(fav), 'vocab_unk': np.array(cfg['V'])}
    with torch.no_grad():
        # (remove_bad_endings in _sample indexes with a uint8 mask, AttModel.py:303, which current torch rejects: the reference itself cannot
        # run that option there, so it has no golden; in beam search the mask is boolean and it works)
        for tag, opt in (('g_plain', {}), ('g_con', {'decoding_constraint': 1}), ('g_tri', {'block_trigrams': 1}),
                         ('g_all', {'decoding_constraint': 1, 'block_trigrams': 1})):
            seq, lp = m(fc, att, None, opt=dict({'sample_method': 'greedy', 'beam_size': 1}, **opt), mode='sample')
            res[tag + '_seq'], res[tag + '_lp'] = seq.numpy(), lp.numpy()
        # block_trigrams with sample_n > 1 only touches the first batch_size rows (the reference loops over range(batch_size))
        torch.manual_seed(3)
        seq, lp = m(fc, att, None, opt={'sample_method': 'sample', 'beam_size': 1, 'sample_n': 2, 'block_trigrams': 1, 'decoding_constraint': 1}, mode='sample')
        res['s_tri_seq'], res['s_tri_lp'] = seq.numpy(), lp.numpy()
        for tag, opt in (('b_unk', {'suppress_UNK': 1}), ('b_temp', {'temperature': 0.7}), ('b_con', {'decoding_constraint': 1}),
                         ('b_bad', {'remove_bad_endings': 1}),
                         ('b_all', {'suppress_UNK': 1, 'decoding_constraint': 1, 'remove_bad_endings': 1, 'temperature': 1.3})):
            seq, lp = m(fc, att, None, opt=dict({'beam_size': b, 'sample_n': 1}, **opt), mode='sample')
            res[tag + '_seq'], res[tag + '_lp'] = seq.numpy(), lp.numpy()
            res[tag + '_done_seq'], res[tag + '_done_len'], res[tag + '_done_p'] = beams_to_arrays(m.done_beams, b, cfg['T'])
    np.savez_compressed(os.path.join(out_dir, 'updown_options.npz'), cfg=np.array([cfg[k] for k in ('V', 'E', 'H', 'A', 'F_fc', 'F_att', 'T')]),
                        meta=np.array([B, R, b, 23]), **res)
    print('updown_options: greedy plain', res['g_plain_seq'][0].tolist(), 'constraint', res['g_con_seq'][0].tolist(), 'all', res['g_all_seq'][0].tolist(),
          '| beam all', res['b_all_seq'][0].tolist(), 'bad words', fav)


def gen_state_dict_keys(out_dir):
    """Names and shapes of the reference modules' parameters: the drop-in must expose exactly these (SURVEY.md 8b)."""
    import json
    res = {}
    for fam in ('updown', 'newfc'):
        cfg = dict(V=60, E=32, H=40, A=16, F_fc=48, F_att=56, T=8)
        W = co.make_weights(fam, cfg['V'], cfg['E'], cfg['H'], cfg['A'], cfg['F_fc'], cfg['F_att'], seed=1)
        m = ref_model(fam, W=W, **cfg)
        res[fam] = {k: list(v.shape) for k, v in m.state_dict().items()}
    W = co.make_weights('transformer', 60, 32, 64, 2, 48, 56, seed=1)
    m = ref_model('transformer', 60, 32, 64, 2, 48, 56, 8, W, num_layers=2, N_enc=2, N_dec=2, d_model=32, d_ff=64, num_att_heads=4, dropout=0.1)
    res['transformer'] = {k: list(v.shape) for k, v in m.state_dict().items()}
    W = co.make_weights('aoa', 60, 32, 32, 16, 48, 56, seed=1)
    m = ref_model('aoa', 60, 32, 32, 16, 48, 56, 8, W, num_layers=2, refine=1, refine_aoa=1, use_ff=0, decoder_type='AoA', use_multi_head=2,
                  num_heads=4, multi_head_scale=1, mean_feats=1, ctx_drop=1, dropout_aoa=0.3)
    res['aoa'] = {k: list(v.shape) for k, v in m.state_dict().items()}
    with open(os.path.join(out_dir, 'state_dict_keys.json'), 'w') as f:
        json.dump({'cfg': cfg, 'keys': res}, f, indent=1, sort_keys=True)
    print('state_dict_keys', {k: len(v) for k, v in res.items()})


def gen_eval_split(out_dir):
    """The reference's eval_split on the stub model / loader of tests/test_eval_cpu.py: loss, predictions and, for sample_n > 1, the
    n_predictions it saves under eval_results/ (one run per sample_n_method)."""
    import json
    sys.path.insert(0, os.path.join(REPO, 'tests'))
    import test_eval_cpu as te
    import captioning.utils.eval_utils as E
    cwd = os.getcwd()
    res = {}
    for name, kwargs in [('n1', te.EVAL_KWARGS)] + [(m, te.eval_n_kwargs(m)) for m in te.N_METHODS]:
        os.chdir(tempfile.mkdtemp(prefix='eval_'))
        loss, preds, _ = E.eval_split(te._StubModel(te.T, te.V1), te._crit, te._StubLoader(10, 4, te.T, te.V1), dict(kwargs))
        res[name] = {'loss': float(loss), 'predictions': [{k: p[k] for k in ('image_id', 'caption', 'perplexity', 'entropy')} for p in preds]}
        if kwargs['sample_n'] > 1:
            _, n_preds = torch.load(os.path.join('eval_results', '.saved_pred_%s_val.pth' % kwargs['id']), weights_only=False)
            res[name]['n_predictions'] = [{k: e[k] for k in ('image_id', 'caption', 'perplexity') if k in e} for e in n_preds]
    os.chdir(cwd)
    with open(os.path.join(out_dir, 'eval_split.json'), 'w') as f:
        json.dump(res, f, indent=1, sort_keys=True)
    print('eval_split', {k: len(v['predictions']) for k, v in res.items()})


def main():
    out_dir = os.path.join(REPO, 'tests', 'golden')
    os.makedirs(out_dir, exist_ok=True)
    scratch = _enter_scratch()
    torch.set_num_threads(os.cpu_count())
    which = sys.argv[1:] or ['small', 'newfc', 'full', 'ciderd', 'rc', 'keys', 'tfm', 'aoa', 'xe', 'dseq', 'pascal', 'penalty', 'b256', 'tfm64', 'aoafull', 'options', 'tfmtrain', 'tfmtrainfull', 'eval']
    if 'small' in which:
        gen_updown_small(out_dir)
    if 'newfc' in which:
        gen_newfc(out_dir)
    if 'penalty' in which:
        gen_updown_penalty(out_dir)
    if 'full' in which:
        gen_updown_full(out_dir)
    if 'ciderd' in which:
        gen_ciderd(out_dir, scratch)
    if 'rc' in which:
        gen_reward_criterion(out_dir)
    if 'dseq' in which:
        gen_decode_sequence(out_dir)
    if 'pascal' in which:
        gen_ciderd_pascal(out_dir, scratch)
    if 'xe' in which:
        gen_xe_struct(out_dir, scratch)            # needs the scratch pickle written by gen_ciderd in the same run
    if 'keys' in which:
        gen_state_dict_keys(out_dir)
    if 'tfm' in which:
        gen_transformer_small(out_dir)
    if 'aoa' in which:
        gen_aoa_small(out_dir)
    if 'options' in which:
        gen_updown_options(out_dir)
    if 'b256' in which:
        gen_updown_b256(out_dir)
    if 'tfm64' in which:
        gen_transformer_b64(out_dir)
    if 'aoafull' in which:
        gen_aoa_scst_full(out_dir, scratch)
    if 'tfmtrain' in which:
        gen_transformer_train(out_dir, scratch)
    if 'tfmtrainfull' in which:
        gen_transformer_train_full(out_dir, scratch)
    if 'eval' in which:
        gen_eval_split(out_dir)


if __name__ == '__main__':
    main()
