"""`python main.py train | evaluation | demo` -- same entry points and arguments as the reference's main.py
(main.py:25,156,193).  `fire` is not installable offline, so a small fire-compatible argv shim dispatches
`--beam-size 5` / `--beam_size=5` style flags.  Without the COCO artefacts (data/<MODEL_NAME>/...) the loops run
on synthetic data of the reference's shapes.  Captions are scored on the GPU from their ids (BLEU-1..4, ROUGE-L, CIDEr,
CIDEr-D: image_caption_b200.CaptionScorer); METEOR needs Java and is not computed."""
import os
import sys
import time

import numpy as np
import torch
from torch.utils.data import DataLoader

from core.models import DEVICE, TRANSFORMER, SelfCriticNetwork
from core.TRANSFORMER.model import PrefetchLoader
from core.config import *          # noqa: F401,F403
from core.dataset import IndexedCaptions, SyntheticCaptionDataset, TestDataset, TrainDataset
from core.utils import save_pickle, write_scores
from image_caption_b200.metrics import MAX_VOCAB, CaptionReward, CaptionScorer     # registered by core.models

MODEL = None


def _model():
    global MODEL
    if MODEL is None:
        # the reference builds it at import time (main.py:19-22)
        MODEL = TRANSFORMER() if CAPTION_MODEL == 'Transformer' else SelfCriticNetwork()
    return MODEL


def _dataset(with_captions, n_images, split='train'):
    """The split's COCO artefacts (data/<MODEL_NAME>/<split>/, utils.py:32-64) when they exist, else synthetic data of
    the same shapes."""
    if os.path.exists(os.path.join(DATA_PATH, split, f'{split}.captions.pkl')):
        return (TrainDataset if with_captions else TestDataset)(data_path=DATA_PATH, split=split)
    seed = {'train': 1234, 'valid': 4321}.get(split, 999)
    return SyntheticCaptionDataset(n_images, NUM_OBJECT, ENCODE_DIM_FEATURES, ENCODE_DIM_POSITIONS, MAX_LENGTH + 2,
                                   _model().num_vocab, with_captions=with_captions, seed=seed)


def _scorer(ds, num_vocab):
    """CaptionScorer over the split's reference captions (None when the vocabulary is too large for the id packing)."""
    if num_vocab > MAX_VOCAB:
        print(f'[scores] a vocabulary of {num_vocab} words is above {MAX_VOCAB}: captions are not scored')
        return None
    return CaptionScorer(ds.data['captions'], ds.data['image_idxs'], num_vocab, DEVICE)


def _score(scorer, id_batches, n_img):
    """Scores of the caption ids decoded per image ([(image numbers, id rows)]) -> (corpus dict, seconds)."""
    t0 = time.time()
    width = id_batches[0][1].shape[1]
    ids = torch.zeros(n_img, width, dtype=torch.long, device=DEVICE)
    for idxs, rows in id_batches:
        ids[torch.as_tensor(idxs).to(DEVICE, torch.long)] = rows.to(DEVICE, torch.long)
    _, corpus = scorer.score(ids, torch.arange(n_img, device=DEVICE))
    return corpus, time.time() - t0


def _scores_line(corpus):
    return '  '.join(f'{k} {v:.4f}' for k, v in corpus.items())


def _collate_idx(items):
    cols = list(zip(*items))
    return tuple(torch.as_tensor(np.asarray(c)) for c in cols)


def train(num_images=64, max_iters=None, region_cache=REGION_CACHE, reward='ngram'):
    """main.py:25-153 without TensorBoard: train_step per batch, train/valid loss every 100 iterations, validation
    captions, their scores (valid_scores.txt) and a checkpoint per epoch.  With `region_cache` (default) both splits'
    region features are packed into HBM once and the loaders yield (image number, caption) only.
    `reward` (RL_Transformer): 'ngram' = the clipped n-gram precision stand-in, 'cider' = the reference's
    CIDER_REWARD_WEIGHT * CIDEr-D + BLEU_REWARD_WEIGHT * BLEU-4 computed on the GPU."""
    if reward not in ('ngram', 'cider'):
        raise ValueError(f"--reward must be 'ngram' or 'cider', not {reward!r}")
    model = _model()
    if reward == 'cider':
        if not isinstance(model, SelfCriticNetwork):
            raise ValueError("--reward cider needs CAPTION_MODEL = 'RL_Transformer' (the Transformer has no reward)")
        model.loss.structure_criterion.reward_fn = CaptionReward(CIDER_REWARD_WEIGHT, BLEU_REWARD_WEIGHT)
    model_dir = os.path.join(OUTPUT_PATH, 'model/')
    target_dir = os.path.join(DATA_PATH, f'valid/{OUTPUT_NAME}/')
    os.makedirs(model_dir, exist_ok=True)
    os.makedirs(target_dir, exist_ok=True)
    train_ds = _dataset(True, num_images, 'train')
    valid_ds = _dataset(True, max(num_images // 4, BATCH_SIZE // 5 + 1), 'valid')
    region_cache = region_cache and hasattr(model, 'cache_regions')     # the RL wrapper feeds tensors, as the reference
    if region_cache:
        t_cache = model.cache_regions(train_ds.data['features'], train_ds.data['positions'])
        v_cache = model.cache_regions(valid_ds.data['features'], valid_ds.data['positions'])
        print(f'[train] region cache: {(t_cache.nbytes + v_cache.nbytes) / 2**20:.1f} MiB in HBM')
        train_loader = DataLoader(IndexedCaptions(train_ds), batch_size=BATCH_SIZE, shuffle=True,
                                  collate_fn=_collate_idx)
        valid_loader = DataLoader(IndexedCaptions(valid_ds), batch_size=BATCH_SIZE, shuffle=False,
                                  collate_fn=_collate_idx)
        step = lambda b: model.train_step_cached(t_cache, b[0], b[1])                                     # noqa: E731
        loss_of = lambda cache, b: model.compute_loss_cached(cache, b[0], b[1])                           # noqa: E731
        caption_of = lambda b: (model.generate_caption_ids_cached(v_cache, b[0])[0], b[0])                # noqa: E731
    else:
        t_cache = v_cache = None
        train_loader = DataLoader(train_ds, batch_size=BATCH_SIZE, shuffle=True)
        valid_loader = DataLoader(valid_ds, batch_size=BATCH_SIZE, shuffle=False)
        step = lambda b: model.train_step(b[0], b[1], b[2])                                               # noqa: E731
        loss_of = lambda cache, b: model.compute_loss(b[0], b[1], b[2])                                   # noqa: E731
        caption_of = lambda b: (model.generate_caption_ids(b[0], b[1])[0], b[3])                          # noqa: E731
    eval_t, eval_v = next(iter(train_loader)), next(iter(valid_loader))
    valid_scorer = _scorer(valid_ds, model.num_vocab)
    it = 0
    for epoch in range(1, NUM_EPOCH + 1):
        print(f'Epoch {epoch}')
        model.model.train()
        for batch in train_loader:
            step(batch)
            it += 1
            if it % 100 == 0 or max_iters:
                model.model.eval()
                tl, vl = loss_of(t_cache, eval_t)['loss'], loss_of(v_cache, eval_v)['loss']
                model.model.train()
                print(f'  iter {it} loss {float(model.last_loss):.4f}  train {float(tl):.4f}  valid {float(vl):.4f}')
            if max_iters and it >= max_iters:
                break
        model.model.eval()
        valid_caption, id_batches = [''] * valid_ds.len_image, []
        for batch in valid_loader:
            ids, idxs = caption_of(batch)
            id_batches.append((idxs, ids))
            for idx, caption in zip(idxs, model.decode_captions(ids.cpu().numpy())):
                valid_caption[int(idx)] = caption
        save_pickle(valid_caption, os.path.join(target_dir, 'valid.candidate.captions.pkl'))
        if valid_scorer is not None:
            corpus, dt = _score(valid_scorer, id_batches, valid_ds.len_image)
            print(f'  valid scores ({dt:.2f}s): {_scores_line(corpus)}')
            write_scores(corpus, target_dir, epoch, 'valid')
        model.save(path=os.path.join(model_dir, f'model_{epoch}.pt'))
        model.save_optimizer(path=os.path.join(model_dir, f'optimizer_{epoch}.pt'))
        if t_cache is not None:
            t_cache.check()
            v_cache.check()
        if max_iters and it >= max_iters:
            break


def evaluation(split='test', epoch=90, beam_size=None, num_images=64, region_cache=REGION_CACHE):
    model = _model()
    model_path = os.path.join(OUTPUT_PATH, f'model/model_{epoch}.pt')
    if os.path.exists(model_path):
        model.load(path=model_path)
    else:
        print(f'[evaluation] {model_path} not found: using the current (random-init) weights')
        model.model.eval()
    ds = _dataset(False, num_images, split)
    captions_out, id_batches = [''] * ds.len_image, []
    t0 = time.time()
    region_cache = region_cache and hasattr(model, 'cache_regions')
    if region_cache:        # every image once (the reference decodes it once per ground-truth caption, dataset.py:36-43)
        cache = model.cache_regions(ds.data['features'], ds.data['positions'])
        loader = DataLoader(IndexedCaptions(ds, with_captions=False, unique_images=True), batch_size=BATCH_SIZE,
                            shuffle=False, collate_fn=_collate_idx)
        for (idxs,) in loader:
            ids, _ = model.generate_caption_ids_cached(cache, idxs, beam_size=beam_size)
            id_batches.append((idxs, ids))
            captions = model.decode_captions(ids.cpu().numpy())
            for i, idx in enumerate(idxs):
                captions_out[int(idx)] = captions[i]
        cache.check()
    else:
        # host -> device copies of batch i + 1 run on a copy stream while batch i decodes
        loader = DataLoader(ds, batch_size=BATCH_SIZE, shuffle=False, pin_memory=True)
        for features, positions, idxs in PrefetchLoader(loader, DEVICE):
            ids, _ = model.generate_caption_ids(object_features=features, position_features=positions,
                                                beam_size=beam_size)
            id_batches.append((idxs, ids))
            captions = model.decode_captions(ids.cpu().numpy())
            for i, idx in enumerate(idxs.tolist()):
                captions_out[int(idx)] = captions[i]
    dt = time.time() - t0
    target_dir = os.path.join(DATA_PATH, f'{split}/{OUTPUT_NAME}/')
    os.makedirs(target_dir, exist_ok=True)
    save_pickle(captions_out, os.path.join(target_dir, f'{split}.candidate.captions.pkl'))
    print(f'[evaluation] {len(captions_out)} captions in {dt:.2f}s ({len(captions_out) / dt:.1f} captions/s); '
          f'METEOR needs Java and is out of scope')
    # the references: the split's caption file, or the synthetic split generated with its captions (same seed, so the
    # same images)
    scorer = _scorer(ds if 'captions' in ds.data else _dataset(True, num_images, split), model.num_vocab)
    if scorer is not None:
        corpus, dt = _score(scorer, id_batches, ds.len_image)
        print(f'[evaluation] scores ({dt:.2f}s): {_scores_line(corpus)}')
        write_scores(corpus, target_dir, epoch, split)
    return captions_out


def demo(image_path=None, beam_size=None, epoch=90, save_img=False, max_obj=False, features_path=None, num_samples=None,
         temperature=1.0, seed=None):
    """The reference runs YOLOv5 + ResNet-101 on `image_path` first (main.py:195-197); offline, pass
    `--features-path file.pt` holding {'features': [R,2048], 'positions': [R,84]} or omit it for a synthetic image.
    `--num-samples N [--temperature T] [--seed S]` prints N captions sampled from the model instead."""
    model = _model()
    start = time.time()
    if features_path:
        blob = torch.load(features_path)
        feature, position = blob['features'].unsqueeze(0), blob['positions'].unsqueeze(0)
    else:
        ds = _dataset(False, 1)                # TestDataset (COCO artefacts) or SyntheticCaptionDataset: first image
        feature, position = (torch.as_tensor(np.asarray(x)).unsqueeze(0) for x in ds[0][:2])
    model_path = os.path.join(OUTPUT_PATH, f'model/model_{epoch}.pt')
    if os.path.exists(model_path):
        model.load(path=model_path)
    else:
        model.model.eval()
    if num_samples is not None:
        ids, logp = model.sample_caption_ids(feature, position, num_samples=int(num_samples),
                                             temperature=float(temperature), seed=seed)
        captions = model.decode_captions(ids[0].cpu().numpy())
        for caption, lp in zip(captions, logp[0].sum(dim=1).tolist()):
            print(f'Sampled Caption: {caption}  (log-probability {lp:.3f})')
        print('Spending Time:', time.time() - start)
        return captions
    caption, attention_list = model.generate_caption(object_features=feature, position_features=position,
                                                     beam_size=beam_size)
    print('Generated Caption:', caption[0])
    print('Spending Time:', time.time() - start)
    return caption[0]


def _fire(argv):
    """fire.Fire() subset: `cmd --flag value`, `--flag=value`, dashes or underscores, ints/None/bools parsed."""
    cmds = {'train': train, 'evaluation': evaluation, 'demo': demo}
    if not argv or argv[0] not in cmds:
        print('usage: main.py {train|evaluation|demo} [--flag value ...]')
        return 2

    def parse(v):
        if v in ('None', 'none'):
            return None
        if v in ('True', 'False'):
            return v == 'True'
        try:
            return int(v)
        except ValueError:
            return v

    kwargs, i, args = {}, 1, argv
    while i < len(args):
        a = args[i]
        assert a.startswith('--'), f'unexpected argument {a}'
        if '=' in a:
            k, v = a[2:].split('=', 1)
            i += 1
        elif i + 1 < len(args) and not args[i + 1].startswith('--'):
            k, v = a[2:], args[i + 1]
            i += 2
        else:
            k, v = a[2:], 'True'
            i += 1
        kwargs[k.replace('-', '_')] = parse(v)
    cmds[argv[0]](**kwargs)
    return 0


if __name__ == '__main__':
    sys.exit(_fire(sys.argv[1:]))
