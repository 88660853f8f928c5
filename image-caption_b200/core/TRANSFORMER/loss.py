"""Losses of the RL fine-tuning mode -- the reference's shipped default CAPTION_MODEL='RL_Transformer'
(core/config.py:14 -> core/models.py:138-211 -> core/TRANSFORMER/loss.py:31-219) -- for the drop-in PolicyNetwork.

The reference's reward is CIDEr-D / BLEU-4 from pycocoevalcap on decoded strings (loss.py:160-186).  Here the reward is an
INJECTABLE callable `reward_fn(target_ids [B, T] ndarray, sample_ids [B, T] ndarray) -> [B] ndarray`; the default is a
clipped n-gram precision on token ids.  `image_caption_b200.CaptionReward(CIDER_REWARD_WEIGHT, BLEU_REWARD_WEIGHT)` is
the reference's reward computed on the GPU from the ids; a reward_fn with an `on_device(target, sample)` method is
called with the device tensors and its [B] result never leaves the device.  Everything differentiable follows the
reference:
  loss = (1 - w) * CrossEntropy(logits, target[:, 1:]; ignore pad)  +  w * structure loss          (loss.py:53-73)
  structure loss = sum(-log p(sample_t) * mask_t * (score - baseline)) / sum(mask)                  (loss.py:127-158)
with mask_t = 1 for t = 0 and for every position after a non-pad sampled token, and the "baseline" of loss.py:146
((sum over the size-1 score axis - score) / 1 = 0).  Tensors stay on the device (the reference moves the [B, T, V]
logits to the CPU first, models.py:190-193); only a host reward_fn makes the sampled ids cross PCIe.
"""
import numpy as np
import torch
import torch.nn as nn
import torch.nn.functional as F


def ngram_precision_reward(target, sequence, max_n=2, end_idx=2, pad_idx=0):
    """Stand-in sentence reward on token ids: geometric mean of the clipped 1..max_n-gram precisions of the sampled
    caption (cut at <END>) against the reference caption, times a brevity penalty (BLEU's form, no smoothing tricks)."""
    def cut(row):
        out = []
        for tok in row:
            tok = int(tok)
            if tok == end_idx:
                break
            if tok != pad_idx:
                out.append(tok)
        return out

    scores = np.zeros(len(sequence), dtype=np.float32)
    for i, (ref_row, hyp_row) in enumerate(zip(target, sequence)):
        ref, hyp = cut(ref_row), cut(hyp_row)
        if not hyp or not ref:
            continue
        logp = 0.0
        for n in range(1, max_n + 1):
            ref_counts = {}
            for j in range(len(ref) - n + 1):
                g = tuple(ref[j:j + n])
                ref_counts[g] = ref_counts.get(g, 0) + 1
            hit, total = 0, max(len(hyp) - n + 1, 0)
            for j in range(total):
                g = tuple(hyp[j:j + n])
                if ref_counts.get(g, 0) > 0:
                    ref_counts[g] -= 1
                    hit += 1
            logp += np.log((hit + 1e-9) / (total + 1e-9)) / max_n
        bp = 1.0 if len(hyp) >= len(ref) else np.exp(1.0 - len(ref) / len(hyp))
        scores[i] = bp * np.exp(logp)
    return scores


class StructureCriterion(nn.Module):
    """loss.py:98-158 with an injectable reward."""

    def __init__(self, reward_fn=None, entropy_reward_weight=0.0):
        super().__init__()
        self.reward_fn = reward_fn or ngram_precision_reward
        self.entropy_reward_weight = entropy_reward_weight

    def forward(self, output, sequence, target):
        mask = (sequence > 0).to(output)
        mask = torch.cat([mask.new_ones(mask.size(0), 1), mask[:, :-1]], 1)
        if hasattr(self.reward_fn, 'on_device'):
            scores = self.reward_fn.on_device(target, sequence).to(output).view(-1, 1).clone()
        else:
            scores = self.reward_fn(target.cpu().numpy(), sequence.cpu().numpy())
            scores = torch.as_tensor(np.asarray(scores, dtype=np.float32)).to(output).view(-1, 1)
        out = {'reward': scores}
        if self.entropy_reward_weight > 0:
            entropy = -(F.softmax(output, dim=2) * F.log_softmax(output, dim=2)).sum(2).detach()
            entropy = (entropy * mask).sum(1) / mask.sum(1)
            scores = scores + self.entropy_reward_weight * entropy.view(-1, 1)
        picked = output.gather(2, sequence.unsqueeze(2)).squeeze(2)
        baseline = (scores.sum(1, keepdim=True) - scores) / scores.shape[1]
        scores = scores - baseline
        out['loss'] = torch.sum(-picked * mask * scores.view(-1, 1)) / torch.sum(mask)
        return out


class ReinforcementLearningLoss(nn.Module):
    """loss.py:31-76.  The reference's scorer weights (cider / bleu / self-cider) configure pycocoevalcap and are
    accepted for signature compatibility; the reward itself comes from `reward_fn` (pass
    `CaptionReward(cider_reward_weight, bleu_reward_weight)` for the reference's reward).

    `forward` receives only `target`, so the reward scores sample i against the single reference target_i[1:]
    (gts = {i: [target_i]} over the batch: document frequencies from the batch's targets, ref_len = log(B)).  The
    reference's loss.py:160-186 is not part of this port; that reading is the one its signature allows.  The self-CIDEr
    weight stays unused: the arg-max sampler draws one sample per image."""

    def __init__(self, structure_loss_weight, cider_reward_weight=0, bleu_reward_weight=0, entropy_reward_weight=0,
                 self_cider_reward_weight=0, word_to_idx_path=None, pad_idx=0, reward_fn=None):
        super().__init__()
        self.criterion = nn.CrossEntropyLoss(ignore_index=pad_idx)
        self.structure_criterion = StructureCriterion(reward_fn=reward_fn, entropy_reward_weight=entropy_reward_weight)
        self.structure_loss_weight = structure_loss_weight

    def forward(self, model_output, sample_sequence, sample_logprobs, target):
        target = target[:, 1:].clone().long().contiguous().to(model_output.device)
        out = {}
        zero = model_output.new_zeros(())
        if self.structure_loss_weight < 1:
            language_model_loss = self.criterion(model_output.reshape(-1, model_output.size(2)), target.reshape(-1))
        else:
            language_model_loss = zero
        if self.structure_loss_weight > 0:
            structure = self.structure_criterion(sample_logprobs, sample_sequence, target)
        else:
            structure = {'loss': zero, 'reward': zero}
        out['loss'] = (1 - self.structure_loss_weight) * language_model_loss + self.structure_loss_weight * structure['loss']
        out['language_model_loss'] = language_model_loss
        out['structure_loss'] = structure['loss']
        out['reward'] = structure['reward']
        return out
