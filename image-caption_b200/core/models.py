"""Drop-in for the caption-model wrapper of the reference's core/models.py:18-135 (`MODEL_init`, `TRANSFORMER`):
same methods, same argument meaning.  train_step runs the fused zero_grad/forward/backward/Adam sequence of
libicap (core/models.py:115-126); inputs arrive as CPU tensors from a DataLoader and are moved to DEVICE here."""
import os
import pickle

import torch
import torch.nn as nn

from core.TRANSFORMER.model import Transformer
from core.TRANSFORMER.model_RL import PolicyNetwork
from core.TRANSFORMER.loss import ReinforcementLearningLoss
from core.config import *          # noqa: F401,F403  (the reference does the same, models.py:12)
from core.utils import decode_captions


# keyword of the model constructors -> the core/config.py constant of the same name in upper case
_CONFIG_KEYWORDS = ("encode_dim_positions", "encode_dim_features", "encode_input_size", "encode_q_k_dim", "encode_v_dim",
                    "encode_hidden_size", "encode_num_blocks", "encode_num_heads", "dim_word_embedding",
                    "decode_input_size", "decode_q_k_dim", "decode_v_dim", "decode_hidden_size", "decode_num_blocks",
                    "decode_num_heads", "dropout", "encode_mask", "pad_idx", "split_position", "split_image_objects")


def _model_kwargs(num_vocab):
    """Constructor arguments of Transformer / PolicyNetwork taken from core/config.py (the reference spells the same 24
    keywords out at both call sites, models.py:68-94 and :141-166)."""
    cfg = globals()
    kw = {name: cfg[name.upper()] for name in _CONFIG_KEYWORDS}
    kw.update(num_vocab=num_vocab, max_length=MAX_LENGTH + 2, device=DEVICE,
              move_first_image_feature=MOVE_FIRST_IMAGE_FAETURE)        # (sic) the constant's spelling in config.py
    return kw


class MODEL_init:

    def __init__(self):
        if os.path.exists(WORD_TO_IDX_PATH):
            word_to_idx = pickle.load(open(WORD_TO_IDX_PATH, 'rb'))
        else:   # offline / synthetic mode: the reference's special tokens (preprocess.py:303) + numbered words
            word_to_idx = {'<NULL>': 0, '<START>': 1, '<END>': 2, '<UNK>': 3}
            word_to_idx.update({f'w{i}': i for i in range(4, SYNTHETIC_VOCAB)})
        self.num_vocab = len(word_to_idx)
        self.idx_to_word = {i: w for w, i in word_to_idx.items()}
        self.model = nn.Module()

    def train_step(self):
        raise NotImplementedError

    def compute_loss(self):
        raise NotImplementedError

    def generate_caption_ids(self, object_features, position_features, beam_size=None):
        """generate_caption without the decoding: (caption id rows on the device, attention list or None), the
        input of image_caption_b200.CaptionScorer."""
        if beam_size in [None, 1]:
            return self.model.generate_caption_vector(object_features=object_features.to(DEVICE),
                                                      position_features=position_features.to(DEVICE))
        elif isinstance(beam_size, int) and beam_size > 1:
            return self.model.beam_search(object_features=object_features.to(DEVICE),
                                          position_features=position_features.to(DEVICE), beam_size=beam_size), None
        else:
            assert isinstance(beam_size, int)
            assert beam_size > 1 or beam_size in [None, 1]

    def generate_caption(self, object_features, position_features, beam_size=None):
        caption_vector, attention_list = self.generate_caption_ids(object_features, position_features, beam_size)
        return self.decode_captions(caption_vector.cpu().numpy()), attention_list

    def sample_caption_ids(self, object_features, position_features, num_samples=1, temperature=1.0, seed=None):
        """num_samples captions per image drawn from the model (Transformer.sample_captions): (ids [B, n, L] and their
        log-probabilities [B, n, L - 1] on the device)."""
        return self.model.sample_captions(object_features.to(DEVICE), position_features.to(DEVICE),
                                          num_samples=num_samples, temperature=temperature, seed=seed)

    def sample_caption_ids_cached(self, cache, image_idxs, num_samples=1, temperature=1.0, seed=None):
        return self.model.sample_captions(cache.batch(image_idxs), None, num_samples=num_samples,
                                          temperature=temperature, seed=seed)

    def generate_caption_ids_nbest(self, object_features, position_features, beam_size=5, n_best=None,
                                   length_penalty=0.0):
        """The n_best captions per image of the beam search that stops at <END> (Transformer.beam_search_nbest): (ids
        [B, n, L], log-probabilities [B, n], lengths [B, n]) on the device, best first."""
        return self.model.beam_search_nbest(object_features.to(DEVICE), position_features.to(DEVICE),
                                            beam_size=beam_size, n_best=n_best, length_penalty=length_penalty)

    def generate_caption_ids_nbest_cached(self, cache, image_idxs, beam_size=5, n_best=None, length_penalty=0.0):
        return self.model.beam_search_nbest(cache.batch(image_idxs), None, beam_size=beam_size, n_best=n_best,
                                            length_penalty=length_penalty)

    def decode_captions(self, caption_vector):
        return decode_captions(captions=caption_vector, index_to_word=self.idx_to_word)

    def save(self, path):
        torch.save(self.model.state_dict(), path)           # the reference's checkpoint format, unchanged

    def load(self, path):
        state_dict = torch.load(path, map_location=DEVICE)
        self.model.load_state_dict(state_dict)
        self.model.eval()

    # resume support (the reference cannot resume: it never saves the optimizer, models.py:62-63)
    def save_optimizer(self, path):
        torch.save(self.model.optimizer_state_dict(), path)

    def load_optimizer(self, path):
        self.model.load_optimizer_state_dict(torch.load(path, map_location="cpu"))

    def preprocess(self, image_path, save_img=False, max_obj=False):
        raise NotImplementedError("image feature extraction (YOLOv5 + ResNet-101, core/preprocess.py:91-138) is the "
                                  "stage BEFORE the hot path and needs pretrained weights that are not available "
                                  "offline; pass precomputed features (SURVEY.md §8f #4)")


class TRANSFORMER(MODEL_init):

    def __init__(self):
        super(TRANSFORMER, self).__init__()
        self.model = Transformer(output_name=OUTPUT_NAME, **_model_kwargs(self.num_vocab)).to(DEVICE)
        # Adam(lr=LEARNING_RATE) state lives in the engine's flat buffers (models.py:111-113)
        self.last_loss = None

    def train_step(self, batch_features, batch_positions, batch_captions):
        self.last_loss = self.model.train_step_fused(batch_features, batch_positions, batch_captions, lr=LEARNING_RATE)

    def compute_loss(self, object_features, position_features, target_caption):
        with torch.no_grad():
            return self.model(object_features=object_features.to(DEVICE),
                              position_features=position_features.to(DEVICE),
                              target_caption=target_caption.to(DEVICE))

    # ---- device-resident region cache (SURVEY.md 8f #2): batches are named by image number, nothing else crosses PCIe
    def cache_regions(self, features, positions, chunk_images=1024):
        """features [n_img, R, 2048] / positions [n_img, R, Dp] of a whole split (ndarray, memmap or CPU tensor) ->
        RegionCache in HBM, packed for the encoder in the model's compute dtype."""
        from image_caption_b200 import RegionCache
        return RegionCache(self.model, features, positions, chunk_images=chunk_images)

    def train_step_cached(self, cache, batch_image_idxs, batch_captions):
        self.last_loss = self.model.train_step_fused(cache.batch(batch_image_idxs), None, batch_captions,
                                                     lr=LEARNING_RATE)

    def compute_loss_cached(self, cache, image_idxs, target_caption):
        with torch.no_grad():
            return self.model(object_features=cache.batch(image_idxs), position_features=None,
                              target_caption=target_caption.to(DEVICE))

    def generate_caption_ids_cached(self, cache, image_idxs, beam_size=None):
        batch = cache.batch(image_idxs)
        if beam_size in [None, 1]:
            return self.model.generate_caption_vector(batch, None)
        assert isinstance(beam_size, int) and beam_size > 1
        return self.model.beam_search(batch, None, beam_size=beam_size), None

    def generate_caption_cached(self, cache, image_idxs, beam_size=None):
        caption_vector, attention_list = self.generate_caption_ids_cached(cache, image_idxs, beam_size)
        return self.decode_captions(caption_vector.cpu().numpy()), attention_list


class SelfCriticNetwork(MODEL_init):
    """core/models.py:138-211: PolicyNetwork (logits out) + ReinforcementLearningLoss, torch.optim.Adam on the flat
    parameter views.  `reward_fn(target_ids, sample_ids) -> [B]` is injectable (default: clipped n-gram precision);
    `image_caption_b200.CaptionReward(CIDER_REWARD_WEIGHT, BLEU_REWARD_WEIGHT)` is the reference's CIDEr-D + BLEU-4
    reward on the GPU.  Forward, the log-softmax/arg-max "sampler" and the whole backward run on libicap."""

    def __init__(self, reward_fn=None):
        super(SelfCriticNetwork, self).__init__()
        self.model = PolicyNetwork(**_model_kwargs(self.num_vocab)).to(DEVICE)
        g = globals()
        self.loss = ReinforcementLearningLoss(word_to_idx_path=WORD_TO_IDX_PATH,
                                              pad_idx=PAD_IDX,
                                              structure_loss_weight=g.get('STRUCTURE_LOSS_WEIGHT', 0.5),
                                              cider_reward_weight=g.get('CIDER_REWARD_WEIGHT', 1),
                                              bleu_reward_weight=g.get('BLEU_REWARD_WEIGHT', 1),
                                              entropy_reward_weight=g.get('ENTROPY_REWARD_WEIGHT', 1),
                                              self_cider_reward_weight=g.get('SELF_CIDER_REWARD_WEIGHT', 1),
                                              reward_fn=reward_fn)
        self.optimizer = torch.optim.Adam((p for p in self.model.parameters() if p.requires_grad), lr=LEARNING_RATE)
        self.last_loss = None

    def _loss(self, features, positions, captions):
        model_output = self.model(object_features=features.to(DEVICE), position_features=positions.to(DEVICE),
                                  target_caption=captions.to(DEVICE))
        sample_sequence, sample_logprobs = self.model.sample(output=model_output)
        return self.loss(model_output=model_output, sample_sequence=sample_sequence, sample_logprobs=sample_logprobs,
                         target=captions)

    def train_step(self, batch_features, batch_positions, batch_captions):
        self.optimizer.zero_grad()
        loss = self._loss(batch_features, batch_positions, batch_captions)['loss'].mean()
        loss.backward()
        self.optimizer.step()
        self.last_loss = loss.detach()

    def compute_loss(self, object_features, position_features, target_caption):
        with torch.no_grad():
            return self._loss(object_features, position_features, target_caption)
