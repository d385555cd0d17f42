"""One DAMSM pretraining step (reference pretrain_damsm.py:110-134) around the native losses.

Only the losses are the hot path of this repository; the text encoder and the two trainable heads of the image
encoder are ordinary PyTorch modules (cuDNN LSTM, 1x1 convolution, linear) kept here with the REFERENCE'S
state-dict names, so ``RNNEncoder.pkl`` / the head entries of ``CNNEncoder.pkl`` (trainers/trainer.py:109-127)
load unchanged:

  TextEncoder   <-> networks/rnn_encoder.py:11-96   keys  embedding.weight, rnn.weight_ih_l0, rnn.weight_hh_l0,
                                                          rnn.bias_ih_l0, rnn.bias_hh_l0 (+ *_reverse)
  RegionHeads   <-> networks/cnn_encoder.py:54-64   keys  emb_features.weight [256,768,1,1], emb_cnn_code.weight
                                                          [256,2048], emb_cnn_code.bias
The frozen Inception-v3 trunk (cnn_encoder.py:37-53,73-96) is out of scope; RegionHeads takes its two outputs
(Mixed_6e features [B,768,17,17] and the pooled [B,2048] vector), which the benchmark synthesises.

DamsmPretrainStep.step() does what the loop body does, in the same order: encoders -> WordsLoss + SentenceLoss ->
zero_grad / backward -> clip_grad_norm_(RNN, 0.25) -> Adam(lr 2e-3, betas (0.5, 0.999)).  Nothing in it
synchronises with the host (packed attention maps, device-resident lengths / class ids, loss returned as a
tensor), so with fixed-length captions the whole step is CUDA-graph capturable (agb_native/graph.py).
"""
from __future__ import annotations

from typing import Optional, Tuple

import torch
import torch.distributed as dist
from torch import nn
from torch.nn.utils import clip_grad_norm_
from torch.nn.utils.rnn import pack_padded_sequence, pad_packed_sequence

from ..losses.damsm_loss import DAMSMLoss
from ..networks.region_head import region_head


class TextEncoder(nn.Module):
    """bidirectional LSTM text encoder with the reference's constructor defaults and state-dict names
    (networks/rnn_encoder.py:11-96)"""

    def __init__(self, vocabsize: int, embdim: int = 300, dropprob: float = 0.5, nhidden: int = 128, nlayers: int = 1,
                 bidirectional: bool = True):
        super().__init__()
        self.vocabsize, self.embdim, self.dropprob, self.nlayers = vocabsize, embdim, dropprob, nlayers
        self.bidirectional = bidirectional
        self.ndirections = 2 if bidirectional else 1
        self.nhidden = nhidden // self.ndirections
        self.embedding = nn.Embedding(vocabsize, embdim)
        self.dropout = nn.Dropout(dropprob)
        # the reference passes dropout=dropprob with nlayers=1 (a no-op that only warns); 0 here for the same maths
        self.rnn = nn.LSTM(input_size=embdim, hidden_size=self.nhidden, num_layers=nlayers, batch_first=True,
                           dropout=dropprob if nlayers > 1 else 0.0, bidirectional=bidirectional)
        self.embedding.weight.data.uniform_(-0.1, 0.1)                     # rnn_encoder.py:48-50

    def forward(self, captions: torch.Tensor, caption_lengths, fixed_length: bool = False
                ) -> Tuple[torch.Tensor, torch.Tensor]:
        """captions [B,T] int64, caption_lengths [B] -> (word_embs [B,nhidden,T] as a transposed view of [B,T,nhidden],
        sent_embs [B,nhidden])                                              (rnn_encoder.py:69-96)
        fixed_length: every caption fills the whole row (the synthetic bedroom captions: 7 tokens) -> no packing,
        no .tolist() host sync; same result as the packed path."""
        x = self.dropout(self.embedding(captions))
        if fixed_length:
            out, (hidden, _) = self.rnn(x)
        else:
            lens = caption_lengths.detach().cpu().tolist()                 # the reference syncs here too (:84)
            packed = pack_padded_sequence(x, lengths=lens, batch_first=True, enforce_sorted=False)
            out, (hidden, _) = self.rnn(packed)
            out = pad_packed_sequence(out, batch_first=True)[0]
        word_embs = out.transpose(1, 2)
        sent_embs = hidden.transpose(0, 1).contiguous().view(-1, self.ndirections * self.nhidden)
        return word_embs, sent_embs


class RegionHeads(nn.Module):
    """the two trainable heads of the reference's CNNEncoder (cnn_encoder.py:54-64,98-102)"""

    def __init__(self, out_dim: int = 256, native: bool = True):
        super().__init__()
        self.out_dim = out_dim
        self.native = native           # emb_features on tcgen05 (networks/region_head.py) instead of an fp32 cuDNN conv
        self.emb_features = nn.Conv2d(768, out_dim, kernel_size=1, stride=1, padding=0, bias=False)   # Layers.conv1x1
        self.emb_cnn_code = nn.Linear(2048, out_dim)
        self.emb_features.weight.data.uniform_(-0.1, 0.1)                  # cnn_encoder.py:60-64
        self.emb_cnn_code.weight.data.uniform_(-0.1, 0.1)

    def forward(self, mixed_6e: torch.Tensor, pooled: torch.Tensor) -> Tuple[torch.Tensor, torch.Tensor]:
        """mixed_6e [B,768,17,17], pooled [B,2048] -> (region features [B,256,17,17], cnn_code [B,256])"""
        if self.native and mixed_6e.is_cuda:
            return region_head(mixed_6e, self.emb_features.weight), self.emb_cnn_code(pooled)
        return self.emb_features(mixed_6e), self.emb_cnn_code(pooled)


class DamsmPretrainStep:
    def __init__(self, vocab_size: int, device, emb_dim: int = 256, lr: float = 2e-3, rnn_grad_clip: float = 0.25,
                 math: str = "auto", process_group=None, fixed_length: bool = True, max_words: Optional[int] = None,
                 seed: int = 0, native_head: bool = True):
        torch.manual_seed(seed)
        self.device = torch.device(device)
        self.rnn = TextEncoder(vocabsize=vocab_size, nhidden=emb_dim).to(self.device)       # pretrain_damsm.py:67
        self.heads = RegionHeads(out_dim=emb_dim, native=native_head).to(self.device)        # :68 (trainable part)
        params = list(self.rnn.parameters()) + [p for p in self.heads.parameters() if p.requires_grad]
        # capturable: the step counter lives on the device, so the optimiser step can sit inside a CUDA graph
        self.optimizer = torch.optim.Adam(params, lr=lr, betas=(0.5, 0.999), capturable=True)   # :74
        self.params = params
        self.rnn_grad_clip = rnn_grad_clip
        self.group = process_group
        self.fixed_length = fixed_length
        self.loss = DAMSMLoss(self.device, math=math, process_group=process_group, att_maps=None, max_words=max_words)

    def modules(self):
        """what `_save_weights` pickles (trainer.py:109-115): {'RNNEncoder': state_dict, heads of 'CNNEncoder'}"""
        return {"RNNEncoder": self.rnn, "CNNEncoder": self.heads}

    def step(self, captions, lengths, class_ids, mixed_6e, pooled, labels) -> torch.Tensor:
        """one optimiser step; returns wloss + sloss (a device tensor: no host sync; pretrain_damsm.py:134 logs
        loss.item(), which is left to the caller).  class_ids: int32 device tensor, numpy array or None."""
        region_features, cnn_code = self.heads(mixed_6e, pooled)                             # :120
        word_embs, sent_embs = self.rnn(captions, lengths, fixed_length=self.fixed_length)   # :124
        self.optimizer.zero_grad(set_to_none=False)                                          # :126
        wloss, sloss, _ = self.loss.get_losses(region_features, cnn_code, word_embs, sent_embs, labels, lengths,
                                               class_ids)                                    # :128-129
        loss = wloss + sloss
        loss.backward()                                                                      # :131
        if self.group is not None and dist.get_world_size(self.group) > 1:
            # data parallel over the ranks: the loss on every rank is the loss of the GLOBAL batch and each rank
            # holds the gradient of its own samples' contribution -> sum over ranks
            flat = torch.cat([p.grad.reshape(-1) for p in self.params])
            dist.all_reduce(flat, group=self.group)
            o = 0
            for p in self.params:
                p.grad.copy_(flat[o:o + p.numel()].view_as(p))
                o += p.numel()
        clip_grad_norm_(self.rnn.parameters(), self.rnn_grad_clip)                           # :132
        self.optimizer.step()                                                                # :133
        return loss.detach()
