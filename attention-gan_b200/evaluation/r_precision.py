"""R-precision of a trained DAMSM, scored on the B200 kernels.

The AttnGAN family evaluates text-to-image models by R-precision: every image is scored against 100 captions,
its own and 99 drawn at random from other classes, and a hit is an image whose own caption scores highest.  Two
scores are available:

  ``DAMSMScorer.sentence``  cosine of the DAMSM global vectors (cnn_code, sent_emb): AttnGAN's published definition
  ``DAMSMScorer.words``     DAMSM's word-level matching score m[b, i] (losses/words_loss.py:77-79), the score that
                            WordsLoss is trained on

Both evaluate only the listed pairs (agb_damsm_cand_fwd / agb_sent_cos_cand_fwd), not the dense N x N matrix.

    scorer = DAMSMScorer(device, gamma1=4.0, gamma2=5.0, math="f16x2")
    cands = mismatched_candidates(class_ids, n_mismatched=99, seed=0)       # [N, 100], column 0 = own caption
    hits = r_precision(scorer.words(img_features, words_emb, cap_lens, cands), r=1)

Text-to-image R-precision ranks every caption against its own image and 99 images of other classes:
``by="caption"`` takes [Nc, K] image indices per caption (column 0 = own image).  Any other list of
(image, caption) pairs is scored by ``words_pairs`` / ``sentence_pairs`` (agb_damsm_pairs_fwd /
agb_sent_cos_pairs_fwd), which can also return the pairs' attention maps.
"""
from __future__ import annotations

from typing import Optional

import numpy as np
import torch

from ..agb_native import native, ops, torch_ops
from ..losses.damsm_core import as_device_i32, chunk_pairs, pair_index

_CAND_MATH = ("f16", "bf16", "f16x2")


class DAMSMScorer:
    """Scores images against per-image lists of candidate captions.  Inference only: the inputs are detached and
    no autograd graph is recorded.  Every input must be on the scorer's CUDA device (there is no CPU fallback);
    cap_lens and the candidate lists may also be host arrays.

    math             "f16x2" (split precision: m as accurate as fp32 arithmetic), "f16" or "bf16"
    workspace_bytes  bound on the workspace of one ``words`` launch; larger image sets are scored in chunks of
                     images, with results identical to one launch
    """

    def __init__(self, device, gamma1: float = 4.0, gamma2: float = 5.0, math: str = "f16x2",
                 workspace_bytes: int = 4 << 30, eps: float = 1e-8):
        if math not in _CAND_MATH:
            raise ValueError(f"math must be one of {_CAND_MATH} (candidate scores run on the tensor cores)")
        self.device = torch.device(device)
        self.gamma1 = float(gamma1)
        self.gamma2 = float(gamma2)
        self.math = native.MATH_NAMES[math]
        self.workspace_bytes = int(workspace_bytes)
        self.eps = float(eps)

    def _chunk_images(self, N: int, K: int, T: int, D: int, R: int, ws_bytes=ops.damsm_cand_workspace_bytes) -> int:
        """the most images whose candidate workspace fits workspace_bytes (the size grows with the image count)"""
        if ws_bytes(1, K, T, D, R, self.math) == 0:
            raise native.NativeError(f"candidate DAMSM shape K={K} T={T} D={D} R={R} is unsupported")
        lo, hi = 0, min(N, 65535)
        while lo < hi:
            mid = (lo + hi + 1) // 2
            nb = ws_bytes(mid, K, T, D, R, self.math)
            if 0 < nb <= self.workspace_bytes:
                lo = mid
            else:
                hi = mid - 1
        if lo == 0:
            need = ws_bytes(1, K, T, D, R, self.math)
            raise native.NativeError(f"workspace_bytes={self.workspace_bytes} is below the {need} bytes one image needs")
        return lo

    def _chunk_pairs(self, N: int, Nc: int, P: int, T: int, D: int, R: int, ws_bytes) -> int:
        """the most pairs whose workspace fits workspace_bytes (the size grows with the pair count)"""
        return chunk_pairs(N, Nc, P, T, D, R, self.math, ws_bytes, self.workspace_bytes)

    @staticmethod
    def _pairs(image_idx, caption_idx, device):
        return pair_index(image_idx, caption_idx, device)

    @staticmethod
    def _by_caption(candidates, Nc: int, device):
        """[Nc,K] image indices per caption -> the pair list in row-major order"""
        cand = as_device_i32(candidates, device)
        if cand.dim() != 2 or cand.shape[0] != Nc:
            raise ValueError(f'candidates must be [Nc={Nc}, K] image indices with by="caption", got {tuple(cand.shape)}')
        K = cand.shape[1]
        caps = torch.arange(Nc, dtype=torch.int32, device=device).repeat_interleave(K)
        return cand.reshape(-1), caps, K

    def words_pairs(self, img_features: torch.Tensor, words_emb: torch.Tensor, cap_lens, image_idx, caption_idx,
                    att_maps: bool = False):
        """The DAMSM word-level score of an arbitrary pair list: image_idx, caption_idx [P] (numpy, int64 or int32;
        any order, duplicates allowed).  img_features [N,D,h,w] or [N,D,R], words_emb [Nc,D,T], cap_lens [Nc].
        Returns m [P] fp32, m[p] = the score of image image_idx[p] and caption caption_idx[p], bit for bit what
        WordsLoss's similarity matrix holds for that pair in the same math mode; NaN for an index out of range or a
        caption of length 0.  att_maps=True also returns the pairs' region-attention maps [P,T,h,w] (or [P,T,R])
        fp32, words_loss.py:63's beta: rows t >= the caption's length are 0, every row of an invalid pair is NaN.
        Lists whose workspace exceeds workspace_bytes are scored in contiguous chunks of pairs, with identical
        results."""
        ops.require_cuda(img_features, words_emb)
        img = img_features.detach()
        map_shape = img.shape[2:]
        img = img.reshape(img.shape[0], img.shape[1], -1).float().contiguous()
        words = words_emb.detach().float()
        N, D, R = img.shape
        Nc, _, T = words.shape
        lens = as_device_i32(cap_lens, img.device)
        pi, pc = self._pairs(image_idx, caption_idx, img.device)
        P = pi.shape[0]
        compiling = torch.compiler.is_compiling()
        ws_bytes = _traced_pairs_workspace_bytes if compiling else ops.damsm_pairs_workspace_bytes
        per = self._chunk_pairs(N, Nc, max(P, 1), T, D, R, ws_bytes)
        g1, g2, mt = self.gamma1, self.gamma2, self.math
        if compiling:
            # traced: the same chunks as agb::damsm_pairs_fwd calls, each with a workspace of its own
            def run(a, b):
                return torch.ops.agb.damsm_pairs_fwd(img, words, lens, a, b, g1, g2, att_maps, mt)
        else:
            ws = ops._ws(ws_bytes(N, Nc, per, T, D, R, mt), img.device)

            def run(a, b):
                return ops.damsm_pairs_fwd(img, words, lens, a, b, g1, g2, mt, att_maps, ws=ws)
        outs = [run(pi[s:s + per], pc[s:s + per]) for s in range(0, max(P, 1), per)]
        m = outs[0][0] if len(outs) == 1 else torch.cat([o[0] for o in outs])
        if not att_maps:
            return m
        att = outs[0][1] if len(outs) == 1 else torch.cat([o[1] for o in outs])
        return m, att.reshape(P, T, *map_shape)

    def sentence_pairs(self, cnn_code: torch.Tensor, sent_emb: torch.Tensor, image_idx, caption_idx) -> torch.Tensor:
        """cnn_code [N,D], sent_emb [Nc,D], image_idx / caption_idx [P] -> cosine [P] fp32 of every listed pair,
        bit for bit what ``sentence`` gives for the same pair; NaN for an index out of range."""
        ops.require_cuda(cnn_code, sent_emb)
        cnn = cnn_code.detach().float().contiguous()
        rnn = sent_emb.detach().float().contiguous()
        pi, pc = self._pairs(image_idx, caption_idx, cnn.device)
        if torch.compiler.is_compiling():
            return torch.ops.agb.sent_cos_pairs_fwd(cnn, rnn, pi, pc, self.eps)
        return ops.sent_cos_pairs_fwd(cnn, rnn, pi, pc, self.eps)

    def words(self, img_features: torch.Tensor, words_emb: torch.Tensor, cap_lens, candidates, *,
              by: str = "image") -> torch.Tensor:
        """img_features [N,D,h,w] or [N,D,R], words_emb [Nc,D,T] (any strides; the RNN's transposed view is read
        coalesced), cap_lens [Nc], candidates [N,K] caption indices (numpy, int64 or int32).
        Returns m [N,K] fp32: m[b,k] = the DAMSM word-level score of image b and caption candidates[b,k], bit for
        bit what WordsLoss's similarity matrix holds for that pair in the same math mode; NaN for an index
        outside [0, Nc).
        by="caption" (text-to-image): candidates [Nc,K] image indices per caption, and m[i,k] = the score of image
        candidates[i,k] and caption i (scored with ``words_pairs``)."""
        if by == "caption":
            ops.require_cuda(img_features, words_emb)
            pi, pc, K = self._by_caption(candidates, words_emb.shape[0], img_features.device)
            return self.words_pairs(img_features, words_emb, cap_lens, pi, pc).reshape(-1, K)
        if by != "image":
            raise ValueError(f'by must be "image" or "caption", got {by!r}')
        ops.require_cuda(img_features, words_emb)
        img = img_features.detach()
        img = img.reshape(img.shape[0], img.shape[1], -1).float().contiguous()
        words = words_emb.detach().float()
        N, D, R = img.shape
        T = words.shape[2]
        lens = as_device_i32(cap_lens, img.device)
        cand = as_device_i32(candidates, img.device)
        if cand.dim() != 2 or cand.shape[0] != N:
            raise ValueError(f"candidates must be [N={N}, K], got {tuple(cand.shape)}")
        K = cand.shape[1]
        if torch.compiler.is_compiling():
            # traced: the same chunks as agb::damsm_cand_fwd calls, each with a workspace of its own
            per = self._chunk_images(N, K, T, D, R, _traced_cand_workspace_bytes)
            parts = [torch.ops.agb.damsm_cand_fwd(img[s:s + per], words, lens, cand[s:s + per], self.gamma1,
                                                  self.gamma2, self.math) for s in range(0, N, per)]
            return parts[0] if len(parts) == 1 else torch.cat(parts)
        per = self._chunk_images(N, K, T, D, R)
        ws = ops._ws(ops.damsm_cand_workspace_bytes(per, K, T, D, R, self.math), img.device)
        parts = [ops.damsm_cand_fwd(img[s:s + per], words, lens, cand[s:s + per], self.gamma1, self.gamma2, self.math,
                                    ws=ws) for s in range(0, N, per)]
        return parts[0] if len(parts) == 1 else torch.cat(parts)

    def sentence(self, cnn_code: torch.Tensor, sent_emb: torch.Tensor, candidates, *, by: str = "image") -> torch.Tensor:
        """cnn_code [N,D], sent_emb [Nc,D], candidates [N,K] -> cosine [N,K] fp32 of every listed pair
        (losses/sentence_loss.py:33-38 before gamma3); NaN for an index outside [0, Nc).
        by="caption": candidates [Nc,K] image indices per caption, cos[i,k] of image candidates[i,k] and caption i."""
        if by == "caption":
            ops.require_cuda(cnn_code, sent_emb)
            pi, pc, K = self._by_caption(candidates, sent_emb.shape[0], cnn_code.device)
            return self.sentence_pairs(cnn_code, sent_emb, pi, pc).reshape(-1, K)
        if by != "image":
            raise ValueError(f'by must be "image" or "caption", got {by!r}')
        ops.require_cuda(cnn_code, sent_emb)
        cnn = cnn_code.detach().float().contiguous()
        rnn = sent_emb.detach().float().contiguous()
        cand = as_device_i32(candidates, cnn.device)
        if cand.dim() != 2 or cand.shape[0] != cnn.shape[0]:
            raise ValueError(f"candidates must be [N={cnn.shape[0]}, K], got {tuple(cand.shape)}")
        if torch.compiler.is_compiling():
            return torch.ops.agb.sent_cos_cand_fwd(cnn, rnn, cand, self.eps)
        return ops.sent_cos_cand_fwd(cnn, rnn, cand, self.eps)


def _traced_cand_workspace_bytes(*args) -> int:
    return torch_ops.host_query("agb_damsm_cand_workspace_bytes", *args)


def _traced_pairs_workspace_bytes(*args) -> int:
    return torch_ops.host_query("agb_damsm_pairs_workspace_bytes", *args)


def mismatched_candidates(class_ids, n_mismatched: int = 99, seed: int = 0, n: Optional[int] = None) -> np.ndarray:
    """Candidate caption lists of the R-precision protocol: [N, 1 + n_mismatched] int64, column 0 = image i's own
    caption i, the other columns drawn uniformly with replacement from the captions whose class differs from
    class_ids[i].  class_ids=None treats every caption as its own class (then ``n`` gives N).  Seeded numpy
    generator on the host.  Raises ValueError when an image has no caption of another class."""
    rng = np.random.default_rng(seed)
    if class_ids is None:
        if n is None:
            raise ValueError("class_ids=None needs the number of captions n")
        N = int(n)
        if N < 2:
            raise ValueError("one caption has no mismatched caption to draw")
        own = np.arange(N)
        u = rng.integers(0, N - 1, size=(N, n_mismatched))
        other = u + (u >= own[:, None])                      # skip caption i itself
    else:
        cls = class_ids.cpu().numpy() if torch.is_tensor(class_ids) else np.asarray(class_ids)
        cls = cls.reshape(-1)
        N = cls.shape[0]
        order = np.argsort(cls, kind="stable")
        uniq, start, count = np.unique(cls[order], return_index=True, return_counts=True)
        ci = np.searchsorted(uniq, cls)
        pool = N - count[ci]                                 # captions of another class
        if (pool == 0).any():
            i = int(np.flatnonzero(pool == 0)[0])
            raise ValueError(f"image {i} has no caption of another class (class {cls[i]} covers every caption)")
        u = rng.integers(0, pool[:, None], size=(N, n_mismatched))
        # position u in the class-sorted order with image i's own class block cut out
        u = u + (u >= start[ci][:, None]) * count[ci][:, None]
        other = order[u]
    return np.concatenate([np.arange(N, dtype=np.int64)[:, None], other.astype(np.int64)], axis=1)


def r_precision(scores: torch.Tensor, r: int = 1) -> torch.Tensor:
    """[N] bool: the own caption (column 0) ranks within the top r of its row.  A tie with a mismatched caption, or
    a NaN on either side, counts against the own caption.  Plain torch ops on the scores' device (CPU too).
    R-precision is hits.float().mean(); the protocol reports mean and std over 10 folds of the images."""
    own = scores[:, :1]
    ahead = (~(scores[:, 1:] < own)).sum(dim=1)              # mismatched captions scoring >= own, or NaN
    return (ahead < r) & ~torch.isnan(own[:, 0])
