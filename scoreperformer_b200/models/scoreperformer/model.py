"""ScorePerformer / Performer models (reference: scoreperformer/models/scoreperformer/model.py:48-407).

Same constructors, forward signatures, output dataclasses, loss keys and state_dict layout as the reference, so the
class drops into `train.py` / the generator; the arithmetic underneath is the sm_100a kernel library.
"""
from __future__ import annotations

from dataclasses import dataclass
from typing import Dict, List, Optional, Union

import os as _os

import torch
from torch import Tensor

from ...config import MISSING, DictConfig
from ...modules.constructor import ModuleConfig
from ...utils import default
from ..base import Model
from ..classifiers.model import (MultiHeadEmbeddingClassifier, MultiHeadEmbeddingClassifierConfig,
                                 MultiHeadEmbeddingClassifierOutput)
from .embeddings import TupleTokenLMHeadConfig
from .mmd_transformer import MMDTupleTransformer, MMDTupleTransformerOutput
from ...utils import SideBranch
from .transformer import TupleTransformer, TupleTransformerConfig, TupleTransformerOutput
from .wrappers import LMWrapper, ScorePerformerLMModes, ScorePerformerLMWrappers


def _get(cfg, key, default_=None):
    if cfg is None:
        return default_
    return cfg.get(key, default_) if hasattr(cfg, "get") else getattr(cfg, key, default_)


@dataclass
class PerformerConfig(ModuleConfig):
    transformer: TupleTransformerConfig = MISSING
    mode: Optional[str] = None


@dataclass
class PerformerOutputs(TupleTransformerOutput):
    loss: Optional[Tensor] = None
    losses: Optional[Dict[str, Tensor]] = None


class _LMMixin:
    _lm_attr = "perf_decoder"

    def _prepare_for_lm(self, mode):
        cur = getattr(self, self._lm_attr)
        if isinstance(cur, TupleTransformer):
            setattr(self, self._lm_attr, ScorePerformerLMWrappers[mode](cur))
        elif isinstance(cur, LMWrapper):
            setattr(self, self._lm_attr, ScorePerformerLMWrappers[mode](cur.model))
        self.mode = mode

    def prepare_for_mlm(self):
        self._prepare_for_lm(ScorePerformerLMModes.MLM)

    def prepare_for_clm(self):
        self._prepare_for_lm(ScorePerformerLMModes.CLM)

    def prepare_for_mixlm(self):
        self._prepare_for_lm(ScorePerformerLMModes.MixedLM)

    def _apply_mode(self, mode):
        self.mode = mode
        if mode == ScorePerformerLMModes.MLM:
            self.prepare_for_mlm()
        elif mode == ScorePerformerLMModes.CLM:
            self.prepare_for_clm()
        elif mode == ScorePerformerLMModes.MixedLM:
            self.prepare_for_mixlm()


class Performer(_LMMixin, Model):
    _lm_attr = "transformer"

    def __init__(self, transformer, mode: Optional[str] = None):
        super().__init__()
        self.transformer = TupleTransformer.init(
            transformer, lm_head=_get(transformer, "lm_head", TupleTokenLMHeadConfig(dim=_get(transformer, "dim"))))
        self._apply_mode(mode)

    def forward(self, perf: Tensor, mask: Optional[Tensor] = None, labels: Optional[Tensor] = None,
                masked_perf: Optional[Tensor] = None):
        return self.transformer(perf, mask=mask, labels=labels, seq_masked=masked_perf)

    def prepare_inputs(self, inputs):
        inputs_dict = {"perf": inputs.performances.tokens, "mask": inputs.performances.mask}
        if hasattr(inputs, "labels") and inputs.labels is not None:
            inputs_dict["labels"] = inputs.labels.tokens
        if hasattr(inputs, "masked_performances") and inputs.masked_performances is not None:
            inputs_dict["masked_perf"] = inputs.masked_performances.tokens
        return inputs_dict


@dataclass
class ScorePerformerConfig(ModuleConfig):
    num_tokens: Dict[str, int] = MISSING
    dim: int = MISSING
    perf_decoder: TupleTransformerConfig = MISSING
    score_encoder: Optional[TupleTransformerConfig] = None
    perf_encoder: Optional[TupleTransformerConfig] = None
    classifiers: Optional[Union[DictConfig, MultiHeadEmbeddingClassifierConfig]] = None
    tie_token_emb: bool = False
    mode: Optional[str] = None
    num_score_tokens: Optional[Dict[str, int]] = None


@dataclass
class ScorePerformerEncoderOutputs:
    score_embeddings: Optional[Tensor] = None
    score_mask: Optional[Tensor] = None
    perf_embeddings: Optional[Tensor] = None
    score_encoder: Optional[TupleTransformerOutput] = None
    perf_encoder: Optional[MMDTupleTransformerOutput] = None


@dataclass
class ScorePerformerOutputs:
    perf_decoder: TupleTransformerOutput
    score_encoder: Optional[TupleTransformerOutput] = None
    perf_encoder: Optional[MMDTupleTransformerOutput] = None
    classifiers: Optional[MultiHeadEmbeddingClassifierOutput] = None
    loss: Optional[Tensor] = None
    losses: Optional[Dict[str, Tensor]] = None


class ScorePerformer(_LMMixin, Model):
    def __init__(self, num_tokens: Dict[str, int], dim: int, perf_decoder, score_encoder=None, perf_encoder=None, classifiers=None,
                 tie_token_emb: bool = False, mode: Optional[str] = None, num_score_tokens: Optional[Dict[str, int]] = None):
        super().__init__()
        self.score_encoder = None
        if score_encoder is not None:
            self.score_encoder = TupleTransformer.init(score_encoder, num_tokens=num_score_tokens or num_tokens, dim=dim, lm_head=None)

        self.perf_encoder = None
        if perf_encoder is not None:
            self.perf_encoder = MMDTupleTransformer.init(perf_encoder, num_tokens=num_tokens, dim=dim, lm_head=None)

        self.classifiers = None
        if classifiers is not None and _get(classifiers, "num_classes") is not None:
            assert self.perf_encoder is not None
            self.classifiers = MultiHeadEmbeddingClassifier.init(classifiers, input_dim=self.perf_encoder.embedding_dim)

        perf_decoder["transformer"]["cross_attend"] = self.score_encoder is not None
        context_emb_dim = None if self.score_encoder is None else self.score_encoder.dim
        style_emb_dim = None if self.perf_encoder is None else self.perf_encoder.embedding_dim
        self.perf_decoder = TupleTransformer.init(
            perf_decoder, num_tokens=num_tokens, dim=dim, context_emb_dim=context_emb_dim, style_emb_dim=style_emb_dim,
            lm_head=_get(perf_decoder, "lm_head", TupleTokenLMHeadConfig(dim=dim)))

        if tie_token_emb:
            for key, emb in self.perf_decoder.token_emb.embs.items():
                if self.score_encoder is not None and key in self.score_encoder.token_emb.embs:
                    self.score_encoder.token_emb.embs[key] = self.perf_decoder.token_emb.embs[key]
                if self.perf_encoder is not None and key in self.perf_encoder.token_emb.embs:
                    self.perf_encoder.token_emb.embs[key] = self.perf_decoder.token_emb.embs[key]

        self._apply_mode(mode)
        # Optional injection points for parity runs (SURVEY B.3): list of N(0, I) prior samples, one per latent level.
        self.z_prior: Optional[List[Tensor]] = None
        # ... and of the (sample, segment) rows MMDLoss subsamples when a level has more than 4096 valid latents
        self.mmd_rows: Optional[List[Optional[Tensor]]] = None

    def forward_encoders(self, perf=None, perf_mask=None, score=None, score_mask=None, bars=None, beats=None, onsets=None,
                         deadpan_mask=None, compute_loss: bool = True, table_cache: Optional[dict] = None, side_branch=None,
                         after_score=None):
        """`after_score(score_embeddings)` (optional) is evaluated right behind the score encoder, on its branch: forward() uses it
        for the decoder's input embedding, which needs the score but not the style embeddings."""
        table_cache = {} if table_cache is None else table_cache
        score_emb = perf_emb = None
        score_enc_out = perf_enc_out = None
        enc_branch = None
        extra = None
        if self.score_encoder is not None:
            # the two encoders are independent: the score encoder runs as a second branch next to the performance encoder
            both = self.perf_encoder is not None and side_branch is not None and _os.environ.get("SPB_ENC_BRANCH", "1") == "1"
            if both:
                enc_branch = SideBranch(score.device, slot=1)
                with enc_branch.run(score, score_mask):
                    score_enc_out = self.score_encoder(score, mask=score_mask, table_cache=table_cache)
                    score_emb = score_enc_out.hidden_state
                    if after_score is not None:
                        extra = after_score(score_emb)
            else:
                score_enc_out = self.score_encoder(score, mask=score_mask, table_cache=table_cache)
                score_emb = score_enc_out.hidden_state
                if after_score is not None:
                    extra = after_score(score_emb)
        if self.perf_encoder is not None:
            perf_enc_out = self.perf_encoder(perf, mask=perf_mask, bars=bars, beats=beats, onsets=onsets, deadpan_mask=deadpan_mask,
                                             compute_loss=compute_loss, z_prior=self.z_prior, table_cache=table_cache,
                                             side_branch=side_branch, mmd_rows=self.mmd_rows)
            perf_emb = perf_enc_out.embeddings
        if enc_branch is not None:
            enc_branch.join(score_emb, *[t for t in (extra or ()) if isinstance(t, torch.Tensor)])
        out = ScorePerformerEncoderOutputs(score_embeddings=score_emb, score_mask=score_mask, perf_embeddings=perf_emb,
                                           score_encoder=score_enc_out, perf_encoder=perf_enc_out)
        out.after_score = extra
        return out

    def forward(self, perf: Tensor, perf_mask: Optional[Tensor] = None, score: Optional[Tensor] = None,
                score_mask: Optional[Tensor] = None, noisy_perf: Optional[Tensor] = None, noisy_perf_mask: Optional[Tensor] = None,
                masked_perf: Optional[Tensor] = None, labels: Optional[Tensor] = None, bars: Optional[Tensor] = None,
                beats: Optional[Tensor] = None, onsets: Optional[Tensor] = None, directions: Optional[Tensor] = None,
                deadpan_mask: Optional[Tensor] = None):
        table_cache: dict = {}
        # MMD terms and the classifier heads are dozens of tiny kernels nothing else waits for: they run on a side stream
        # (a parallel branch of the captured graph) underneath the decoder and are joined just before the losses are summed
        branch = SideBranch(perf.device)
        # the (tied) performance table is built here, before any branch forks off: every stack of the step then finds it -- or a
        # prefix of it -- in the cache, on a stream that already waits for this one
        self.perf_decoder.model.token_emb.table(table_cache)
        # the decoder's input embedding needs the score embeddings but not the latents: it runs behind the score encoder, next to
        # the performance encoder, instead of after both
        pre_embed = None
        if self.score_encoder is not None and hasattr(self.perf_decoder, "pre_embed"):
            pre_embed = lambda score_emb: self.perf_decoder.pre_embed(perf, masked_perf, score_emb, table_cache)
        enc_out = self.forward_encoders(
            perf=default(noisy_perf, perf), perf_mask=default(noisy_perf_mask, perf_mask), score=score, score_mask=score_mask,
            bars=bars, beats=beats, onsets=onsets, deadpan_mask=deadpan_mask, table_cache=table_cache, side_branch=branch,
            after_score=pre_embed)

        clf_out = None
        if self.classifiers is not None:
            clf_mask = perf_mask if deadpan_mask is None else perf_mask & (~deadpan_mask[:, None])
            # fused replacement of `full_embeddings[clf_mask]` / `directions[clf_mask]` (model.py:323-329): rows are
            # selected inside the kernel, so no dynamic-shape gather and no host sync
            with branch.run(enc_out.perf_encoder.full_embeddings, directions, clf_mask):
                clf_out = self.classifiers(embeddings=enc_out.perf_encoder.full_embeddings, labels=directions, rowmask=clf_mask,
                                           with_logits=not self.training)

        perf_dec_out = self.perf_decoder(perf, mask=perf_mask, style_embeddings=enc_out.perf_embeddings,
                                         context=enc_out.score_embeddings, context_mask=enc_out.score_mask, labels=labels,
                                         seq_masked=masked_perf, table_cache=table_cache,
                                         **({} if enc_out.after_score is None else {"pre_embedded": enc_out.after_score}))
        loss, losses = perf_dec_out.loss, perf_dec_out.losses

        side_out = []
        if enc_out.perf_encoder is not None and enc_out.perf_encoder.loss is not None:
            side_out += list(enc_out.perf_encoder.losses.values())
        if clf_out is not None:
            side_out += [clf_out.loss] + list(clf_out.losses.values()) + [getattr(clf_out, "logits", None)]
        branch.join(*[t for t in side_out if isinstance(t, torch.Tensor)])

        if enc_out.perf_encoder is not None and enc_out.perf_encoder.loss is not None:
            loss = loss + enc_out.perf_encoder.loss
            losses.update(**enc_out.perf_encoder.losses)

        if clf_out is not None:
            if clf_out.loss is not None:
                loss = loss + clf_out.loss
                losses.update(**clf_out.losses)

        return ScorePerformerOutputs(perf_decoder=perf_dec_out, score_encoder=enc_out.score_encoder, perf_encoder=enc_out.perf_encoder,
                                     classifiers=clf_out, loss=loss, losses=losses)

    def prepare_inputs(self, inputs):
        inputs_dict = {"perf": inputs.performances.tokens, "perf_mask": inputs.performances.mask,
                       "score": inputs.scores.tokens, "score_mask": inputs.scores.mask}
        if getattr(inputs, "labels", None) is not None:
            inputs_dict["labels"] = inputs.labels.tokens
        if getattr(inputs, "noisy_performances", None) is not None:
            inputs_dict["noisy_perf"] = inputs.noisy_performances.tokens
            inputs_dict["noisy_perf_mask"] = inputs.noisy_performances.mask
        if getattr(inputs, "masked_performances", None) is not None:
            inputs_dict["masked_perf"] = inputs.masked_performances.tokens
        if getattr(inputs, "segments", None) is not None:
            inputs_dict["bars"] = inputs.segments.bar
            inputs_dict["beats"] = inputs.segments.beat
            inputs_dict["onsets"] = inputs.segments.onset
        if getattr(inputs, "directions", None) is not None:
            inputs_dict["directions"] = inputs.directions
        if getattr(inputs, "deadpan_mask", None) is not None:
            inputs_dict["deadpan_mask"] = inputs.deadpan_mask
        return inputs_dict

    @staticmethod
    def inject_data_config(config, dataset):
        config["num_tokens"] = dataset.tokenizer.performance_sizes
        config["num_score_tokens"] = dataset.tokenizer.score_sizes
        for key in ["score_encoder", "perf_encoder", "perf_decoder"]:
            if config.get(key) is not None:
                config[key]["token_embeddings"]["token_values"] = {
                    k: v.tolist() for k, v in dataset.tokenizer.token_values(normalize=True).items()}
        if config.get("classifiers") is not None and dataset.performance_directions is not None:
            config["classifiers"]["num_classes"] = dict(dataset.performance_direction_sizes)
            config["classifiers"]["class_samples"] = dict(dataset.get_direction_class_weights()[1])
        return config

    @staticmethod
    def cleanup_config(config):
        for key in ["score_encoder", "perf_encoder", "perf_decoder"]:
            if config.get(key) is not None:
                del config[key]["token_embeddings"]["token_values"]
        if config.get("classifiers") is not None:
            del config["classifiers"]["class_samples"]
        return config
