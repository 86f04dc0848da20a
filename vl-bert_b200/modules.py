"""Drop-in nn.Modules: same constructor arguments, forward signatures, return structures and
state_dict keys as the reference classes they replace, with the compute routed to libvlbert_b200.so.

  VisualLinguisticBert                <- common/visual_linguistic_bert.py:31-241
  VisualLinguisticBertForPretraining  <- common/visual_linguistic_bert.py:312-380 (heads: torch for now, SURVEY 8f.1)
  FastRCNN                            <- common/fast_rcnn.py:17-203
  ROIAlign / C_ROIPooling             <- common/lib/roi_pooling/roi_align.py:46-78, vision.cpp:6-11

There is no CPU / eager fallback: a forward on CPU tensors raises.
"""
import math
import types

import torch
import torch.nn as nn
import torch.nn.functional as F

from . import functional as VF

NUM_SPECIAL_WORDS = 1000


def default_config(**over):
    """NETWORK.VLBERT defaults for VL-BERT-base (reference: pretrain/function/config.py:87-115, cfgs/pretrain/base_*.yaml):
    hidden_dropout_prob = attention_probs_dropout_prob = 0.1 like every shipped cfg."""
    cfg = dict(vocab_size=30522, hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072,
               hidden_act="gelu", hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1, max_position_embeddings=512,
               type_vocab_size=3, initializer_range=0.02, visual_size=768, visual_scale_text_init=1.0,
               visual_scale_object_init=1.0, visual_ln=True, word_embedding_frozen=False, with_pooler=True,
               position_padding_idx=-1, obj_pos_id_relative=True)
    cfg.update(over)
    return types.SimpleNamespace(**cfg)


class BertLayerNorm(nn.Module):
    """Parameter holder with the reference's names (modeling.py:222-229); compute happens in the kernels.
    Calling it directly (heads) uses the TF-style formula in torch."""

    def __init__(self, hidden_size, eps=1e-12):
        super().__init__()
        self.weight = nn.Parameter(torch.ones(hidden_size))
        self.bias = nn.Parameter(torch.zeros(hidden_size))
        self.variance_epsilon = eps

    def forward(self, x):
        u = x.mean(-1, keepdim=True)
        s = (x - u).pow(2).mean(-1, keepdim=True)
        return self.weight * ((x - u) / torch.sqrt(s + self.variance_epsilon)) + self.bias


class _SelfAttention(nn.Module):
    def __init__(self, H):
        super().__init__()
        self.query, self.key, self.value = nn.Linear(H, H), nn.Linear(H, H), nn.Linear(H, H)


class _DenseLN(nn.Module):
    def __init__(self, fan_in, H):
        super().__init__()
        self.dense = nn.Linear(fan_in, H)
        self.LayerNorm = BertLayerNorm(H, eps=1e-12)


class _Attention(nn.Module):
    def __init__(self, H):
        super().__init__()
        self.self = _SelfAttention(H)
        self.output = _DenseLN(H, H)


class _Intermediate(nn.Module):
    def __init__(self, H, I):
        super().__init__()
        self.dense = nn.Linear(H, I)


class BertLayer(nn.Module):
    def __init__(self, H, I):
        super().__init__()
        self.attention = _Attention(H)
        self.intermediate = _Intermediate(H, I)
        self.output = _DenseLN(I, H)

    def flat_params(self):
        a, o = self.attention, self.output
        return [a.self.query.weight, a.self.query.bias, a.self.key.weight, a.self.key.bias, a.self.value.weight,
                a.self.value.bias, a.output.dense.weight, a.output.dense.bias, a.output.LayerNorm.weight,
                a.output.LayerNorm.bias, self.intermediate.dense.weight, self.intermediate.dense.bias, o.dense.weight,
                o.dense.bias, o.LayerNorm.weight, o.LayerNorm.bias]


class BertEncoder(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.layer = nn.ModuleList([BertLayer(config.hidden_size, config.intermediate_size)
                                    for _ in range(config.num_hidden_layers)])


class BertPooler(nn.Module):
    """modeling.py:424-436: tanh(dense(first token)) -- the dense layer runs on the library's tcgen05 GEMM (VF.LinearFn)."""

    def __init__(self, config):
        super().__init__()
        self.dense = nn.Linear(config.hidden_size, config.hidden_size)

    def forward(self, hidden_states):
        return torch.tanh(VF.LinearFn.apply(hidden_states[:, 0], self.dense.weight, self.dense.bias))


class BaseModel(nn.Module):
    def __init__(self, config, **kwargs):
        self.config = config
        super().__init__()

    def init_weights(self, module):
        """common/visual_linguistic_bert.py:14-25"""
        if isinstance(module, (nn.Linear, nn.Embedding)):
            module.weight.data.normal_(mean=0.0, std=self.config.initializer_range)
        elif isinstance(module, BertLayerNorm):
            module.bias.data.zero_()
            module.weight.data.fill_(1.0)
        if isinstance(module, nn.Linear) and module.bias is not None:
            module.bias.data.zero_()


class VisualLinguisticBert(BaseModel):
    def __init__(self, config, language_pretrained_model_path=None):
        super().__init__(config)
        H = config.hidden_size
        if config.hidden_act != "gelu":
            raise ValueError("vlbert_b200: only hidden_act='gelu' (erf form) is implemented")
        if H % config.num_attention_heads != 0 or H // config.num_attention_heads != 64:
            raise ValueError("vlbert_b200: attention head size must be 64 (hidden %d, heads %d)" % (H, config.num_attention_heads))
        if getattr(config, "word_embedding_frozen", False):
            raise ValueError("vlbert_b200: word_embedding_frozen is not implemented")
        if not config.visual_ln:
            raise ValueError("vlbert_b200: visual_ln=False (scalar visual scale) is not implemented")
        if not config.obj_pos_id_relative:
            raise AssertionError("Don't use position id 510/511 for objects and [END]!!!")  # visual_linguistic_bert.py:229
        for nm in ("hidden_dropout_prob", "attention_probs_dropout_prob"):
            if not (0.0 <= getattr(config, nm) < 1.0):
                raise ValueError("dropout probability has to be between 0 and 1, but got {}".format(getattr(config, nm)))
        self.word_embeddings = nn.Embedding(config.vocab_size, H)
        self.end_embedding = nn.Embedding(1, H)
        self.position_embeddings = nn.Embedding(config.max_position_embeddings, H)
        self.token_type_embeddings = nn.Embedding(config.type_vocab_size, H)
        self.embedding_LayerNorm = BertLayerNorm(H, eps=1e-12)
        self.position_padding_idx = config.position_padding_idx
        self.visual_1x1_text = None
        self.visual_1x1_object = None
        if config.visual_size != H:
            self.visual_1x1_text = nn.Linear(config.visual_size, H)
            self.visual_1x1_object = nn.Linear(config.visual_size, H)
        self.visual_ln_text = BertLayerNorm(H, eps=1e-12)
        self.visual_ln_object = BertLayerNorm(H, eps=1e-12)
        self.encoder = BertEncoder(config)
        if config.with_pooler:
            self.pooler = BertPooler(config)
        self.apply(self.init_weights)
        self.visual_ln_text.weight.data.fill_(config.visual_scale_text_init)
        self.visual_ln_object.weight.data.fill_(config.visual_scale_object_init)
        if language_pretrained_model_path is not None:
            self.load_language_pretrained_model(language_pretrained_model_path)
        # Upper bound for the packed length; when set, no device->host sync is needed to size the outputs
        # (the reference's `max_length = (...).max() + 1`, visual_linguistic_bert.py:202, syncs every forward).
        self.max_length_hint = None
        self._weights = None
        self._last_pidx = None
        # Residual stream precision (csrc/encoder.cu): fp32 like the reference under autocast (default; what the parity tests
        # pin) or bf16 (VLB_RESIDUAL=bf16: ~2 % faster, ~1.7x the rounding error after 12 layers).
        import os
        self.fp32_residual_stream = os.environ.get("VLB_RESIDUAL", "fp32") != "bf16"
        # Dropout (modeling.py:283,310,331,376 / visual_linguistic_bert.py:75,239) is fused into the kernels as counter-based
        # masks: (seed, step) live in this DEVICE buffer, non-persistent so the state_dict keys stay the reference's.  The
        # default seed derives from torch.initial_seed() without consuming torch's generator (the reference's masks follow
        # torch.manual_seed(RNG_SEED) too, and every rank of a DDP job uses the same stream there as well).
        seed = (torch.initial_seed() * 0x9E3779B97F4A7C15 + 0x1234567) & 0x7FFFFFFFFFFFFFFF
        self.register_buffer("_rng_state", torch.tensor([seed, 0], dtype=torch.int64), persistent=False)

    def set_dropout_seed(self, seed, step=0):
        """(Re)seed the dropout stream: the masks of training step n are a pure function of (seed, step0 + n, site, element)."""
        self._rng_state.copy_(torch.tensor([int(seed) & 0x7FFFFFFFFFFFFFFF, int(step)], dtype=torch.int64))

    def dropout_state(self):
        """(seed, step) of the most recent training forward (one device->host sync; tests and checkpointing)."""
        v = self._rng_state.tolist()
        return int(v[0]), int(v[1])

    def _dropout_rng(self):
        """Advance the step counter on the device and return a snapshot tensor for this forward (its backward re-reads the
        same snapshot, so interleaved forwards / gradient accumulation keep their own masks).  None when dropout is off."""
        cfg = self.config
        if not self.training or (cfg.hidden_dropout_prob == 0 and cfg.attention_probs_dropout_prob == 0):
            return None
        self._rng_state[1] += 1
        return self._rng_state.clone()

    def check_errors(self):
        """Deferred index check of the most recent forward (the graph-friendly path never syncs by itself): raises IndexError
        if `max_length_hint` was too small or token / position / type ids were out of range.  One device->host sync."""
        if self._last_pidx is not None:
            self._last_pidx.check()

    # -- helpers -----------------------------------------------------------------------------------
    def _encoder_meta(self, all_layers, device):
        cfg = self.config
        if self._weights is None or self._weights.w_qkv.device != device:
            self._weights = VF.EncoderWeights(cfg.num_hidden_layers, cfg.hidden_size, cfg.intermediate_size, device)
        return types.SimpleNamespace(L=cfg.num_hidden_layers, H=cfg.hidden_size, heads=cfg.num_attention_heads,
                                     I=cfg.intermediate_size, eps=1e-12, all_layers=all_layers, weights=self._weights,
                                     reducer=getattr(self, "_grad_reducer", None), drop=None)

    def _packed_length(self, text_mask, object_mask):
        T, R = text_mask.shape[1], object_mask.shape[1]
        if self.max_length_hint is not None:
            return min(int(self.max_length_hint), T + R + 1)
        S = int((text_mask.sum(1) + object_mask.sum(1)).max().item()) + 1
        if S > 256:
            raise ValueError("vlbert_b200: packed sequence length %d > 256 is not supported by the fused attention" % S)
        return S

    def embedding(self, text_input_ids, text_token_type_ids, text_visual_embeddings, text_mask, object_vl_embeddings,
                  object_mask):
        emb, emb32, pidx = self._embedding_impl(text_input_ids, text_token_type_ids, text_visual_embeddings, text_mask,
                                                object_vl_embeddings, object_mask, self._dropout_rng())
        kind = pidx.kind
        return emb32, (kind != 3).to(text_mask.dtype), kind == 0, kind == 1

    def _embedding_impl(self, text_input_ids, text_token_type_ids, text_visual_embeddings, text_mask, object_vl_embeddings,
                        object_mask, rng=None):
        cfg = self.config
        VS = cfg.visual_size
        if self.visual_1x1_text is not None:
            text_visual_embeddings = self.visual_1x1_text(text_visual_embeddings)
            object_vl_embeddings = torch.cat((self.visual_1x1_object(object_vl_embeddings[:, :, :VS]),
                                              object_vl_embeddings[:, :, VS:]), -1)
        S = self._packed_length(text_mask, object_mask)
        pidx = VF.PackIndex(text_mask, object_mask, text_token_type_ids, S, self.position_padding_idx + 1)
        drop = None
        if rng is not None and cfg.hidden_dropout_prob > 0:
            drop = VF.DropSite(cfg.hidden_dropout_prob, 0, rng)            # site 0: embedding_dropout (:75, :239)
        emb, emb32 = VF.EmbeddingFn.apply(text_visual_embeddings, object_vl_embeddings, self.word_embeddings.weight,
                                          self.end_embedding.weight, self.position_embeddings.weight,
                                          self.token_type_embeddings.weight, self.embedding_LayerNorm.weight,
                                          self.embedding_LayerNorm.bias, self.visual_ln_text.weight, self.visual_ln_text.bias,
                                          self.visual_ln_object.weight, self.visual_ln_object.bias, text_input_ids, pidx, 1e-12,
                                          drop)
        self._last_pidx = pidx
        if self.max_length_hint is None:
            pidx.check()      # this path already synchronised for the packed length; surface bad ids like the reference does
        return emb, emb32, pidx

    def forward(self, text_input_ids, text_token_type_ids, text_visual_embeddings, text_mask, object_vl_embeddings,
                object_mask, output_all_encoded_layers=True, output_text_and_object_separately=False,
                output_attention_probs=False):
        if output_attention_probs:
            raise NotImplementedError("vlbert_b200: the fused attention never materialises probabilities "
                                      "(output_attention_probs is a visualisation-only path of the reference)")
        rng = self._dropout_rng()
        emb, emb32, pidx = self._embedding_impl(text_input_ids, text_token_type_ids, text_visual_embeddings, text_mask,
                                                object_vl_embeddings, object_mask, rng)
        if not self.fp32_residual_stream:
            emb32 = None
        meta = self._encoder_meta(bool(output_all_encoded_layers), emb.device)
        if rng is not None:
            meta.drop = types.SimpleNamespace(p_attn=float(self.config.attention_probs_dropout_prob),
                                              p_hidden=float(self.config.hidden_dropout_prob), rng=rng)
        params = []
        for layer in self.encoder.layer:
            params += layer.flat_params()
        outs = VF.EncoderFn.apply(emb, emb32, pidx.add_mask, meta, *params)
        encoded_layers = list(outs)
        sequence_output = encoded_layers[-1]
        pooled_output = self.pooler(sequence_output) if self.config.with_pooler else None
        if not output_all_encoded_layers:
            encoded_layers = encoded_layers[-1]
        if not output_text_and_object_separately:
            return encoded_layers, pooled_output
        lst = encoded_layers if output_all_encoded_layers else [encoded_layers]
        B, S, H = lst[0].shape
        T, R = text_input_ids.shape[1], object_vl_embeddings.shape[1]
        texts, objs = [], []
        for enc in lst:
            texts.append(enc[:, :T])
            objs.append(VF.GatherRowsFn.apply(enc.reshape(B * S, H), pidx.obj_row.view(-1), B * R).view(B, R, H))
        if not output_all_encoded_layers:
            texts, objs = texts[0], objs[0]
        return texts, objs, pooled_output

    def load_language_pretrained_model(self, language_pretrained_model_path):
        """Initialise from a HuggingFace BERT / RoBERTa checkpoint (common/visual_linguistic_bert.py:243-309; the pre-training
        subclass also takes the `cls.seq_relationship.*` / `cls.predictions.*` / `lm_head.*` heads, :382-470)."""
        sd = torch.load(language_pretrained_model_path, map_location="cpu")
        own = {"encoder": self.encoder.state_dict(), "ln": self.embedding_LayerNorm.state_dict(),
               "pooler": self.pooler.state_dict() if self.config.with_pooler else {}}
        rel_head = getattr(self, "relationsip_head", None) if getattr(self, "with_rel_head", False) else None
        mlm_head = getattr(self, "mlm_head", None) if getattr(self, "with_mlm_head", False) else None
        picked = {"encoder": {}, "ln": {}, "pooler": {}, "rel": {}, "mlm": {}}
        unexpected = []

        def rename(k):  # TF-style parameter names of old checkpoints
            return k.replace("gamma", "weight").replace("beta", "bias")

        def put(table, k, v, raw, known):
            if k in known:
                picked[table][k] = v
            else:
                unexpected.append(raw)

        for raw, v in sd.items():
            if raw.startswith(("bert.", "roberta.")):
                k = rename(raw.split(".", 1)[1])
                if k.startswith("encoder."):
                    put("encoder", k[len("encoder."):], v, raw, own["encoder"])
                elif k.startswith("embeddings."):
                    k = k[len("embeddings."):]
                    if k == "word_embeddings.weight":
                        self.word_embeddings.weight.data = v.to(self.word_embeddings.weight.data)
                    elif k == "position_embeddings.weight":
                        self.position_embeddings.weight.data = v.to(self.position_embeddings.weight.data)
                    elif k == "token_type_embeddings.weight":
                        w = self.token_type_embeddings.weight.data
                        w[:v.size(0)] = v.to(w)
                        if v.size(0) == 1:      # RoBERTa has one token type: replicate it (:280-287; the pre-training class
                            w[1] = v[0].to(w)   # fills only row 1, :415-419)
                            if rel_head is None and mlm_head is None and not isinstance(self, VisualLinguisticBertForPretraining):
                                w[2] = v[0].to(w)
                    elif k.startswith("LayerNorm."):
                        put("ln", k[len("LayerNorm."):], v, raw, own["ln"])
                    else:
                        unexpected.append(raw)
                elif self.config.with_pooler and k.startswith("pooler."):
                    put("pooler", k[len("pooler."):], v, raw, own["pooler"])
                # (anything else under bert./roberta. is silently ignored, like the reference)
            elif rel_head is not None and raw.startswith("cls.seq_relationship."):
                put("rel", rename(raw[len("cls.seq_relationship."):]), v, raw, rel_head.caption_image_relationship.state_dict())
            elif mlm_head is not None and raw.startswith(("cls.predictions.", "lm_head.")):
                if raw.startswith("lm_head."):  # RoBERTa naming of the LM head
                    k = raw[len("lm_head."):]
                    if "dense" in k or "layer_norm" in k:
                        k = "transform." + k
                    k = k.replace("layer_norm", "LayerNorm")
                else:
                    k = raw[len("cls.predictions."):]
                put("mlm", rename(k), v, raw, mlm_head.predictions.state_dict())
            else:
                unexpected.append(raw)
        if unexpected:
            print("Warnings: Unexpected keys: {}.".format(unexpected))
        self.embedding_LayerNorm.load_state_dict(picked["ln"])
        self.encoder.load_state_dict(picked["encoder"])
        if self.config.with_pooler and picked["pooler"]:
            self.pooler.load_state_dict(picked["pooler"])
        if rel_head is not None and picked["rel"]:
            rel_head.caption_image_relationship.load_state_dict(picked["rel"])
        if mlm_head is not None:
            mlm_head.predictions.load_state_dict(picked["mlm"])


# ------------------------------------------------------------------------------------------------
# pre-training heads (reference: common/visual_linguistic_bert.py:312-380, :473-502; modeling.py:439-472).
# Torch ops for now -- SURVEY.md 8(f) ranks the fused vocab GEMM + CE as the first "next" row.
# ------------------------------------------------------------------------------------------------
def _gelu(x):
    return x * 0.5 * (1.0 + torch.erf(x / math.sqrt(2.0)))


class BertPredictionHeadTransform(nn.Module):
    def __init__(self, config):
        super().__init__()
        self.dense = nn.Linear(config.hidden_size, config.hidden_size)
        self.LayerNorm = BertLayerNorm(config.hidden_size, eps=1e-12)

    def forward(self, x):
        return self.LayerNorm(_gelu(self.dense(x)))


class BertLMPredictionHead(nn.Module):
    def __init__(self, config, bert_model_embedding_weights):
        super().__init__()
        self.transform = BertPredictionHeadTransform(config)
        self.decoder = nn.Linear(bert_model_embedding_weights.size(1), bert_model_embedding_weights.size(0), bias=False)
        self.decoder.weight = bert_model_embedding_weights
        self.bias = nn.Parameter(torch.zeros(bert_model_embedding_weights.size(0)))

    def forward(self, x):
        return self.decoder(self.transform(x)) + self.bias


class BertOnlyMLMHead(nn.Module):
    def __init__(self, config, bert_model_embedding_weights):
        super().__init__()
        self.predictions = BertLMPredictionHead(config, bert_model_embedding_weights)

    def forward(self, x):
        return self.predictions(x)


class VisualLinguisticBertMVRCHeadTransform(BaseModel):
    def __init__(self, config):
        super().__init__(config)
        self.dense = nn.Linear(config.hidden_size, config.hidden_size)
        self.apply(self.init_weights)

    def forward(self, x):
        return _gelu(self.dense(x))


class VisualLinguisticBertMVRCHead(BaseModel):
    def __init__(self, config):
        super().__init__(config)
        self.transform = VisualLinguisticBertMVRCHeadTransform(config)
        self.region_cls_pred = nn.Linear(config.hidden_size, config.visual_region_classes)
        self.apply(self.init_weights)

    def forward(self, x):
        return self.region_cls_pred(self.transform(x))


class VisualLinguisticBertRelationshipPredictionHead(BaseModel):
    def __init__(self, config):
        super().__init__(config)
        self.caption_image_relationship = nn.Linear(config.hidden_size, 2)
        self.apply(self.init_weights)

    def forward(self, pooled_rep):
        return self.caption_image_relationship(pooled_rep)


class VisualLinguisticBertForPretraining(VisualLinguisticBert):
    def __init__(self, config, language_pretrained_model_path=None, with_rel_head=True, with_mlm_head=True,
                 with_mvrc_head=True):
        super().__init__(config, language_pretrained_model_path=None)
        self.with_rel_head, self.with_mlm_head, self.with_mvrc_head = with_rel_head, with_mlm_head, with_mvrc_head
        if with_rel_head:
            self.relationsip_head = VisualLinguisticBertRelationshipPredictionHead(config)  # (sic) reference key name
        if with_mlm_head:
            self.mlm_head = BertOnlyMLMHead(config, self.word_embeddings.weight)
        if with_mvrc_head:
            self.mvrc_head = VisualLinguisticBertMVRCHead(config)
        self.apply(self.init_weights)
        self.visual_ln_text.weight.data.fill_(config.visual_scale_text_init)
        self.visual_ln_object.weight.data.fill_(config.visual_scale_object_init)
        if language_pretrained_model_path is not None:
            self.load_language_pretrained_model(language_pretrained_model_path)
        if getattr(config, "pos_embedding_frozen", False):  # common/visual_linguistic_bert.py:341-343
            for p in self.position_embeddings.parameters():
                p.requires_grad = False

    def forward(self, text_input_ids, text_token_type_ids, text_visual_embeddings, text_mask, object_vl_embeddings,
                object_mask, output_all_encoded_layers=True, output_text_and_object_separately=False):
        text_out, object_out, pooled_rep = super().forward(text_input_ids, text_token_type_ids, text_visual_embeddings,
                                                           text_mask, object_vl_embeddings, object_mask,
                                                           output_all_encoded_layers=False,
                                                           output_text_and_object_separately=True)
        relationship_logits = self.relationsip_head(pooled_rep) if self.with_rel_head else None
        mlm_logits = self.mlm_head(text_out) if self.with_mlm_head else None
        mvrc_logits = self.mvrc_head(object_out) if self.with_mvrc_head else None
        return relationship_logits, mlm_logits, mvrc_logits

    def mlm_loss(self, text_out, mlm_labels, max_labelled=None):
        """Fused masked-LM loss (SURVEY 8(f) rank 1) for callers that need the LOSS, not the [B, T, V] logits:
        == F.cross_entropy(self.mlm_head(text_out).view(-1, V), mlm_labels.view(-1), ignore_index=-1)
        (pretrain/modules/resnet_vlbert_for_pretraining.py:165-189) evaluated on the labelled positions only: they are compacted
        on the device, the transform + tied-decoder GEMMs run on those rows, the cross-entropy is one pass over bf16 logits.
        Returns (loss, n_correct, n_labelled) -- the two counters feed the trainer's MLMAccuracy metric without logits.
        max_labelled: static upper bound of labelled positions (no host sync; CUDA-graph friendly); None = counted on the host."""
        p = self.mlm_head.predictions
        if max_labelled is None:
            max_labelled = max(8, int((mlm_labels != -1).sum().item()))
        return VF.MLMLossFn.apply(text_out, mlm_labels, p.transform.dense.weight, p.transform.dense.bias,
                                  p.transform.LayerNorm.weight, p.transform.LayerNorm.bias, p.decoder.weight, p.bias,
                                  int(max_labelled), 1e-12)

    def mvrc_loss(self, object_out, mvrc_labels, max_valid=None, norm_in_batch_first=False):
        """Fused masked-region-classification loss for callers that need the LOSS, not the [B, R, C] logits:
        == soft_cross_entropy(self.mvrc_head(object_out).view(-1, C), mvrc_labels.view(-1, C)) (common/utils/misc.py:124-151,
        pretrain/modules/resnet_vlbert_for_pretraining.py:191-203), or its MVRC_LOSS_NORM_IN_BATCH_FIRST form, evaluated on the
        valid regions only (target row sum within 0.1 of 1): they are compacted on the device, the transform + classifier GEMMs
        run on those rows, the soft-target cross-entropy is one pass over bf16 logits and the fp32 targets.
        Returns (loss, n_correct, n_valid) -- n_correct counts what MVRCAccuracy counts (logit arg-max == target arg-max).
        max_valid: static upper bound of valid regions (no host sync; CUDA-graph friendly); None = counted on the host.  If more
        regions are valid than max_valid, the first max_valid (ascending flat order) are used and the loss is normalised by
        the regions used (per sample in batch-first mode); n_valid reports the true count, so callers can detect it."""
        h = self.mvrc_head
        if max_valid is None:
            max_valid = max(8, int(((mvrc_labels.sum(-1) - 1).abs() < 0.1).sum().item()))
        return VF.MVRCLossFn.apply(object_out, mvrc_labels, h.transform.dense.weight, h.transform.dense.bias,
                                   h.region_cls_pred.weight, h.region_cls_pred.bias, int(max_valid), bool(norm_in_batch_first))


# ------------------------------------------------------------------------------------------------
# region-feature front end
# ------------------------------------------------------------------------------------------------
class ROIAlign(nn.Module):
    """common/lib/roi_pooling/roi_align.py:46-78"""

    def __init__(self, output_size, spatial_scale, sampling_ratio=1):
        super().__init__()
        self.output_size = output_size
        self.spatial_scale = spatial_scale
        self.sampling_ratio = sampling_ratio

    def forward(self, input, rois):
        return VF.RoIAlignFn.apply(input.float(), rois.float(), self.output_size, self.spatial_scale, self.sampling_ratio)

    def __repr__(self):
        return "%s(output_size=%s, spatial_scale=%s, sampling_ratio=%s)" % (self.__class__.__name__, self.output_size,
                                                                            self.spatial_scale, self.sampling_ratio)


def _roi_pool_unavailable(*a, **k):
    raise RuntimeError("vlbert_b200: roi_pool_* is dead code on the reference's hot path and is not provided")


#: module object with the reference extension's function names (common/lib/roi_pooling/vision.cpp:6-11)
C_ROIPooling = types.SimpleNamespace(roi_align_forward=VF.roi_align_forward, roi_align_backward=VF.roi_align_backward,
                                     roi_pool_forward=_roi_pool_unavailable, roi_pool_backward=_roi_pool_unavailable)


class Flattener(nn.Module):
    """common/utils/flatten.py:4-13 (parameter-free; kept so `head.*` state_dict keys match the reference)"""

    def forward(self, x):
        return x.view(x.size(0), -1)


_RESNET_LAYERS = {50: (3, 4, 6), 101: (3, 4, 23), 152: (3, 8, 36)}


class FastRCNN(nn.Module):
    """common/fast_rcnn.py:17-203.  Both paths run on the library: the precomputed-feature path
    (IMAGE_FEAT_PRECOMPUTED, BASELINE configs 1-4) is region-operand + one GEMM; the end-to-end path (config 5) is
    ResNet-C4 (NHWC bf16, frozen BN folded into the conv GEMM epilogue) -> RoIAlign 14x14 @ 1/16 -> dilated res5 head ->
    mean pool -> the same region projection.

    `compact_rois` (default True) gathers the valid boxes with one host sync like the reference (`box_mask.nonzero()`,
    :135); set it False to run every [B, R] slot with static shapes (no sync; padded slots are computed and discarded)."""

    def __init__(self, config, average_pool=True, final_dim=768, enable_cnn_reg_loss=False):
        super().__init__()
        self.average_pool = average_pool
        self.enable_cnn_reg_loss = enable_cnn_reg_loss
        self.final_dim = final_dim
        self.image_feat_precomputed = config.NETWORK.IMAGE_FEAT_PRECOMPUTED
        self.compact_rois = True
        if config.NETWORK.IMAGE_SEMANTIC:
            raise ValueError("vlbert_b200: IMAGE_SEMANTIC (object class embedding) is not implemented")
        self.object_embed = None
        if not self.image_feat_precomputed:
            from .resnet import ResNetC4, make_layer
            self.stride_in_1x1 = config.NETWORK.IMAGE_STRIDE_IN_1x1
            self.c5_dilated = config.NETWORK.IMAGE_C5_DILATED
            self.num_layers = config.NETWORK.IMAGE_NUM_LAYERS
            self.pretrained_model_path = '{}-{:04d}.model'.format(
                config.NETWORK.IMAGE_PRETRAINED, config.NETWORK.IMAGE_PRETRAINED_EPOCH) if config.NETWORK.IMAGE_PRETRAINED != '' else None
            self.output_conv5 = config.NETWORK.OUTPUT_CONV5
            if self.output_conv5:
                raise NotImplementedError("vlbert_b200: OUTPUT_CONV5 is not implemented (false in every reference cfg)")
            if self.num_layers not in _RESNET_LAYERS:
                raise NotImplementedError("vlbert_b200: only Bottleneck backbones (50/101/152) are implemented")
            if not average_pool:
                raise NotImplementedError("vlbert_b200: average_pool=False is not implemented")
            self.backbone = ResNetC4(_RESNET_LAYERS[self.num_layers], stride_in_1x1=self.stride_in_1x1)
            if self.pretrained_model_path is not None:
                import os
                if not os.path.exists(self.pretrained_model_path):
                    # the reference fails inside torch.load on a missing checkpoint (common/backbone/resnet/resnet.py:279-283);
                    # a silently random-initialised backbone with frozen stages must not happen
                    raise FileNotFoundError("vlbert_b200.FastRCNN: IMAGE_PRETRAINED checkpoint %s not found" % self.pretrained_model_path)
                sd = torch.load(self.pretrained_model_path, map_location="cpu")
                own = self.backbone.state_dict()
                missing = [k for k in own if k not in sd]
                if missing:
                    print("Warnings: Missing keys: {}.".format(missing))
                self.backbone.load_state_dict({k: sd.get(k, v) for k, v in own.items()})
            else:
                import warnings
                warnings.warn("vlbert_b200.FastRCNN: IMAGE_PRETRAINED is empty -- the backbone keeps its random (Kaiming) "
                              "initialisation (the reference would download the model-zoo weights; there is no network here)")
            self.mask_upsample = None
            self.roi_head_feature_extractor, _ = make_layer(self.backbone.inplanes, 512, 3,
                                                            stride=2 if not self.c5_dilated else 1,
                                                            dilation=1 if not self.c5_dilated else 2,
                                                            stride_in_1x1=self.stride_in_1x1)
            for m in self.roi_head_feature_extractor.modules():
                if isinstance(m, nn.Conv2d):
                    nn.init.kaiming_normal_(m.weight, mode="fan_out", nonlinearity="relu")
            self.head = torch.nn.Sequential(self.roi_head_feature_extractor,
                                            nn.AvgPool2d(7 if not self.c5_dilated else 14, stride=1), Flattener())
            if config.NETWORK.IMAGE_FROZEN_BN:
                for m in self.roi_head_feature_extractor.modules():
                    if isinstance(m, nn.BatchNorm2d):
                        for p in m.parameters():
                            p.requires_grad = False
            frozen_stages = list(config.NETWORK.IMAGE_FROZEN_BACKBONE_STAGES)
            if 5 in frozen_stages:
                for p in self.roi_head_feature_extractor.parameters():
                    p.requires_grad = False
                frozen_stages = [s for s in frozen_stages if s != 5]
            self.backbone.frozen_parameters(frozen_stages=frozen_stages, frozen_bn=config.NETWORK.IMAGE_FROZEN_BN)
            if self.enable_cnn_reg_loss:
                self.regularizing_predictor = torch.nn.Linear(2048, 81)
        self.obj_downsample = torch.nn.Sequential(
            torch.nn.Dropout(p=0.1),
            torch.nn.Linear(2 * 2048, final_dim),
            torch.nn.ReLU(inplace=True),
        )
        # obj_downsample[0] (Dropout(0.1), common/fast_rcnn.py:104-109) is fused into the kernel that writes the GEMM operand:
        # counter-based masks from this device-resident (seed, step) state (non-persistent: not a state_dict key)
        seed = (torch.initial_seed() * 0xD1B54A32D192ED03 + 0x7654321) & 0x7FFFFFFFFFFFFFFF
        self.register_buffer("_rng_state", torch.tensor([seed, 0], dtype=torch.int64), persistent=False)

    #: dropout call-site id of obj_downsample (the encoder uses 0 .. 3L)
    DROP_SITE = 1000

    def set_dropout_seed(self, seed, step=0):
        self._rng_state.copy_(torch.tensor([int(seed) & 0x7FFFFFFFFFFFFFFF, int(step)], dtype=torch.int64))

    def dropout_state(self):
        v = self._rng_state.tolist()
        return int(v[0]), int(v[1])

    def init_weight(self):
        """common/fast_rcnn.py:111-120: the res5 head starts from the checkpoint's layer4.* (no model-zoo download here)."""
        if not self.image_feat_precomputed and self.pretrained_model_path is not None:
            sd = torch.load(self.pretrained_model_path, map_location="cpu")
            self.roi_head_feature_extractor.load_state_dict({k[len("layer4."):]: v for k, v in sd.items() if k.startswith("layer4.")})

    def bn_eval(self):
        if not self.image_feat_precomputed:
            for m in self.modules():
                if isinstance(m, nn.BatchNorm2d):
                    m.eval()

    def _region_features(self, images, boxes, box_mask, segms):
        """images -> per-slot res5 features f32 [B, R, 2048] (zeros in invalid slots); common/fast_rcnn.py:143-158.
        `segms` [B, R, 14, 14] (VCR instance masks): the res5 map is multiplied by the box's mask before the mean pool (:151-156)."""
        B, R = box_mask.shape
        feat = self.backbone(images)["body4"]
        b4 = boxes[:, :, :4].float()
        if self.compact_rois:
            inds = box_mask.nonzero()
            assert inds.shape[0] > 0
            rois = torch.cat((inds[:, 0, None].float(), b4[inds[:, 0], inds[:, 1]]), 1)
        else:
            inds = None
            bidx = torch.arange(B, device=boxes.device, dtype=torch.float32).view(B, 1, 1).expand(B, R, 1)
            rois = torch.cat((bidx, b4), 2).view(B * R, 5)
        pooled = VF.RoIAlignNHWCFn.apply(feat, rois, 14, 14, 1.0 / 16, 1)          # ROIAlign(sampling_ratio=1), roi_align.py:51
        x = self.roi_head_feature_extractor(pooled)
        if x.shape[1] != (7 if not self.c5_dilated else 14):
            raise NotImplementedError("vlbert_b200: AvgPool2d window must cover the whole res5 map")
        if segms is not None:
            m = segms[inds[:, 0], inds[:, 1]] if inds is not None else segms.reshape(B * R, *segms.shape[2:])
            if tuple(m.shape[1:]) != tuple(x.shape[1:3]):
                raise ValueError("vlbert_b200: segms of size %s do not match the res5 map %s" % (tuple(m.shape[1:]), tuple(x.shape[1:3])))
            x = x * m.to(x.dtype).unsqueeze(-1)                                      # NHWC: mask broadcast over channels
        post = VF.AvgPoolFn.apply(x)                                              # [K, 2048] f32
        if inds is None:
            return post.view(B, R, -1), post, None
        full = post.new_zeros((B, R, post.shape[1]))
        full = full.index_put((inds[:, 0], inds[:, 1]), post)
        return full, post, inds

    def forward(self, images, boxes, box_mask, im_info, classes=None, segms=None, mvrc_ops=None, mask_visual_embed=None):
        drop = None
        if self.training and self.obj_downsample[0].p > 0:
            self._rng_state[1] += 1
            drop = VF.DropSite(self.obj_downsample[0].p, self.DROP_SITE, self._rng_state.clone())
        lin = self.obj_downsample[1]
        extra = {}
        if self.image_feat_precomputed:
            feats = boxes[:, :, 4:]                      # (segms are unused on the precomputed path, as in the reference)
        else:
            feats, post, inds = self._region_features(images, boxes, box_mask, segms)
            if self.enable_cnn_reg_loss:
                if inds is None:
                    inds = box_mask.nonzero()
                    post = feats[inds[:, 0], inds[:, 1]]
                obj_labels = classes[inds[:, 0], inds[:, 1]].type(torch.long)
                obj_logits = self.regularizing_predictor(post)
                extra = {"obj_logits": obj_logits, "obj_labels": obj_labels,
                         "cnn_regularization_loss": F.cross_entropy(obj_logits, obj_labels)[None]}
        if mvrc_ops is not None and mask_visual_embed is not None:
            feats = feats.clone()
            feats[mvrc_ops == 1] = mask_visual_embed
        packed = torch.cat((boxes[:, :, :4].to(feats.dtype), feats), -1)
        obj_reps, raw = VF.RegionFn.apply(packed, lin.weight, lin.bias, box_mask, im_info, drop)
        out = {"obj_reps_raw": raw, "obj_reps": obj_reps}
        out.update(extra)
        return out
