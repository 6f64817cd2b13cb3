"""
The noise predictor, with the reference's loading surface and a CUDA-only forward.

Drop-in for the parts of /root/reference/foldingdiff/modelling.py that the sampler uses:
  * `BertForDiffusionBase.from_dir(dirname, ft_is_angular=None, load_weights=True, idx=-1,
    best_by="valid", copy_to="", **kwargs)`                         (reference :297-382)
  * `model(inputs, timestep, attention_mask=..., position_ids=None)`  (reference :384-484)
  * `.to(device) / .eval() / .parameters() / .state_dict()`, `.n_inputs`, `.ft_is_angular`,
    `.ft_names`, `.config`
  * `BertForDiffusion` - in the reference a pytorch-lightning training wrapper (:487-804); here
    the same loader/forward plus the evaluation half of training: the reference's constructor kwargs,
    `_get_loss_terms` and `validation_step` on the device (the backward pass is out of scope).

What is different by design: there is no HuggingFace `BertEncoder` and no PyTorch eager forward.
The module only *holds* the parameters under the reference's state-dict names (so checkpoints
load strictly); `forward` hands device pointers to the hand-written sm_100a kernels behind the C
ABI (`engine.Engine`).  On a CPU device `forward` raises: there is no fallback path.
"""
from __future__ import annotations

import glob
import json
import logging
import os
import re
import shutil
from pathlib import Path
from typing import Dict, List, Literal, Optional, Sequence, Union

import torch
from torch import nn

from . import _native, engine, losses
from .datasets import FEATURE_SET_NAMES_TO_ANGULARITY

TIME_ENCODING = Literal["gaussian_fourier", "sinusoidal"]
DECODER_HEAD = Literal["mlp", "linear"]
DEFAULT_GEMM = os.environ.get("FOLDINGDIFF_B200_GEMM", "tc3x")


class BertConfig:
    """Minimal stand-in for transformers.BertConfig: the keys of the model dir's config.json."""

    _defaults = dict(hidden_size=768, num_hidden_layers=12, num_attention_heads=12, intermediate_size=3072,
                     hidden_act="gelu", hidden_dropout_prob=0.1, attention_probs_dropout_prob=0.1,
                     max_position_embeddings=512, initializer_range=0.02, layer_norm_eps=1e-12,
                     position_embedding_type="absolute", is_decoder=False, model_type="bert")

    def __init__(self, **kwargs):
        self.__dict__.update(self._defaults)
        self.__dict__.update(kwargs)

    @classmethod
    def from_json_file(cls, path: str) -> "BertConfig":
        with open(path) as f:
            return cls(**json.load(f))

    def to_dict(self) -> dict:
        return dict(self.__dict__)

    def save_pretrained(self, dirname) -> None:
        os.makedirs(dirname, exist_ok=True)
        with open(os.path.join(dirname, "config.json"), "w") as f:
            json.dump(self.to_dict(), f, indent=2, sort_keys=True)


class _Holder(nn.Module):
    """Parameter container; exists only so state-dict keys match the reference checkpoint."""


def _linear(i: int, o: int) -> nn.Linear:
    return nn.Linear(i, o)


def mask_layout(attention_mask: torch.Tensor):
    """
    -> (lengths, mask_cpu, is_prefix) of a (B, N) attention mask: per-chain valid-token counts, the mask as fp32 on the
    host, and whether every row is a prefix mask (tokens [0, lengths[b]) valid, lengths[b] >= 1) - the layout the
    packed-row path of fd_set_batch serves without a key mask.
    """
    mask_cpu = attention_mask.detach().to("cpu", torch.float32)
    N = mask_cpu.shape[1]
    lengths = mask_cpu.sum(dim=1).to(torch.int64)
    prefix = torch.arange(N)[None, :] < lengths[:, None]
    is_prefix = bool(torch.equal(prefix, mask_cpu > 0.5)) and bool((lengths >= 1).all())
    return lengths.tolist(), mask_cpu, is_prefix


class BertForDiffusionBase(nn.Module):
    """BERT-style epsilon predictor on continuous angle inputs; compute runs in native CUDA."""

    def __init__(self, config: BertConfig, ft_is_angular: List[bool] = [False, True, True, True],
                 ft_names: Optional[List[str]] = None, time_encoding: TIME_ENCODING = "gaussian_fourier",
                 decoder: DECODER_HEAD = "mlp", gemm: Optional[str] = None, **_training_kwargs) -> None:
        super().__init__()
        self.config = config
        if getattr(config, "is_decoder", False):
            raise NotImplementedError
        if config.position_embedding_type != "relative_key":
            raise NotImplementedError(
                f"position_embedding_type={config.position_embedding_type!r}: every shipped foldingdiff config "
                "uses 'relative_key' (config_jsons/*.json); other types are not implemented in the CUDA path")
        if decoder != "mlp":
            raise NotImplementedError(f"decoder={decoder!r}: only the 'mlp' head (AnglesPredictor) is implemented")
        if config.hidden_act != "gelu":
            raise NotImplementedError(f"hidden_act={config.hidden_act!r}")
        self.ft_is_angular = list(ft_is_angular)
        self.n_inputs = len(self.ft_is_angular)
        self.ft_names = list(ft_names) if ft_names is not None else [f"ft{i}" for i in range(self.n_inputs)]
        assert len(self.ft_names) == self.n_inputs
        self.time_encoding = time_encoding
        self.gemm = gemm or DEFAULT_GEMM

        H, I = config.hidden_size, config.intermediate_size
        dh = H // config.num_attention_heads
        self.inputs_to_hidden_dim = _linear(self.n_inputs, H)
        self.embeddings = _Holder()
        self.embeddings.LayerNorm = nn.LayerNorm(H, eps=config.layer_norm_eps)
        self.encoder = _Holder()
        self.encoder.layer = nn.ModuleList()
        for _ in range(config.num_hidden_layers):
            lyr = _Holder()
            lyr.attention = _Holder()
            lyr.attention.self = _Holder()
            lyr.attention.self.query = _linear(H, H)
            lyr.attention.self.key = _linear(H, H)
            lyr.attention.self.value = _linear(H, H)
            lyr.attention.self.distance_embedding = nn.Embedding(2 * config.max_position_embeddings - 1, dh)
            lyr.attention.output = _Holder()
            lyr.attention.output.dense = _linear(H, H)
            lyr.attention.output.LayerNorm = nn.LayerNorm(H, eps=config.layer_norm_eps)
            lyr.intermediate = _Holder()
            lyr.intermediate.dense = _linear(H, I)
            lyr.output = _Holder()
            lyr.output.dense = _linear(I, H)
            lyr.output.LayerNorm = nn.LayerNorm(H, eps=config.layer_norm_eps)
            self.encoder.layer.append(lyr)
        self.token_decoder = _Holder()
        self.token_decoder.dense1 = _linear(H, H)
        self.token_decoder.layer_norm = nn.LayerNorm(H, eps=1e-12)
        self.token_decoder.dense2 = _linear(H, self.n_inputs)
        self.time_embed = _Holder()
        if time_encoding == "gaussian_fourier":
            self.time_embed.register_buffer("W", torch.randn(H // 2) * 2 * torch.pi)
        elif time_encoding != "sinusoidal":
            raise ValueError(f"Unknown time encoding: {time_encoding}")
        self._init_weights()
        for p in self.parameters():
            p.requires_grad_(False)
        self._engine: Optional[engine.Engine] = None
        self._engine_key = None

    def _init_weights(self):
        # BertPreTrainedModel._init_weights: N(0, initializer_range) weights, zero biases, unit LayerNorm
        std = self.config.initializer_range
        for m in self.modules():
            if isinstance(m, (nn.Linear, nn.Embedding)):
                m.weight.data.normal_(mean=0.0, std=std)
                if isinstance(m, nn.Linear) and m.bias is not None:
                    m.bias.data.zero_()
            elif isinstance(m, nn.LayerNorm):
                m.bias.data.zero_()
                m.weight.data.fill_(1.0)

    # ------------------------------------------------------------------------------------------
    @classmethod
    def from_dir(cls, dirname: str, ft_is_angular: Optional[Sequence[bool]] = None, load_weights: bool = True,
                 idx: int = -1, best_by: Literal["train", "valid"] = "valid", copy_to: str = "", **kwargs):
        """Build the model from a training output directory (config.json, training_args.json, models/)."""
        with open(os.path.join(dirname, "training_args.json")) as f:
            train_args = json.load(f)
        config = BertConfig.from_json_file(os.path.join(dirname, "config.json"))
        if ft_is_angular is None:
            ft_is_angular = FEATURE_SET_NAMES_TO_ANGULARITY[train_args["angles_definitions"]]
            logging.info(f"Auto constructed ft_is_angular: {ft_is_angular}")
        time_key = "time_encoding" if "time_encoding" in train_args else "seq_len_encoding"
        model = cls(config=config, ft_is_angular=ft_is_angular, time_encoding=train_args[time_key],
                    decoder=train_args["decoder"], **kwargs)
        subfolder = f"best_by_{best_by}"
        ckpt_name = None
        if load_weights:
            def epoch_of(path):
                return int(re.findall(r"epoch=[0-9]+", os.path.basename(path)).pop().split("=")[-1])
            ckpts = sorted(glob.glob(os.path.join(dirname, "models", subfolder, "*.ckpt")), key=epoch_of)
            logging.info(f"Found {len(ckpts)} checkpoints")
            ckpt_name = ckpts[idx]  # IndexError when the folder is empty, like the reference
            logging.info(f"Loading weights from {ckpt_name}")
            loaded = torch.load(ckpt_name, map_location=torch.device("cpu"), weights_only=True)
            model.load_state_dict(loaded["state_dict"])
        else:
            logging.info(f"Loaded unitialized model from {dirname}")
        if copy_to:
            logging.info(f"Copying minimal model file set to: {copy_to}")
            dst = Path(copy_to)
            os.makedirs(dst, exist_ok=True)
            with open(dst / "training_args.json", "w") as f:
                json.dump(train_args, f)
            config.save_pretrained(dst)
            if load_weights:
                os.makedirs(dst / "models" / subfolder, exist_ok=True)
                shutil.copyfile(ckpt_name, dst / "models" / subfolder / os.path.basename(ckpt_name))
        return model

    # ------------------------------------------------------------------------------------------
    def _time_rows(self, t: torch.Tensor) -> torch.Tensor:
        if self.time_encoding == "gaussian_fourier":
            return engine.gaussian_fourier_rows(self.time_embed.W, t)
        return engine.sinusoidal_rows(self.config.hidden_size, t)

    def native_engine(self) -> engine.Engine:
        """The native handle for the parameters' current device (built lazily, rebuilt on change)."""
        p = next(self.parameters())
        if p.device.type != "cuda":
            raise _native.NativeError(
                f"model is on {p.device}; foldingdiff_b200 computes on CUDA (sm_100a) only - "
                "move it with .to('cuda:0'). There is no CPU fallback.")
        key = (p.device, tuple(int(q._version) for q in self.parameters()), self.gemm)
        if self._engine is None or self._engine_key != key:
            if self._engine is not None:
                self._engine.close()
            cfg = self.config
            self._engine = engine.Engine(
                self.state_dict(), hidden=cfg.hidden_size, layers=cfg.num_hidden_layers,
                heads=cfg.num_attention_heads, intermediate=cfg.intermediate_size,
                max_pos=cfg.max_position_embeddings, n_features=self.n_inputs, ln_eps=cfg.layer_norm_eps,
                time_rows_fn=self._time_rows, device=p.device, gemm=self.gemm)
            self._engine_key = key
        return self._engine

    def set_gemm(self, gemm: str) -> "BertForDiffusionBase":
        """'tc3x' (tensor cores, error-compensated; default), 'fp32' (CUDA-core reference), 'tc1x'."""
        assert gemm in _native.GEMM_MODES
        self.gemm = gemm
        if self._engine is not None:
            self._engine.set_gemm(gemm)
            self._engine_key = self._engine_key[:2] + (gemm,)
        return self

    @torch.no_grad()
    def forward(self, inputs: torch.Tensor, timestep: torch.Tensor, attention_mask: torch.Tensor,
                position_ids: Optional[torch.Tensor] = None, **_hf_kwargs) -> torch.Tensor:
        """
        eps_hat (B, N, F) for inputs (B, N, F), timestep (B,) or (B, 1), attention_mask (B, N) in {0, 1}.
        `position_ids` is accepted for signature compatibility; relative_key attention ignores it
        (reference modelling.py:164-166).  Every row is computed, like the reference.
        """
        assert attention_mask is not None
        assert attention_mask.dim() == 2, \
            f"Attention mask expected in shape (batch_size, seq_length), got {attention_mask.shape}"
        assert inputs.dim() == 3
        eng = self.native_engine()
        B, N, _ = inputs.shape
        lengths, mask_cpu, is_prefix = mask_layout(attention_mask)
        if is_prefix:
            eng.set_batch(lengths, N, all_rows=True)
        else:
            eng.set_batch([N] * B, N, all_rows=True, key_mask=mask_cpu)
        t = timestep.detach().reshape(-1).to("cpu")
        temb = self._time_rows(t).to(inputs.device)
        x = inputs.detach().to(torch.float32).contiguous()
        return eng.forward(x, temb)


class BertForDiffusion(BertForDiffusionBase):
    """
    The reference's training wrapper (modelling.py:487-804) as far as evaluation goes: it takes the training kwargs of
    bin/train.py:446-459 and evaluates the training objective on the device (`_get_loss_terms`, `validation_step`;
    kernels in csrc/loss.cuh).  The backward pass, the optimizer and dropout are not implemented: `training_step` raises.
    `lr`, `l1`, `l2`, `epochs`, `steps_per_epoch` and `lr_scheduler` are stored for signature compatibility only.
    """

    def __init__(self, lr: float = 5e-5, loss: str = "smooth_l1",
                 use_pairwise_dist_loss: Union[float, Sequence[float]] = 0.0, l2: float = 0.0, l1: float = 0.0,
                 circle_reg: float = 0.0, epochs: int = 1, steps_per_epoch: int = 250, lr_scheduler=None,
                 write_preds_to_dir: Optional[str] = None, **kwargs):
        super().__init__(**kwargs)
        if callable(loss) or not isinstance(loss, str):
            raise NotImplementedError(f"loss={loss!r}: only the named losses {sorted(losses.LOSS_KINDS)} (and the "
                                      "autocorrected 'radian_l1_smooth') have device kernels; a callable loss does not")
        loss = losses.LOSS_AUTOCORRECT.get(loss, loss)  # modelling.py:515-521
        if loss not in losses.LOSS_KINDS:
            raise ValueError(f"loss={loss!r}: expected one of {sorted(losses.LOSS_KINDS)} or 'radian_l1_smooth'")
        if write_preds_to_dir:
            raise NotImplementedError("write_preds_to_dir: writing validation predictions is not implemented")
        self.loss = loss
        self.learning_rate = lr
        self.use_pairwise_dist_loss = list(use_pairwise_dist_loss) if isinstance(use_pairwise_dist_loss, (list, tuple)) \
            else float(use_pairwise_dist_loss)
        self.l1_lambda, self.l2_lambda = l1, l2
        self.circle_lambda = float(circle_reg)
        self.epochs, self.steps_per_epoch, self.lr_scheduler = epochs, steps_per_epoch, lr_scheduler
        self.write_preds_to_dir = None

    @property
    def pdist_enabled(self) -> bool:
        """modelling.py:610-613: the list form, or a positive scalar, switches the pairwise-distance term on."""
        return isinstance(self.use_pairwise_dist_loss, list) or self.use_pairwise_dist_loss > 0

    def _circle_mask(self) -> torch.Tensor:
        """1.0 for the features whose loss carries the circle penalty (angular smooth-L1), else 0.0."""
        on = self.loss == "smooth_l1" and self.circle_lambda > 0
        return torch.tensor([1.0 if (a and on) else 0.0 for a in self.ft_is_angular], dtype=torch.float64)

    @torch.no_grad()
    def _loss_terms_detail(self, batch):
        """_get_loss_terms plus the per-chain sums the terms were reduced from (validation_loss builds its per-timestep
        table from them): -> (terms, {"eps_hat", "chain_sums"[, "pdist_chain_sums"]})."""
        eng = self.native_engine()
        dev = next(self.parameters()).device
        corrupted = batch["corrupted"].detach().to(dev, torch.float32).contiguous()
        known = batch["known_noise"].detach().to(dev, torch.float32).contiguous()
        assert corrupted.dim() == 3 and known.shape == corrupted.shape, f"{known.shape} != {corrupted.shape}"
        attn_mask = batch["attn_mask"]
        assert attn_mask.dim() == 2
        B, N, _ = corrupted.shape
        lengths, mask_cpu, is_prefix = mask_layout(attn_mask)
        pdist_lengths = None
        if self.pdist_enabled:
            pdist_lengths = [int(l) for l in batch["lengths"].reshape(-1).tolist()]
        # Only the rows the loss reads are computed: padded rows enter no term (the pairwise term reads rows below
        # batch["lengths"], which a dataset item sets to the mask's length).
        if is_prefix and (pdist_lengths is None or all(p <= l for p, l in zip(pdist_lengths, lengths))):
            eng.set_batch(lengths, N, all_rows=False)
        else:
            eng.set_batch([N] * B, N, all_rows=True, key_mask=mask_cpu)
        t = batch["t"].detach().reshape(-1).to("cpu")
        temb = self._time_rows(t).to(dev)
        eps_hat = eng.forward(corrupted, temb)
        terms, chain = losses.loss_terms(eps_hat, known, attn_mask.to(dev), self.ft_is_angular, self.loss,
                                         self.circle_lambda)
        detail = {"eps_hat": eps_hat, "chain_sums": chain}
        if self.pdist_enabled:
            tt = batch["t"].detach().to(dev)
            coef = losses.pdist_coefficients(self.use_pairwise_dist_loss, tt)
            pd, pchain = losses.pdist_loss(corrupted, eps_hat, batch["angles"].to(dev),
                                           batch["sqrt_alphas_cumprod_t"].to(dev),
                                           batch["sqrt_one_minus_alphas_cumprod_t"].to(dev), coef, pdist_lengths,
                                           self.ft_names)
            terms = torch.cat([terms, pd.reshape(1)])
            detail["pdist_chain_sums"] = pchain
        return terms, detail

    def _get_loss_terms(self, batch, write_preds: Optional[str] = None) -> torch.Tensor:
        """
        The reference's _get_loss_terms (modelling.py:553-677) on the device: (F,) per-feature terms, (F+1,) with the
        pairwise-distance term, fp32 on the model's device.  `batch` is the default_collate of NoisedAnglesDataset
        items (corrupted, t, known_noise, attn_mask, position_ids, lengths, angles, sqrt_*_t), on CPU or CUDA.
        The network runs on the valid rows only when the mask is a prefix mask (exact: padded rows enter no term).
        """
        if write_preds is not None:
            raise NotImplementedError("write_preds: writing validation predictions is not implemented")
        return self._loss_terms_detail(batch)[0]

    def validation_step(self, batch, batch_idx) -> Dict[str, torch.Tensor]:
        """modelling.py:719-750, without the logging: {"val_loss": mean of the terms}."""
        return {"val_loss": torch.mean(self._get_loss_terms(batch))}

    def training_step(self, batch, batch_idx):
        raise NotImplementedError("training_step needs the backward pass (gradient of the loss through the network) and "
                                  "the optimizer, which foldingdiff_b200 does not implement; evaluate with "
                                  "_get_loss_terms / validation_step / losses.validation_loss")
