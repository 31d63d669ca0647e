"""Architecture contract of the Xception-UQ classifier -- mirrors reference biscuit/hp.py:3-24
(`nature2022 = sf.model.ModelParams(...)`).  Only the fields that define INFERENCE are kept; the
training fields of the reference (optimizer, learning rate, augmentation, early stopping;
hp.py:9-18,23) are out of scope."""
from __future__ import annotations

from dataclasses import dataclass, replace


@dataclass(frozen=True)
class ModelConfig:
    model: str = "xception"            # hp.py:4
    tile_px: int = 299                 # hp.py:5
    tile_um: int = 302                 # hp.py:6
    batch_size: int = 128              # hp.py:7  (reference inference batch)
    dropout: float = 0.1               # hp.py:11
    uq: bool = True                    # hp.py:12 (enabled in the UQ sub-experiments, experiment.py:849); the GPU
                                       # interface only does MC-dropout inference: UncertaintyInterface rejects False
    hidden_layer_width: int = 1024     # hp.py:13; a multiple of 64, at most 1024 (the fused head's limit)
    normalizer: str | None = None      # hp.py:19 'reinhard_fast' -- stain normalisation is a "next" row
    include_top: bool = False          # hp.py:20
    hidden_layers: int = 2             # hp.py:21
    pooling: str = "avg"               # hp.py:22
    n_classes: int = 2                 # 2..8
    uq_samples: int = 30               # Slideflow's hard-coded MC-dropout sample count
    # where Dropout(rate) fires at inference when `uq` is on: (after the pooled 2048-d features, after hidden_0,
    # after hidden_1).  hp.py:11-12 fix only the rate and the `uq` flag; the placement is Slideflow's and differs
    # between its versions (INTEGRATION.md): (False, True, True) = after every hidden layer (default here),
    # (True, True, True) = additionally right after `post_convolution`.  At least one site must be on: a model
    # without dropout has no uncertainty to estimate (`dropout_site_mask` raises ValueError).
    dropout_sites: tuple = (False, True, True)

    @property
    def dropout_site_mask(self) -> int:
        sites = tuple(bool(x) for x in self.dropout_sites)
        if len(sites) != self.hidden_layers + 1:
            raise ValueError("dropout_sites needs one flag per site: pooled features + each hidden layer")
        if not any(sites):
            raise ValueError("dropout_sites needs at least one enabled site")
        return sum(1 << i for i, on in enumerate(sites) if on)

    def replace(self, **kw) -> "ModelConfig":
        return replace(self, **kw)


nature2022 = ModelConfig()
