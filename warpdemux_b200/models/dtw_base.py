"""`BaseDTWModel` — same fields and methods as the reference's
(warpdemux/models/dtw_base.py:13-77), holding plain arrays instead of an
sklearn estimator, plus the lazily created device replica."""
import logging
from abc import ABC, abstractmethod
from typing import Dict, Optional, Tuple, Union

import numpy as np
import pandas as pd

from ..model_io import ModelParams
from .utils import process_probs as _process_probs


class BaseDTWModel(ABC):
    def __init__(self, params: Optional[ModelParams] = None, device: Optional[int] = None):
        self.params: Optional[ModelParams] = params
        self.device: Optional[int] = device
        self._dev = None  # DeviceModel, created in the calling process on first predict

    # -- the reference's attribute names, served from the arrays ------------
    @property
    def _X(self):
        return None if self.params is None else self.params.sv

    @property
    def model(self):
        """The reference stores an sklearn SVC here; this backend stores its
        arrays (`self.params`).  Truthy when trained."""
        return self.params

    @property
    def window(self):
        return self.params.window

    @property
    def penalty(self):
        return self.params.penalty

    @property
    def block_size(self):
        return self.params.block_size

    @property
    def thresholds(self):
        return self.params.thresholds

    @thresholds.setter
    def thresholds(self, v):
        self.params.thresholds = np.ascontiguousarray(v, dtype=np.float64)
        self._drop_device()

    @property
    def label_mapper(self) -> Dict[int, int]:
        return self.params.label_mapper

    @property
    def noise_class(self) -> bool:
        return self.params.noise_class

    @property
    def n_classes(self) -> int:
        return self.params.k

    @property
    def is_trained(self):
        return self.params is not None and self.params.sv is not None

    @property
    def num_bcs(self):
        if self.params is None:
            msg = "Model not trained yet."
            logging.error(msg)
            raise ValueError(msg)
        return self.params.k

    @abstractmethod
    def predict(self, X: np.ndarray, nproc: int = -1, block_size: Optional[int] = None, pbar: bool = False,
                pbar_kwargs: dict = {}, return_df: bool = False
                ) -> Union[Tuple[np.ndarray, np.ndarray], pd.DataFrame]:
        ...

    def get_thresholds(self) -> np.ndarray:
        return self.thresholds

    def process_probs(self, y_prob: np.ndarray) -> Tuple[np.ndarray, np.ndarray]:
        if self.params is None or self.params.label_map is None:
            msg = "Label mapper not set."
            logging.error(msg)
            raise ValueError(msg)
        return _process_probs(y_prob, self.label_mapper, self.get_thresholds())

    # -- device replica -------------------------------------------------------
    def _drop_device(self):
        if self._dev is not None:
            self._dev.close()
            self._dev = None

    def _device_model(self):
        # the thresholds are applied on the device: when another holder of the same params replaced them (the lanes of
        # MinibatchDemuxer share lane 0's params), this replica rebuilds too
        if self._dev is not None and self._dev.thresholds is not self.params.thresholds:
            self._drop_device()
        if self._dev is None:
            from ..device_model import DeviceModel
            from ..sharding import default_device

            self._dev = DeviceModel(self.params, default_device() if self.device is None else self.device)
        return self._dev

    # pickling: the reference pickles the model into every worker task
    # (file_proc.py:1232-1243); carry host arrays only, rebuild on the device lazily.
    def __getstate__(self):
        st = dict(self.__dict__)
        st["_dev"] = None
        return st

    def __setstate__(self, st):
        self.__dict__.update(st)
        self._dev = None
