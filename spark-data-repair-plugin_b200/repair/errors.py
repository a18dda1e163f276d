"""Error detectors: same class names, constructors and ``setUp(...).detect()`` protocol as the
reference (``python/repair/errors.py:37-312``), evaluated by CUDA scans instead of Spark SQL.

A detector is a small value object; ``spec()`` lowers it to the dict the device pipeline
(``engine.Engine.detect``) consumes.  ``detect()`` on a detector that was ``setUp`` against an
input registered in the catalog returns a pandas frame ``(row_id, attribute)``.
"""
from abc import ABCMeta, abstractmethod
from typing import Any, Callable, Dict, List, Optional

from .utils import get_option_value


class ErrorDetector(metaclass=ABCMeta):

    def __init__(self, targets: List[str] = []) -> None:
        self.row_id: Optional[str] = None
        self.qualified_input_name: Optional[Any] = None
        self.continous_cols: List[str] = []
        self.targets: List[str] = targets

    def setUp(self, row_id: str, qualified_input_name: Any, continous_cols: List[str],
              targets: List[str]) -> "ErrorDetector":
        self.row_id = row_id
        self.qualified_input_name = qualified_input_name
        self.continous_cols = continous_cols
        self._targets = [t for t in targets if t in set(self.targets)] if self.targets else list(targets)
        return self

    @abstractmethod
    def spec(self) -> Dict[str, Any]:
        """The detector as a plain dict for the device pipeline."""

    def detect(self) -> Any:
        assert self.row_id is not None and self.qualified_input_name is not None
        from .model import detect_with
        return detect_with(self)


class NullErrorDetector(ErrorDetector):

    def __init__(self) -> None:
        ErrorDetector.__init__(self)

    def __str__(self) -> str:
        return "{}()".format(self.__class__.__name__)

    def spec(self):
        return {"type": "null"}


class DomainValues(ErrorDetector):

    def __init__(self, attr: str, values: List[str] = [], autofill: bool = False, min_count_thres: int = 12) -> None:
        ErrorDetector.__init__(self)
        self.attr = attr
        self.values = values if not autofill else []
        self.autofill = autofill
        self.min_count_thres = min_count_thres

    def __str__(self) -> str:
        return '{}(attr="{}",size={},autofill={},min_count_thres={})'.format(
            self.__class__.__name__, self.attr, len(self.values), self.autofill, self.min_count_thres)

    def spec(self):
        return {"type": "domain", "attr": self.attr, "values": list(self.values), "autofill": self.autofill,
                "min_count_thres": self.min_count_thres}


class RegExErrorDetector(ErrorDetector):

    def __init__(self, attr: str, regex: str) -> None:
        ErrorDetector.__init__(self)
        self.attr = attr
        self.regex = regex

    def __str__(self) -> str:
        return '{}(pattern="{}")'.format(self.__class__.__name__, self.regex)

    def spec(self):
        return {"type": "regex", "attr": self.attr, "regex": self.regex}


class ConstraintErrorDetector(ErrorDetector):

    def __init__(self, constraint_path: str = "", constraints: str = "", targets: List[str] = []) -> None:
        ErrorDetector.__init__(self, targets)
        if not constraint_path and not constraints:
            raise ValueError("At least one of `constraint_path` or `constraints` should be specified")
        self.constraint_path = constraint_path
        self.constraints = constraints

    def __str__(self) -> str:
        params = []
        if self.constraint_path:
            params.append("constraint_path={}".format(self.constraint_path))
        if self.constraints:
            params.append("constraints={}".format(self.constraints))
        if self.targets:
            params.append("targets={}".format(",".join(self.targets)))
        return "{}({})".format(self.__class__.__name__, ",".join(params))

    def spec(self):
        return {"type": "constraint", "path": self.constraint_path, "constraints": self.constraints,
                "targets": list(self.targets)}


class GaussianOutlierErrorDetector(ErrorDetector):

    def __init__(self, approx_enabled: bool = False) -> None:
        ErrorDetector.__init__(self)
        self.approx_enabled = approx_enabled

    def __str__(self) -> str:
        return "{}(approx_enabled={})".format(self.__class__.__name__, self.approx_enabled)

    def spec(self):
        return {"type": "outlier", "approx": self.approx_enabled}


class ScikitLearnBasedErrorDetector(ErrorDetector):
    """Per-column outlier detection over the continuous targets (errors.py:193-279).  The reference scores
    random partitions of tables with at least `parallel_mode_threshold` rows; here the whole column is scored
    at any size, so `parallel_mode_threshold` and `num_parallelism` are validated and kept but change
    nothing."""

    def __init__(self, parallel_mode_threshold: int = 10000, num_parallelism: Optional[int] = None) -> None:
        ErrorDetector.__init__(self)

        if num_parallelism is not None and int(num_parallelism) <= 0:
            raise ValueError(f'`num_parallelism` must be positive, got {num_parallelism}')

        self.parallel_mode_threshold = parallel_mode_threshold
        self.num_parallelism = num_parallelism

    def __str__(self) -> str:
        return f'{self.__class__.__name__}()'

    # An instance with a scikit-learn-like `fit_predict(X)` returning 1 (inlier) or -1 (outlier) per row.
    @abstractmethod
    def _outlier_detector_impl(self) -> Any:
        pass


class ScikitLearnBackedErrorDetector(ScikitLearnBasedErrorDetector):
    """A user-supplied estimator, fitted on the host per target column (NULLs filled with the median)."""

    def __init__(self, error_detector_cls: Callable[[], Any], parallel_mode_threshold: int = 10000,
                 num_parallelism: Optional[int] = None) -> None:
        ScikitLearnBasedErrorDetector.__init__(self, parallel_mode_threshold, num_parallelism)

        if not hasattr(error_detector_cls, "__call__"):
            raise ValueError('`error_detector_cls` should be callable')
        if not hasattr(error_detector_cls(), "fit_predict"):
            raise ValueError('An instance that `error_detector_cls` returns should have a `fit_predict` method')

        self.error_detector_cls = error_detector_cls

    def _outlier_detector_impl(self) -> Any:
        return self.error_detector_cls()

    def spec(self):
        return {"type": "sklearn", "factory": self._outlier_detector_impl}


class LOFOutlierErrorDetector(ScikitLearnBasedErrorDetector):
    """LocalOutlierFactor(novelty=False) per continuous target, computed exactly on the GPU (dr_lof_flag):
    k = min(20, n - 1), a cell is an error iff its local outlier factor exceeds 1.5."""

    def __init__(self, parallel_mode_threshold: int = 10000, num_parallelism: Optional[int] = None) -> None:
        ScikitLearnBasedErrorDetector.__init__(self, parallel_mode_threshold, num_parallelism)

    def _outlier_detector_impl(self) -> Any:
        from sklearn.neighbors import LocalOutlierFactor
        return LocalOutlierFactor(novelty=False)

    def spec(self):
        return {"type": "lof"}


class ErrorModelOptions:
    """Option carriers of the reference's ``ErrorModel`` (errors.py:321-346), keys kept verbatim."""
    _defs = [
        ("error.attr_freq_ratio_threshold", 0.0, float, lambda v: 0.0 <= v <= 1.0, "`{}` should be in [0.0, 1.0]"),
        ("error.pairwise_freq_ratio_threshold", 0.05, float, lambda v: 0.0 <= v <= 1.0,
         "`{}` should be in [0.0, 1.0]"),
        ("error.max_attrs_to_compute_pairwise_stats", 3, int, lambda v: v >= 2, "`{}` should be greater than 1"),
        ("error.max_attrs_to_compute_domains", 2, int, lambda v: v >= 2, "`{}` should be greater than 1"),
        ("error.domain_threshold_alpha", 0.0, float, lambda v: 0.0 <= v < 1.0, "`{}` should be in [0.0, 1.0)"),
        ("error.domain_threshold_beta", 0.70, float, lambda v: 0.0 <= v < 1.0, "`{}` should be in [0.0, 1.0)"),
    ]
    option_keys = set(d[0] for d in _defs)

    @classmethod
    def resolve(cls, opts):
        return {d[0]: get_option_value(opts, *d) for d in cls._defs}


def default_detectors(targets, columns):
    """errors.py:389-396: NULL + DomainValues(autofill, min_count_thres=4) per attribute."""
    dets: List[ErrorDetector] = [NullErrorDetector()]
    for c in (targets if targets else columns):
        dets.append(DomainValues(attr=c, autofill=True, min_count_thres=4))
    return dets
