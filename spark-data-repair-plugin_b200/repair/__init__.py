"""B200-native drop-in for the hot path of maropu/spark-data-repair-plugin's ``repair`` package:
``delphi.repair.setInput(..).setRowId(..).setErrorDetectors([..]).run()`` backed by hand-written
sm_100a CUDA (``libb200repair.so``) instead of Spark SQL + pandas UDFs."""
from .api import Delphi  # noqa: F401
from .errors import (ConstraintErrorDetector, DomainValues, ErrorDetector,  # noqa: F401
                     GaussianOutlierErrorDetector, LOFOutlierErrorDetector, NullErrorDetector, RegExErrorDetector,
                     ScikitLearnBackedErrorDetector, ScikitLearnBasedErrorDetector)
from .model import RepairModel  # noqa: F401

delphi = Delphi.getOrCreate()
