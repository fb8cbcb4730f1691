"""Mirror of ``Quanta.nn`` (Quanta/nn/__init__.py exports Linear8bitLt, Linear4bit)."""
from .linear import Linear8bitLt, Linear4bit
from .functional import (linear_wna16, linear_nf4a16, linear_wna16_dgrad, linear_nf4a16_dgrad, int8_outlier_matmul,
                         int8_outlier_dgrad, rowwise_quantize_sym)

__all__ = ["Linear8bitLt", "Linear4bit", "linear_wna16", "linear_nf4a16", "linear_wna16_dgrad", "linear_nf4a16_dgrad",
           "int8_outlier_matmul", "int8_outlier_dgrad", "rowwise_quantize_sym"]
