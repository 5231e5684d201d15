"""Same module name as the reference's ``poor_man_gplvm/test.py`` (shuffle tests of a fitted model; NOT pytest tests);
implementation in ``batched.py``."""
from .batched import (circular_shuffle_data, compute_entropy, draw_shifts, normalize_shifts,  # noqa: F401
                      quantile_rows, shuffle_and_decode, shuffle_test, test_one_model)
