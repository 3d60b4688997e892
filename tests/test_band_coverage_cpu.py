"""The synthetic band models of tests/band_models.py reach every template bound of the banded KKT kernels and the first
half bandwidth past each, in the exact-Hessian mode and in the knot-block mode (host-only `kkt.analyze`, no GPU). If the
ordering changes, this fails here instead of the GPU coverage of tests/test_kkt_band_coverage_gpu.py quietly shrinking."""
import os
import re

import pytest

import dto_b200 as D
from dto_b200 import _lib
from dto_b200 import kkt as PK

from band_models import BAND_CASES, band_kwargs, build_band, case_id

HERE = os.path.dirname(os.path.abspath(__file__))


def compiled_bounds():
    """The bounds BW of `dto_kkt_bw_bound` (csrc/dto_kkt_dev.h) per row width W: {16: [6, 9, 12, 15], 32: [20, 31]}"""
    src = open(os.path.join(HERE, "..", "directtrajectoryoptimization.jl_b200", "csrc", "dto_kkt_dev.h")).read()
    body = re.search(r"static inline int dto_kkt_bw_bound\(int W, int bw\)\s*\{(.*?)\n\}", src, re.S).group(1)
    narrow, wide = re.findall(r"return ([^;]*);", body)
    values = lambda expr: sorted({int(v) for v in re.findall(r"(?:\?|:)\s*(\d+)", expr)})   # noqa: E731
    return {16: values(narrow), 32: values(wide)}


@pytest.mark.parametrize("key", list(BAND_CASES), ids=[case_id(k) for k in BAND_CASES])
def test_band_model_bandwidth(key):
    exact, blocks = BAND_CASES[key]
    pn = D.solver_from(build_band(D, **band_kwargs(key)), batch=1).nlp
    assert PK.analyze(pn)[1] == exact
    if blocks is None:
        with pytest.raises(_lib.DtoError) as e:
            PK.analyze(pn, hessian="knot-blocks")
        assert e.value.status == -7
    else:
        assert PK.analyze(pn, hessian="knot-blocks")[1] == blocks
    # the bandwidth is a property of the knot pattern, not of the horizon
    pn6 = D.solver_from(build_band(D, **band_kwargs(key, T=6)), batch=1).nlp
    assert PK.analyze(pn6)[1] == exact


def test_band_table_covers_every_compiled_bound():
    bounds = compiled_bounds()
    assert bounds == {16: [6, 9, 12, 15], 32: [20, 31]}
    every = bounds[16] + bounds[32]
    first_past = [b + 1 for b in every[:-1]]                  # 7, 10, 13, 16, 21
    for mode in (0, 1):
        have = {v[mode] for v in BAND_CASES.values() if v[mode] is not None}
        assert set(every) <= have, (mode, sorted(set(every) - have))
        assert set(first_past) <= have, (mode, sorted(set(first_past) - have))
    assert any(v[0] == 32 for v in BAND_CASES.values())       # the exact mode's refusal
    assert any(v[1] is None for v in BAND_CASES.values())     # the knot-block mode's refusal
