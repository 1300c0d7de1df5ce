"""The SM-pair (cta_group::2) schedule of the 256-row dataflow tower launches gives the bits the single-CTA kernel
gave, at the shapes where its schedule has edge cases: a null tile (odd tile count), an odd CTA limit, fewer pair
items than pairs, the bench's 1024 boards, and the two-stream PipelinedSearchPlan with the confined tree kernel of
one sub-batch beside the tower of the other.  tests/golden/pair_golden.npz was recorded with the single-CTA kernel
(tests/golden/make_golden_pair.py)."""
import os

import numpy as np
import pytest

from conftest import GOLDEN
from pair_cases import CASES, build_net, run_case, run_search

pytestmark = pytest.mark.gpu


@pytest.fixture(scope='module')
def net():
    return build_net()


@pytest.fixture(scope='module')
def golden():
    return np.load(os.path.join(GOLDEN, 'pair_golden.npz'))


@pytest.mark.parametrize('name,batch,cta_limit,rows', CASES, ids=[c[0] for c in CASES])
def test_pair_tower_bits_equal_the_single_cta_kernel(net, golden, name, batch, cta_limit, rows):
    got = run_case(net, batch, cta_limit, rows)
    for k, v in got.items():
        assert np.array_equal(v, golden[f'{name}_{k}']), f'{name}: {k} differs'


def test_two_stream_search_equals_single_plan_and_recording(net, golden):
    piped = run_search(net, parts=2)
    single = run_search(net, parts=1)
    for k in piped:
        assert np.array_equal(piped[k], single[k]), f'pipelined vs single plan: {k} differs'
        assert np.array_equal(piped[k], golden[f'search_{k}']), f'{k} differs from the recording'
