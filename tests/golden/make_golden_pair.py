"""Seeded Gomoku tower outputs at the shapes whose 256-row dataflow launches exercise the edge cases of the SM-pair
schedule (run on a GPU with the build whose results are the reference, i.e. the single-CTA tower kernel):

    python tests/golden/make_golden_pair.py [OUT.npz]

Writes tests/golden/pair_golden.npz: for every case of pair_cases.CASES, the SHA-256 of the hidden-state slots, policy,
value and reward that initial_inference_batch followed by recurrent_inference_batch return (the recurrent inference
runs the 33-conv dynamics + prediction tower as ONE launch), and the same digests for one batched search through the
two-sub-batch PipelinedSearchPlan.  tests/test_conv_pair_gpu.py compares against them byte for byte.
"""
from __future__ import annotations

import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.dirname(HERE))
sys.path.insert(0, os.path.dirname(os.path.dirname(HERE)))

from pair_cases import CASES, build_net, run_case, run_search  # noqa: E402


def main(out: str) -> None:
    net = build_net()
    rec = {}
    for name, batch, cta_limit, rows in CASES:
        for k, v in run_case(net, batch, cta_limit, rows).items():
            rec[f'{name}_{k}'] = v
    for k, v in run_search(net, parts=2).items():
        rec[f'search_{k}'] = v
    np.savez(out, **rec)
    print(f'wrote {out}: {len(rec)} digests')


if __name__ == '__main__':
    main(sys.argv[1] if len(sys.argv) > 1 else os.path.join(HERE, 'pair_golden.npz'))
