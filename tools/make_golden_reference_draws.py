"""Write tests/golden/reference_augmentation_draws.json from the reference's OWN augment_audio_signal
(open_seq2seq/data/speech2text/speech_utils.py:225-268), executed from a checkout of the reference: for seeded
global np.random streams, the output length and the drawn noise level of every call.
The reference module is loaded by path with resampy replaced by the oracle's restatement (only the LENGTH of its
result enters the fixture); see tests/test_reference_executed_cpu.py.

    python tools/make_golden_reference_draws.py <checkout of NVIDIA/OpenSeq2Seq>
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))
sys.path.insert(0, ROOT)
from tests.test_reference_executed_cpu import load_reference_speech_utils  # noqa: E402

AUGS = [
    {"speed_perturbation_ratio": [0.9, 1.0, 1.1]},
    {"speed_perturbation_ratio": 0.1},
    {"speed_perturbation_ratio": [0.9, 1.1], "noise_level_min": -90, "noise_level_max": -46},
    {"noise_level_min": -60, "noise_level_max": -50},
]


def main():
    ref = load_reference_speech_utils(sys.argv[1])
    n, sr = 23456, 16000
    cases = []
    for aug in AUGS:
        for seed in range(8):
            np.random.seed(seed)
            drawn = []
            orig = np.random.randint

            def spy(*a, **k):
                v = orig(*a, **k)
                drawn.append(int(v))
                return v
            np.random.randint = spy
            try:
                out = ref.augment_audio_signal(np.zeros(n, dtype=np.float32), sr, aug)
            finally:
                np.random.randint = orig
            cases.append({"seed": seed, "augmentation": aug, "n_out": int(len(out)),
                          "noise_level_db": drawn[0] if drawn else None})
    path = os.path.join(ROOT, "tests", "golden", "reference_augmentation_draws.json")
    with open(path, "w") as f:
        json.dump({"source": "open_seq2seq/data/speech2text/speech_utils.py:225-268 executed by "
                             "tools/make_golden_reference_draws.py", "n_samples": n, "sample_freq": sr, "cases": cases},
                  f, indent=1)
    print(path, len(cases), "cases")


if __name__ == "__main__":
    main()
