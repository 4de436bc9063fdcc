"""CPU oracle of the speaker normalisation around the mel front-end / back-end (reference data_utils.py:35-47).  TEST
INFRASTRUCTURE ONLY: attack.py normalises file2mel's output with the checkpoint's attr.pkl statistics before the attack and
denormalises the result before mel2wav.  Pinned against the reference's own functions in test_defend_cpu.py when
ATTACK_VC_REFERENCE is set."""
import numpy as np


def normalize(mel: np.ndarray, mean: np.ndarray, std: np.ndarray) -> np.ndarray:
    """data_utils.py:35-40: (mel - mean) / std per mel bin over the frames of [n_frames, n_mels]."""
    return (mel - mean) / std


def denormalize(mel: np.ndarray, mean: np.ndarray, std: np.ndarray) -> np.ndarray:
    """data_utils.py:43-47: mel * std + mean."""
    return mel * std + mean
