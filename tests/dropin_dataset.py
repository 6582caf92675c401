"""Inference dataset through which tests/golden/make_golden.py feeds clips to the reference's inferencer: the interface of its
fullsubnet/dataset/dataset_inference.py:10-45 (``__getitem__`` -> (float32 waveform, basename)) without librosa: the clips come
from one .npy file."""
import numpy as np
from torch.utils import data


class Dataset(data.Dataset):
    def __init__(self, npy_path, sr):
        super().__init__()
        self.clips = np.load(npy_path).astype(np.float32)
        self.sr = sr

    def __len__(self):
        return len(self.clips)

    def __getitem__(self, item):
        return self.clips[item], f"clip{item}"
