"""CPU: the 2x2 neighbour regrouping of the mirror against the oracle and the reference's stored output, and the
`.safetensors` feature-file contract of README.md:151-161 (what the reference's loaders read back)."""
import os

import numpy as np
import pytest
import torch

from flash_vstream_b200 import feature_io
from flash_vstream_b200.vstream_arch import FlashVStreamB200, NeuralTuringMachine
from oracle import fvs_oracle as O

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")


def make_model(**cfg):
    return FlashVStreamB200(None, NeuralTuringMachine(64, 32), **cfg)


@pytest.mark.parametrize("B,g,D", [(3, 24, 16), (1, 16, 8), (2, 2, 4)])
def test_reshape_2x2_matches_oracle(B, g, D):
    x = torch.randn(B, g * g, D, generator=torch.Generator().manual_seed(g)).half()
    got = make_model().reshape_2x2_image_features(x)
    assert got.shape == (B, (g // 2) ** 2, 4 * D)
    assert np.array_equal(got.numpy(), O.reshape_2x2(x.numpy()))


def test_reshape_2x2_matches_reference():
    """the original reshape_2x2_image_features only moves elements: tests/golden/seams.npz holds its output on an
    index-coded [2, 576, 32] input, i.e. which input element lands where (tests/golden/make_golden_seams.py)"""
    gather = torch.from_numpy(np.load(os.path.join(G, "seams.npz"))["reshape_2x2_gather"]).long()
    x = torch.randn(2, 576, 32, generator=torch.Generator().manual_seed(5))
    ref = x.reshape(-1)[gather]
    assert torch.equal(make_model().reshape_2x2_image_features(x), ref)


def test_feature_file_round_trip_and_reference_loader_call(tmp_path):
    from safetensors.torch import load_file
    feat = torch.randn(7, 256, 1024, generator=torch.Generator().manual_seed(1)).half()
    path = tmp_path / "videos" / "v_0001.safetensors"
    feature_io.save_video_features(path, feat)
    assert torch.equal(load_file(str(path))["feature"], feat)          # the reference's own read (featuresloader.py:64)
    back = feature_io.load_video_features(path, dtype=torch.float32)
    assert back.dtype == torch.float32 and torch.equal(back, feat.float())
    img = feat[0]
    feature_io.save_video_features(tmp_path / "img.safetensors", img)   # [P, D] for an image (README.md:160)
    assert feature_io.load_video_features(tmp_path / "img.safetensors").shape == (256, 1024)
    with pytest.raises(AssertionError):
        feature_io.save_video_features(tmp_path / "bad.safetensors", feat[None])
    assert feature_io.feature_path_for("clips/v_0001.mp4") == "clips/v_0001.safetensors"


def test_extract_video_features_batches_through_the_tower(tmp_path):
    class FakeTower:            # stands in for CLIPVisionTower on the CPU box: counts calls, checks micro-batching
        device, dtype, num_patches, hidden_size = torch.device("cpu"), torch.float16, 4, 8
        calls = []

        def __call__(self, x):
            self.calls.append(x.shape[0])
            assert x.dtype == self.dtype
            return x.flatten(1)[:, :32].reshape(-1, 4, 8)

    tower = FakeTower()
    frames = torch.randn(70, 3, 4, 4)
    out = feature_io.extract_video_features(tower, frames, batch=32)
    assert tower.calls == [32, 32, 6] and out.shape == (70, 4, 8)
    assert feature_io.extract_video_features(tower, frames[:0]).shape == (0, 4, 8)
    paths = feature_io.extract_to_files(tower, [("a.mp4", frames[:3]), ("b.avi", frames[:5])], tmp_path)
    assert [os.path.basename(p) for p in paths] == ["a.safetensors", "b.safetensors"]
    assert feature_io.load_video_features(paths[1]).shape == (5, 4, 8)


def test_encode_video_memory_argument_contract():
    m = make_model()
    with pytest.raises(AssertionError):
        m.encode_video_memory()
    with pytest.raises(AssertionError):
        m.encode_video_memory(images=[torch.zeros(1, 3, 4, 4)], features=[torch.zeros(1, 4, 8)])
