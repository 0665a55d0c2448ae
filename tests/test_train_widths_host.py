"""run.py's early width check: the vanilla image model trains and samples at the widths the AdaGN kernels cover."""
import types

import pytest


def _args(mode, unets_channels, model="vanilla"):
    return types.SimpleNamespace(model=model, mode=mode, is_latent=False, unets_channels=unets_channels)


@pytest.mark.parametrize("mode", ["train", "eval", "eval_fid"])
def test_vanilla_widths_check_is_the_same_for_training_and_inference(mode):
    import run as idf_run
    from infodiffusion_b200 import engine
    assert engine.MAX_GN_CHANNELS == 1024 and not hasattr(engine, "MAX_TRAIN_GN_CHANNELS")
    idf_run._check_widths(_args(mode, 64))                # ch_mult [1,2,4,8] at 64 channels: GroupNorm over 1024
    with pytest.raises(NotImplementedError, match="2048"):
        idf_run._check_widths(_args(mode, 128))           # 1024 channels, GroupNorm over 2048
    idf_run._check_widths(_args(mode, 128, model="diff"))  # the InfoDiff model is not the vanilla UNet
