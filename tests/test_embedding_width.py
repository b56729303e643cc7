"""Host-side checks of the embedding-width support (no GPU)."""
import pytest


def test_width_not_a_multiple_of_4_is_rejected_before_any_gpu_work():
    from types import SimpleNamespace
    from musediffusion_b200.initialization import create_model_and_diffusion
    args = SimpleNamespace(hidden_dim=50, hidden_t_dim=128, vocab_size=729, seq_len=64, dropout=0.1, noise_schedule="sqrt",
                           diffusion_steps=2000, timestep_respacing="", rescale_timesteps=True, predict_xstart=True)
    with pytest.raises(ValueError, match="multiple of 4"):
        create_model_and_diffusion(args)


def test_padded_width():
    from musediffusion_b200 import ops
    assert [ops.padded_width(d) for d in (4, 16, 64, 100, 128, 200, 500, 512, 768)] == [64, 64, 64, 128, 128, 256, 512, 512, 768]
