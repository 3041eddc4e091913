"""CPU: the host surface of InfoNCE training -- the loss objects, the head scratch sizes the step needs, and the argument
checks of the new entry points (no GPU needed: they refuse before touching the device)."""
import ctypes

import pytest

import dib_b200
from dib_b200 import _lib
from dib_b200.keras_compat import resolve_loss


def test_infonce_loss_objects_resolve_and_check_their_arguments():
    loss = dib_b200.losses.InfoNCE()
    assert (loss.similarity_type, loss.temperature, loss.output_encoder_architecture) == ("l2", 1.0, [128, 128])
    assert resolve_loss(loss) == "infonce"
    assert resolve_loss("infonce") == resolve_loss("InfoNCE") == "infonce"
    assert resolve_loss(dib_b200.losses.InfoNCE("cosine", 0.5, (64,))) == "infonce"
    with pytest.raises(ValueError, match="Similarity type not implemented"):
        dib_b200.losses.InfoNCE("dot")
    for t in (0.0, -1.0):
        with pytest.raises(ValueError, match="temperature"):
            dib_b200.losses.InfoNCE(temperature=t)
    with pytest.raises(ValueError):
        dib_b200.losses.InfoNCE(output_encoder_architecture=(8, 0))


def test_infonce_scratch_bytes():
    lib = _lib.load()
    for kind in (0, 1, 4):
        for n in (1, 5, 129, 4096, 40000, 65536, 1 << 20):
            for d in (1, 3, 64, 256):
                assert lib.dib_infonce_scratch_bytes(kind, n, d) == lib.dib_infonce_head_tc_scratch_bytes(n, d) > 0
        assert lib.dib_infonce_scratch_bytes(kind, 1024, 257) == -1
    for kind in (2, 3):
        for n in (1, 7, 4096, 32768):
            assert lib.dib_infonce_scratch_bytes(kind, n, 64) == (n * n + 4 * n) * 4
        assert lib.dib_infonce_scratch_bytes(kind, 32769, 64) == -1
        assert lib.dib_infonce_scratch_bytes(kind, 40000, 64) == -1
    assert lib.dib_infonce_scratch_bytes(5, 16, 8) == -1
    assert lib.dib_infonce_scratch_bytes(-1, 16, 8) == -1


def test_infonce_entry_points_refuse_null_handles_and_arguments():
    lib = _lib.load()
    err = lambda: lib.dib_last_error().decode()
    assert lib.dib_attach_output_encoder(None, None) != 0 and "null" in err()
    cfg = _lib.DibOutputEncoderConfig(input_dimensionality=1, number_layers=0, architecture=None)
    assert lib.dib_attach_output_encoder(None, ctypes.byref(cfg)) != 0 and "null" in err()
    assert lib.dib_output_encoder_param_count(None) == -1
    assert lib.dib_output_encoder_param_layout(None, None, None, None, 0) == -1 and "no output encoder" in err()
    assert lib.dib_output_encoder_forward(None, None, None, 1, None, None, None) != 0 and "null model handle" in err()
    # (handle, params, x, y, n, beta_dev, kind, temperature, eps, seed, step, sample_offset, head_scratch, ...)
    args = (None, None, None, None, 4, None, 1, 1.0, None, 0, 0, 0, None)
    assert lib.dib_infonce_train_step(*args, None, None, None, None) != 0 and "null model handle" in err()
    assert lib.dib_infonce_forward(*args, None, None, None) != 0 and "null model handle" in err()
