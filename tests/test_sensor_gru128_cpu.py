"""Which sensor-encoder sizes take the native path, and the hidden-128 encoder off it (no GPU needed)."""
import torch

from leak_det_gnn_b200 import ops
from leak_det_gnn_b200.models.detector import SharedSensorGRUEncoder


def test_gru_supported_sizes():
    assert ops.gru_supported(64, 9) and ops.gru_supported(128, 9) and ops.gru_supported(128, 0)
    assert ops.gru_supported(128, 30) and not ops.gru_supported(128, 31) and not ops.gru_supported(128, -1)
    assert not ops.gru_supported(96, 9) and not ops.gru_supported(256, 9)


def test_hidden_128_encoder_on_cpu_is_the_reference_gru():
    torch.manual_seed(0)
    enc = SharedSensorGRUEncoder(hidden_size=128)
    r, tf = torch.randn(2, 5, 3), torch.randn(2, 5, 9)
    seq = torch.cat([r.transpose(1, 2).reshape(6, 5, 1), tf.unsqueeze(1).expand(2, 3, 5, 9).reshape(6, 5, 9)], dim=-1)
    out, _ = enc.gru(seq)
    assert torch.equal(enc(r, tf), out[:, -1, :].view(2, 3, 128))
