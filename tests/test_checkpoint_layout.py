"""The checkpoint layout (engine.encoder_layout / decoder_layout) names exactly the state-dict keys the engines read."""
import pytest

from oracle.synth import config_for, synth_state_dict


def _named_keys(record, out):
    """Every key string in a layout record; TimeHead.name is a TimeProjector column name, not a key."""
    if isinstance(record, str):
        out.add(record)
    elif isinstance(record, dict):
        for v in record.values():
            _named_keys(v, out)
    elif hasattr(record, "_fields"):
        for f, v in zip(record._fields, record):
            if f != "name":
                _named_keys(v, out)
    elif isinstance(record, tuple):
        for v in record:
            _named_keys(v, out)
    return out


@pytest.mark.parametrize("ck", [dict(n_lr=1), dict(n_lr=2, geo=True, seasons=True), dict(use_resize_conv=False, norm="instance"),
                                dict(block_layers=(3, 4, 6, 3), activation="gelu", n_heads=2)])
def test_layout_names_every_key_the_engines_read(ck):
    from sbgm_danra_b200 import engine
    from sbgm_danra_b200._smoke import build_model
    cfg = config_for(**ck)
    net = build_model(cfg, synth_state_dict(cfg), "bf16x3", "cpu")
    spec = net.spec()
    named = _named_keys(engine.encoder_layout(spec), set()) | _named_keys(engine.decoder_layout(spec), set())
    sd = set(net.state_dict())
    assert named <= sd, sorted(named - sd)
    # unread: BatchNorm's step counters, and the final layer's time projection (it runs without a time input)
    unread = {k for k in sd if k.endswith("num_batches_tracked") or k.startswith(("decoder.final_layer.sinusoidal_embedding.",
                                                                                   "decoder.final_layer.time_projection_layer.1."))}
    assert sd - named == unread
