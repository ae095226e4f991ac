"""Argument checks of the tensor-output encode calls (Tokenizer.encode_to_tensor / encode_batch_to_tensor / encode_batch_padded): every bad
argument raises ValueError / TypeError before the device is touched, so these run without a GPU."""
import pytest

import _bootstrap  # noqa: F401
from transformer_lm_b200 import _lib
from transformer_lm_b200.tokenizer import Tokenizer


@pytest.fixture
def tok(monkeypatch):
    def no_device(self):
        raise AssertionError("the device was touched before the arguments were checked")
    monkeypatch.setattr(Tokenizer, "_device_tok", no_device)
    return Tokenizer({i: bytes([i]) for i in range(256)}, [], ["<|endoftext|>"])


@pytest.mark.parametrize("kwargs,exc", [
    (dict(max_length=0), ValueError),
    (dict(max_length=-3), ValueError),
    (dict(max_length=2**32), ValueError),
    (dict(max_length=1.5), TypeError),
    (dict(max_length="8"), TypeError),
    (dict(max_length=True), TypeError),
    (dict(pad_to="max"), ValueError),
    (dict(pad_to=None), ValueError),
    (dict(pad_to="max_length"), ValueError),               # without max_length
    (dict(padding_side="center"), ValueError),
    (dict(truncation_side="middle"), ValueError),
    (dict(padding_side=None), ValueError),
    (dict(offsets="token"), ValueError),
    (dict(offsets=1), ValueError),
    (dict(dropout=1.5), ValueError),
    (dict(dropout=0.1, seed=-1), ValueError),
])
def test_padded_argument_errors(tok, kwargs, exc):
    with pytest.raises(exc):
        tok.encode_batch_padded(["a b", "c"], pad_id=0, **kwargs)


@pytest.mark.parametrize("pad_id,exc", [(None, TypeError), (1.0, TypeError), ("0", TypeError), (False, TypeError),
                                        (2**63, ValueError), (-2**63 - 1, ValueError)])
def test_pad_id_is_a_required_int64(tok, pad_id, exc):
    with pytest.raises(TypeError):
        tok.encode_batch_padded(["a"])                      # no default
    with pytest.raises(exc):
        tok.encode_batch_padded(["a"], pad_id=pad_id)


@pytest.mark.parametrize("kwargs", [dict(offsets="bytes"), dict(offsets="CHAR"), dict(dropout=-0.1), dict(dropout=float("nan")),
                                    dict(seed=2**64), dict(seed=1.0)])
def test_to_tensor_argument_errors(tok, kwargs):
    with pytest.raises(ValueError):
        tok.encode_to_tensor(b"a b", **kwargs)
    with pytest.raises(ValueError):
        tok.encode_batch_to_tensor(["a b"], **kwargs)


def test_binding_declares_the_new_abi():
    assert "bpe_pad_rows_dev" in _lib.EXPORTS
    assert (_lib.PAD_LEFT, _lib.TRUNC_LEFT) == (1, 2)
    names = [f[0] for f in _lib.EncodeOpts._fields_]
    assert names[-1] == "out_device"                        # appended: a zero-filled struct keeps meaning bpe_encode
    assert _lib.EncodeOpts().out_device == 0
