"""CPU tests of variable-length MelGAN batches (``Generator.forward(x, lengths=...)``, pipeline.vocode_utterances): the
host-side validation, the tile prefix tables of the fused ResnetBlocks, and the ragged forward on the CPU stand-ins of
tests/emulate.py plus the stand-ins below for the lengths-aware entry points, compared per utterance with the oracle on
the cropped utterance."""
import warnings

import pytest
import torch
import torch.nn.functional as F

from oracle import rel_l2, templates
from oracle.melgan import melgan_forward
from oracle.seeded import seeded_state_dict, synthetic_mel
from tests import emulate

warnings.filterwarnings("ignore", category=FutureWarning)


# ------------------------------------------------------------------------------------------------ stand-ins for lengths
def _emu_zero_tail(buf, row0, T, lengths):
    for b, n in enumerate(lengths.tolist()):
        buf[b, row0 + n:row0 + T] = 0
    return buf


def _emu_reflect_halo(buf, row0, L, reflect, lengths=None):
    if lengths is None:
        return emulate._emu_reflect_halo(buf, row0, L, reflect)
    for b, n in enumerate(lengths.tolist()):
        assert reflect < n <= L
        for k in range(1, reflect + 1):
            buf[b, row0 - k] = buf[b, row0 + k]
            buf[b, row0 + n - 1 + k] = buf[b, row0 + n - 1 - k]
    return buf


def _emu_conv_to_mono_tanh(x, w, bias, lengths=None):
    if lengths is None:
        return emulate._emu_conv_to_mono_tanh(x, w, bias)
    out = torch.zeros(x.shape[0], x.shape[1])
    for b, n in enumerate(lengths.tolist()):
        out[b, :n] = emulate._emu_conv_to_mono_tanh(x[b:b + 1, :n].contiguous(), w, bias)[0]
    return out


def _emu_resblock2(self, x, B, L, y=None, y_row0=0, y_reflect=0, y_act=False, out2=None, wav=None, mono=None,
                   lengths=None):
    """The kernel's ragged contract: only the tiles that hold a valid row are computed and stored (the fixed-length
    arithmetic on them); wav reflects at each utterance's end and is 0 past it in the last tile."""
    if lengths is None:
        return emulate._emu_resblock2_call(self, x, B, L, y, y_row0, y_reflect, y_act, out2, wav, mono)
    rows = lengths.host
    if wav is not None:
        w_out, b_out = mono
        K, lead = w_out.shape[0], w_out.shape[0] // 2
        stride = 128 - (K - 1)
        a = torch.empty(B * L, self.C)
        emulate._emu_resblock2_call(self, x, B, L, out2=a)                      # LeakyReLU(y), exact fp32
        a = a.view(B, L, -1).double()
        for b, n in enumerate(rows):
            tau = torch.arange(n)[:, None] + torch.arange(K)[None, :] - lead
            tau = torch.where(tau < 0, -tau, tau)
            tau = torch.where(tau >= n, 2 * (n - 1) - tau, tau)
            acc = (a[b][tau] * w_out.double()[None]).sum(dim=(1, 2)) + b_out
            wav[b, :n] = torch.tanh(acc).float()
            wav[b, n:min(L, -(-n // stride) * stride)] = 0
        return wav
    full = y.clone() if y is not None else out2.clone()
    emulate._emu_resblock2_call(self, x, B, L, full if y is not None else None, y_row0, y_reflect, y_act,
                                full if out2 is not None else None)
    for b, n in enumerate(rows):
        end = -(-n // 128) * 128                                                # rows of the tiles that run
        if y is not None:
            y[b, y_row0 - y_reflect:y_row0 + end] = full[b, y_row0 - y_reflect:y_row0 + end]
            if end >= L:
                y[b, y_row0 + L:y_row0 + L + y_reflect] = full[b, y_row0 + L:y_row0 + L + y_reflect]
        else:
            out2[b * L:b * L + end] = full[b * L:b * L + end]
    return y if y is not None else out2


class _Recorder:
    def __init__(self):
        self.calls = []

    def wrap(self, name, fn):
        def rec(*a, **kw):
            self.calls.append((name, tuple(sorted(kw))))
            return fn(*a, **kw)
        return rec


@pytest.fixture
def rec(monkeypatch):
    from autoformer_b200 import ops
    emulate.install_cpu_kernels(monkeypatch)
    r = _Recorder()
    for name, fn in (("zero_tail", _emu_zero_tail), ("reflect_halo", _emu_reflect_halo),
                     ("conv_to_mono_tanh", _emu_conv_to_mono_tanh)):
        monkeypatch.setattr(ops, name, r.wrap(name, fn))
    rb2 = r.wrap("resblock2", _emu_resblock2)
    monkeypatch.setattr(ops.Resblock2, "__call__", lambda self, *a, **kw: rb2(self, *a, **kw))
    return r


def _generator(precision, seed=4):
    from autoformer_b200.melgan.modules import Generator
    sd = seeded_state_dict(templates.melgan_template(), seed)
    g = Generator(80, 32, 3)
    g.load_state_dict(sd)
    g.precision = precision
    return g, sd


# ------------------------------------------------------------------------------------------------ host validation
@pytest.mark.parametrize("lengths,what", [([16, 16], "entries"), ([16, 3, 8], "at least 4"), ([16, 17, 8], r"\[1, T"),
                                          ([16, 0, 8], r"\[1, T"), (torch.tensor([16, 12]), "entries"),
                                          (torch.tensor([16, 2, 9]), "at least 4")])
def test_generator_lengths_validation(rec, lengths, what):
    g, _ = _generator("fp16s")
    with pytest.raises(ValueError, match=what):
        g(synthetic_mel(3, 16, 1).transpose(1, 2), lengths=lengths)
    assert not rec.calls


def test_generator_lengths_with_taps(rec):
    g, _ = _generator("fp32")
    g.collect_taps = True
    with pytest.raises(NotImplementedError):
        g(synthetic_mel(2, 8, 1).transpose(1, 2), lengths=[8, 5])


# ------------------------------------------------------------------------------------------------ tile tables
def test_ragged_tile_tables():
    from autoformer_b200 import ops
    lengths = [1000, 4, 513, 128, 999]
    scales, strides = (1, 8, 64, 128, 256), (128, 122)
    tables = ops.ragged_rows(lengths, scales, strides, "cpu")
    assert len(tables) == len(scales)
    for s, t in zip(scales, tables):
        rows = [s * n for n in lengths]
        assert t.host == rows and t.rows.dtype == torch.int32 and t.rows.tolist() == rows
        for S in strides:
            start, total = t.tiles[S]
            counts = [-(-r // S) for r in rows]
            assert total == sum(counts) and start.tolist() == [sum(counts[:b]) for b in range(len(rows) + 1)]
    # one upload: every view shares one storage
    assert len({t.rows.untyped_storage().data_ptr() for t in tables}) == 1


# ------------------------------------------------------------------------------------------------ fixed-length calls
@pytest.mark.parametrize("precision,halos", [("fp32", 0), ("fp16s", 4)])
def test_fixed_length_calls_are_unchanged(rec, precision, halos):
    """lengths=None: no ops function gets a `lengths` keyword and nothing is zero-tailed -- the fixed-length forward
    launches exactly what it launched before variable-length batches existed."""
    g, _ = _generator(precision)
    g(synthetic_mel(2, 16, 1).transpose(1, 2))
    names = [name for name, _ in rec.calls]
    assert "zero_tail" not in names and names.count("reflect_halo") == halos
    assert all("lengths" not in kw for _, kw in rec.calls)


# ------------------------------------------------------------------------------------------------ ragged forward
@pytest.mark.parametrize("precision,tol", [("fp32", 1e-4), ("tf32", 3e-3), ("bf16", 3e-2), ("fp16x2", 2e-3),
                                           ("fp16s", 1e-3)])
def test_generator_ragged_matches_cropped_oracle(rec, precision, tol):
    g, sd = _generator(precision)
    lengths = [16, 9, 4, 12]
    B, T = len(lengths), max(lengths)
    mel = synthetic_mel(B, T, 6).transpose(1, 2).contiguous()
    for b, n in enumerate(lengths):
        mel[b, :, n:] = float("nan")                    # whatever the padded frames hold is ignored
    wav = g(mel, lengths=torch.tensor(lengths))
    assert wav.shape == (B, 1, 256 * T) and torch.isfinite(wav).all()
    names = [name for name, _ in rec.calls]
    assert names.count("zero_tail") == 4
    for b, n in enumerate(lengths):
        ref = melgan_forward(sd, mel[b:b + 1, :, :n])
        assert rel_l2(wav[b:b + 1, :, :256 * n], ref) < tol, (b, n)
        assert not wav[b, :, 256 * n:].any()


def test_generator_ragged_fused_tiles_skip(rec):
    """fp16s at an even T: the three narrow stages run fused with the compacted tiles (the wav of the last one
    included)."""
    g, sd = _generator("fp16s")
    lengths = [4, 10]
    mel = synthetic_mel(2, 10, 8).transpose(1, 2).contiguous()
    wav = g(mel, lengths=lengths)
    kws = [kw for name, kw in rec.calls if name == "resblock2"]
    assert len(kws) == 9 and all("lengths" in kw for kw in kws) and any("wav" in kw for kw in kws)
    ref = melgan_forward(sd, mel[:1, :, :4])
    assert rel_l2(wav[:1, :, :1024], ref) < 1e-3 and not wav[0, :, 1024:].any()


def test_padded_batch_without_lengths_is_wrong_at_the_edge(rec):
    """Negative control: the padded batch run without lengths and trimmed misses the oracle on the short utterance."""
    g, sd = _generator("fp32")
    mel = synthetic_mel(2, 12, 3).transpose(1, 2).contiguous()
    mel[1, :, 6:] = 0
    wav = g(mel)
    ref = melgan_forward(sd, mel[1:, :, :6])
    assert rel_l2(wav[1:, :, 256 * 5:256 * 6], ref[:, :, 256 * 5:]) > 1e-2


# ------------------------------------------------------------------------------------------------ pipeline
def test_vocode_utterances_order_and_lengths(rec):
    from autoformer_b200 import pipeline
    g, _ = _generator("fp32")
    lens = [7, 12, 4, 9, 12]
    mels = [synthetic_mel(1, n, 20 + i)[0] for i, n in enumerate(lens)]
    wavs = pipeline.vocode_utterances(g, mels, max_batch=2)
    assert len(wavs) == len(mels)
    for i, (m, w) in enumerate(zip(mels, wavs)):
        ref = g(m.t()[None].contiguous()).view(-1)
        assert w.shape == (256 * lens[i],) and rel_l2(w, ref) < 1e-5, i


def test_vocode_utterances_pads_batches_to_even_length(monkeypatch):
    from autoformer_b200 import pipeline

    class _Stub:
        hop_length = 256

        def __init__(self):
            self.shapes = []

        def __call__(self, x, lengths):
            self.shapes.append((tuple(x.shape), list(lengths)))
            # sample j of utterance b carries (b, j) so that any mix-up shows
            B, _, T = x.shape
            return (x[:, 0, :].repeat_interleave(256, dim=1) + 0 * torch.arange(256 * T)).unsqueeze(1)

    stub = _Stub()
    lens = [5, 8, 7, 5]
    mels = [torch.full((n, 80), float(i)) for i, n in enumerate(lens)]
    wavs = pipeline.vocode_utterances(stub, mels, max_batch=3)
    assert [s[0][2] for s in stub.shapes] == [8, 6] and all(s[0][1] == 80 for s in stub.shapes)
    assert stub.shapes[0][1] == [8, 7, 5] and stub.shapes[1][1] == [5]
    for i, w in enumerate(wavs):
        assert w.shape == (256 * lens[i],) and bool((w == i).all())
