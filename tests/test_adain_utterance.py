"""CPU tests of per-utterance AdaIN statistics (``adain_stats = "utterance"``) on AutoVC2 / MetaPool2 / MetaConv2: the
real model classes on the CPU stand-ins of tests/emulate.py and tests/test_ragged.py plus stand-ins for the two new
entry points below, each utterance of a padded batch compared with the oracle on that utterance alone."""
import warnings

import pytest
import torch

from oracle import rel_l2, templates
from oracle.adain import autovc2_forward
from oracle.seeded import seeded_state_dict, synthetic_mel, synthetic_speaker
from autoformer_b200 import packing
from tests import emulate
from tests.test_ragged import _Recorder, _emu_bilstm_small, _emu_lstm_seq, _emu_lstm_seq_ws, _emu_lstm_stack_ws, \
    _emu_zero_tail

warnings.filterwarnings("ignore", category=FutureWarning)
ARGS = (32, 256, 512, 32)


# ------------------------------------------------------------------------------------------------ stand-ins
def _emu_segment_stats(x, lengths=None, out=None):
    B, T, _ = x.shape
    lens = lengths.tolist() if lengths is not None else [T] * B
    r = torch.stack([torch.stack([x[b, :n].double().mean(), x[b, :n].double().std()]) for b, n in enumerate(lens)])
    if out is not None:
        out.copy_(r.float())
        return out
    return r.float()


def _emu_adain_segmented(x, x_stats, t_stats, precision, lengths=None, want_f32=False):
    B, T, _ = x.shape
    xs = x_stats.double().view(B, 1, 1, 2)
    ts = t_stats.double().expand(B, 2).reshape(B, 1, 1, 2)
    y = ((x.double() - xs[..., 0]) / xs[..., 1] * ts[..., 1] + ts[..., 0]).float()
    if lengths is not None:
        for b, n in enumerate(lengths.tolist()):
            y[b, n:] = 0
    return packing.to_act(y, precision), (y if want_f32 else None)


@pytest.fixture
def rec(monkeypatch):
    from autoformer_b200 import ops
    emulate.install_cpu_kernels(monkeypatch)
    r = _Recorder()
    for name, fn in (("zero_tail", _emu_zero_tail), ("bilstm_small", _emu_bilstm_small), ("lstm_seq", _emu_lstm_seq),
                     ("lstm_seq_ws", _emu_lstm_seq_ws), ("lstm_stack_ws", _emu_lstm_stack_ws),
                     ("segment_stats", _emu_segment_stats), ("adain_segmented", _emu_adain_segmented),
                     ("global_stats", emulate._emu_global_stats), ("adain", emulate._emu_adain)):
        monkeypatch.setattr(ops, name, r.wrap(name, fn))
    return r


def adain2(kind, args, seed, precision="fp32", adain_stats="utterance"):
    from tests.test_host_logic import _adain_model
    tpl = templates.autovc2_template(*args) if kind is None else templates.meta2_template(kind, *args)
    sd = seeded_state_dict(tpl, seed)
    m = _adain_model(kind, args, sd)
    m.precision = precision
    m.adain_stats = adain_stats
    return m, sd


def ragged_inputs(lengths, seed):
    B, T = len(lengths), max(lengths)
    x, c_org, c_trg = synthetic_mel(B, T, seed), synthetic_speaker(B, seed, "org"), synthetic_speaker(B, seed, "trg")
    for b, n in enumerate(lengths):
        x[b, n:] = 1e3                                  # whatever the padded frames hold is ignored
    return x, c_org, c_trg


def check_against_cropped_oracle(m, sd, x, c_org, c_trg, lengths, tol, feat_tol, target_feature=None, ref_tf=None,
                                 codes_tol=None):
    """Each utterance's mel / mel_postnet / codes (and features) against the oracle on x[b:b+1, :lengths[b]] alone;
    zeros past its end.  target_feature: the batch's argument, ref_tf(b): utterance b's target_feature for the oracle."""
    B, T = x.shape[:2]
    F = ARGS[3]
    kw = {} if lengths is None else {"lengths": lengths}
    lens = lengths if lengths is not None else [T] * B
    _, feats = m(x, c_org, None, **kw)
    mel, post, codes = m(x, c_org, c_trg, target_feature, **kw)
    codes = codes.view(B, T // F, -1)
    for b, n in enumerate(lens):
        xb = x[b:b + 1, :n].cpu()
        codes_ref, feats_ref = autovc2_forward(sd, xb, c_org[b:b + 1].cpu(), None, ARGS[0], F)
        ref = autovc2_forward(sd, xb, c_org[b:b + 1].cpu(), c_trg[b:b + 1].cpu(), ARGS[0], F,
                              target_feature=ref_tf(b) if ref_tf else None)
        got = torch.tensor([[float(f[0][b]), float(f[1][b])] for f in feats])
        want = torch.tensor([[float(mu), float(sd_)] for mu, sd_ in feats_ref])
        assert (got - want).abs().max() < feat_tol, (b, got, want)
        for key, t, r in (("mel", mel[b:b + 1, :, :n], ref[0]), ("mel_postnet", post[b:b + 1, :, :n], ref[1]),
                          ("codes", codes[b:b + 1, :n // F].reshape(1, -1), ref[2])):
            assert rel_l2(t, r) < (codes_tol or tol if key == "codes" else tol), (b, key, rel_l2(t, r))
        assert not mel[b, :, n:].any() and not post[b, :, n:].any() and not codes[b, n // F:].any()
    return mel, post, codes


# ------------------------------------------------------------------------------------------------ AutoVC2
@pytest.mark.parametrize("lengths", [[96, 32, 64], None], ids=["ragged", "fixed"])
def test_autovc2_utterance_matches_cropped_oracle(rec, lengths):
    m, sd = adain2(None, ARGS, 3)
    x, c_org, c_trg = ragged_inputs(lengths or [96] * 3, 8)
    if lengths is None:
        x = synthetic_mel(3, 96, 8) * torch.tensor([1.0, 0.5, 2.0]).view(3, 1, 1)  # utterances of distinct statistics
    check_against_cropped_oracle(m, sd, x, c_org, c_trg, lengths, 2e-4, 1e-5)
    names = [name for name, _ in rec.calls]
    assert "global_stats" not in names and "adain" not in names
    assert names.count("segment_stats") == 2 * 3 + 3 and names.count("adain_segmented") == 3
    # the codes-only call: 3 in the pre-extract + 3 in the encoder; the conversion: those and AutoVC's other 10
    assert names.count("zero_tail") == (0 if lengths is None else 6 + 16)


def test_autovc2_per_utterance_target_feature(rec):
    """target_feature of (B,) tensors: utterance b is styled with the features of utterance perm[b] of another batch; a
    0-dim entry styles every utterance alike."""
    m, sd = adain2(None, ARGS, 3)
    lengths = [64, 96, 32]
    x, c_org, c_trg = ragged_inputs(lengths, 9)
    xo = synthetic_mel(3, 96, 77)
    _, fo = m(xo, c_org, None)
    perm = [2, 0, 1]
    tf = [[mu[perm], s[perm]] for mu, s in fo]
    tf[1] = [fo[1][0][0], fo[1][1][0]]                   # entry 1: 0-dim, one style for all
    ref_tf = lambda b: [[tf[0][0][b], tf[0][1][b]], [tf[1][0], tf[1][1]], [tf[2][0][b], tf[2][1][b]]]
    check_against_cropped_oracle(m, sd, x, c_org, c_trg, lengths, 2e-4, 1e-5, tf, ref_tf)


def test_default_mode_never_calls_the_new_ops(rec):
    m, _ = adain2(None, ARGS, 3, adain_stats="batch")
    x, c_org, c_trg = ragged_inputs([64, 64], 4)
    m(x, c_org, c_trg)
    _, feats = m(x, c_org, None)
    assert all(f.dim() == 0 for pair in feats for f in pair)
    names = {name for name, _ in rec.calls}
    assert {"global_stats", "adain"} <= names
    assert not names & {"segment_stats", "adain_segmented", "zero_tail"}
    assert all("lengths" not in kw for _, kw in rec.calls)


# ------------------------------------------------------------------------------------------------ Meta2 golden rows
def golden_row_call(m, inputs, row=1, B=3, seed=31):
    """check_adain_outputs' `call` with the golden fixture's utterance as row `row` of a batch of B other utterances:
    returns that row's outputs (and features)."""
    others = synthetic_mel(B, 176, seed) * torch.linspace(0.5, 1.5, B).view(B, 1, 1)
    co, ct = synthetic_speaker(B, seed, "org"), synthetic_speaker(B, seed, "trg")
    dev = next(m.parameters()).device

    def call(xk, conv, tf):
        x, c_org, c_trg = others.clone(), co.clone(), ct.clone()
        x[row], c_org[row], c_trg[row] = inputs[xk][0], inputs["c_org"][0], inputs["c_trg"][0]
        out = m(x.to(dev), c_org.to(dev), c_trg.to(dev) if conv else None, tf)
        pick = lambda f: f if f.dim() == 0 else f[row]
        if not conv:
            return out[0][row:row + 1], [[pick(mu), pick(s)] for mu, s in out[1]]
        return tuple(t[row:row + 1] for t in out)
    return call


@pytest.mark.parametrize("name,kind", [("metapool2_b1_t176", "pool"), ("metaconv2_b1_t176", "conv")])
def test_meta2_golden_row_in_a_batch(rec, name, kind):
    """The golden utterance as one row of a batch of three: "utterance" statistics give the reference's outputs and
    features for it; "batch" statistics (the negative control) do not."""
    from tests.test_host_logic import _adain_model
    from tests.test_oracle_golden import adain_case, check_adain_outputs
    g, args, sd, i, _ = adain_case(name, kind)
    m = _adain_model(kind, args, sd)
    m.adain_stats = "utterance"
    check_adain_outputs(g, golden_row_call(m, i), 2e-4, 1e-4)
    m.adain_stats = "batch"
    with pytest.raises(AssertionError):
        check_adain_outputs(g, golden_row_call(m, i), 2e-4, 1e-4)
    assert rel_l2(golden_row_call(m, i)("x", True, None)[1], torch.from_numpy(g["own_mel_postnet"])) > 1e-2


# ------------------------------------------------------------------------------------------------ pipeline
def test_convert_utterances_adain(rec):
    """pipeline.convert_utterances on AutoVC2: each utterance self-styled (the Evaluator's isAdain recipe) and equal to
    the oracle on it alone, padded to a multiple of freq and trimmed; "batch" statistics are refused."""
    from autoformer_b200 import pipeline
    m, sd = adain2(None, ARGS, 5)
    lens = [40, 64, 17, 96]
    mels = [synthetic_mel(1, n, 20 + i)[0] for i, n in enumerate(lens)]
    c_org, c_trg = synthetic_speaker(len(lens), 6, "org"), synthetic_speaker(len(lens), 6, "trg")
    outs = pipeline.convert_utterances(m, mels, c_org, c_trg, max_batch=2)
    for i, (mel, o) in enumerate(zip(mels, outs)):
        x, _ = pipeline.pad_to_multiple(mel[None], ARGS[3])
        ref = autovc2_forward(sd, x, c_org[i:i + 1], c_trg[i:i + 1], ARGS[0], ARGS[3])[1].squeeze(1)[0, :lens[i]]
        assert o.shape == (lens[i], 80) and rel_l2(o, ref) < 2e-4
    m.adain_stats = "batch"
    with pytest.raises(ValueError, match="adain_stats"):
        pipeline.convert_utterances(m, mels, c_org, c_trg)


# ------------------------------------------------------------------------------------------------ validation
def test_validation_errors(rec):
    m, _ = adain2(None, ARGS, 0)
    x, c_org, c_trg = ragged_inputs([64, 32, 64], 1)
    m.adain_stats = "batch"
    with pytest.raises(ValueError, match="adain_stats"):
        m(x, c_org, c_trg, lengths=[64, 32, 64])
    m.adain_stats = "global"
    with pytest.raises(ValueError, match="adain_stats"):
        m(x, c_org, c_trg)
    m.adain_stats = "utterance"
    m.bn_stats = "batch"
    with pytest.raises(ValueError, match="bn_stats"):
        m(x, c_org, c_trg)
    m.bn_stats = "running"
    with pytest.raises(ValueError, match="multiples of freq"):
        m(x, c_org, c_trg, lengths=[64, 40, 64])
    with pytest.raises(ValueError, match=r"\[1, T"):
        m(x, c_org, c_trg, lengths=[64, 0, 64])
    for bad in (torch.zeros(2), torch.zeros(3, 1), torch.zeros(1)):
        with pytest.raises(ValueError, match="target_feature"):
            m(x, c_org, c_trg, [[bad, torch.ones(3)], [0.0, 1.0], [0.0, 1.0]])
    meta, _ = adain2("pool", (44, 256, 512, 22), 0)
    with pytest.raises(ValueError, match="lengths"):
        meta(synthetic_mel(2, 176, 1), synthetic_speaker(2, 1), synthetic_speaker(2, 2), lengths=[176, 88])
    assert not rec.calls
