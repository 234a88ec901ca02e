"""FarmerLstm move histories, without a GPU: the float64 statement of tests/history_reference.py against torch float64 autograd
of nn.LSTM on pack_padded_sequence and against the C oracle, the packer, and the C ABI of the option (struct layout, default,
the configurations fi_learner_create refuses before it looks for a device, the new inference entry point's refusals).

The rule (include/fi_learner.h, FI_REC_WORD_LENGTH): slot b holds a history of L_b = (W == 0 || W > T) ? T : W records, W being
word 183 of its record 0; the step is the reference's train_step on each sample cut to its first L_b records, one mean over
the batch."""
import ctypes as C
import os
import subprocess

import numpy as np
import pytest

import _util as U
import history_reference as H
from oracle import pyoracle as po

HEADER = os.path.join(U.ROOT, "include", "fi_learner.h")


def _case(seed, m, t, lengths):
    z, x, tg = U.farmer_batch(seed, m, t)
    return z, x, tg, np.asarray(lengths, np.int64)


def _torch_reference(params, z, x, tg, lengths, loss="mse"):
    """Loss and flat gradient in torch float64: nn.LSTM on pack_padded_sequence (h_n is each sequence's h at its own last
    step), then the dense stack and the criterion, mean over the batch."""
    import torch
    from torch.nn.utils.rnn import pack_padded_sequence
    torch.manual_seed(0)
    lstm = torch.nn.LSTM(162, 128, batch_first=True).double()
    dense = [torch.nn.Linear(612 if i == 0 else 512, 512).double() for i in range(5)] + [torch.nn.Linear(512, 1).double()]
    ps = [lstm.weight_ih_l0, lstm.weight_hh_l0, lstm.bias_ih_l0, lstm.bias_hh_l0] + [q for d in dense for q in (d.weight, d.bias)]
    off = 0
    with torch.no_grad():
        for q, shp in zip(ps, U.FARMER_SHAPES):
            n = int(np.prod(shp))
            q.copy_(torch.from_numpy(np.asarray(params[off:off + n], np.float64).reshape(shp)))
            off += n
    packed = pack_padded_sequence(torch.from_numpy(z.astype(np.float64)), torch.from_numpy(lengths), batch_first=True,
                                  enforce_sorted=False)
    _, (h_n, _) = lstm(packed)
    a = torch.cat([h_n[0], torch.from_numpy(x.astype(np.float64))], 1)
    for d in dense[:5]:
        a = torch.relu(d(a))
    y = dense[5](a)[:, 0]
    tgt = torch.from_numpy(tg.astype(np.float64))
    fn = {"mse": torch.nn.functional.mse_loss, "mae": torch.nn.functional.l1_loss,
          "huber": torch.nn.functional.smooth_l1_loss}[loss]
    out = fn(y, tgt)
    out.backward()
    return out.item(), np.concatenate([q.grad.numpy().ravel() for q in ps])


@pytest.mark.parametrize("name,m,t,lengths", [
    ("mixed", 6, 9, [1, 9, 4, 4, 7, 2]),
    ("all-L1", 4, 7, [1, 1, 1, 1]),
    ("all-LT", 3, 8, [8, 8, 8]),
])
@pytest.mark.parametrize("loss", ["mse", "huber"])
def test_history_reference_matches_torch_autograd(oracle, name, m, t, lengths, loss):
    z, x, tg, L = _case(len(name) + m * t, m, t, lengths)
    params = U.farmer_params(11)
    got_l, got_g = H.loss_grad_history(oracle.farmer(params, loss=loss), z, x, tg, L)
    want_l, want_g = _torch_reference(params, z, x, tg, L, loss)
    assert abs(got_l - want_l) <= 1e-12 * abs(want_l), (got_l, want_l)
    assert U.rel_max(got_g, want_g) <= 1e-12, U.rel_max(got_g, want_g)


def test_full_length_is_the_oracles_full_batch_step(oracle):
    m, t = 5, 12
    z, x, tg, _ = _case(3, m, t, [t] * m)
    params = U.farmer_params(12)
    o = oracle.farmer(params)
    want_l = o.loss_grad(z, x, tg)
    want_g = o.grads()
    for words in ([0] * m, [t] * m, [t + 1, 1 << 31, 0xFFFFFFFF, 0, t]):
        got_l, got_g = H.loss_grad_history(oracle.farmer(params), z, x, tg, H.lengths_of(words, t))
        assert abs(got_l - want_l) <= 1e-12 * abs(want_l) and U.rel_max(got_g, want_g) <= 1e-12, words


def test_history_past_its_length_is_never_read(oracle):
    """NaN in z past each length leaves the statement unchanged, bit for bit."""
    m, t = 4, 10
    z, x, tg, L = _case(4, m, t, [3, 10, 1, 8])
    params = U.farmer_params(13)
    want = H.loss_grad_history(oracle.farmer(params), z, x, tg, L)
    z2 = z.copy()
    z2[np.arange(t)[None, :] >= L[:, None]] = np.nan
    got = H.loss_grad_history(oracle.farmer(params), z2, x, tg, L)
    assert got[0] == want[0] and np.array_equal(got[1], want[1])


@pytest.mark.skipif(not po.ref_available(), reason="needs the reference compiled into oracle/_ref")
def test_history_statement_is_the_references_step_at_the_cut_length(oracle):
    """Every L = 37 in 100-record slots: the reference's own libtorch train_step at T = 37."""
    m, t, n = 4, 100, 37
    z, x, tg, L = _case(5, m, t, [n] * m)
    ref = po.RefNN(seed=1234)
    params = ref.params()
    want_l = ref.train_step(np.ascontiguousarray(z[:, :n]), x, tg)
    got_l, got_g = H.loss_grad_history(oracle.farmer(params), z, x, tg, L)
    assert abs(got_l - want_l) <= 1e-5 * abs(want_l) + 1e-7
    assert U.rel_l2(got_g, ref.grads()) < 2e-5


def test_packer_writes_length_and_pads_only_the_unread_region():
    m, t = 3, 12
    z, x, tg = U.farmer_batch(6, m, t)
    words = np.array([0, 3, 10], np.uint32)   # L = 12, 3, 10
    plain = po.pack_farmer_slots(z, x, tg).view(np.uint32).reshape(m, t, po.REC_WORDS)
    for pad in ("zeros", "garbage"):
        w = H.pack_history_slots(z, x, tg, words, pad=pad).view(np.uint32).reshape(m, t, po.REC_WORDS)
        assert np.array_equal(w[:, 0, H.WORD], words)
        assert np.array_equal(w[0], plain[0])                          # full length: nothing padded
        for b, n in ((1, 3), (2, 10)):   # z of records 0..L-1, x of records 0..7 and the target stay
            assert np.array_equal(w[b, :n, :162], plain[b, :n, :162])
            assert np.array_equal(w[b, :8, 192:], plain[b, :8, 192:]) and w[b, 0, 181] == plain[b, 0, 181]
    f = H.pack_history_slots(z, x, tg, words, pad="garbage").view(np.float32).reshape(m, t, po.REC_WORDS)
    assert not np.isfinite(f[1, 3:, :162]).all() and not np.isfinite(f[1, 8:]).all()


# ------------------------------------------------------------------------------- C ABI
def test_header_field_matches_ctypes(fi, tmp_path):
    from freeimpala_b200 import _lib
    c = tmp_path / "h.c"
    c.write_text('#include <stdio.h>\n#include <stddef.h>\n#include "fi_learner.h"\n'
                 'int main(void){printf("%zu %zu %zu\\n", sizeof(fi_learner_config), offsetof(fi_learner_config, history_length),'
                 'offsetof(fi_learner_config, variable_length));return 0;}\n')
    exe = tmp_path / "h"
    subprocess.run(["gcc", "-std=c99", "-Wall", "-Werror", "-I", os.path.dirname(HEADER), str(c), "-o", str(exe)], check=True)
    size, off, off_prev = map(int, subprocess.check_output([str(exe)]).split())
    K = _lib.FiLearnerConfig
    assert C.sizeof(K) == size and K.history_length.offset == off
    assert off == off_prev + C.sizeof(C.c_int)   # appended right after variable_length


def test_config_default_leaves_histories_off(fi):
    from freeimpala_b200 import _lib
    cfg = _lib.FiLearnerConfig()
    cfg.history_length = 7
    fi.load_library().fi_learner_config_default(C.byref(cfg))
    assert cfg.history_length == 0


@pytest.mark.parametrize("model,value", [("farmer_lstm", 2), ("farmer_lstm", -1), ("mlp_actor_critic", 1)])
def test_create_rejects_invalid_history_length_before_the_device_check(fi, model, value):
    from freeimpala_b200 import _lib
    lib = fi.load_library()
    cfg = _lib.FiLearnerConfig()
    lib.fi_learner_config_default(C.byref(cfg))
    cfg.num_players, cfg.buffer_capacity, cfg.entry_size, cfg.batch_size = 1, 4, 8, 2
    cfg.model = _lib.MODEL[model]
    cfg.loss = _lib.LOSS["vtrace" if model == "mlp_actor_critic" else "mse"]
    cfg.history_length = value
    assert not lib.fi_learner_create(C.byref(cfg))
    msg = _lib.last_error()
    assert msg.startswith("fi_learner_create: history_length") and "no CUDA device" not in msg, msg


def test_learner_keyword_reaches_the_config(fi):
    with pytest.raises(fi.FiError, match="history_length"):
        fi.Learner(1, 4, 8, 2, model="mlp_actor_critic", history_length=True)


def test_variable_length_is_still_refused_for_the_farmer_model(fi):
    with pytest.raises(fi.FiError, match="variable_length is for the actor-critic model"):
        fi.Learner(1, 4, 8, 2, model="farmer_lstm", variable_length=True, history_length=True)
