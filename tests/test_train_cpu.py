"""Contact-classifier training step against the reference's own module (tests/golden/make_contact_train_golden.py: three Adam
steps of `OpenPoseModel` in training mode), and a small end-to-end run whose weights load into the inference path."""
import os
import sys

import numpy as np
import pytest

G = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
sys.path.insert(0, G)


def test_three_adam_steps_match_reference_module(chd):
    """In fp64 like the golden run (see its generator): in fp32 the steps of the biases in front of a BatchNorm depend on the
    host's thread count and SIMD width."""
    import torch
    from make_contact_golden import contact_weights
    T = chd.train
    g = np.load(os.path.join(G, "contact", "train_golden.npz"))
    rng = np.random.default_rng(11)
    xs = rng.normal(0, 0.6, (3, 64, 9, 13, 3))
    xs[..., 2] = rng.uniform(0, 1, xs[..., 2].shape)
    ys = (rng.uniform(size=(3, 64, 5, 4)) < 0.4).astype(np.float64)
    sd = {k: torch.from_numpy(v.astype(np.float64) if v.dtype == np.float32 else v.copy()) for k, v in contact_weights(5).items()}
    tr = T.Trainer(sd=sd)
    torch.manual_seed(7)
    for s in range(3):
        loss, conf = tr.step(torch.from_numpy(xs[s]), torch.from_numpy(ys[s]))
        assert abs(loss - float(g["losses"][s])) < 1e-12
        np.testing.assert_array_equal(conf, g["confusion"][s])
    for k, v in tr.state_dict_numpy().items():
        f = np.asarray(v, dtype=np.float64).reshape(-1)
        pos = np.random.default_rng(len(f)).integers(0, len(f), 512)
        dig = np.concatenate([[f.sum(), (f * f).sum()], f[pos]])
        np.testing.assert_allclose(dig, g["final/" + k], rtol=1e-9, atol=1e-11, err_msg=k)
    with torch.no_grad():
        ev = T.forward(tr.sd, torch.from_numpy(xs[0]), False).numpy()
    np.testing.assert_allclose(ev, g["eval_logits"], atol=1e-11)


def test_window_construction_matches_inference_windows(chd):
    """make_window (training) builds the same 9 x 13 x 3 window the inference path / reference dataset builds (no noise)."""
    from oracle import contact as oc
    g = np.load(os.path.join(G, "contact", "contact_golden.npz"), allow_pickle=True)
    n = list(g["names"])[0]
    fr = g["proc_" + n]
    win = oc.windows_from_frames(fr[None])          # (1 * nwin, 9, 13, 3) float32: window w covers frames [w, w + 9)
    for tgt in (4, 10, fr.shape[0] - 5):
        w, lab = chd.train.make_window(fr, np.zeros((fr.shape[0], 4)), tgt)
        np.testing.assert_array_equal(w, win.reshape(-1, 9, 13, 3)[tgt - 4])
        assert lab.shape == (5, 4)


def test_training_learns_and_weights_load(chd):
    import torch
    T = chd.train
    rng = np.random.default_rng(0)
    # sequences whose contact labels are a simple function of the ankle heights: learnable in a few epochs
    frames, labels = [], []
    for i in range(96):
        F = 40
        fr = rng.normal(0, 0.3, (F, 25, 3))
        fr[:, :, 2] = rng.uniform(0.3, 1.0, (F, 25))
        ph = rng.uniform(0, 2 * np.pi)
        lift_l, lift_r = np.sin(np.arange(F) * 0.4 + ph), -np.sin(np.arange(F) * 0.4 + ph)
        fr[:, [14, 19, 20, 21], 1] += lift_l[:, None]
        fr[:, [11, 22, 23, 24], 1] += lift_r[:, None]
        lab = np.stack([lift_l < 0, lift_l < 0, lift_r < 0, lift_r < 0], axis=1).astype(np.float32)
        frames.append(fr)
        labels.append(lab)
    tr0 = T.Trainer(seed=1)
    xs, ys = zip(*[T.make_window(frames[i], labels[i], 20) for i in range(96)])
    x, y = torch.as_tensor(np.stack(xs)), torch.as_tensor(np.stack(ys))
    l0, _ = tr0.evaluate(x, y)
    tr = T.train(frames, labels, epochs=60, batch_size=32, seed=1)
    l1, c1 = tr.evaluate(x, y)
    assert l1 < 0.8 * l0 and T.metrics(c1)[0] > 0.75
    sd = tr.state_dict_numpy()
    assert set(sd) == set(T.init_state(0)) and sd["model.0.weight"].shape == (1024, 351)
    w, b, bn = chd.contact.pack_state_dict(sd)                        # what chd_contact_create takes
    assert w.size == 953984 and b.size == 1716 and bn.size == 4 * (1024 + 512 + 128 + 32)
