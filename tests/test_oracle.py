"""CPU tests: the oracle against every pin that exists (golden vectors from the
reference's own glue, literal graph execution, known answers)."""
import os

import numpy as np
import pytest

from conftest import REFERENCE, WEIGHTS, load_weights
from oracle import restated as R

HAVE_REF = bool(REFERENCE) and os.path.isdir(os.path.join(REFERENCE, "tf_lite_models"))
NO_REF = "needs the reference's .tflite files: set WWB_REFERENCE to a checkout of the reference project"


def test_known_answers(w_crnn, w_crnn_softmax, w_wavenet):
    # SURVEY.md Appendix A4
    z = np.zeros((1, 151, 40), np.float32)
    assert abs(float(R.posterior(z, w_crnn)[0]) - 0.00343328) < 1e-6
    np.testing.assert_allclose(R.detect(R.encode(z, w_crnn_softmax), w_crnn_softmax)[0],
                               [0.8681737, 0.13182628], atol=1e-6)
    zw = np.zeros((1, 182, 40), np.float32)
    np.testing.assert_allclose(R.detect(R.encode(zw, w_wavenet), w_wavenet)[0],
                               [0.87389916, 0.12610082], atol=1e-6)
    # digital silence -> mel exactly 0.0
    assert np.all(R.mel_from_magnitude(np.zeros((2, 257), np.float32), w_crnn) == 0.0)


def test_mel_matrix_is_slaney(w_crnn):
    W = w_crnn["mel_w"]
    assert W.shape == (40, 257)
    assert np.count_nonzero(W) == 490
    assert np.all(W[:, 0] == 0) and np.all(W[:, 256] == 0)
    assert (np.count_nonzero(W, axis=1)).max() <= 36


def test_golden_filter(golden, w_crnn):
    for tag, a in (("pe0", 0.0), ("pe97", 0.97)):
        n = int(golden["filter_consumed_" + tag])
        mel = R.mel_stream(golden["filter_in"][:n], w_crnn, a)
        ref = golden["filter_mel_" + tag]
        assert mel.shape == ref.shape
        np.testing.assert_allclose(mel, ref, atol=2e-6)
        assert int(golden["filter_counts_" + tag].sum()) == ref.shape[0]


@pytest.mark.parametrize("name", ["crnn", "wavenet"])
def test_golden_trigger(golden, name):
    w = load_weights("CRNN" if name == "crnn" else "Wavenet")
    t = R.TriggerOracle(w)
    pcm, sp = golden["trig_%s_pcm" % name], golden["trig_%s_speech" % name]
    at = -1
    for i in range(len(sp)):
        t(pcm[i * 320:(i + 1) * 320], bool(sp[i]))
        if t.active:
            at = i
            break
    assert at == int(golden["trig_%s_active_at" % name]) and at > 0
    ref = golden["trig_%s_post" % name]
    assert len(t.posteriors) == len(ref)
    np.testing.assert_allclose(np.array(t.posteriors, np.float32), ref, atol=5e-6)
    assert abs(t.post_max - float(golden["trig_%s_post_max" % name])) < 5e-6


@pytest.mark.parametrize("name", ["crnn", "wavenet"])
def test_golden_get_posterior_and_sweep(golden, name):
    w = load_weights("CRNN_arik_original" if name == "crnn" else "Wavenet")
    clips = [golden["gp_%s_clip%d" % (name, i)] for i in range(3)]
    fn = np.array(R.get_posterior(clips, w, "false_negatives"))
    fa = np.array(R.get_posterior(clips, w, "false_accepts"))
    np.testing.assert_allclose(fn, golden["gp_%s_frr_max" % name], atol=5e-6)
    assert fa.shape == golden["gp_%s_far_traj" % name].shape
    np.testing.assert_allclose(fa, golden["gp_%s_far_traj" % name], atol=5e-6)
    thr = R.thresholds_eval()
    np.testing.assert_array_equal(thr, golden["sweep_%s_thr" % name])
    acc, edg = R.far_frr_counts(golden["gp_%s_frr_max" % name], golden["gp_%s_far_traj" % name], thr)
    np.testing.assert_array_equal((3 - acc) / 3, golden["sweep_%s_frr" % name])
    np.testing.assert_array_equal(edg / 0.5, golden["sweep_%s_far" % name])
    assert acc.max() >= 1 and (name == "crnn" or edg.max() >= 1)   # the fixtures do exercise the counters


def test_golden_threshold_accepts(golden):
    acc = np.array([R.rising_edges(golden["pm_traj"], t) for t in golden["pm_thr"]])
    np.testing.assert_array_equal(acc, golden["pm_accepts"])
    np.testing.assert_array_equal(R.thresholds_plot(), golden["pm_thr"])


def test_window_counts():
    # SURVEY.md Appendix C: 10 s clip padded to 11 s -> F = 1097 -> 474 CRNN / 458 WaveNet windows
    assert R.num_frames(176000) == 1097
    assert R.eval_windows(1097, 151) == 474 and R.eval_windows(1097, 182) == 458
    assert R.num_frames(511) == 0 and R.num_frames(512) == 1 and R.eval_windows(150, 151) == 0


@pytest.mark.skipif(not HAVE_REF, reason=NO_REF)
def test_restated_equals_literal():
    from oracle.tflite_literal import LiteralInterpreter
    ref = os.path.join(REFERENCE, "tf_lite_models")
    rng = np.random.default_rng(0)
    w = load_weights("CRNN")
    e, d = LiteralInterpreter(ref + "/CRNN/encode.tflite"), LiteralInterpreter(ref + "/CRNN/detect.tflite")
    mel = (rng.random((3, 151, 40)) * 6).astype(np.float32)
    enc_l = np.stack([e(m.T[None, :, :, None])[0][0] for m in mel])
    np.testing.assert_allclose(R.crnn_encode(mel, w), enc_l, atol=5e-6)
    np.testing.assert_allclose(R.crnn_detect(enc_l, w), np.stack([d(x[None])[0][0] for x in enc_l]), atol=1e-6)
    ww = load_weights("Wavenet")
    e, d = LiteralInterpreter(ref + "/Wavenet/encode.tflite"), LiteralInterpreter(ref + "/Wavenet/detect.tflite")
    mel = (rng.random((2, 182, 40)) * 6).astype(np.float32)
    enc_l = np.stack([e(m[None])[0][0] for m in mel])
    np.testing.assert_allclose(R.wavenet_encode(mel, ww), enc_l, atol=5e-6)
    np.testing.assert_allclose(R.wavenet_detect(enc_l, ww), np.stack([d(x[None])[0][0] for x in enc_l]), atol=1e-6)
    f = LiteralInterpreter(ref + "/CRNN/filter.tflite")
    mag = (rng.random((4, 257)) * 3).astype(np.float32)
    np.testing.assert_allclose(R.mel_from_magnitude(mag, w), np.stack([f(m[None])[0][0] for m in mag]), atol=2e-6)


@pytest.mark.skipif(not HAVE_REF, reason=NO_REF)
def test_committed_weights_match_reference_files():
    from wakeword_detection_b200 import weights as W
    for name, sub, typ in (("CRNN", "tf_lite_models/CRNN", "CRNN"), ("Wavenet", "tf_lite_models/Wavenet", "Wavenet")):
        a = W.load_model_dir(os.path.join(REFERENCE, sub), typ)
        b = W.load_model_dir(os.path.join(WEIGHTS, name), typ)
        assert set(a) == set(b)
        for k in a:
            np.testing.assert_array_equal(a[k], b[k])
    geo = W.geometry(W.load_model_dir(os.path.join(WEIGHTS, "Wavenet"), "Wavenet"))
    assert geo["mel_length"] == 182 and geo["fft"] == 512 and geo["encode_width"] == 32
