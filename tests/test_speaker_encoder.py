"""Row N3: speaker encoder.  CPU: the oracle restatement against the golden vectors produced by the reference's own
SpeakerEncoder class; GPU: the device implementation (mel front-end, LSTM, averaging) through the C ABI against both."""
import numpy as np
import pytest
import torch

from mvb200 import synth
from oracle import speaker_port as P


def test_oracle_network_and_slicing_match_reference_golden(golden_dir):
    g = np.load(f"{golden_dir}/speaker.npz")
    sd = synth.speaker_encoder_state_dict(3)
    assert synth.state_dict_checksum(sd) == pytest.approx(float(g["checksum"]), abs=1e-9)
    o = P.SpeakerOracle(sd)
    emb = o.forward(torch.from_numpy(g["mels"]))
    assert np.abs(emb.numpy() - g["emb"]).max() < 2e-6                      # reference forward(): pinned
    e, partials = o.embed_utterance(g["wav"])
    assert partials.shape == g["partials"].shape and np.abs(partials - g["partials"]).max() < 2e-6
    assert np.abs(e - g["utt_embed"]).max() < 2e-6                          # reference embed_utterance(): slicing + mean pinned
    from mvb200.speaker_encoder import SpeakerEncoder, slaney_mel_filterbank
    ws, ms = SpeakerEncoder.compute_partial_slices(len(g["wav"]), 1.3, 0.75)
    assert [(s.start, s.stop) for s in ms] == [tuple(x) for x in g["mel_slices"].tolist()]
    assert np.array_equal(slaney_mel_filterbank(16000, 400, 40), P.mel_filterbank())


def test_partial_slices_match_live_reference(golden_dir):
    """The slices the reference's own SpeakerEncoder.compute_partial_slices returns, as recorded by
    oracle/make_golden_reference.py."""
    from mvb200.speaker_encoder import SpeakerEncoder
    g = np.load(f"{golden_dir}/reference_checks.npz")
    for n in (16000, 25601, 102400, 480000, 777777):
        for rate, cov in ((1.3, 0.75), (2.0, 0.5)):
            a, b = (g[f"spk_{n}_{rate}_{cov}_wav"], g[f"spk_{n}_{rate}_{cov}_mel"]), SpeakerEncoder.compute_partial_slices(n, rate, cov)
            assert [tuple(s) for s in a[0].tolist()] == [(s.start, s.stop) for s in b[0]]
            assert [tuple(s) for s in a[1].tolist()] == [(s.start, s.stop) for s in b[1]]


def test_wav_reader_resampler_trimmer(tmp_path):
    from mvb200 import audio_out as A
    from mvb200.speaker_encoder import check_audio_file, read_wav, resample, trim_silence
    wav = np.concatenate([np.zeros(8000, np.float32), synth.synthetic_waveform(1.0, 24000, seed=2), np.zeros(12000, np.float32)])
    p = A.audio_write_wav(str(tmp_path / "ref"), torch.from_numpy(wav)[None], 24000, strategy="clip")
    x, sr = read_wav(p)
    assert sr == 24000 and x.shape == wav.shape and np.abs(x - wav).max() < 2.0 / 32768
    y = resample(x, 24000, 16000)
    assert abs(y.size - wav.size * 2 // 3) <= 1
    t = trim_silence(y, top_db=20)
    assert 0.8 * 16000 < t.size < 1.25 * 16000                      # the two silent flanks are gone
    with pytest.raises(Exception, match="too short"):
        check_audio_file(p)


@pytest.mark.gpu
def test_device_speaker_encoder_vs_reference_golden(golden_dir):
    from mvb200.speaker_encoder import SpeakerEncoder
    g = np.load(f"{golden_dir}/speaker.npz")
    enc = SpeakerEncoder(model_state=synth.speaker_encoder_state_dict(3), device="cuda:0", verbose=False)
    wav = g["wav"]
    ws, ms = enc.compute_partial_slices(len(wav), 1.3, 0.75)
    padded = np.pad(wav, (0, max(0, ws[-1].stop - len(wav))))
    mel = enc.wav_to_mel_spectrogram(padded).cpu().numpy()
    ref_mel = g["mel"]
    assert mel.shape == ref_mel.shape
    err_mel = np.abs(mel - ref_mel).max() / np.abs(ref_mel).max()
    embed, partials, _ = enc.embed_utterance(wav, return_partials=True)
    err_p = np.abs(partials - g["partials"]).max()
    err_e = np.abs(embed - g["utt_embed"]).max()
    print(f"speaker encoder on device: mel rel err {err_mel:.2e}, partial embeddings abs err {err_p:.2e}, utterance embedding {err_e:.2e}")
    assert err_mel < 1e-4 and err_p < 1e-4 and err_e < 1e-4
    assert abs(np.linalg.norm(embed) - 1.0) < 1e-5
