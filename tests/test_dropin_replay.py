"""Drop-in boundary, stage B (see oracle/dropin.py): the reference's UNMODIFIED Inference_*.py scripts run here with a
session that answers every run() with what the vadx sessions produced on the B200 for exactly that call
(tests/golden/dropin_vadx_outputs.npz, written by tests/test_gpu_dropin.py) -- after checking that the feed the script
built is bit-for-bit the one stage A fed -- and the two text files each script writes must equal the files of the
all-reference run.  The replay needs a checkout of the upstream reference project (oracle/ref_loader.py) and skips
without one; the check of the committed transcript runs everywhere."""
import os

import numpy as np
import pytest

from oracle import ref_loader as RL

GOLD = os.path.join(os.path.dirname(os.path.abspath(__file__)), "golden")
needs_reference = pytest.mark.skipif(not RL.reference_available(),
                                     reason="replays into the upstream reference scripts, which are not part of this repository")


@pytest.fixture(scope="module")
def replayed():
    from oracle import dropin
    tr = np.load(os.path.join(GOLD, "dropin_transcript.npz"))
    vx = np.load(os.path.join(GOLD, "dropin_vadx_outputs.npz"))
    return tr, vx, dropin.replay_scripts(tr, vx)


@needs_reference
@pytest.mark.parametrize("family,n_calls", [("firered", 6), ("fsmn", 8), ("silero", 175)])
def test_unmodified_script_on_vadx_outputs_writes_the_reference_files(replayed, family, n_calls):
    tr, vx, res = replayed
    ns, files, calls = res[family]
    assert calls == n_calls                                      # every recorded call was consumed, none was extra
    assert files["timestamps_second.txt"] == str(tr[f"{family}_file_second"])
    assert files["timestamps_indices.txt"] == str(tr[f"{family}_file_indices"])
    assert len(files["timestamps_second.txt"].strip().splitlines()) >= 1


def test_transcript_files_are_the_committed_script_goldens():
    """the all-reference text files in the transcript are the same ones the per-family goldens hold"""
    tr = np.load(os.path.join(GOLD, "dropin_transcript.npz"))
    fr = np.load(os.path.join(GOLD, "firered_script.npz"))
    fs = np.load(os.path.join(GOLD, "fsmn.npz"))
    si = np.load(os.path.join(GOLD, "silero.npz"))
    assert str(tr["firered_file_second"]) == str(fr["vad_file_second"]) and str(tr["firered_file_indices"]) == str(fr["vad_file_indices"])
    assert str(tr["fsmn_file_second"]) == str(fs["c16000_file_second"]) and str(tr["fsmn_file_indices"]) == str(fs["c16000_file_indices"])
    assert str(tr["silero_file_second"]) == str(si["sample_file_second"]) and str(tr["silero_file_indices"]) == str(si["sample_file_indices"])
