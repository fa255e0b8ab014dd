"""The environment switches that remain in the library select code paths the default run never takes (the padded residue
axis, the dense adjacency walk, the separate pooling kernel, the full-square contact-map kernel, the fused LSTM kernel without
CTA pairs ...).  Each one is exercised here against the exact-fp32 engine / the oracle so that it cannot
rot; the measured-and-rejected experiments of round 1 (CTA-pair adjacency kernel, N = 256 adjacency MMA, tile-dithered weights,
CNN weight multicast) were deleted instead."""
import os
import subprocess
import sys

import pytest

pytestmark = pytest.mark.gpu
ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))

SWITCHES = [{}, {"MDF_COMPACT": "0"}, {"MDF_ADJ_SPARSE": "0"}, {"MDF_POOL_FUSED": "0"}, {"MDF_ADJ_LEAN": "0"}, {"MDF_ADJ_EXPAND": "0"},
            {"MDF_GEMM_PAIR": "0"}, {"MDF_EMBED_STAGED": "0"}, {"MDF_HEAD_TC": "0"}, {"MDF_CMAP_SYM": "0"}, {"MDF_XW_MEAN": "0"}, {"MDF_LSTM_COOP": "0"},
            {"MDF_LSTM_PAIR": "0"}, {"MDF_LSTM_CELL": "0"}, {"MDF_LSTM_ABLATE": "64"}, {"MDF_LSTM_ABLATE": "384"}, {"MDF_LSTM_CLUSTER": "8"}, {"MDF_LSTM_PRECISE_LEN": "100"}, {"MDF_HOST_THREADS": "1"}]


@pytest.mark.parametrize("env", SWITCHES, ids=lambda e: ",".join(f"{k}={v}" for k, v in e.items()) or "defaults")
def test_switch_path_matches_exact_engine(env):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "_switch_worker.py")], env=dict(os.environ, **env),
                       capture_output=True, text=True, timeout=600)
    assert r.returncode == 0 and "SWITCH_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]


# the LSTM switches again on the full-size head: H = 512 selects the fused kernel's straight-line CTA-pair issuer (the small shape
# above runs its generic loop), so the alternative paths of THAT code are the ones exercised here
LSTM_FULL = [{}, {"MDF_LSTM_CELL": "0"}, {"MDF_LSTM_ABLATE": "64"}, {"MDF_LSTM_ABLATE": "384"}, {"MDF_LSTM_CLUSTER": "8"},
             {"MDF_LSTM_PRECISE_LEN": "100"}, {"MDF_LSTM_PAIR": "0"}, {"MDF_LSTM_PHASES": "8"}]


@pytest.mark.parametrize("env", LSTM_FULL, ids=lambda e: "full," + (",".join(f"{k}={v}" for k, v in e.items()) or "defaults"))
def test_lstm_switch_on_full_size_head(env):
    r = subprocess.run([sys.executable, os.path.join(ROOT, "tests", "_switch_worker.py")],
                       env=dict(os.environ, MDF_TEST_FULL_MODEL="1", **env), capture_output=True, text=True, timeout=900)
    assert r.returncode == 0 and "SWITCH_OK" in r.stdout, r.stdout[-2000:] + r.stderr[-4000:]
