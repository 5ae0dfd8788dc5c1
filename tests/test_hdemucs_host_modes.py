"""HDemucsEngine's host logic in the tensor-core modes, through the ABI emulator (CPU).  These modes take their own host
paths: the 3-tap form of the transposed convolutions, the 16-column padded DConv weights and the arithmetic handed to
the register-level thin-layer kernels.  The emulator computes in fp32, so this checks wiring, geometry and workspaces,
not rounding."""
import pytest
import torch

from _fixtures import golden, rel_l2, synth_mix
from abi_emulator import emulated_abi
from demucs_b200 import hdemucs as HD
from demucs_b200.hdemucs_engine import HDemucsEngine
from oracle.hdemucs_oracle import hdemucs_forward
from oracle.make_golden import hdemucs_small_config


@pytest.mark.parametrize("mode", ["tf32", "tf32x3", "strict", "bf16"])
def test_engine_host_logic_matches_oracle(mode):
    g = golden("hdemucs_small_odd.npz")          # odd length: the padded pair rows of layer 5 and the odd time lengths
    cfg = hdemucs_small_config()
    W = HD.init_weights(cfg, int(g["seed"]), float(g["layer_scale"]))
    mix = synth_mix(1, int(g["length"]), 4321 + int(g["seed"]))
    with torch.no_grad():
        want = hdemucs_forward(W, cfg, mix)
    with emulated_abi():
        got = HDemucsEngine(cfg, W, "cpu", mode=mode).forward(mix)
    assert rel_l2(got, want) < 1e-5
