"""Device memory of a domain and its companion objects (luw_domain_bytes, the reference's Device_Info::memory_used): a fresh domain counts its lattice
arrays; each companion object adds exactly its own arrays while it lives and gives all of them back when it is destroyed."""
import numpy as np
import pytest

from latticeurbanwind_b200 import _cabi as A
from latticeurbanwind_b200.domain import CellSet, Domain, Probes, Stats, VkInlet, WallLoads, WindStats

SHAPE = (20, 12, 8)
N_DEV = 32 * 12 * 8  # cells of a device array: rows padded to 32
K = 50  # listed cells
CELLS = np.arange(0, 5 * K, 5, dtype=np.uint64)
LABELS = np.array([0] * 40 + [2] * 10, np.uint32)  # label 1 has no cells
L, CAPACITY, THRESHOLDS, MODES, MODE_STRIDE = 3, 16, (0.01, 0.02, 0.05), 5, 6


def _lattice_bytes(ddf_size, thermal):
    b = 19 * N_DEV * ddf_size + 4 * N_DEV + 12 * N_DEV + N_DEV + 16  # fi rho u flags sched
    return b + (7 * N_DEV * ddf_size + 4 * N_DEV + 12 * N_DEV if thermal else 0)  # gi T upre


def _companions(dom, thermal):
    """(name, constructor, bytes of its device arrays)"""
    rng = np.random.default_rng(3)
    # wall loads: label 0 = 2 chunks of at most 32 cells, label 2 = 1 chunk; one group of chunks per label
    nchunks, ngroups = 3, 2
    wall = 3 * L * 8 + (L + 1) * 8 + CAPACITY * L * 6 * 8 + K * (8 + 4 + 12 + 24) + (nchunks + 1) * 8 + nchunks * 4 + 6 * nchunks * 8 + (ngroups + 1) * 8 + 6 * ngroups * 8
    return [
        ("CellSet", lambda: CellSet(dom, CELLS), 8 * K + 4 * 3 * K * 4),
        ("Stats", lambda: Stats(dom), (3 + 3 + 1 + thermal) * N_DEV * 4),
        ("WindStats", lambda: WindStats(dom, CELLS, THRESHOLDS), 8 * K + 12 * K * 4 + len(THRESHOLDS) * K * 4),
        ("WallLoads", lambda: WallLoads(dom, CELLS, LABELS, L, rng.random((L, 3)), capacity=CAPACITY), wall),
        ("Probes", lambda: Probes(dom, CELLS, capacity=CAPACITY), 8 * K + CAPACITY * (5 if thermal else 4) * K * 4),
        ("VkInlet", lambda: VkInlet(dom, CELLS, np.zeros(K, np.uint8), rng.random(7 * K), rng.random(10 * MODE_STRIDE), MODES, MODE_STRIDE),
         8 * K + K + 7 * K * 4 + 10 * MODE_STRIDE * 4 + 6 * MODE_STRIDE * 4),
    ]


@pytest.mark.gpu
@pytest.mark.parametrize("precision,thermal", [(A.FP16S, False), (A.FP32, True)], ids=["fp16s", "fp32-thermal"])
def test_companion_bytes_are_given_back(precision, thermal):
    with Domain(*SHAPE, precision=precision, features=A.TEMPERATURE if thermal else 0) as dom:
        assert dom.device_bytes() == _lattice_bytes(4 if precision == A.FP32 else 2, thermal)
        for name, make, nbytes in _companions(dom, thermal):
            before = dom.device_bytes()
            obj = make()
            assert dom.device_bytes() - before == nbytes, f"{name} while alive"
            obj.close()
            assert dom.device_bytes() == before, f"{name}: {dom.device_bytes() - before} bytes still counted after destroy"
