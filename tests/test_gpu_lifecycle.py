"""Engine lifecycle: a failed fmgpu_engine_create reports its CUDA error and clears it, so the
next engine in the same process computes exactly what an engine before the failure computed."""
import numpy as np
import pytest

import fmtuner_sdr_b200 as fm
from oracle import orc

pytestmark = pytest.mark.gpu

C, NBLK = 40, 2


def _process(cfg, iq):
    eng = fm.Engine(cfg, C, 0)
    try:
        return eng.process_host(iq, NBLK)
    finally:
        eng.close()


def test_failed_create_leaves_no_error_for_the_next_engine():
    cfg = fm.make_config(max_blocks=NBLK)
    n = NBLK * cfg.block_samples * cfg.decimation
    iq = np.stack([orc.config3_signal(c).generate(n) for c in range(C)])
    before = _process(cfg, iq)
    # 2,000,000 channels: the IQ staging buffer alone would be about 1.3 TB, so the first
    # cudaMalloc fails (an ordinary error return; nothing is allocated)
    with pytest.raises(fm.EngineError, match=r"failed \(-3\)"):
        fm.Engine(fm.make_config(), 2_000_000, 0)
    after = _process(cfg, iq)
    for name, a, b in zip(("audio", "n_audio", "groups", "n_groups", "status"), before, after):
        assert a.tobytes() == b.tobytes(), name
