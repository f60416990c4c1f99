"""bench.py --dump-outputs: the last timed step's results are written so that two runs, or two builds, can be compared
entry for entry.  CPU only: a small stand-in model in place of the detector."""
import numpy as np
import torch

import bench


def test_dump_outputs_is_reproducible_and_samples_large_tensors(tmp_path):
    torch.manual_seed(0)
    m = torch.nn.Sequential(torch.nn.Linear(300, 200), torch.nn.Linear(200, 3))
    with torch.no_grad():
        m[0].weight.copy_(torch.arange(60000.0).view(200, 300))      # value == flat position: the sample shows its positions
    for d in ("a", "b"):
        bench.dump_outputs(tmp_path / d, m, [torch.tensor(1.5), torch.tensor(-2.0)])
    a, b = ({k: np.load(tmp_path / d / f"{k}.npy") for k in ("losses", "params")} for d in ("a", "b"))
    for k in a:
        assert a[k].dtype == np.float32 and np.array_equal(a[k], b[k]), k
    assert a["losses"].tolist() == [1.5, -2.0]
    cap = bench.DUMP_PER_TENSOR
    assert cap < 60000 and len(a["params"]) == cap + 200 + 600 + 3
    pos = a["params"][:cap]
    assert (np.diff(pos) > 0).all() and pos[0] >= 0 and pos[-1] < 60000             # distinct positions, in order
    rest = torch.cat([m[0].bias, m[1].weight.flatten(), m[1].bias]).detach().numpy()
    np.testing.assert_array_equal(a["params"][cap:], rest)                             # small tensors whole
