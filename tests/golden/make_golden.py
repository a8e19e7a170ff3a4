"""Write tests/golden/pytorch_reference_<name>*.npz from the reference's own PyTorch golden files.

    python tests/golden/make_golden.py <DLRM.jl checkout>

Source fixtures: ref/pytorch_reference_single.hdf5 and ref/pytorch_reference_multi.hdf5,
the files `test/integration.jl:4-41` and `src/validation.jl:1-44` of the reference check
against (58 datasets each).  Every value is kept verbatim, in a layout that keeps each file
under 1 MB; tests/helpers.py:load_golden rebuilds all 58 datasets, names and dtypes as in
the HDF5 files, so the tests need no HDF5 library at run time:

  * the model's parameters before the step (emb_*, bot_l.*, top_l.*) are not stored: they are
    regenerated from the reference's seed (helpers.reference_parameters), and the file holds
    their SHA-256 (params_sha256) so that a regeneration that differs by one bit fails;
  * update_emb_<k> keeps only the rows the batch looks up (update_emb_<k>_rows, in the order
    of np.unique(input_emb_<k>)): the step changes no other row;
  * the MLP updates go to pytorch_reference_<name>_update_bot.npz and _update_top.npz.
"""
import os
import sys

import numpy as np

HERE = os.path.dirname(os.path.abspath(__file__))
sys.path.insert(0, os.path.join(HERE, "..", ".."))
from dlrm_jl_b200.hdf5_min import read_hdf5  # noqa: E402
from tests.helpers import load_golden, params_sha256, reference_parameters  # noqa: E402


def write(name: str, data: dict) -> None:
    """Store the 58 datasets of one golden file in the compact layout, then check the round trip."""
    params = reference_parameters()
    for k, v in params.items():
        assert np.array_equal(data[k], v) and data[k].dtype == v.dtype, f"{k} is not the seeded initial value"
    main = {k: v for k, v in data.items() if k not in params and not k.startswith("update_")}
    main["params_sha256"] = np.array(params_sha256(params))
    for k in range(7):
        rows = np.unique(data[f"input_emb_{k}"])
        untouched = np.ones(len(data[f"emb_{k}"]), dtype=bool)
        untouched[rows] = False
        assert np.array_equal(data[f"update_emb_{k}"][untouched], data[f"emb_{k}"][untouched])
        main[f"update_emb_{k}_rows"] = data[f"update_emb_{k}"][rows]
    np.savez_compressed(os.path.join(HERE, f"pytorch_reference_{name}.npz"), **main)
    for part in ("bot", "top"):
        np.savez_compressed(os.path.join(HERE, f"pytorch_reference_{name}_update_{part}.npz"),
                            **{k: v for k, v in data.items() if k.startswith(f"update_{part}_")})
    again = load_golden(name)
    assert sorted(again) == sorted(data)
    for k, v in data.items():
        assert np.array_equal(again[k], v) and again[k].dtype == v.dtype, k


def main(ref_root: str) -> None:
    for name in ("single", "multi"):
        src = os.path.join(ref_root, "ref", f"pytorch_reference_{name}.hdf5")
        data = read_hdf5(src)
        assert len(data) == 58, len(data)
        write(name, data)
        print(f"{src} -> tests/golden/pytorch_reference_{name}*.npz: {len(data)} datasets")


if __name__ == "__main__":
    if len(sys.argv) != 2:
        raise SystemExit(__doc__)
    main(sys.argv[1])
