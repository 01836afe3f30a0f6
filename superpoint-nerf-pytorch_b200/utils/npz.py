"""Deterministic .npz writer shared by the evaluation and matching outputs."""
import io
import zipfile

import numpy as np


def write_npz(path, arrays):
    """np.savez without the zip members' wall-clock timestamps, so that equal arrays give equal bytes."""
    with zipfile.ZipFile(path, "w", zipfile.ZIP_STORED) as z:
        for k in sorted(arrays):
            buf = io.BytesIO()
            np.lib.format.write_array(buf, np.asanyarray(arrays[k]), allow_pickle=False)
            z.writestr(zipfile.ZipInfo(f"{k}.npy", date_time=(1980, 1, 1, 0, 0, 0)), buf.getvalue())
