"""Fixtures shared by the command-line tests.  Kept apart from _data.py, which bench.py, smoke() and scripts/ import
without pytest."""
import os

import numpy as np
import pytest

from _data import GOLD


@pytest.fixture()
def crumb_csv(tmp_path, monkeypatch):
    """data/crumb_data.csv rebuilt from the packaged fixture in a temporary directory, which becomes the working
    directory: the command lines write their output tree there."""
    z = np.load(os.path.join(GOLD, "datasets.npz"))
    os.makedirs(tmp_path / "data")
    f = tmp_path / "data" / "crumb_data.csv"
    with open(f, "w") as out:
        out.write("Compound,Channel,Experiment,Dose,Response\n")
        for row in zip(z["crumb_data__drug"], z["crumb_data__channel"], z["crumb_data__experiment"],
                       z["crumb_data__dose"], z["crumb_data__response"]):
            out.write("%s,%s,%d,%r,%r\n" % (row[0], row[1], row[2], float(row[3]), float(row[4])))
    monkeypatch.chdir(tmp_path)
    return str(f)
