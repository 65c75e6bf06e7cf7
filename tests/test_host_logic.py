"""Host-side logic of the drop-in layer that needs no GPU: CSV text, argument parsing, the
reference's bookkeeping quirks (SURVEY.md Appendix C)."""
import csv
import os

import numpy as np

from tests.conftest import GOLDEN, run_without_gpu


def test_hue_row_text_matches_reference_layout():
    from opticalflowclustering_b200.drawGridsAndOutputCSV import hue_row_text
    txt = hue_row_text(np.array([60, 0, 179], np.uint8), True)
    assert txt == "cell_0,cell_1,cell_2\n60.0,0.0,179.0\n"
    assert hue_row_text([5], False) == "5.0\n"


def test_outcsv_rows(tmp_path):
    from opticalflowclustering_b200.KmeanGrids import write_outcsv_row
    p = tmp_path / "x.csv"
    hues = list(range(350))
    write_outcsv_row(str(p), hues, True)
    write_outcsv_row(str(p), hues, False)
    rows = list(csv.reader(open(p)))
    assert len(rows) == 3 and len(rows[0]) == 350 and rows[0][349] == "cell_349" and rows[2][7] == "7"
    # golden OutCSV of the reference has the same shape of text
    ref_rows = None
    g = os.path.join(GOLDEN, "g23_cells.npz")
    z = np.load(g)
    write_outcsv_row(str(p), z["outcsv_hues"][0], True)
    ref_rows = list(csv.reader(open(p)))
    assert ref_rows[1] == [str(int(v)) for v in z["outcsv_hues"][0]]


def test_magnitude_csv_text():
    from opticalflowclustering_b200.computeOpticalFlow import magnitude_csv_text
    txt = magnitude_csv_text([0.5, 1.25])
    assert txt.splitlines() == [",Frame,Average Magnitude", "0,0,0.5", "1,1,1.25"]


def test_read_hue_column_bom_and_ints():
    from opticalflowclustering_b200.findCosineDifferentVectors import read_hue_column
    v = read_hue_column(os.path.join(GOLDEN, "bounce.csv"))          # starts with a UTF-8 BOM
    assert v.dtype == np.int64 and len(v) == 16


def test_kmeangrids_flags_are_store_false():
    from opticalflowclustering_b200.KmeanGrids import get_number, parse_arguments
    a = parse_arguments(["-d", "OutImgs/v", "-c", "1", "-f", "x.csv", "--noyolo", "--nocontour", "--path", "v.mp4"])
    assert a["noyolo"] is False and a["nocontour"] is False and a["clusters"] == 1
    a = parse_arguments(["-d", "OutImgs/v", "-c", "2", "-f", "x.csv", "--path", "v.mp4"])
    assert a["noyolo"] is True
    assert get_number("crop_of0012.png") == 12 and get_number("abc") is None


def test_grid_lines_host_match_oracle_rectangles():
    from opticalflowclustering_b200.KmeanGrids import draw_grid_lines_host
    from oracle import grid_np as G
    rng = np.random.default_rng(0)
    for (h, w, rows, cols) in [(720, 1280, 14, 25), (60, 100, 3, 4), (50, 50, 5, 5)]:
        a = rng.integers(0, 200, (h, w, 3), dtype=np.uint8)
        b = a.copy()
        draw_grid_lines_host(a, rows, cols)
        for (x1, y1, x2, y2) in G.grid_cells(h, w, rows, cols):
            G.draw_rect_1px(b, x1, y1, x2, y2)
        assert (a == b).all()


def test_dropins_fail_loudly_without_gpu():
    out = run_without_gpu("""
import numpy as np
import torch
assert not torch.cuda.is_available()
from opticalflowclustering_b200 import _lib, cosine, kmeans
for call in (lambda: kmeans.kmeans_fit(np.zeros((8, 4), np.uint8), np.zeros((2, 4))),
             lambda: cosine.sliding_cosine([1, 2], [1, 2, 3])):
    try:
        call()
    except _lib.OfcError:
        print("raised")
""")
    assert out.split() == ["raised", "raised"]
