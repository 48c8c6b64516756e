"""Full-neighbourhood PBR priorities, host side (no GPU): the driver's --priority_neighbourhood flag."""
import importlib.util
import os

import pytest

ROOT = os.path.dirname(os.path.dirname(os.path.abspath(__file__)))


def _driver():
    spec = importlib.util.spec_from_file_location("ogl_train_main_prio", os.path.join(ROOT, "train", "__main__.py"))
    m = importlib.util.module_from_spec(spec)
    spec.loader.exec_module(m)
    return m


def test_driver_priority_neighbourhood_flag():
    m = _driver()
    base = ["pubmed", "pytorch", "o.csv", "t", "--cuda"]
    data = m.parse(base)[1]
    assert data["priority_neighbourhood"] == "sampled" and data["eval_neighbourhood"] == "sampled"
    data = m.parse(base + ["--priority_neighbourhood", "full"])[1]
    assert data["priority_neighbourhood"] == "full" and data["eval_neighbourhood"] == "sampled"
    # the two options are independent
    data = m.parse(base + ["--eval_neighbourhood", "full"])[1]
    assert data["priority_neighbourhood"] == "sampled" and data["eval_neighbourhood"] == "full"
    for bad in ("exact", "Full", ""):
        with pytest.raises(SystemExit):
            m.parse(base + ["--priority_neighbourhood", bad])
