"""run.py's --deterministic_training switch (host side, no GPU)."""


def test_run_py_parses_deterministic_training_and_defaults_off():
    import run as idf_run
    base = ["--model", "diff", "--mode", "train", "--prior", "regular", "--dataset", "celeba", "--a_dim", "32"]
    assert idf_run.parse_args(base).deterministic_training is False
    assert idf_run.parse_args(base + ["--deterministic_training"]).deterministic_training is True
