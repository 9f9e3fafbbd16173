"""Test double for the reference's datasets/pair_folders.py (see ../custom_transforms.py).  train.py imports PairFolder for
every real dataset; the tests train on the sequence layout only."""


class PairFolder:
    def __init__(self, *args, **kwargs):
        raise NotImplementedError("the pair-folder layout is not part of the test double")
