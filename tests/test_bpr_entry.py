"""The command line of BPR training (main_rec --loss bpr) and the shape of its epoch, without a GPU."""
import pytest


def test_bpr_flags_stay_out_of_the_reference_namespace():
    from spex_b200.lg_parser import parse_args_r

    plain = vars(parse_args_r([]))
    assert not {"loss", "decay", "bpr_batch"} & set(plain)
    a = parse_args_r(["--loss", "bpr", "--decay", "0.001", "--bpr_batch", "512"])
    assert (a.loss, a.decay, a.bpr_batch) == ("bpr", 0.001, 512)
    assert {k: v for k, v in vars(a).items() if k in plain} == plain
    assert parse_args_r(["--loss", "bce"]).loss == "bce"
    with pytest.raises(SystemExit):
        parse_args_r(["--loss", "hinge"])


def test_bpr_epoch_draws_n_train_triples_in_ceil_steps():
    from spex_b200.main_rec import bpr_epoch_steps

    assert bpr_epoch_steps(5000, 2048) == [2048, 2048, 904]
    assert bpr_epoch_steps(4096, 2048) == [2048, 2048]
    assert bpr_epoch_steps(668, 2048) == [668]
    assert bpr_epoch_steps(0, 2048) == []
