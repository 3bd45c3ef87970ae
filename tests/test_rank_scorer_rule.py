"""FullRanker.scorer_for for a rank query (k=None), with the near-tie probe's verdict injected: no GPU needed."""
import pytest
import torch


@pytest.mark.parametrize("verdict", [False, True])
@pytest.mark.parametrize("probe", [False, True])
def test_rank_scorer_rule_table(monkeypatch, probe, verdict):
    """"f16" ranks with the f16 rank kernel unless probe=True and the probe finds the filter not selective (then
    "fp32"); "fp32" ranks with fp32 at any D and never asks the probe; "bf16" has no rank kernel (ValueError)."""
    from spex_b200 import ops

    asked = []

    def fake_probe(U, I, users):
        asked.append((U, I, users))
        return verdict

    monkeypatch.setattr(ops, "f16_filter_is_selective", fake_probe)
    U, users = torch.zeros(8, 1), torch.arange(8)
    for precision, dims in (("f16", (64, 128)), ("bf16", (64,)), ("fp32", (40, 64, 128, 192))):
        for D in dims:
            I = torch.zeros(16, D)
            ranker = ops.FullRanker(I, precision, probe=probe)
            asked.clear()
            if precision == "bf16":
                with pytest.raises(ValueError, match="bf16"):
                    ranker.scorer_for(None, U, users)
                assert not asked
                continue
            consulted = precision == "f16" and probe
            want = "fp32" if consulted and not verdict else precision
            assert ranker.scorer_for(None, U, users) == want, (precision, D)
            assert len(asked) == consulted, (precision, D)
            assert all(a[0] is U and a[1] is I and a[2] is users for a in asked)
