"""runner.FlatAdam host logic (no kernels): the launch table of the update and torch's Adam / AdamW state-dict
layout in both directions."""
import copy

import torch


def _nets():
    torch.manual_seed(0)
    net = torch.nn.Sequential(torch.nn.Linear(100, 90), torch.nn.Linear(90, 3), torch.nn.Linear(7, 1))  # [2] unused
    return net, copy.deepcopy(net)


def test_flat_adam_launch_table_covers_the_live_parameters_once():
    from spgnn_b200.runner import FlatAdam
    net, _ = _nets()
    opt = FlatAdam(net.parameters())
    assert opt.step_t.tolist() == [0] * 6 and opt.max_exp_avg_sq is None
    live = [0, 1, 3]
    table, n = opt._table(live)
    assert table.dtype == torch.int64 and table[3 * n:].tolist() == live
    assert opt._table(live)[0] is table                                   # built once per set of live parameters
    covered = []
    for o, k, i in table[:3 * n].view(n, 3).tolist():
        po, pk = opt.offsets[i]
        assert po <= o and o + k <= po + pk and 0 < k <= opt.CHUNK       # a chunk lies inside one parameter
        covered += range(o, o + k)
    want = [e for i in live for e in range(opt.offsets[i][0], sum(opt.offsets[i]))]
    assert covered == want and n == 3 + 1 + 1                             # the 9000-element weight is 3 chunks
    assert opt._table([0, 1, 2, 3])[1] == 3 + 1 + 1 + 1 and len(opt._tables) == 2


def test_flat_adam_loads_torch_state_dicts_and_torch_loads_its_own():
    """A CPU torch.optim.Adam / AdamW state dict (one ``step`` given as a number) loads into FlatAdam with the saved
    group's hyper-parameters; FlatAdam's state dict loads back into torch and reproduces torch's state."""
    from spgnn_b200.runner import FlatAdam
    for cls, decoupled in ((torch.optim.Adam, False), (torch.optim.AdamW, True)):
        net, ref = _nets()
        opt = FlatAdam(net.parameters())
        t_opt = cls(ref.parameters(), lr=0.02, betas=(0.8, 0.99), amsgrad=True, weight_decay=0.1)
        for _ in range(3):
            t_opt.zero_grad()
            ref[1](ref[0](torch.randn(4, 100))).square().sum().backward()
            t_opt.step()
        sd = copy.deepcopy(t_opt.state_dict())
        sd["state"][1]["step"] = float(sd["state"][1]["step"])
        opt.load_state_dict(sd)
        assert (opt.lr, opt.betas, opt.weight_decay, opt.amsgrad, opt.decoupled) == (0.02, (0.8, 0.99), 0.1, True,
                                                                                     decoupled)
        assert opt.step_t.tolist() == [3, 3, 3, 3, 0, 0] and opt.max_exp_avg_sq is not None
        for i, (o, k) in enumerate(opt.offsets[:4]):
            for name, buf in (("exp_avg", opt.exp_avg), ("exp_avg_sq", opt.exp_avg_sq),
                              ("max_exp_avg_sq", opt.max_exp_avg_sq)):
                assert torch.equal(buf[o:o + k], t_opt.state_dict()["state"][i][name].reshape(-1)), (i, name)
        assert torch.equal(opt.exp_avg[opt.offsets[4][0]:], torch.zeros(8))
        back = cls(copy.deepcopy(ref).parameters())
        back.load_state_dict(opt.state_dict())
        bsd, tsd = back.state_dict(), t_opt.state_dict()
        assert bsd["param_groups"] == tsd["param_groups"]
        assert set(bsd["state"]) == set(tsd["state"]) == {0, 1, 2, 3}
        for i, st in tsd["state"].items():
            assert set(bsd["state"][i]) == set(st)
            for name, t in st.items():
                assert torch.equal(bsd["state"][i][name], t), (i, name)
