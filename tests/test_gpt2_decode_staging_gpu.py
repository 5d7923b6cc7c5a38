"""GPU tier: the fp32 online loop stages the K/V stream in one of two ways, chosen from the batch size alone -- register-staged
global loads when more than 24 env-warps land on an SM, bulk-async copies through a shared-memory ring (1-, 2- or 4-warp
CTAs) otherwise.  Every draw is keyed by the global env id, so a slice of the envs run on its own (env_id0 = first env)
must reproduce its columns of the full run bit for bit, whichever staging either run used."""
import pytest
import torch

pytestmark = pytest.mark.gpu

CTX = ("context_states", "context_actions", "context_next_states", "context_rewards")


@pytest.fixture(scope="module")
def model(dpt):
    from dpt_b200.models.net import Transformer
    torch.manual_seed(0)
    m = Transformer({"horizon": 500, "state_dim": 1, "action_dim": 5, "n_layer": 4, "n_embd": 32, "n_head": 1, "dropout": 0.0,
                     "test": True})
    with torch.no_grad():   # move off the init so that the softmax is far from uniform
        for k, p in m.named_parameters():
            if "wte" not in k:
                p.add_(0.15 * torch.randn_like(p))
    return m


@pytest.mark.parametrize("H", [77, 500])
@pytest.mark.parametrize("reward_type", ["uniform", "bernoulli"])
@pytest.mark.parametrize("sample", [True, False])
def test_online_loop_kv_stagings_agree(dpt, model, sample, reward_type, H):
    sms = torch.cuda.get_device_properties(0).multi_processor_count
    N, seed, var = 32 * sms, 23, 0.3
    means, _, _ = dpt.kernels.bandit_sample_means(N, 5, seed, 0)
    full = model.online_loop(means, H, var, sample, seed, 0, dump=True, reward_type=reward_type)   # register-staged
    for per_sm, lo in ((8, 5), (16, sms + 3), (24, 8 * sms - 7)):   # ring with 1-, 2- and 4-warp CTAs
        n = per_sm * sms
        part = model.online_loop(means[lo:lo + n], H, var, sample, seed, lo, dump=True, reward_type=reward_type)
        cols = slice(lo, lo + n)
        assert torch.equal(part["cum_means"], full["cum_means"][:, cols]), per_sm
        for k in CTX:
            assert torch.equal(part[k], full[k][cols]), (per_sm, k)
        for k in ("logits", "reward_z", "ctrl_u"):
            assert torch.equal(part["noise"][k], full["noise"][k][:, cols]), (per_sm, k)
