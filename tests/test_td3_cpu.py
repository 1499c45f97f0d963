"""CPU: TD3 host mirror vs goldens produced by the reference's own td3.py + shipped checkpoint (scripts/make_td3_golden.py)."""
import os

import numpy as np
import torch

GOLD = os.path.join(os.path.dirname(__file__), "golden", "td3_golden.npz")


def load_actor():
    from plen_ml_walk_b200.td3 import Actor
    g = np.load(GOLD)
    a = Actor()
    a.load_state_dict({k: torch.from_numpy(g["actor_" + k.replace(".", "_")]) for k in a.state_dict().keys()})
    return a, g


def test_actor_mirror_reproduces_reference_checkpoint_outputs():
    a, g = load_actor()
    with torch.no_grad():
        out = a(torch.from_numpy(g["obs"])).numpy()
    # fp32 GEMM summation order differs between host CPUs (oneDNN/MKL kernel choice): 2e-5 absolute on tanh outputs
    assert np.abs(out - g["actor_out"]).max() < 2e-5
    # SURVEY.md section 4 known answers (fp32 CPU, torch 2.11)
    assert np.allclose(out[0, :4], [-0.2388544, -0.9999999, 0.9836175, -0.2882677], atol=2e-5)
    assert np.allclose(out[1, :4], [0.1014272, -1.0, 0.9964353, -0.9608743], atol=2e-5)
    assert abs(float(g["q1"][1, 0]) + 30.3603668) < 1e-4 and abs(float(g["q2"][1, 0]) + 32.2503319) < 1e-4
    assert sum(p.numel() for p in a.parameters()) == 77330                    # SURVEY.md Appendix D


def test_replay_oracle_matches_reference_ring_order():
    from oracle.replay_oracle import ReplayRing
    g = np.load(GOLD)
    rb = ReplayRing(3)
    for k in range(5):
        rb.add((k, k, k + 0.5, float(k), 0.0))
    assert [t[3] for t in rb.storage] == list(g["ring_rewards"]) == [3.0, 4.0, 2.0] and rb.ptr == int(g["ring_ptr"]) == 2


def test_state_dict_keys_match_reference_checkpoints():
    from plen_ml_walk_b200.td3 import Actor, Critic
    assert list(Actor().state_dict().keys()) == ["fc%d.%s" % (i, p) for i in (1, 2, 3) for p in ("weight", "bias")]
    assert list(Critic().state_dict().keys()) == ["fc%d.%s" % (i, p) for i in range(1, 7) for p in ("weight", "bias")]
    assert sum(p.numel() for p in Critic().parameters()) == 155138


def test_agent_host_logic_without_a_gpu(tmp_path):
    """Host side of TD3Agent that needs no device: argument checking, the reference's four-file checkpoint round trip and its
    load() semantics (td3.py:366-376 leaves the TARGET networks untouched), and the loud failure of train() off the GPU."""
    import pytest
    from plen_ml_walk_b200.td3 import TD3Agent
    with pytest.raises(ValueError):
        TD3Agent(device="cpu", precision="bf16")
    torch.manual_seed(1)
    a = TD3Agent(device="cpu")
    a.save(str(tmp_path / "ck"))
    torch.manual_seed(2)
    b = TD3Agent(device="cpu")
    tgt0 = b._flat["actor_target"].clone()
    b.load(str(tmp_path / "ck"))
    assert torch.equal(b._flat["actor"], a._flat["actor"]) and torch.equal(b._flat["critic"], a._flat["critic"])
    assert torch.equal(b._flat["actor_target"], tgt0)                       # as the reference: targets keep their old values
    b.load(str(tmp_path / "ck"), sync_targets=True)
    assert torch.equal(b._flat["actor_target"], a._flat["actor"]) and torch.equal(b._flat["critic_target"], a._flat["critic"])
    with pytest.raises(RuntimeError):
        a.train(None, batch=(torch.zeros(4, 26), torch.zeros(4, 18), torch.zeros(4, 26), torch.zeros(4, 1), torch.ones(4, 1)))


def test_td3_gemm_harness_compiles_and_loads():
    """tests/cuda/td3_gemm_harness.cu includes the learner's sources: it must keep compiling for sm_100a and load without
    undefined symbols, or the GPU tests of the learner's GEMM kernels would break unnoticed when those sources change."""
    import ctypes
    import pytest
    import td3_gemm_util
    if not os.path.exists(td3_gemm_util.nvcc()):
        pytest.skip("nvcc not available")
    lib = ctypes.CDLL(td3_gemm_util.build_harness())
    assert lib.harness_gemm and lib.harness_tc_timed_out
