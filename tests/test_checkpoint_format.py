"""CPU: the checkpoint format's rules (xuanpolicy_b200/checkpoint.py) — which runs may resume from a checkpoint, and that a
save cut off part-way keeps the previous file."""
import os
from argparse import Namespace

import pytest
import torch

from xuanpolicy_b200 import checkpoint
from xuanpolicy_b200.configs import ppo_config


def _meta(**changes):
    cfg = checkpoint.plain_config(ppo_config("CartPole-v1", parallels=64, n_steps=32))
    meta = {"format_version": checkpoint.FORMAT_VERSION, "agent_class": "PPOCLIP_Agent", "env_id": "CartPole-v1",
            "n_envs": 64, "n_steps": 32, "obs_row": 4, "world_size": 1, "rank": 0,
            "params": [("representation.model.0.weight", [128, 4]), ("representation.model.0.bias", [128])], "config": cfg}
    for k, v in changes.items():
        if k.startswith("config."):
            meta["config"] = dict(meta["config"], **{k[len("config."):]: v})
        else:
            meta[k] = v
    return meta


@pytest.mark.parametrize("field,value", [("format_version", 0), ("agent_class", "A2C_Agent"), ("env_id", "Acrobot-v1"),
                                         ("n_envs", 128), ("n_steps", 16), ("obs_row", 8), ("world_size", 2), ("rank", 1)])
def test_identity_fields_are_refused_by_name(field, value):
    with pytest.raises(ValueError, match=field):
        checkpoint.check_compatible(_meta(**{field: value}), _meta())


def test_world_size_refusal_says_resharding_is_unsupported():
    with pytest.raises(ValueError, match="re-sharding"):
        checkpoint.check_compatible(_meta(world_size=2, rank=1), _meta())


def test_parameter_names_and_shapes_are_refused():
    with pytest.raises(ValueError, match="parameter names"):
        checkpoint.check_compatible(_meta(params=[("a", [128, 4]), ("representation.model.0.bias", [128])]), _meta())
    with pytest.raises(ValueError, match="'representation.model.0.weight' has shape"):
        checkpoint.check_compatible(_meta(params=[("representation.model.0.weight", [256, 4]),
                                                  ("representation.model.0.bias", [128])]), _meta())


def test_seed_is_refused_with_its_own_reason():
    with pytest.raises(ValueError, match="seed.*sampling"):
        checkpoint.check_compatible(_meta(**{"config.seed": 2}), _meta())


@pytest.mark.parametrize("key,value", [("learning_rate", 1e-3), ("gamma", 0.99), ("use_obsnorm", True), ("shuffle", "device"),
                                       ("representation_hidden_size", [256])])
def test_config_keys_are_refused_by_name(key, value):
    with pytest.raises(ValueError, match="config key '%s'" % key):
        checkpoint.check_compatible(_meta(**{"config." + key: value}), _meta())


def test_a_config_key_present_on_one_side_only_is_refused():
    cur = _meta(**{"config.value_clip": 0.2})
    with pytest.raises(ValueError, match="config key 'value_clip'.*<absent>"):
        checkpoint.check_compatible(_meta(), cur)


def test_place_and_logging_keys_may_differ():
    changed = {"config.model_dir": "/elsewhere/models", "config.log_dir": "/elsewhere/logs", "config.device": "cuda:3",
               "config.feeder_threads": 2, "config.sync_info": False}
    checkpoint.check_compatible(_meta(**changed), _meta())
    assert set(checkpoint.PLACE_KEYS) == {k[len("config."):] for k in changed}


def test_plain_config_keeps_what_a_weights_only_load_reads():
    cfg = checkpoint.plain_config(Namespace(a=1, b=[128, (2, 3)], c=None, d=torch.float32, e="x"))
    assert cfg == {"a": 1, "b": [128, [2, 3]], "c": None, "d": "torch.float32", "e": "x"}


def _payload(value):
    return {"meta": _meta(), "tensors": {"ctr": torch.tensor([value])}, "host": {"t": 0, "last_info": {}}}


def test_interrupted_save_keeps_the_previous_checkpoint(tmp_path, monkeypatch):
    f = checkpoint.rank_file(str(tmp_path), 0, 1)
    checkpoint.write_atomic(_payload(7), f)
    real_save = torch.save

    def failing_save(obj, fh, *a, **kw):
        real_save(obj, fh, *a, **kw)          # a partial file: the bytes are written, then the process is "cut off"
        fh.truncate(fh.tell() // 2)
        raise KeyboardInterrupt

    monkeypatch.setattr(torch, "save", failing_save)
    with pytest.raises(KeyboardInterrupt):
        checkpoint.write_atomic(_payload(8), f)
    monkeypatch.setattr(torch, "save", real_save)
    assert sorted(os.listdir(tmp_path)) == [os.path.basename(f)]          # no partial file under any name
    back = checkpoint.read(str(tmp_path), 0, 1)
    assert int(back["tensors"]["ctr"][0]) == 7 and back["meta"] == _meta()


def test_a_directory_of_another_world_size_is_refused_by_name(tmp_path):
    for r in range(2):
        checkpoint.write_atomic(_payload(r), checkpoint.rank_file(str(tmp_path), r, 2))
    with pytest.raises(ValueError, match="world_size.*rank0-of-2.pt"):
        checkpoint.read(str(tmp_path), 0, 1)
    with pytest.raises(FileNotFoundError):
        checkpoint.read(str(tmp_path / "missing"), 0, 1)


def test_tensor_names_shapes_and_dtypes_are_checked():
    live = {"ctr": torch.zeros(1, dtype=torch.int64), "x0": torch.zeros(4, 4)}
    checkpoint.check_tensors({"ctr": torch.ones(1, dtype=torch.int64), "x0": torch.ones(4, 4)}, live)
    with pytest.raises(ValueError, match="'x0' is missing"):
        checkpoint.check_tensors({"ctr": torch.ones(1, dtype=torch.int64)}, live)
    with pytest.raises(ValueError, match="'x0' is \\(8, 4\\)"):
        checkpoint.check_tensors({"ctr": torch.ones(1, dtype=torch.int64), "x0": torch.ones(8, 4)}, live)
    with pytest.raises(ValueError, match="'ctr' is \\(1,\\) torch.int32"):
        checkpoint.check_tensors({"ctr": torch.ones(1, dtype=torch.int32), "x0": torch.ones(4, 4)}, live)
    with pytest.raises(ValueError, match="'extra' is not held"):
        checkpoint.check_tensors({"ctr": torch.ones(1, dtype=torch.int64), "x0": torch.ones(4, 4), "extra": torch.ones(1)}, live)


def test_replicated_part_includes_optimizer_state_but_not_local_state():
    payload = {"tensors": {"learner.flat_param": torch.ones(4), "learner.scalars": torch.ones(8), "env.state": torch.ones(2),
                           "obs_rms0": torch.ones(9), "buffer.obs": torch.ones(1, 2, 4)},
               "host": {"learner": {"optimizer": {"state": {0: {"step": torch.tensor(3.0), "exp_avg": torch.ones(2)}},
                                                  "param_groups": []}}}}
    names = [n for n, _ in checkpoint.replicated(payload)]
    assert names == ["learner.flat_param", "obs_rms0", "optimizer.state.0.exp_avg", "optimizer.state.0.step"]
