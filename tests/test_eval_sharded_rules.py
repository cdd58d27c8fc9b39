"""CPU: the host rules of the env-sharded `test()`: the (step, rank, env) order of the gathered scores, and the check that every
rank takes the device path with the same env count, env kind and episode target."""
import pytest

from xuanpolicy_b200.agent import agree_eval_plan, order_eval_scores


def test_scores_come_back_in_step_rank_env_order():
    # rank 0 finished envs (2, 5) at step 3 and env 1 at step 9; rank 1 finished env 0 at step 3 and envs (4, 6) at step 4
    scores = [[0.32, 0.35, 0.91], [1.30, 1.44, 1.46]]
    steps = [[3, 3, 9], [3, 4, 4]]
    assert order_eval_scores(scores, steps) == [0.32, 0.35, 1.30, 1.44, 1.46, 0.91]


def test_order_keeps_each_ranks_env_order_within_a_step():
    """Equal scores and equal steps: the env order inside a rank is the queue order, never the value order."""
    scores = [[5.0, 1.0, 3.0], [4.0, 2.0], []]
    steps = [[7, 7, 7], [7, 7], []]
    assert order_eval_scores(scores, steps) == [5.0, 1.0, 3.0, 4.0, 2.0]


def test_order_of_one_rank_is_its_queue():
    assert order_eval_scores([[2.0, 1.0, 3.0]], [[0, 0, 1]]) == [2.0, 1.0, 3.0]
    assert order_eval_scores([[]], [[]]) == []
    out = order_eval_scores([[2.5]], [[0]])
    assert all(isinstance(s, float) for s in out)


def test_order_refuses_inconsistent_queues():
    with pytest.raises(ValueError):
        order_eval_scores([[1.0, 2.0]], [[0]])                   # a score without a step tag
    with pytest.raises(ValueError):
        order_eval_scores([[1.0], [2.0]], [[0]])                 # a rank without tags
    with pytest.raises(ValueError):
        order_eval_scores([[1.0, 2.0]], [[4, 3]])                # a queue out of step order


def test_plan_agreement():
    assert agree_eval_plan([(1, 64, 0, 100), (1, 64, 0, 100)]) is True
    assert agree_eval_plan([(0, 0, -1, 100), (0, 0, -1, 7)]) is False      # all on the host loop: each rank on its own
    assert agree_eval_plan([(1, 16, 3, 5)]) is True


@pytest.mark.parametrize("plans,what", [
    ([(1, 64, 0, 100), (0, 0, -1, 100)], "host loop"),            # one rank has compat envs
    ([(1, 64, 0, 100), (1, 32, 0, 100)], "env counts"),
    ([(1, 64, 0, 100), (1, 64, 1, 100)], "env kinds"),
    ([(1, 64, 0, 100), (1, 64, 0, 99)], "test_episode"),
    ([(1, 64, 0, 100), (1, 64, 0, 100), (1, 64, 0, 100), (0, 0, -1, 100)], "host loop"),
])
def test_plan_mismatch_raises(plans, what):
    with pytest.raises(ValueError, match=what):
        agree_eval_plan(plans)
