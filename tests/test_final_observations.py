"""Final observations of the autoreset (``keep_final_observations=True``) without a GPU: which rows each domain keeps,
that the observation views and both host downloads read those rows only, the constructor's checks, and the argument
errors of ``frz_autoreset`` with ``keep`` arrays set."""
import ast
import ctypes
import inspect
import os
import textwrap

import pytest
import torch

from free_range_zoo_b200 import _lib, presets
from free_range_zoo_b200.envs.cybersecurity.env import cybersecurity
from free_range_zoo_b200.envs.rideshare.env import rideshare
from free_range_zoo_b200.envs.wildfire.env import wildfire
from free_range_zoo_b200.utils.env import BatchedAECEnv

DOMAINS = {'wildfire': (wildfire.raw_env, presets.wildfire_large), 'rideshare': (rideshare.raw_env, presets.rideshare_c2),
           'cybersecurity': (cybersecurity.raw_env, presets.cyber_c3)}
FINAL = {
    'wildfire': {'self_obs', 'task_obs', 'action_mask', 'env_task_count', 'agent_task_count'},
    'rideshare': {'self_obs', 'task_obs', 'task_mask', 'env_task_count', 'agent_task_count'},
    'cybersecurity': {'attacker_self', 'defender_self', 'task_obs', 'monitored', 'env_task_count', 'agent_task_count'},
}
# the hooks that build observations from a name -> tensor mapping (live or final)
BUILDERS = ('_observation_views', '_observation_download', '_compact_schema', '_tasks_for')
# live observation arrays and the properties over them: a builder that read one would ignore the mapping it was given
LIVE = {'_self_obs', '_task_obs', '_action_mask', '_task_mask', '_attacker_self', '_defender_self', '_monitored',
        'environment_task_count', '_agent_task_count', 'action_mask', 'task_mask', 'task_store'}


@pytest.fixture(scope='module')
def lib():
    if not os.path.exists(_lib.LIBRARY_PATH):
        import __graft_entry__
        __graft_entry__.build()
    return _lib.library()


def builder_reads(env_class):
    """(names read from the mapping, live attributes read) by the domain's observation builders."""
    names, live = set(), set()
    for method in BUILDERS:
        if method not in vars(env_class):
            continue
        tree = ast.parse(textwrap.dedent(inspect.getsource(vars(env_class)[method])))
        function = tree.body[0]
        mapping = {'buffers', 'b'}
        for node in ast.walk(function):
            if (isinstance(node, ast.Subscript) and isinstance(node.value, ast.Name) and node.value.id in mapping
                    and isinstance(node.slice, ast.Constant)):
                names.add(node.slice.value)
            if isinstance(node, ast.Attribute) and isinstance(node.value, ast.Name) and node.value.id == 'self' \
                    and node.attr in LIVE:
                live.add(f'{method}: self.{node.attr}')
    return names, live


@pytest.mark.parametrize('domain', sorted(DOMAINS))
def test_final_rows_are_observation_rows_a_restart_restores(domain):
    rows = DOMAINS[domain][0]._autoreset_rows()
    assert len(rows.final) == len(set(rows.final))
    assert set(rows.final) == FINAL[domain]
    restored = set(rows.init) | set(rows.snapshot) | set(rows.zero)
    assert set(rows.final) <= restored, set(rows.final) - restored
    assert 'passengers' not in rows.final  # rideshare's passenger table is state, not observation


@pytest.mark.parametrize('domain', sorted(DOMAINS))
def test_the_observation_builders_read_the_final_rows_only(domain):
    """The views and both download hooks take every array from the mapping they are given, and the final rows cover
    all of them; the download counts are the mapping's ``env_task_count`` (``BatchedAECEnv._download_counts``)."""
    env_class = DOMAINS[domain][0]
    names, live = builder_reads(env_class)
    assert not live, f'builders read live buffers: {sorted(live)}'
    assert names | {'env_task_count'} == set(env_class._autoreset_rows().final)
    assert "_final_buffers['env_task_count']" in inspect.getsource(BatchedAECEnv._download_counts)


@pytest.mark.parametrize('domain', sorted(DOMAINS))
def test_keep_final_observations_needs_autoreset(domain):
    """Refused before any device work, so also where there is no GPU."""
    env_class, config = DOMAINS[domain]
    with pytest.raises(ValueError, match='autoreset=True'):
        env_class(configuration=config(), parallel_envs=2, max_steps=5, device=torch.device('cuda', 0),
                  keep_final_observations=True)


@pytest.mark.parametrize('domain', sorted(DOMAINS))
def test_final_observations_need_the_keyword(domain):
    env = DOMAINS[domain][0].__new__(DOMAINS[domain][0])
    env.keep_final_observations = False
    with pytest.raises(RuntimeError, match='keep_final_observations=True'):
        env.final_observations
    with pytest.raises(RuntimeError, match='keep_final_observations=True'):
        env._download_buffers(final=True)


def test_the_row_mirror_ends_with_keep():
    assert [name for name, _ in _lib.AutoresetRow._fields_] == ['dst', 'src', 'bytes', 'keep']
    assert ctypes.sizeof(_lib.AutoresetRow) == 32


def test_null_and_shape_errors_are_reported_with_keep_arrays(lib):
    dummy = ctypes.create_string_buffer(256)
    address = ctypes.addressof(dummy)
    block = _lib.Autoreset()
    for name in ('terminated', 'truncated', 'step_terminated', 'step_truncated', 'done', 'cumulative_rewards',
                 'episode_return', 'num_moves', 'episode_length', 'control', 'finished', 'finished_count', 'scratch'):
        setattr(block, name, address)
    block.num_agents = 2
    rows = (_lib.AutoresetRow * 2)()
    for row in rows:
        row.keep, row.bytes = address, 8
    block.rows, block.row_count = rows, 2
    assert lib.frz_autoreset(ctypes.byref(block), 4, None) == 1  # FRZ_ERR_NULL: a kept row without a destination
    assert b'NULL destination' in lib.frz_last_error()
    for row in rows:
        row.dst = address
    rows[1].bytes = 0
    assert lib.frz_autoreset(ctypes.byref(block), 4, None) == 2  # FRZ_ERR_SHAPE
    assert b'bytes per environment' in lib.frz_last_error()
    rows[1].bytes = 4
    for change in (dict(parallel_envs=0), dict(num_agents=0), dict(row_count=_lib.AUTORESET_MAX_ROWS + 1)):
        B = change.pop('parallel_envs', 4)
        saved = {name: getattr(block, name) for name in change}
        for name, value in change.items():
            setattr(block, name, value)
        assert lib.frz_autoreset(ctypes.byref(block), B, None) == 2, change
        assert b'unsupported' in lib.frz_last_error()
        for name, value in saved.items():
            setattr(block, name, value)
