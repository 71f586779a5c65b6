"""Generates tests/golden/*.npz by RUNNING THE UNMODIFIED REFERENCE.

Run in the build container only (needs /root/reference):

    python tests/golden/make_golden.py

The reference is imported through oracle/refshim (alias patches + stand-ins for the
absent matplotlib/dm_env; SURVEY.md App. E).  Nothing here is used at test time except
the .npz files it writes; /root/reference does not exist on the GPU box.

Fixtures
  render_cases.npz   scenes (sprite factor arrays) + the frames PILRenderer produced
  episodes_<cfg>.npz per-env scene pools, action scripts and the per-step outputs of
                     Environment.step (positions, reward, step_type, success, frames)
"""
import json
import os
import sys

import numpy as np

ROOT = os.path.dirname(os.path.dirname(os.path.dirname(os.path.abspath(__file__))))
sys.path.insert(0, ROOT)
from oracle.refshim import load_reference  # noqa: E402

load_reference()
from spriteworld import action_spaces, constants, environment, tasks  # noqa: E402
from spriteworld import factor_distributions as distribs  # noqa: E402
from spriteworld import renderers as sw_renderers  # noqa: E402
from spriteworld import sprite as sprite_lib  # noqa: E402
from spriteworld import sprite_generators  # noqa: E402
from spriteworld.configs.cobra import (clustering, goal_finding_more_targets,  # noqa: E402
                                       goal_finding_new_position, sorting)
from spriteworld.configs.examples import goal_finding_clustering, goal_finding_embodied  # noqa

OUT = os.environ.get('SWB_GOLDEN_OUT') or os.path.dirname(os.path.abspath(__file__))
SHAPE_IDS = {name: int(constants.ShapeType[name]) for name in constants.SHAPES}

FIELDS = ('x', 'y', 'pos_f32', 'shape', 'angle', 'scale', 'c0', 'c1', 'c2', 'color_f32',
          'vx', 'vy', 'member', 'rgb')


def collect_filters(task):
  """Filter distributions of a task tree in first-appearance order."""
  out = []

  def add(d):
    if d is not None and all(d is not o for o in out):
      out.append(d)

  def walk(t):
    if isinstance(t, tasks.FindGoalPosition):
      add(t._filter_distrib)
    elif isinstance(t, tasks.Clustering):
      for d in t._cluster_distribs:
        add(d)
    elif isinstance(t, tasks.MetaAggregated):
      for st in t._subtasks:
        walk(st)

  walk(task)
  return out


def task_nodes(task, filters):
  """Post-order POD description of the task tree (root last)."""
  nodes = []

  def slot(d):
    if d is None:
      return -1
    return [i for i, o in enumerate(filters) if o is d][0]

  def walk(t):
    if isinstance(t, tasks.FindGoalPosition):
      nodes.append(dict(
          kind='find_goal', filter_slot=slot(t._filter_distrib),
          goal=[float(v) for v in t._goal_position],
          weights=[float(v) for v in t._weights_dimensions],
          terminate_distance=float(t._terminate_distance),
          terminate_bonus=float(t._terminate_bonus),
          raw_reward_multiplier=float(t._raw_reward_multiplier),
          sparse_reward=bool(t._sparse_reward)))
    elif isinstance(t, tasks.Clustering):
      nodes.append(dict(
          kind='clustering', cluster_slots=[slot(d) for d in t._cluster_distribs],
          termination_threshold=float(t._termination_threshold),
          terminate_bonus=float(t._terminate_bonus), sparse_reward=bool(t._sparse_reward),
          reward_range=float(t._reward_range)))
    elif isinstance(t, tasks.MetaAggregated):
      kids = []
      for st in t._subtasks:
        walk(st)
        kids.append(len(nodes) - 1)
      agg = [k for k, v in tasks.MetaAggregated.REWARD_AGGREGATOR.items()
             if v is t._reward_aggregator][0]
      crit = [k for k, v in tasks.MetaAggregated.TERMINATION_CRITERION.items()
              if v is t._termination_criterion][0]
      nodes.append(dict(kind='meta', children=kids, aggregator=agg, criterion=crit,
                        terminate_bonus=float(t._terminate_bonus)))
    elif isinstance(t, tasks.NoReward):
      nodes.append(dict(kind='no_reward'))
    else:
      raise TypeError(t)
    return len(nodes) - 1

  walk(task)
  return nodes


def action_desc(a):
  if isinstance(a, action_spaces.Embodied):
    return dict(kind='embodied', scale=float(a._step_size), motion_cost=float(a._motion_cost))
  kind = 'drag_and_drop' if isinstance(a, action_spaces.DragAndDrop) else 'select_move'
  assert not a._noise_scale
  return dict(kind=kind, scale=float(a._scale), motion_cost=float(a._motion_cost))


def sprites_to_arrays(sprites, n_slots, filters, color_to_rgb):
  """Pads at the FRONT so the last sprite (Embodied body) is always slot S-1."""
  n = len(sprites)
  assert n <= n_slots
  a = dict(
      x=np.zeros(n_slots), y=np.zeros(n_slots), pos_f32=np.zeros(n_slots, np.uint8),
      shape=np.zeros(n_slots, np.uint8), angle=np.zeros(n_slots), scale=np.zeros(n_slots),
      c0=np.zeros(n_slots), c1=np.zeros(n_slots), c2=np.zeros(n_slots),
      color_f32=np.zeros(n_slots, np.uint8), vx=np.zeros(n_slots), vy=np.zeros(n_slots),
      member=np.zeros(n_slots, np.uint32), rgb=np.zeros((n_slots, 3), np.uint8))
  for i, s in enumerate(sprites):
    k = n_slots - n + i
    a['x'][k], a['y'][k] = float(s.position[0]), float(s.position[1])
    a['pos_f32'][k] = s.position.dtype == np.float32
    a['shape'][k] = SHAPE_IDS[s.shape]
    a['angle'][k], a['scale'][k] = float(s.angle), float(s.scale)
    a['c0'][k], a['c1'][k], a['c2'][k] = [float(c) for c in s.color]
    a['color_f32'][k] = all(isinstance(c, np.float32) for c in s.color)
    a['vx'][k], a['vy'][k] = float(s.velocity[0]), float(s.velocity[1])
    m = 0
    for bit, d in enumerate(filters):
      if d.contains(s.factors):
        m |= 1 << bit
    a['member'][k] = m
    rgb = color_to_rgb(s.color) if color_to_rgb is not None else s.color
    a['rgb'][k] = [int(c) for c in rgb]
    # the centred path the reference built must equal (scale then rotate) . SHAPES[shape]
    import math
    th = math.radians(s.angle)
    ca, sa, sc = math.cos(th), math.sin(th), float(s.scale)
    v = constants.SHAPES[s.shape]
    cx = (ca * sc) * v[:, 0] + ((-sa) * sc) * v[:, 1] + 0.0
    cy = (sa * sc) * v[:, 0] + (ca * sc) * v[:, 1] + 0.0
    assert np.array_equal(np.stack([cx, cy], 1), s._centered_path.vertices), s.shape
  return a


def positions(sprites, n_slots):
  p = np.zeros((n_slots, 2))
  n = len(sprites)
  for i, s in enumerate(sprites):
    p[n_slots - n + i] = [float(s.position[0]), float(s.position[1])]
  return p


def shapes_blob():
  return {('shape_' + k): np.asarray(v, np.float64) for k, v in constants.SHAPES.items()}


# ---------------------------------------------------------------------------
# render_cases.npz
# ---------------------------------------------------------------------------

def render_cases():
  cases = []

  def add(name, sprites, renderer_kwargs, color_map):
    ctr = sw_renderers.color_maps.hsv_to_rgb if color_map == 'hsv' else None
    r = sw_renderers.PILRenderer(color_to_rgb=ctr, **renderer_kwargs)
    frame = r.render(sprites)
    arrs = sprites_to_arrays(sprites, len(sprites), [], ctr)
    size = renderer_kwargs.get('image_size', (64, 64))
    cases.append(dict(
        name=name, width=int(size[0]), height=int(size[1]),
        aa=int(renderer_kwargs.get('anti_aliasing', 1)),
        bg=[int(c) for c in (renderer_kwargs.get('bg_color') or (0, 0, 0))],
        color_map=color_map or 'none', frame=frame, **arrs))

  def fixture():  # tests/renderers/pil_renderer_test.py:31-43
    return [
        sprite_lib.Sprite(x=0.75, y=0.95, shape='spoke_6', scale=0.2, c0=20, c1=50, c2=80),
        sprite_lib.Sprite(x=0.2, y=0.3, shape='triangle', scale=0.1, c0=150, c1=255, c2=100),
        sprite_lib.Sprite(x=0.7, y=0.5, shape='square', scale=0.3, c0=0, c1=255, c2=0),
        sprite_lib.Sprite(x=0.5, y=0.5, shape='square', scale=0.3, c0=255, c1=0, c2=0),
    ]

  add('ref_test_basic_64', fixture(), dict(image_size=(64, 64)), None)
  add('ref_test_bg_64', fixture(), dict(image_size=(64, 64), bg_color=(5, 6, 7)), None)
  add('ref_test_aa5_16', fixture(), dict(image_size=(16, 16), anti_aliasing=5), None)
  add('ref_test_aa1_16', fixture(), dict(image_size=(16, 16), anti_aliasing=1), None)
  add('ref_test_hsv_64',
      [sprite_lib.Sprite(x=0.5, y=0.5, shape='square', c0=0.2, c1=0.5, c2=0.5)],
      dict(image_size=(64, 64)), 'hsv')
  add('fixture_aa5_64', fixture(), dict(image_size=(64, 64), anti_aliasing=5), None)
  add('fixture_aa5_128', fixture(), dict(image_size=(128, 128), anti_aliasing=5), None)
  add('fixture_aa3_48', fixture(), dict(image_size=(48, 48), anti_aliasing=3), None)
  add('fixture_aa5_96x64', fixture(), dict(image_size=(96, 64), anti_aliasing=5), None)
  add('fixture_aa2_bg', fixture(), dict(image_size=(32, 32), anti_aliasing=2,
                                        bg_color=(200, 10, 90)), None)

  # scenes sampled from the shipped configs (HSV float32 colours, 64x64 aa=5)
  np.random.seed(11)
  cfgs = [('more_targets', goal_finding_more_targets.get_config('test')),
          ('clustering', clustering.get_config('train')),
          ('sorting', sorting.get_config('train')),
          ('new_position', goal_finding_new_position.get_config('train')),
          ('embodied', goal_finding_embodied.get_config())]
  for name, cfg in cfgs:
    for i in range(6):
      add('%s_%d' % (name, i), cfg['init_sprites'](),
          dict(image_size=(64, 64), anti_aliasing=5), 'hsv')
  cfg = goal_finding_embodied.get_config()
  for i in range(3):
    add('embodied128_%d' % i, cfg['init_sprites'](),
        dict(image_size=(128, 128), anti_aliasing=5), 'hsv')
  # rotated stars / spokes with integer RGB colours (examples/goal_finding_clustering.py)
  cfg = goal_finding_clustering.get_config()
  for i in range(8):
    add('gfc_%d' % i, cfg['init_sprites'](), dict(image_size=(64, 64), anti_aliasing=5), None)
  # every shape at random angle/scale, sprites partly out of frame, random velocities
  rng = np.random.RandomState(5)
  for i in range(12):
    sprites = []
    for shape in rng.permutation(sorted(constants.SHAPES))[:6]:
      sprites.append(sprite_lib.Sprite(
          x=np.float32(rng.uniform(-0.05, 1.05)), y=np.float32(rng.uniform(-0.05, 1.05)),
          shape=str(shape), angle=int(rng.randint(0, 360)), scale=float(rng.uniform(0.03, 0.4)),
          c0=int(rng.randint(256)), c1=int(rng.randint(256)), c2=int(rng.randint(256))))
    add('allshapes_%d' % i, sprites, dict(image_size=(64, 64), anti_aliasing=5), None)
  for i in range(4):
    sprites = [sprite_lib.Sprite(
        x=float(rng.uniform(0, 1)), y=float(rng.uniform(0, 1)),
        shape=str(rng.choice(sorted(constants.SHAPES))), angle=float(rng.uniform(0, 360)),
        scale=float(rng.uniform(0.01, 0.6)), c0=int(rng.randint(256)), c1=int(rng.randint(256)),
        c2=int(rng.randint(256))) for _ in range(9)]
    add('float_angle_%d' % i, sprites, dict(image_size=(40, 24), anti_aliasing=4), None)

  blob = dict(names=np.array([c['name'] for c in cases]))
  for i, c in enumerate(cases):
    blob['meta_%d' % i] = np.array(json.dumps(
        {k: c[k] for k in ('name', 'width', 'height', 'aa', 'bg', 'color_map')}))
    blob['frame_%d' % i] = c['frame']
    for f in FIELDS:
      blob['%s_%d' % (f, i)] = c[f]
  blob.update(shapes_blob())
  np.savez_compressed(os.path.join(OUT, 'render_cases.npz'), **blob)
  print('render_cases.npz: %d cases' % len(cases))


# ---------------------------------------------------------------------------
# episodes_<cfg>.npz
# ---------------------------------------------------------------------------

def run_episodes(name, make_config, n_envs, n_steps, n_slots, action_dtype, frame_envs,
                 seed_base=1000, env_overrides=None):
  """Steps `n_envs` independent reference Environments in lockstep."""
  rng = np.random.RandomState(7)
  scene_log = [[] for _ in range(n_envs)]
  envs = []
  meta = None
  for e in range(n_envs):
    np.random.seed(seed_base + e)
    cfg = make_config()
    cfg.update(env_overrides or {})
    base_gen = cfg['init_sprites']
    filters = collect_filters(cfg['task'])
    rend = cfg['renderers']['image']

    def logged_gen(_base=base_gen, _log=scene_log[e], _f=filters, _r=rend):
      sprites = _base()
      _log.append(sprites_to_arrays(sprites, n_slots, _f, _r._color_to_rgb
                                    if _r._color_to_rgb.__name__ != '<lambda>' else None))
      return sprites

    cfg['init_sprites'] = logged_gen
    env = environment.Environment(**cfg)
    envs.append(env)
    if meta is None:
      meta = dict(
          name=name, n_slots=n_slots, action=action_desc(cfg['action_space']),
          keep_in_frame=bool(env._keep_in_frame),
          max_episode_length=int(env._max_episode_length),
          nodes=task_nodes(cfg['task'], filters), n_filters=len(filters),
          width=int(rend._image_size[0]), height=int(rend._image_size[1]),
          aa=int(rend._anti_aliasing), bg=[0, 0, 0], action_dtype=action_dtype,
          frame_envs=list(frame_envs))
  embodied = meta['action']['kind'] == 'embodied'
  if embodied:
    actions = np.stack([rng.randint(0, 2, (n_steps, n_envs)),
                        rng.randint(0, 4, (n_steps, n_envs))], -1).astype(np.int32)
  else:
    actions = rng.uniform(0, 1, (n_steps, n_envs, 4)).astype(action_dtype)
    # aim half of the clicks at a sprite centre so that sprites actually move
    aim = rng.uniform(size=(n_steps, n_envs)) < 0.6
  pos = np.zeros((n_steps, n_envs, n_slots, 2))
  reward = np.zeros((n_steps, n_envs))
  step_type = np.zeros((n_steps, n_envs), np.int8)
  success = np.zeros((n_steps, n_envs), np.uint8)
  scene_idx = np.zeros((n_steps, n_envs), np.int32)
  frames = np.zeros((n_steps, len(frame_envs), meta['height'], meta['width'], 3), np.uint8)
  for t in range(n_steps):
    for e, env in enumerate(envs):
      if not embodied and aim[t, e] and env._sprites:
        s = env._sprites[rng.randint(len(env._sprites))]
        jitter = rng.uniform(-0.03, 0.03, 2)
        actions[t, e, :2] = np.clip(s.position + jitter, 0, 1).astype(action_dtype)
      a = actions[t, e]
      ts = env.step(a if not embodied else [int(a[0]), int(a[1])])
      pos[t, e] = positions(env._sprites, n_slots)
      reward[t, e] = 0.0 if ts.reward is None else float(ts.reward)
      step_type[t, e] = int(ts.step_type)
      success[t, e] = bool(env.success())
      scene_idx[t, e] = len(scene_log[e]) - 1
      if e in frame_envs:
        frames[t, list(frame_envs).index(e)] = ts.observation['image']
  n_scenes = max(len(l) for l in scene_log)
  blob = dict(meta=np.array(json.dumps(meta)), actions=actions, pos=pos, reward=reward,
              step_type=step_type, success=success, scene_idx=scene_idx, frames=frames,
              n_scenes=np.array([len(l) for l in scene_log], np.int32))
  for f in FIELDS:
    proto = scene_log[0][0][f]
    arr = np.zeros((n_envs, n_scenes) + proto.shape, proto.dtype)
    for e in range(n_envs):
      for k, sc in enumerate(scene_log[e]):
        arr[e, k] = sc[f]
    blob['scene_' + f] = arr
  blob.update(shapes_blob())
  path = os.path.join(OUT, 'episodes_%s.npz' % name)
  np.savez_compressed(path, **blob)
  print('%s: %d envs x %d steps, %d scenes max, LAST=%d, success=%d, %.0f KB' % (
      os.path.basename(path), n_envs, n_steps, n_scenes, (step_type == 2).sum(),
      success.sum(), os.path.getsize(path) / 1024))


def bench_like_goal_finding():
  """C2-shaped scene: 2 targets + 3 distractors (SURVEY.md 8d)."""
  cfg = goal_finding_more_targets.get_config('test')
  shared = distribs.Product([
      distribs.Continuous('x', 0.1, 0.9), distribs.Continuous('y', 0.1, 0.9),
      distribs.Discrete('shape', ['square', 'triangle', 'circle']),
      distribs.Discrete('scale', [0.13]), distribs.Continuous('c1', 0.3, 1.),
      distribs.Continuous('c2', 0.9, 1.)])
  target_hue = cfg['task']._filter_distrib
  gen = sprite_generators.shuffle(sprite_generators.chain_generators(
      sprite_generators.generate_sprites(distribs.Product([target_hue, shared]), 2),
      sprite_generators.generate_sprites(
          distribs.Product([distribs.Continuous('c0', 0.5, 0.9), shared]), 3)))
  cfg['init_sprites'] = gen
  return cfg


def moving_sprites_config():
  """Sprites with velocities, keep_in_frame=False, motion cost, bonus, DragAndDrop."""
  factors = distribs.Product([
      distribs.Continuous('x', 0.2, 0.8), distribs.Continuous('y', 0.2, 0.8),
      distribs.Discrete('shape', ['pentagon', 'star_5', 'spoke_4', 'hexagon']),
      distribs.Continuous('scale', 0.08, 0.2), distribs.Discrete('angle', [0, 30, 77]),
      distribs.Continuous('c0', 0., 1.), distribs.Continuous('c1', 0.3, 1.),
      distribs.Continuous('c2', 0.9, 1.),
      distribs.Continuous('x_vel', -0.07, 0.07), distribs.Discrete('y_vel', [0.0, 0.01, -0.05]),
  ])
  task = tasks.MetaAggregated([
      tasks.FindGoalPosition(filter_distrib=distribs.Continuous('c0', 0., 0.5),
                             goal_position=(0.3, 0.6), terminate_distance=0.2,
                             terminate_bonus=3.0, weights_dimensions=(1, 0.5)),
      tasks.FindGoalPosition(filter_distrib=distribs.Continuous('c0', 0.5, 1.),
                             goal_position=(0.7, 0.4), terminate_distance=0.3,
                             sparse_reward=True, raw_reward_multiplier=10),
      tasks.FindGoalPosition(filter_distrib=distribs.Continuous('c0', 2., 3.)),  # empty: NaN
  ], reward_aggregator='mean', termination_criterion='all', terminate_bonus=1.5)
  return dict(
      task=task, action_space=action_spaces.DragAndDrop(scale=0.5, motion_cost=0.7),
      renderers={'image': sw_renderers.PILRenderer(
          image_size=(64, 64), anti_aliasing=5,
          color_to_rgb=sw_renderers.color_maps.hsv_to_rgb)},
      init_sprites=sprite_generators.generate_sprites(factors, num_sprites=4),
      keep_in_frame=False, max_episode_length=12)


CONFIG_MODES = [
    ('cobra', 'goal_finding_more_targets', ('train', 'test')),
    ('cobra', 'goal_finding_more_distractors', ('train', 'test')),
    ('cobra', 'goal_finding_new_position', ('train', 'test')),
    ('cobra', 'goal_finding_new_shape', ('train', 'test')),
    ('cobra', 'clustering', ('train', 'test')),
    ('cobra', 'sorting', ('train', 'test')),
    ('cobra', 'exploration', (None,)),
    ('examples', 'goal_finding_embodied', (None,)),
    ('examples', 'goal_finding_clustering', ('train', 'test')),
]
TYPE_CODES = {float: 0, np.float64: 1, np.float32: 2, int: 3, np.int32: 4, np.uint8: 5,
              np.int64: 6, str: 7}


def sampling_cases(seed=5, n_scenes=12):
  """What init_sprites() of every shipped config draws from np.random.seed(seed): pins the
  RNG call order of factor_distributions / sprite_generators."""
  import contextlib
  import importlib
  import io
  blob = {}
  for pkg, name, modes in CONFIG_MODES:
    mod = importlib.import_module('spriteworld.configs.%s.%s' % (pkg, name))
    for mode in modes:
      with contextlib.redirect_stdout(io.StringIO()):
        cfg = mod.get_config(mode) if mode else mod.get_config()
      np.random.seed(seed)
      counts, values, types, shapes = [], [], [], []
      for _ in range(n_scenes):
        sprites = cfg['init_sprites']()
        counts.append(len(sprites))
        for s in sprites:
          f = s.factors
          shapes.append(SHAPE_IDS[f['shape']])
          values.append([float(v) for k, v in f.items() if k != 'shape'])
          types.append([TYPE_CODES[type(v)] for k, v in f.items() if k != 'shape'])
      key = '%s.%s.%s' % (pkg, name, mode)
      blob[key + '.count'] = np.array(counts, np.int32)
      blob[key + '.values'] = np.array(values, np.float64).reshape(-1, 9)
      blob[key + '.types'] = np.array(types, np.uint8).reshape(-1, 9)
      blob[key + '.shapes'] = np.array(shapes, np.uint8)
      blob[key + '.max_episode_length'] = np.array(cfg['max_episode_length'])
      blob[key + '.task'] = np.array(json.dumps(
          task_nodes(cfg['task'], collect_filters(cfg['task']))))
      blob[key + '.action'] = np.array(json.dumps(action_desc(cfg['action_space'])))
  blob['seed'] = np.array(seed)
  np.savez_compressed(os.path.join(OUT, 'sampling.npz'), **blob)
  print('sampling.npz: %d config/mode pairs' % (len(blob) // 7))


def reference_probes():
  """reference_probes.npz: the records of tests/reference_probes.py against the reference, keyed
  '<probe>:<record>', and its public surface under 'surface'."""
  import importlib
  import types
  from spriteworld_b200 import gym_wrapper as own_gym_wrapper
  # by path: the reference's own `tests` package is ahead of ours on sys.path
  spec = importlib.util.spec_from_file_location(
      'reference_probes', os.path.join(ROOT, 'tests', 'reference_probes.py'))
  probes = importlib.util.module_from_spec(spec)
  spec.loader.exec_module(probes)
  if importlib.util.find_spec('gym') is None and importlib.util.find_spec('gymnasium') is None:
    # the reference's gym_wrapper only builds spaces from specs; gym is absent here
    gym, spaces = types.ModuleType('gym'), types.ModuleType('gym.spaces')
    for name in ('Box', 'Discrete', 'Dict', 'Tuple'):
      setattr(spaces, name, getattr(own_gym_wrapper._MiniSpaces, name))
    gym.spaces = spaces
    sys.modules.update({'gym': gym, 'gym.spaces': spaces})
  sw = lambda name: importlib.import_module('spriteworld.' + name)
  blob = dict(surface=np.array(json.dumps(probes.public_surface(sw))))
  for name in sorted(probes.HOST) + sorted(probes.ENGINE):
    for key, v in probes.run(name, sw).items():
      blob['%s:%s' % (name, key)] = np.asarray(v)
  np.savez_compressed(os.path.join(OUT, 'reference_probes.npz'), **blob)
  print('reference_probes.npz: %d records' % len(blob))


def main():
  sampling_cases()
  render_cases()
  run_episodes('goal_finding', bench_like_goal_finding, n_envs=12, n_steps=60, n_slots=5,
               action_dtype='float32', frame_envs=(0, 1, 2))
  run_episodes('more_targets_f64', lambda: goal_finding_more_targets.get_config('test'),
               n_envs=8, n_steps=45, n_slots=4, action_dtype='float64', frame_envs=(0,))
  run_episodes('clustering', lambda: clustering.get_config('train'), n_envs=10, n_steps=70,
               n_slots=4, action_dtype='float32', frame_envs=(0, 1))
  run_episodes('sorting', lambda: sorting.get_config('train'), n_envs=10, n_steps=70,
               n_slots=2, action_dtype='float32', frame_envs=(0, 1))
  run_episodes('embodied', goal_finding_embodied.get_config, n_envs=10, n_steps=80,
               n_slots=7, action_dtype='int32', frame_envs=(0, 1))
  run_episodes('moving', moving_sprites_config, n_envs=8, n_steps=40, n_slots=4,
               action_dtype='float32', frame_envs=(0,))
  reference_probes()


if __name__ == '__main__':
  main()
