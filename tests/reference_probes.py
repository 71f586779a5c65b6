"""Seeded probes of the public API that spriteworld_b200 shares with the original Spriteworld
package (test infrastructure).

Every probe takes `sw`, a function from a module name ('sprite', 'renderers.handcrafted', ...) to
that module of one of the two packages, and records what the calls return.  Run against the
original package, the records are stored in tests/golden/reference_probes.npz
(tests/golden/make_golden.py); tests/test_reference_suite.py runs the same probes
against this package and compares record for record.  The probes of tasks, action spaces, the PIL
renderer, environments and the gym wrapper need the engine; on the CPU they run on the
oracle-backed double (tests/oracle_engine.py).
"""
import json

import numpy as np


def encode(v):
  """A JSON-able canonical form of a returned value: exact float values, array dtypes and shapes;
  a NumPy scalar counts as the Python number or bool it holds, an object array as a list."""
  if isinstance(v, np.ndarray) and v.dtype == object:
    return [encode(x) for x in v]
  if isinstance(v, np.ndarray):
    return {'ndarray': v.dtype.str, 'shape': list(v.shape), 'v': [encode(x) for x in v.reshape(-1).tolist()]}
  if isinstance(v, np.generic):
    return encode(v.item())
  if isinstance(v, (bool, int, float, str)) or v is None:
    return v
  if isinstance(v, dict):
    return {'dict': sorted([str(k), encode(x)] for k, x in v.items())}
  if isinstance(v, (list, tuple)):
    return [encode(x) for x in v]
  if hasattr(v, 'factors') and hasattr(v, 'position'):   # a Sprite
    return {'sprite': encode(v.factors), 'position': encode(v.position)}
  return {'type': type(v).__name__}


def attempt(fn, *args, **kwargs):
  """fn(*args, **kwargs), or the name of the exception it raised."""
  try:
    return fn(*args, **kwargs)
  except Exception as ex:  # the exception type is part of the behaviour under test
    return {'raised': type(ex).__name__}


class Record(dict):
  """key -> JSON string; integer images are kept as arrays."""

  def __setitem__(self, key, value):
    if isinstance(value, np.ndarray) and value.size > 256:
      super().__setitem__(key, value)
    else:
      super().__setitem__(key, json.dumps(encode(value), sort_keys=True))


def _sprites(sw, seed, n, shapes=('square', 'triangle', 'circle', 'star_5', 'spoke_4'), rgb=False):
  """n seeded sprites; colours in HSV [0, 1], or integer RGB with `rgb`.  Factor values are
  float32 numbers, as the factor distributions draw them."""
  sprite = sw('sprite')
  rng = np.random.RandomState(seed)
  u = lambda lo, hi: float(np.float32(rng.uniform(lo, hi)))
  out = []
  for _ in range(n):
    kw = dict(x=u(0.05, 0.95), y=u(0.05, 0.95), shape=str(shapes[rng.randint(len(shapes))]),
              angle=int(rng.randint(0, 360)), scale=u(0.05, 0.3), c0=u(0, 1), c1=u(0.3, 1),
              c2=u(0.5, 1), x_vel=u(-0.05, 0.05), y_vel=u(-0.05, 0.05))
    if rgb:
      kw.update(c0=int(255 * kw['c0']), c1=int(255 * kw['c1']), c2=int(255 * kw['c2']))
    out.append(sprite.Sprite(**kw))
  return out


def _spec(spec):
  """[shape, dtype] of an array spec, or of each spec of a list / dict of them."""
  if isinstance(spec, dict):
    return {k: _spec(v) for k, v in spec.items()}
  if isinstance(spec, (list, tuple)):
    return [_spec(v) for v in spec]
  return [spec.shape, str(np.dtype(spec.dtype))]


# ---------------------------------------------------------------------------------------------
# host modules
# ---------------------------------------------------------------------------------------------

def factor_distributions(sw, R):
  fd = sw('factor_distributions')
  c, d = fd.Continuous('x', 0.2, 0.8), fd.Discrete('shape', ['square', 'triangle', 'circle'])
  c64 = fd.Continuous('y', -1, 1, dtype='float64')
  dp = fd.Discrete('c0', [0, 0.5, 1], probs=[0.2, 0.3, 0.5])
  dists = dict(
      continuous=c, continuous64=c64, discrete=d, discrete_probs=dp,
      mixture=fd.Mixture([fd.Continuous('x', 0, 0.3), fd.Continuous('x', 0.7, 1)], probs=[0.25, 0.75]),
      product=fd.Product([c, c64, d, dp]),
      intersection=fd.Intersection([fd.Continuous('x', 0, 0.6), fd.Continuous('x', 0.4, 1)],
                                   index_for_sampling=1),
      setminus=fd.SetMinus(fd.Product([c, d]), fd.Discrete('shape', ['square'])),
      selection=fd.Selection(fd.Product([fd.Continuous('x', 0, 1), d]), fd.Continuous('x', 0.5, 0.6)),
      nested=fd.Mixture([fd.Product([c, d]), fd.Product([fd.Continuous('x', 0.9, 1),
                                                          fd.Discrete('shape', ['star_5'])])]))
  specs = [dict(x=0.1, shape='square'), dict(x=0.5, shape='circle'),
           dict(x=0.65, y=0.0, shape='triangle', c0=0.5), dict(x=0.95, y=2.0, shape='star_5', c0=1),
           dict(x=0.2, y=-1, shape='circle', c0=0)]
  for name, dist in sorted(dists.items()):
    rng = np.random.RandomState(3)
    R[name + '.samples'] = [dist.sample(rng) for _ in range(25)]
    np.random.seed(4)
    R[name + '.samples_global'] = [dist.sample() for _ in range(5)]
    R[name + '.keys'] = sorted(dist.keys)
    R[name + '.contains'] = [attempt(dist.contains, s) for s in specs]
    R[name + '.str'] = str(dist)
  R['errors'] = [
      attempt(fd.Discrete, 'x', [1, 2], probs=[1.0]),
      attempt(fd.Mixture, [fd.Continuous('x', 0, 1), fd.Continuous('y', 0, 1)]),
      attempt(fd.Product, [fd.Continuous('x', 0, 1), fd.Continuous('x', 0, 1)]),
      attempt(fd.Intersection, [fd.Continuous('x', 0, 1), fd.Continuous('y', 0, 1)]),
      attempt(lambda: fd.SetMinus(c, fd.Continuous('x', 0, 1)).sample(np.random.RandomState(0)))]


def sprite_generators(sw, R):
  fd, sg = sw('factor_distributions'), sw('sprite_generators')
  a = fd.Product([fd.Continuous('x', 0, 0.5), fd.Continuous('y', 0, 1),
                  fd.Discrete('shape', ['square', 'triangle']), fd.Continuous('c0', 0, 1)])
  b = fd.Product([fd.Continuous('x', 0.5, 1), fd.Discrete('shape', ['circle']),
                  fd.Discrete('scale', [0.2])])
  gens = dict(
      single=sg.generate_sprites(a, num_sprites=3),
      chain=sg.chain_generators(sg.generate_sprites(a, 2), sg.generate_sprites(b, 1)),
      sample=sg.sample_generator([sg.generate_sprites(a, 1), sg.generate_sprites(b, 2)], p=[0.3, 0.7]),
      sample_uniform=sg.sample_generator([sg.generate_sprites(a, 1), sg.generate_sprites(b, 2)]),
      shuffle=sg.shuffle(sg.chain_generators(sg.generate_sprites(a, 2), sg.generate_sprites(b, 2))),
      callable_count=sg.generate_sprites(a, num_sprites=lambda: np.random.randint(1, 4)))
  for name, gen in sorted(gens.items()):
    np.random.seed(6)
    R[name] = [gen() for _ in range(4)]


def shapes(sw, R):
  sh = sw('shapes')
  for n in (3, 4, 5, 8, 30):
    for theta in (0.0, 0.3, np.pi / 4):
      R['polygon.%d.%g' % (n, theta)] = sh.polygon(n, theta_0=theta)
  for n in (3, 4, 6):
    for h in (0.3, 1, 2.5):
      R['star.%d.%g' % (n, h)] = sh.star(n, point_height=h, theta_0=0.2)
      R['spokes.%d.%g' % (n, h)] = sh.spokes(n, spoke_height=h, theta_0=0.2)


def sprite(sw, R):
  sprites = _sprites(sw, 1, 8, shapes=sorted(sw('constants').SHAPES))
  points = np.random.RandomState(2).uniform(0, 1, (200, 2))
  for i, s in enumerate(sprites):
    k = 's%d.' % i
    R[k + 'factors'] = s.factors
    R[k + 'props'] = [s.x, s.y, s.shape, s.angle, s.scale, s.c0, s.c1, s.c2, s.x_vel, s.y_vel,
                      s.color, s.position, s.velocity, s.out_of_frame]
    R[k + 'vertices'] = s.vertices
    R[k + 'contains'] = np.array([bool(s.contains_point(p)) for p in points])
    np.random.seed(10 + i)
    R[k + 'sample_contained'] = [s.sample_contained_position() for _ in range(5)]
    s.move(np.array([0.4, -0.7]), keep_in_frame=i % 2 == 0)
    R[k + 'moved'] = [s.position, s.out_of_frame, s.vertices]
    s.update_position(keep_in_frame=i % 3 == 0)
    s.shape, s.angle, s.scale = 'pentagon', 33, 0.15
    R[k + 'changed'] = [s.position, s.factors, s.vertices, s.contains_point(s.position)]
  R['default'] = sw('sprite').Sprite().factors
  R['factor_names'] = list(sw('sprite').FACTOR_NAMES)


def renderers_handcrafted(sw, R):
  hc = sw('renderers.handcrafted')
  sprites = _sprites(sw, 3, 4)
  for name, r in [('factors', hc.SpriteFactors()),
                  ('factors_subset', hc.SpriteFactors(factors=('x', 'shape', 'c1'))),
                  ('passthrough', hc.SpritePassthrough())]:
    R[name] = r.render(sprites=sprites)
    R[name + '.spec'] = _spec(r.observation_spec())
  R['factors.error'] = attempt(hc.SpriteFactors, factors=('x', 'not_a_factor'))
  s = hc.Success()
  R['success'] = [s.render(global_state=dict(success=v)) for v in (True, False)]
  R['success.spec'] = _spec(s.observation_spec())
  R['success.no_key'] = attempt(s.render, global_state={})


HOST = dict(factor_distributions=factor_distributions, sprite_generators=sprite_generators,
            shapes=shapes, sprite=sprite, renderers_handcrafted=renderers_handcrafted)


# ---------------------------------------------------------------------------------------------
# modules that drive the engine
# ---------------------------------------------------------------------------------------------

def tasks(sw, R):
  fd, tk = sw('factor_distributions'), sw('tasks')
  red, blue = fd.Continuous('c0', 0, 0.5), fd.Continuous('c0', 0.5, 1)
  all_tasks = dict(
      no_reward=tk.NoReward(),
      goal=tk.FindGoalPosition(),
      goal_filtered=tk.FindGoalPosition(filter_distrib=red, goal_position=(0.3, 0.7),
                                        terminate_distance=0.2, terminate_bonus=2.0,
                                        weights_dimensions=(1, 0.5)),
      goal_sparse=tk.FindGoalPosition(filter_distrib=blue, terminate_distance=0.3,
                                      sparse_reward=True, raw_reward_multiplier=10),
      clustering=tk.Clustering([red, blue], termination_threshold=1.5, terminate_bonus=1.0),
      clustering_sparse=tk.Clustering([red, blue], sparse_reward=True, reward_range=5),
      meta_sum=tk.MetaAggregated([tk.FindGoalPosition(filter_distrib=red),
                                  tk.FindGoalPosition(filter_distrib=blue, goal_position=(0.8, 0.2))]),
      meta_mean_any=tk.MetaAggregated(
          [tk.FindGoalPosition(filter_distrib=red, terminate_distance=0.3),
           tk.FindGoalPosition(filter_distrib=blue)],
          reward_aggregator='mean', termination_criterion='any', terminate_bonus=1.5),
      meta_max=tk.MetaAggregated([tk.FindGoalPosition(filter_distrib=red),
                                  tk.Clustering([red, blue])], reward_aggregator='max'),
      meta_min=tk.MetaAggregated([tk.FindGoalPosition(filter_distrib=red),
                                  tk.FindGoalPosition(filter_distrib=blue)], reward_aggregator='min'))
  scenes = [_sprites(sw, 20 + i, n) for i, n in enumerate((1, 2, 4, 6, 6, 8))]
  for name, task in sorted(all_tasks.items()):
    R[name] = [[attempt(task.reward, s), attempt(task.success, s)] for s in scenes]


def action_spaces(sw, R):
  asp = sw('action_spaces')
  spaces = dict(select_move=asp.SelectMove(), select_move_cost=asp.SelectMove(scale=0.5, motion_cost=0.3),
                drag_and_drop=asp.DragAndDrop(scale=0.7, motion_cost=0.1),
                select_move_noise=asp.SelectMove(scale=0.5, noise_scale=0.05),
                drag_and_drop_noise=asp.DragAndDrop(noise_scale=0.1),
                embodied=asp.Embodied(step_size=0.1, motion_cost=0.2))
  for name, space in sorted(spaces.items()):
    R[name + '.spec'] = _spec(space.action_spec())
    rng = np.random.RandomState(30)
    np.random.seed(31)   # the action noise
    out = []
    for t in range(12):
      sprites = _sprites(sw, 40 + t, 4)
      if name == 'embodied':
        action = np.array([t % 2, t % 4])
      else:
        action = rng.uniform(0, 1, 4)
        if t % 2 == 0:   # aim at a sprite so that it moves
          action[:2] = sprites[t % 4].position
      cost = attempt(space.step, action, sprites, keep_in_frame=t % 3 != 0)
      out.append([cost, [np.array(s.position) for s in sprites]])
    R[name + '.steps'] = out
  R['embodied.bad_action'] = attempt(spaces['embodied'].step, np.array([0, 7]), _sprites(sw, 9, 3), True)


def renderers_pil_renderer(sw, R):
  pil, cm = sw('renderers.pil_renderer'), sw('renderers.color_maps')
  for name, kw in [('default', {}), ('aa5_bg', dict(anti_aliasing=5, bg_color=(20, 30, 40))),
                   ('hsv_48x32', dict(image_size=(48, 32), anti_aliasing=3, color_to_rgb=cm.hsv_to_rgb))]:
    r = pil.PILRenderer(**kw)
    R[name] = r.render(sprites=_sprites(sw, 50, 6, rgb='color_to_rgb' not in kw))
    R[name + '.spec'] = _spec(r.observation_spec())


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


def _episode(env, actions):
  out, ts = [], env.reset()
  for a in actions:
    ts = env.step(a)
    # copies: this package updates a sprite's position array in place, the reference rebinds it
    out.append([int(ts.step_type), ts.reward, bool(env.success()),
                [np.array(s.position) for s in env.state()['sprites']]])
  return out, ts


def configs(sw, R):
  import contextlib
  import io
  env_lib = sw('environment')
  for pkg, name, modes in CONFIG_MODES:
    mod = sw('configs.%s.%s' % (pkg, name))
    for mode in modes:
      with contextlib.redirect_stdout(io.StringIO()):
        cfg = mod.get_config(mode) if mode else mod.get_config()
      np.random.seed(12)
      env = env_lib.Environment(**cfg)
      spec = env.action_spec()
      rng = np.random.RandomState(13)
      if isinstance(spec, (list, tuple)):   # Embodied: (carry, direction)
        actions = [np.array([rng.randint(0, 2), rng.randint(0, 4)], np.int32) for _ in range(6)]
      else:
        actions = [rng.uniform(0, 1, 4).astype(spec.dtype) for _ in range(6)]
      key = '%s.%s.%s' % (pkg, name, mode)
      R[key + '.episode'], ts = _episode(env, actions)
      R[key + '.observation_keys'] = sorted(ts.observation)
      R[key + '.image'] = ts.observation['image']
      R[key + '.max_episode_length'] = cfg['max_episode_length']


def _env(sw, **kw):
  fd, sg, tk, asp, rd = (sw('factor_distributions'), sw('sprite_generators'), sw('tasks'),
                         sw('action_spaces'), sw('renderers'))
  factors = fd.Product([fd.Continuous('x', 0.1, 0.9), fd.Continuous('y', 0.1, 0.9),
                        fd.Discrete('shape', ['square', 'triangle', 'circle']),
                        fd.Discrete('scale', [0.15]), fd.Continuous('c0', 0, 1),
                        fd.Continuous('c1', 0.3, 1), fd.Discrete('c2', [0.9])])
  args = dict(task=tk.FindGoalPosition(filter_distrib=fd.Continuous('c0', 0, 0.5),
                                       terminate_distance=0.15),
              action_space=asp.SelectMove(scale=0.5),
              renderers={'image': rd.PILRenderer(image_size=(32, 32), anti_aliasing=3,
                                                 color_to_rgb=rd.color_maps.hsv_to_rgb),
                         'factors': rd.SpriteFactors(), 'success': rd.Success()},
              init_sprites=sg.generate_sprites(factors, num_sprites=3), max_episode_length=7)
  args.update(kw)
  return sw('environment').Environment(**args)


def environment(sw, R):
  for name, kw in [('default', {}), ('free', dict(keep_in_frame=False))]:
    np.random.seed(14)
    env = _env(sw, **kw)
    R[name + '.action_spec'] = _spec(env.action_spec())
    R[name + '.observation_spec'] = sorted(env.observation_spec())
    rng = np.random.RandomState(15)
    ts = env.reset()
    out = [[int(ts.step_type), ts.reward, ts.discount, ts.observation['factors'],
            ts.observation['success']]]
    for t in range(16):
      a = rng.uniform(0, 1, 4).astype(np.float32)
      if t % 2 == 0 and env.state()['sprites']:
        a[:2] = env.state()['sprites'][t % 3].position
      ts = env.step(a)
      out.append([int(ts.step_type), ts.reward, ts.discount, ts.observation['factors'],
                  ts.observation['success'], env.success(), env.should_terminate()])
    R[name + '.steps'] = out
    R[name + '.image'] = ts.observation['image']
    np.random.seed(16)
    R[name + '.sample_contained_position'] = [env.sample_contained_position() for _ in range(3)]


def _space(space):
  """Kind, shape, dtype and (for float boxes) the distinct bounds of a gym space."""
  kind = type(space).__name__
  if hasattr(space, 'n'):
    return [kind, int(space.n)]
  if isinstance(getattr(space, 'spaces', None), dict):
    return [kind, {k: _space(v) for k, v in space.spaces.items()}]
  if hasattr(space, 'spaces'):
    return [kind, [_space(v) for v in space.spaces]]
  bounds = ([np.unique(space.low).tolist(), np.unique(space.high).tolist()]
            if np.dtype(space.dtype).kind == 'f' else None)
  return [kind, list(space.shape), str(np.dtype(space.dtype)), bounds]


def gym_wrapper(sw, R):
  asp, rd = sw('action_spaces'), sw('renderers')
  for name, space in [('select_move', asp.SelectMove(scale=0.5)), ('embodied', asp.Embodied(step_size=0.1))]:
    np.random.seed(17)
    renderers = {'image': rd.PILRenderer(image_size=(16, 16), anti_aliasing=2,
                                         color_to_rgb=rd.color_maps.hsv_to_rgb),
                 'success': rd.Success()}
    env = sw('gym_wrapper').GymWrapper(_env(sw, action_space=space, renderers=renderers,
                                            max_episode_length=5))
    R[name + '.observation_space'] = _space(env.observation_space)
    R[name + '.action_space'] = _space(env.action_space)
    out = []
    for _ in range(2):   # one step past the episode's end: LAST, then a new episode
      obs = env.reset()
      out.append([sorted(obs), str(obs['image'].dtype), int(obs['image'].sum()), obs['success']])
      for _ in range(6):
        obs, reward, done, info = env.step(env.action_space.sample())
        out.append([str(obs['image'].dtype), int(obs['image'].sum()), obs['success'], reward, done, info])
    R[name + '.episodes'] = out
    R[name + '.render'] = env.render()


ENGINE = dict(tasks=tasks, action_spaces=action_spaces, renderers_pil_renderer=renderers_pil_renderer,
              configs=configs, environment=environment, gym_wrapper=gym_wrapper)


SURFACE_MODULES = [
    'action_spaces', 'constants', 'environment', 'factor_distributions', 'gym_wrapper', 'shapes',
    'sprite', 'sprite_generators', 'tasks', 'renderers', 'renderers.abstract_renderer',
    'renderers.color_maps', 'renderers.handcrafted', 'renderers.pil_renderer',
    'configs.cobra.common']


def public_surface(sw):
  """[module, name, public attributes of a class, constructor or function parameters] for every
  public class, function and value defined in SURFACE_MODULES of the package behind `sw`
  (`renderers` re-exports its classes on purpose)."""
  import inspect
  out = []
  for m in SURFACE_MODULES:
    mod = sw(m)
    for name, obj in sorted(vars(mod).items()):
      if name.startswith('_') or inspect.ismodule(obj) or type(obj).__name__ == '_Feature':
        continue   # private, submodule, `from __future__ import ...`
      if getattr(obj, '__module__', mod.__name__) != mod.__name__ and (
          inspect.isclass(obj) or inspect.isfunction(obj)) and m != 'renderers':
        continue   # imported helper
      attrs, params = [], None
      if inspect.isclass(obj):
        attrs = sorted(a for a in vars(obj) if not a.startswith('_'))
        if '__init__' in vars(obj):
          params = [p for p in inspect.signature(obj.__init__).parameters if p != 'self']
      elif inspect.isfunction(obj):
        params = list(inspect.signature(obj).parameters)
      out.append([m, name, attrs, params])
  return out


def run(name, sw):
  """The records of probe `name` (a key of HOST or ENGINE) against the package behind `sw`."""
  R = Record()
  (HOST.get(name) or ENGINE[name])(sw, R)
  return R
