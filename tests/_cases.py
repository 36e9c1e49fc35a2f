"""Shared small test cases (graph + params + inputs) for CPU and GPU tests."""
import functools

import numpy as np
import pytest

from graphcast_b200 import graph as graph_lib
from oracle import gnn as oracle_gnn


@pytest.fixture
def cluster(request):
  """CTAs per cluster of the tensor-core layer kernel for one test (parametrize it with
  indirect=True).  The setting is process-global, so the library default of 2 is restored
  however the test ends: a leaked value would move every later test onto another schedule."""
  from graphcast_b200 import _native
  lib = _native.lib()
  _native.check(lib.gcb_set_cluster_size(request.param), "gcb_set_cluster_size")
  try:
    yield request.param
  finally:
    _native.check(lib.gcb_set_cluster_size(2), "gcb_set_cluster_size")


@functools.lru_cache(maxsize=None)
def small_graph(res: float = 4.0, mesh_size: int = 3):
  n_lat = int(round(180 / res)) + 1
  lat = np.linspace(-90, 90, n_lat)
  lon = np.arange(0, 360, res)
  return graph_lib.build_static_graph(grid_lat=lat, grid_lon=lon, mesh_size=mesh_size,
                                      radius_query_fraction_edge_length=0.6)


def small_case(c_in=31, n_out=23, msg_steps=3, batch=1, seed=0, res=4.0, mesh_size=3,
               randomize_affine=True):
  g = small_graph(res, mesh_size)
  params = oracle_gnn.init_params(c_in=c_in, n_out=n_out, latent=512, msg_steps=msg_steps,
                                  seed=seed + 1, randomize_affine=randomize_affine)
  x = np.random.default_rng(seed).standard_normal(
      (g.num_grid_nodes, batch, c_in)).astype(np.float32)
  return g, params, x
