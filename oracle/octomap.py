"""CPU restatement of the OctoMap occupancy-tree operations the reference's grid producer calls.

TEST INFRASTRUCTURE ONLY (see oracle/__init__.py): imported by tests/, by
oracle/ref_harness (as the stand-in ``octomap`` module under the reference's own
``MultiInstanceOctreeMapping``) and by bench.py's cpu_baseline leg.  Never by the product.

**PARITY UNPINNED.**  The reference's producer, ``morefusion/contrib/multi_instance_octree_mapping.py``,
delegates to the third-party ``octomap-python`` binding (``requirements.txt:11``,
``octomap-python>=1.8.0.post12``, which wraps OctoMap 1.9.x).  Neither is under /root/reference
or installable here, and the reference holds no test or fixture for this path.  What follows is
the published OctoMap 1.9 algorithm (Hornung et al., "OctoMap", Autonomous Robots 2013; class
and method names below are the library's), restated for exactly the calls the reference makes:

  reference call site (multi_instance_octree_mapping.py)        restated here
  :18  octomap.OcTree(pitch)                                     OcTree.__init__
  :24  octree.insertPointCloud(pcd[mask & nonnan], origin=...)   OcTree.insertPointCloud
       -> OccupancyOcTreeBase::computeUpdate / updateNode,
          OcTreeBaseImpl::computeRayKeys (Amanatides & Woo DDA)
  :30-31 octree.updateNodes(occupied, True, lazy_eval=True); updateInnerOccupancy()
                                                                 OcTree.updateNodes / updateInnerOccupancy
  :78-83 octree.search(point); node.getOccupancy(); NullPointerException for unknown space
                                                                 OcTree.search / OcTreeNode.getOccupancy
  :118 octree.extractPointCloud()                                OcTree.extractPointCloud

Semantics kept from the library: point3d is three *floats*; keys are 16 bit per axis,
``key = floor(coord / resolution) + 32768``; a scan updates every cell at most once and a cell
that holds an end point is not also updated as free; log-odds are float32, hit 0.7 / miss 0.4,
clamped to [0.1192, 0.971]; ``getOccupancy`` is evaluated in double.  An octree with pruning is
observationally a flat key -> log-odds map for ``search`` at depth 0 (a pruned parent carries its
children's common value and unknown cells stay unknown), which is what this class stores.

The assembly of the three grids from these primitives IS pinned: oracle/ref_harness/gen_golden.py
runs the reference's own ``get_target_grids`` / ``integrate`` code on top of this module into
tests/golden/octree_mapping*.npz, which tests/test_oracle_golden.py compares with
``get_target_grids`` below.
"""

import math

import numpy as np

TREE_DEPTH = 16
TREE_MAX_VAL = 32768


def logodds(p):
    return math.log(p / (1.0 - p))


def probability(lo):
    """octomap::probability(float logodds): evaluated in double."""
    return 1.0 - (1.0 / (1.0 + math.exp(float(lo))))


class NullPointerException(Exception):
    """octomap-python raises this from accessors of a node that wraps a NULL pointer."""


class OcTreeNode:
    def __init__(self, lo):
        self._lo = lo

    def getOccupancy(self):
        if self._lo is None:
            raise NullPointerException
        return probability(self._lo)

    def getLogOdds(self):
        if self._lo is None:
            raise NullPointerException
        return float(self._lo)


class OcTree:
    def __init__(self, resolution):
        self.resolution = float(resolution)
        self.resolution_factor = 1.0 / self.resolution
        self.prob_hit_log = np.float32(logodds(0.7))
        self.prob_miss_log = np.float32(logodds(0.4))
        self.clamping_thres_min = np.float32(logodds(0.1192))
        self.clamping_thres_max = np.float32(logodds(0.971))
        self.cells = {}                      # (kx, ky, kz) -> np.float32 log-odds

    def getResolution(self):
        return self.resolution

    # ---- OcTreeBaseImpl::coordToKeyChecked / keyToCoord
    def coord_to_key(self, c):
        f = self.resolution_factor * float(c)
        if not math.isfinite(f):                  # library: (int) of NaN / inf lands outside the range
            return None
        k = int(math.floor(f)) + TREE_MAX_VAL
        return k if 0 <= k < 2 * TREE_MAX_VAL else None

    def coords_to_key(self, p):
        k = tuple(self.coord_to_key(c) for c in p)
        return None if None in k else k

    def key_to_coord(self, k):
        return (float(int(k) - TREE_MAX_VAL) + 0.5) * self.resolution

    # ---- OcTreeBaseImpl::computeRayKeys: the cells a ray crosses, first cell included, last excluded
    def computeRayKeys(self, origin, end):
        """origin, end: float32[3].  Returns the list of keys, or None when an end is outside the
        addressable volume (the library returns false and the ray is skipped)."""
        origin = np.asarray(origin, np.float32)
        end = np.asarray(end, np.float32)
        key_origin = self.coords_to_key(origin)
        key_end = self.coords_to_key(end)
        if key_origin is None or key_end is None:
            return None
        if key_origin == key_end:
            return []
        ray = [key_origin]
        direction = (end - origin).astype(np.float32)                      # float vector
        nsq = np.float32(np.float32(direction[0] * direction[0] + direction[1] * direction[1])
                         + direction[2] * direction[2])                   # Vector3::norm_sq, float
        length = np.float32(math.sqrt(float(nsq)))                         # (float) sqrt(double)
        direction = (direction / length).astype(np.float32)
        step = [0, 0, 0]
        tmax = [0.0, 0.0, 0.0]
        tdelta = [0.0, 0.0, 0.0]
        cur = list(key_origin)
        dmax = float(np.finfo(np.float64).max)
        for i in range(3):
            d = float(direction[i])
            step[i] = 1 if d > 0.0 else (-1 if d < 0.0 else 0)
            if step[i] != 0:
                border = self.key_to_coord(cur[i])
                border += float(np.float32(step[i] * self.resolution * 0.5))
                tmax[i] = (border - float(origin[i])) / d
                tdelta[i] = self.resolution / abs(d)
            else:
                tmax[i] = dmax
                tdelta[i] = dmax
        flen = float(length)
        while True:
            if tmax[0] < tmax[1]:
                dim = 0 if tmax[0] < tmax[2] else 2
            else:
                dim = 1 if tmax[1] < tmax[2] else 2
            cur[dim] += step[dim]
            tmax[dim] += tdelta[dim]
            if tuple(cur) == key_end:
                break
            if min(tmax[0], tmax[1], tmax[2]) > flen:
                break
            if not (0 <= cur[dim] < 2 * TREE_MAX_VAL):                     # library: assert
                break
            ray.append(tuple(cur))
        return ray

    # ---- OccupancyOcTreeBase::updateNode(key, occupied)
    def _update(self, key, occupied):
        upd = self.prob_hit_log if occupied else self.prob_miss_log
        v = np.float32(self.cells.get(key, np.float32(0.0)) + upd)         # float add
        if v < self.clamping_thres_min:
            v = self.clamping_thres_min
        if v > self.clamping_thres_max:
            v = self.clamping_thres_max
        self.cells[key] = v

    # ---- OccupancyOcTreeBase::insertPointCloud (computeUpdate + updates), maxrange = -1
    def insertPointCloud(self, pointcloud, origin, maxrange=-1.0, lazy_eval=False, discretize=False):
        assert maxrange < 0 and not discretize
        pts = np.asarray(pointcloud, dtype=np.float64).astype(np.float32).reshape(-1, 3)
        org = np.asarray(origin, dtype=np.float64).astype(np.float32)
        free, occ = set(), set()
        for p in pts:
            ray = self.computeRayKeys(org, p)
            if ray is not None:
                free.update(ray)
            k = self.coords_to_key(p)
            if k is not None:
                occ.add(k)
        for k in free - occ:
            self._update(k, False)
        for k in occ:
            self._update(k, True)

    # ---- octomap-python updateNodes: one updateNode per row, doubles, no de-duplication
    def updateNodes(self, values, update, lazy_eval=False):
        for v in np.asarray(values, dtype=np.float64).reshape(-1, 3):
            k = self.coords_to_key(v)
            if k is not None:
                self._update(k, bool(update))

    def updateInnerOccupancy(self):
        pass                                     # inner nodes are not observable through search(depth=0)

    # ---- OcTreeBaseImpl::search(x, y, z, depth=0) (double coordinates)
    def search(self, point, depth=0):
        assert depth == 0
        k = self.coords_to_key(np.asarray(point, dtype=np.float64))
        return OcTreeNode(None if k is None else self.cells.get(k))

    # ---- octomap-python extractPointCloud: centres of occupied / free leaves (key order here)
    def extractPointCloud(self):
        occupied, empty = [], []
        for k in sorted(self.cells):
            c = [float(np.float32(self.key_to_coord(a))) for a in k]        # getCoordinate(): floats
            (occupied if self.cells[k] >= 0.0 else empty).append(c)
        return (np.asarray(occupied, dtype=np.float64).reshape(-1, 3),
                np.asarray(empty, dtype=np.float64).reshape(-1, 3))


# --------------------------------------------------------------------------------------------
# restatement of the reference's MultiInstanceOctreeMapping (multi_instance_octree_mapping.py:7-133)
# --------------------------------------------------------------------------------------------
class MultiInstanceOctreeMapping:
    def __init__(self):
        self._octrees = {}

    @property
    def instance_ids(self):
        return list(self._octrees.keys())

    def initialize(self, instance_id, *, pitch):                            # :16-19
        if instance_id in self._octrees:
            raise ValueError("instance {instance_id} already exists")
        self._octrees[instance_id] = OcTree(pitch)

    def integrate(self, instance_id, mask, pcd, origin=(0, 0, 0)):          # :21-27
        origin = np.asarray(origin, dtype=float)
        nonnan = ~np.isnan(pcd).any(axis=2)
        self._octrees[instance_id].insertPointCloud(pcd[mask & nonnan], origin=origin)

    def update(self, instance_id, occupied):                                # :29-34
        self._octrees[instance_id].updateNodes(occupied, True, lazy_eval=True)

    def get_target_grids(self, target_id, *, dimensions, pitch, origin):    # :35-94
        origin = np.asarray(origin, dtype=np.float64)
        X, Y, Z = dimensions
        grid_target = np.zeros(dimensions, np.float32)
        grid_nontarget = np.zeros(dimensions, np.float32)
        grid_empty = np.zeros(dimensions, np.float32)
        ii, jj, kk = np.meshgrid(np.arange(X), np.arange(Y), np.arange(Z), indexing="ij")
        idx = np.stack([ii.ravel(), jj.ravel(), kk.ravel()], 1)
        centers = idx * pitch + origin                                       # trimesh matrix_to_points
        for ins_id, octree in self._octrees.items():
            occ = np.full(len(centers), -1.0)
            for n, c in enumerate(centers):
                k = octree.coords_to_key(c)
                lo = None if k is None else octree.cells.get(k)
                if lo is not None:
                    occ[n] = probability(lo)
            q = occ >= 0.5
            g = grid_target if ins_id == target_id else grid_nontarget
            g[idx[q, 0], idx[q, 1], idx[q, 2]] = occ[q]
            q = (0 <= occ) & (occ < 0.5)
            grid_empty[idx[q, 0], idx[q, 1], idx[q, 2]] = 1 - occ[q]
        return grid_target, grid_nontarget, grid_empty

    def get_target_pcds(self, target_id, aabb_min=None, aabb_max=None):      # :96-133
        occupied, empty = self._octrees[target_id].extractPointCloud()
        if aabb_min is not None:
            occupied = occupied[(occupied >= aabb_min).all(axis=1)]
            empty = empty[(empty >= aabb_min).all(axis=1)]
        if aabb_max is not None:
            occupied = occupied[(occupied < aabb_max).all(axis=1)]
            empty = empty[(empty < aabb_max).all(axis=1)]
        return occupied, empty
